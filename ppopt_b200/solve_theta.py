"""Fixed-parameter QP and LP solves on the GPU and the explicit-vs-implicit check of a solution.

For a fixed theta an mpQP is an ordinary QP and an mpLP an ordinary LP; the reference solves them with an external backend
(``MPQP_Program.solve_theta`` / ``MPLP_Program.solve_theta`` -> daqp / gurobi / GLPK / ..., returning a ``SolverOutput``) and
uses them to seed the graph algorithms (``sample_theta_space``).  Here a whole batch of points is ONE kernel launch, one point
per warp: K8 (csrc/k8_theta_qp.cu, ``ppgpu_solve_theta_batch``) runs a dual active-set iteration on the Gram data of an mpQP
handle, K9 (csrc/k9_theta_lp.cu, ``ppgpu_solve_theta_lp_batch``) a dictionary simplex from the start dictionary of an mpLP
handle.

    solver = ThetaSolver(program)               # mpQP;  ThetaLPSolver(program) for an mpLP, same surface
    out = solver.solve_batch(thetas)            # device tensors: status, x, dual, active, iters, slack, obj
    rec = solver.solve_theta(theta)             # SolverOutput(obj, sol, slack, active_set, dual) or None (no optimum)
    seeds = solver.sample_theta_space(100)      # distinct optimal active sets of sampled points
    report = verify_solution(solution)          # explicit law (K7 point location) against the implicit solve (K8 / K9)

Not covered (NotImplementedError): an mpQP whose Hessian is not positive definite on the space the equalities leave
(``use_gram == 0``), and an mpLP whose reduced inequality rows have rank below n - n_eq (the LP has no vertex).  The rows of
Theta (A_t theta <= b_t) do not constrain x and are not imposed: a point outside Theta is solved as given.  No CPU fallback.
"""
import ctypes
from dataclasses import dataclass
from typing import Dict, List, Optional

import numpy
import torch

from . import _lib
from . import engine as _engine

# per-point status of the kernels (PPG_QP_* / PPG_TLP_* of csrc/tolerances.h)
QP_OPTIMAL, QP_INFEASIBLE, QP_ITERLIM, QP_NUMERIC = 0, 1, 2, 3
LP_OPTIMAL, LP_INFEASIBLE, LP_ITERLIM, LP_NUMERIC, LP_UNBOUNDED = 0, 1, 2, 3, 4


@dataclass
class SolverOutput:
    """Field names of the reference's SolverOutput (solver_interface/solver_interface_utils.py)."""
    obj: float
    sol: numpy.ndarray
    slack: Optional[numpy.ndarray]
    active_set: numpy.ndarray
    dual: numpy.ndarray


def _solver_output_class(program):
    """ppopt's own SolverOutput when the program is a ppopt object (as engine._region_classes does), else the mirror."""
    root = type(program).__module__.split('.mpqp_program')[0].split('.mplp_program')[0]
    if root != 'ppopt_b200' and root.endswith('ppopt'):
        import importlib
        try:
            return importlib.import_module(root + '.solver_interface.solver_interface_utils').SolverOutput
        except Exception:
            pass
    return SolverOutput


def theta_box(A_t, b_t):
    """(lo, hi) of the box that the single-variable rows of A_t theta <= b_t give Theta.  A side that no such row bounds
    is placed 10 (1 + the largest finite bound or |b_t| entry) away from the origin: uniform sampling needs a finite box,
    and the region structure of a program lives at the scale of its data."""
    A_t, b_t = numpy.asarray(A_t, dtype=numpy.float64), numpy.asarray(b_t, dtype=numpy.float64).ravel()
    t = A_t.shape[1]
    lo, hi = numpy.full(t, -numpy.inf), numpy.full(t, numpy.inf)
    for a, b in zip(A_t, b_t):
        nz = numpy.nonzero(a)[0]
        if len(nz) == 1:
            j = nz[0]
            if a[j] > 0:
                hi[j] = min(hi[j], b / a[j])
            else:
                lo[j] = max(lo[j], b / a[j])
    fin = numpy.r_[lo[numpy.isfinite(lo)], hi[numpy.isfinite(hi)], b_t]
    reach = 10.0 * (1.0 + numpy.abs(fin).max(initial=0.0))
    return numpy.where(numpy.isfinite(lo), lo, -reach), numpy.where(numpy.isfinite(hi), hi, reach)


def _attr(program, name, shape):
    v = getattr(program, name, None)
    return numpy.zeros(shape) if v is None else numpy.asarray(v, dtype=numpy.float64).reshape(shape)


class _FixedThetaSolver:
    """What ThetaSolver and ThetaLPSolver share: one program handle (``engine.Engine``), the objective / constraint data on
    the device, slack and objective of a batch, the SolverOutput record, sampling and distinct active sets.  A subclass
    sets ``_entry`` (its C entry point), ``_iters_shape`` and ``OPTIMAL``."""
    _entry = ''
    _iters_shape = ()
    OPTIMAL = 0

    def _setup(self, program, arrays, eng):
        self.program, self.eng = program, eng
        e = eng
        self.n, self.t, self.m, self.n_eq, self.W = e.n, e.t, e.m, e.n_eq, e.W
        dev = lambda a: torch.from_numpy(numpy.ascontiguousarray(a, dtype=numpy.float64)).to(e.tdev)  # noqa: E731
        self._A, self._b, self._F = dev(arrays['A']), dev(arrays['b']), dev(arrays['F'])
        self._Q = None if arrays['Q'] is None else dev(arrays['Q'])
        self._H, self._c = dev(arrays['H']), dev(arrays['c'])
        self._c_c = float(_attr(program, 'c_c', (1,))[0])
        self._c_t = dev(_attr(program, 'c_t', (self.t,)))
        self._Q_t = dev(_attr(program, 'Q_t', (self.t, self.t)))
        self.A_t, self.b_t = arrays['A_t'], arrays['b_t']
        self._out_cls = _solver_output_class(program)

    def close(self):
        self.eng.close()

    def _thetas(self, thetas) -> torch.Tensor:
        if torch.is_tensor(thetas):
            th = thetas.to(self.eng.tdev, dtype=torch.float64)
        else:
            th = torch.from_numpy(numpy.ascontiguousarray(thetas, dtype=numpy.float64)).to(self.eng.tdev)
        return th.reshape(-1, self.t).contiguous()

    def objective(self, thetas: torch.Tensor, x: torch.Tensor) -> torch.Tensor:
        """evaluate_objective(x, theta) of every row (device tensors)"""
        obj = ((thetas @ self._H.T) * x).sum(1)
        if self._Q is not None:
            obj = 0.5 * ((x @ self._Q) * x).sum(1) + obj
        return obj + x @ self._c + self._c_c + thetas @ self._c_t + 0.5 * ((thetas @ self._Q_t) * thetas).sum(1)

    def solve_batch(self, thetas) -> Dict[str, torch.Tensor]:
        """thetas (n_points x t, host or device) -> device tensors: status (uint8), x (n_points x n), dual (n_points x m:
        equality multipliers, then the inequality multipliers; Q x + H theta + c + A' dual = 0, Q = 0 for an mpLP), active
        (n_points x words int64 candidate masks of the final working set or basis), iters (int32), slack = b + F theta - A x
        and obj = evaluate_objective(x, theta).  x, dual, slack and obj are NaN where the status is not optimal."""
        e = self.eng
        th = self._thetas(thetas)
        k = th.shape[0]
        status = e.empty((k,), torch.uint8)
        x, dual = e.empty((k, self.n), torch.float64), e.empty((k, self.m), torch.float64)
        active, iters = e.empty((k, self.W), torch.int64), e.empty((k,) + self._iters_shape, torch.int32)
        if k:
            with torch.cuda.device(e.tdev):
                _lib.check(getattr(e.lib, self._entry)(e.h, th.data_ptr(), k, status.data_ptr(), x.data_ptr(), dual.data_ptr(),
                                                       active.data_ptr(), iters.data_ptr(), e._stream()), self._entry[6:])
        slack = self._b + th @ self._F.T - x @ self._A.T
        return dict(status=status, x=x, dual=dual, active=active, iters=iters, slack=slack, obj=self.objective(th, x))

    def active_sets(self, active: torch.Tensor) -> List[List[int]]:
        """working-set / basis masks -> full active sets (equality rows first), as the graph drivers take them"""
        return self.eng.lists_from_masks(active.cpu().numpy())

    def _record(self, out):
        """SolverOutput of point 0 of a solve_batch result"""
        aset = numpy.array(self.active_sets(out['active'][:1])[0], dtype=numpy.int64)
        return self._out_cls(obj=float(out['obj'][0]), sol=out['x'][0].cpu().numpy(), slack=out['slack'][0].cpu().numpy(),
                             active_set=aset, dual=out['dual'][0].cpu().numpy())

    def sample_thetas(self, num_samples: int, seed: int = 0) -> numpy.ndarray:
        """uniform draws in theta_box(A_t, b_t), kept where every row of A_t theta <= b_t holds"""
        lo, hi = theta_box(self.A_t, self.b_t)
        th = numpy.random.default_rng(seed).uniform(lo, hi, size=(int(num_samples), self.t))
        return th[(th @ self.A_t.T <= self.b_t[None, :]).all(1)]

    def sample_theta_space(self, num_samples: int = 100, seed: int = 0) -> List[tuple]:
        """the reference's sample_theta_space: distinct optimal active sets (equality rows first) of sampled points in
        Theta, in first-seen order - the reference's sampling is random too, only the kind of output is mirrored"""
        th = self.sample_thetas(num_samples, seed)
        out = self.solve_batch(th)
        ok = (out['status'] == self.OPTIMAL).cpu().numpy()
        seen, order = set(), []
        for a in self.active_sets(out['active'][torch.from_numpy(ok).to(self.eng.tdev)]):
            a = tuple(a)
            if a not in seen:
                seen.add(a)
                order.append(a)
        return order


class ThetaSolver(_FixedThetaSolver):
    """Fixed-theta QPs of a strictly convex mpQP (K8).  ``iters`` of solve_batch: steps (adds + drops) per point."""
    _entry = 'ppgpu_solve_theta_batch'
    OPTIMAL = QP_OPTIMAL

    def __init__(self, program, device: Optional[int] = None):
        arrays = _engine.program_arrays(program)
        if not arrays['is_qp']:
            raise NotImplementedError('ThetaSolver covers mpQPs only (an mpLP at fixed theta: ThetaLPSolver)')
        eng = _engine.Engine(arrays, device)
        if not eng.use_gram:
            eng.close()
            raise NotImplementedError('solve_theta needs a Hessian that is positive definite on the reduced space (use_gram == 0)')
        self._setup(program, arrays, eng)

    def solve_theta(self, theta_point):
        """the reference's solve_theta: SolverOutput(obj, sol, slack, active_set, dual) at one theta, None when the QP is
        infeasible; RuntimeError on the iteration cap or a numerical breakdown"""
        out = self.solve_batch(numpy.asarray(theta_point, dtype=numpy.float64).reshape(1, -1))
        st = int(out['status'][0])
        if st == QP_INFEASIBLE:
            return None
        if st != QP_OPTIMAL:
            raise RuntimeError(f'fixed-theta QP failed: {"iteration cap" if st == QP_ITERLIM else "numerical breakdown"}')
        return self._record(out)


class ThetaLPSolver(_FixedThetaSolver):
    """Fixed-theta LPs of an mpLP (K9).  The basis it returns is the set of n - n_eq nonbasic inequality rows of the
    optimal vertex; ``iters`` of solve_batch is n_points x 2: pivots of both phases, pivots of Phase 1."""
    _entry = 'ppgpu_solve_theta_lp_batch'
    _iters_shape = (2,)
    OPTIMAL = LP_OPTIMAL

    def __init__(self, program, device: Optional[int] = None):
        arrays = _engine.program_arrays(program)
        if arrays['is_qp']:
            raise NotImplementedError('ThetaLPSolver covers mpLPs only (an mpQP at fixed theta: ThetaSolver)')
        eng = _engine.Engine(arrays, device)
        # a zero-point call runs no kernel, only the handle's checks: -2 when the reduced rows have no vertex
        rc = eng.lib.ppgpu_solve_theta_lp_batch(eng.h, None, 0, None, None, None, None, None, eng._stream())
        if rc != 0:
            msg = eng.lib.ppgpu_last_error().decode()
            eng.close()
            raise NotImplementedError(msg)
        self._setup(program, arrays, eng)

    def solve_theta(self, theta_point):
        """the reference's solve_theta: SolverOutput(obj, sol, slack, active_set, dual) at one theta, None when the LP is
        infeasible or unbounded; RuntimeError on the iteration cap or a numerical breakdown"""
        out = self.solve_batch(numpy.asarray(theta_point, dtype=numpy.float64).reshape(1, -1))
        st = int(out['status'][0])
        if st in (LP_INFEASIBLE, LP_UNBOUNDED):
            return None
        if st != LP_OPTIMAL:
            raise RuntimeError(f'fixed-theta LP failed: {"iteration cap" if st == LP_ITERLIM else "numerical breakdown"}')
        return self._record(out)


def solver_for(program, device: Optional[int] = None):
    """ThetaLPSolver for an mpLP, ThetaSolver for an mpQP"""
    return ThetaSolver(program, device) if _engine.program_arrays(program)['is_qp'] else ThetaLPSolver(program, device)


def _mask_bits(words: numpy.ndarray, rows: int) -> numpy.ndarray:
    """candidate masks (k x words) -> k x rows booleans"""
    w = numpy.ascontiguousarray(words).view(numpy.uint64)
    r = numpy.arange(rows)
    return ((w[:, r >> 6] >> (r & 63).astype(numpy.uint64)) & numpy.uint64(1)).astype(bool)


def verify_solution(solution, thetas=None, num_samples: int = 100000, seed: int = 0, tol: float = 1e-5,
                    solver: Optional[_FixedThetaSolver] = None) -> Dict:
    """Explicit against implicit: per point, the region the solution's own rule locates (K7, the solution's overlap rule
    and point_location_tolerance) and its law, against the program solved at that point (K8 for an mpQP, K9 for an mpLP).
    Points: ``thetas`` or ``num_samples`` draws in Theta.  Report:
        n_points, n_feasible      points checked / with an optimum
        holes, hole_thetas        an optimum but no region located
        spurious, spurious_thetas, spurious_regions   no optimum (infeasible, or an unbounded LP) but a region located
        max_dx, worst_theta       largest |x_explicit - x_implicit|_inf / max(1, |x_implicit|_inf) over the feasible points
                                  whose located region contains them without the tolerance
        n_dx_over_tol             such points where that relative difference exceeds ``tol``
        n_band, max_dx_band       feasible points located only through the tolerance band (a region they lie outside of by
                                  less than point_location_tolerance: its law is extrapolated there, and the first-hit rule
                                  may pick it before the region that contains the point) and their largest difference
        n_failed                  points where the solve hit the iteration cap or broke down (excluded from the above)
    For an mpLP also:
        max_dobj                  largest |obj_explicit - obj_implicit| / max(1, |obj_implicit|) over the points of max_dx
                                  (the optimal value is unique even where x is not)
        n_unbounded               points where the LP is unbounded
        n_dual_degenerate         points of max_dx where a multiplier of the basis is <= 1e-9 (1 + max |dual|): x need not be
                                  unique there, so max_dx and n_dx_over_tol are taken over the other points only"""
    from .point_location import PointLocation
    own = solver is None
    solver = solver_for(solution.program) if own else solver
    is_lp = isinstance(solver, ThetaLPSolver)
    try:
        th = solver.sample_thetas(num_samples, seed) if thetas is None else numpy.asarray(thetas, dtype=numpy.float64).reshape(-1, solver.t)
        pl = PointLocation(solution, device=solver.eng.device)
        region, x_exp = pl.evaluate_batch(th, tol=float(getattr(solution, 'point_location_tolerance', 1e-5)))
        exact = pl.locate_batch(th)
        out = solver.solve_batch(th)
        status, x_imp = out['status'].cpu().numpy(), out['x'].cpu().numpy()
        if is_lp:
            obj_imp = out['obj'].cpu().numpy()
            x_dev = torch.from_numpy(numpy.ascontiguousarray(x_exp, dtype=numpy.float64)).to(solver.eng.tdev)
            obj_exp = solver.objective(solver._thetas(th), x_dev).cpu().numpy()
            dual, basis = out['dual'].cpu().numpy(), _mask_bits(out['active'].cpu().numpy(), solver.m - solver.n_eq)
    finally:
        if own:
            solver.close()
    feas, inf = status == QP_OPTIMAL, status == QP_INFEASIBLE
    unb = status == LP_UNBOUNDED if is_lp else numpy.zeros(len(th), dtype=bool)
    holes, spurious = feas & (region < 0), (inf | unb) & (region >= 0)
    located = feas & (region >= 0)
    rel = numpy.zeros(len(th))
    if located.any():
        rel[located] = numpy.abs(x_exp[located] - x_imp[located]).max(1) / numpy.maximum(1.0, numpy.abs(x_imp[located]).max(1))
    band = located & (exact != region)
    both = located & ~band
    extra = {}
    if is_lp:
        lam = numpy.where(feas[:, None], dual[:, solver.n_eq:], 0.0)
        scale = 1.0 + numpy.abs(numpy.where(feas[:, None], dual, 0.0)).max(1, initial=0.0)
        degen = both & (basis & (lam <= 1e-9 * scale[:, None])).any(1)
        dobj = numpy.zeros(len(th))
        dobj[both] = numpy.abs(obj_exp[both] - obj_imp[both]) / numpy.maximum(1.0, numpy.abs(obj_imp[both]))
        extra = dict(max_dobj=float(dobj[both].max()) if both.any() else 0.0, n_unbounded=int(unb.sum()),
                     n_dual_degenerate=int(degen.sum()))
        both = both & ~degen
    worst = int(numpy.argmax(numpy.where(both, rel, -1.0))) if both.any() else -1
    return dict(n_points=int(len(th)), n_feasible=int(feas.sum()), holes=int(holes.sum()), hole_thetas=th[holes],
                spurious=int(spurious.sum()), spurious_thetas=th[spurious], spurious_regions=region[spurious],
                max_dx=float(rel[both].max()) if both.any() else 0.0, worst_theta=th[worst] if worst >= 0 else None,
                n_dx_over_tol=int((rel[both] > tol).sum()), n_band=int(band.sum()),
                max_dx_band=float(rel[band].max()) if band.any() else 0.0, n_failed=int((~feas & ~inf & ~unb).sum()), **extra)
