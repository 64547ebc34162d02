"""Fixed-parameter QP solves on the GPU and the explicit-vs-implicit check of a solution.

For a fixed theta an mpQP is an ordinary QP; the reference solves it with an external backend (``MPQP_Program.solve_theta``
-> daqp / gurobi / ..., returning a ``SolverOutput``) and uses it to seed the graph algorithms (``sample_theta_space``).
Here a whole batch of points is ONE launch of the K8 kernel (csrc/k8_theta_qp.cu, through ``ppgpu_solve_theta_batch``): a
dual active-set iteration on the Gram data of the program handle, one point per warp.

    solver = ThetaSolver(program)
    out = solver.solve_batch(thetas)            # device tensors: status, x, dual, active, iters, slack, obj
    rec = solver.solve_theta(theta)             # SolverOutput(obj, sol, slack, active_set, dual) or None (infeasible)
    seeds = solver.sample_theta_space(100)      # distinct optimal active sets of sampled points
    report = verify_solution(solution)          # explicit law (K7 point location) against the implicit solve (K8)

Only strictly convex programs are covered: an mpLP, or an mpQP whose Hessian is not positive definite on the space the
equalities leave (``use_gram == 0``), raises NotImplementedError.  The rows of Theta (A_t theta <= b_t) do not constrain x
and are not imposed: a point outside Theta is solved as given.  No CPU fallback.
"""
import ctypes
from dataclasses import dataclass
from typing import Dict, List, Optional

import numpy
import torch

from . import _lib
from . import engine as _engine

# per-point status of the kernel (PPG_QP_* of csrc/tolerances.h)
QP_OPTIMAL, QP_INFEASIBLE, QP_ITERLIM, QP_NUMERIC = 0, 1, 2, 3


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


class ThetaSolver:
    """Owns one program handle (``engine.Engine``) and the objective / constraint data on the device."""

    def __init__(self, program, device: Optional[int] = None):
        arrays = _engine.program_arrays(program)
        if not arrays['is_qp']:
            raise NotImplementedError('solve_theta on the GPU covers mpQPs only (an mpLP at fixed theta is not implemented)')
        self.program = program
        self.eng = _engine.Engine(arrays, device)
        if not self.eng.use_gram:
            self.eng.close()
            raise NotImplementedError('solve_theta needs a Hessian that is positive definite on the reduced space (use_gram == 0)')
        e = self.eng
        self.n, self.t, self.m, self.n_eq, self.W = e.n, e.t, e.m, e.n_eq, e.W
        dev = lambda a: torch.from_numpy(numpy.ascontiguousarray(a, dtype=numpy.float64)).to(e.tdev)  # noqa: E731
        self._A, self._b, self._F = dev(arrays['A']), dev(arrays['b']), dev(arrays['F'])
        self._Q, self._H, self._c = dev(arrays['Q']), dev(arrays['H']), dev(arrays['c'])
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

    def solve_batch(self, thetas) -> Dict[str, torch.Tensor]:
        """thetas (n_points x t, host or device) -> device tensors: status (uint8, QP_*), x (n_points x n), dual
        (n_points x m: equality multipliers, then the inequality multipliers; Q x + H theta + c + A' dual = 0), active
        (n_points x words int64 candidate masks of the working set), iters (int32), slack = b + F theta - A x and
        obj = evaluate_objective(x, theta).  x, dual, slack and obj are NaN where the status is not optimal."""
        e = self.eng
        th = self._thetas(thetas)
        k = th.shape[0]
        status = e.empty((k,), torch.uint8)
        x, dual = e.empty((k, self.n), torch.float64), e.empty((k, self.m), torch.float64)
        active, iters = e.empty((k, self.W), torch.int64), e.empty((k,), torch.int32)
        if k:
            with torch.cuda.device(e.tdev):
                _lib.check(e.lib.ppgpu_solve_theta_batch(e.h, th.data_ptr(), k, status.data_ptr(), x.data_ptr(), dual.data_ptr(),
                                                         active.data_ptr(), iters.data_ptr(), e._stream()), 'solve_theta_batch')
        slack = self._b + th @ self._F.T - x @ self._A.T
        obj = 0.5 * ((x @ self._Q) * x).sum(1) + ((th @ self._H.T) * x).sum(1) + x @ self._c + self._c_c \
            + th @ self._c_t + 0.5 * ((th @ self._Q_t) * th).sum(1)
        return dict(status=status, x=x, dual=dual, active=active, iters=iters, slack=slack, obj=obj)

    def active_sets(self, active: torch.Tensor) -> List[List[int]]:
        """working-set masks -> full active sets (equality rows first), as the graph drivers take them"""
        return self.eng.lists_from_masks(active.cpu().numpy())

    def solve_theta(self, theta_point):
        """the reference's solve_theta: SolverOutput(obj, sol, slack, active_set, dual) at one theta, None when the QP is
        infeasible; RuntimeError on the iteration cap or a numerical breakdown"""
        out = self.solve_batch(numpy.asarray(theta_point, dtype=numpy.float64).reshape(1, -1))
        st = int(out['status'][0])
        if st == QP_INFEASIBLE:
            return None
        if st != QP_OPTIMAL:
            raise RuntimeError(f'fixed-theta QP failed: {"iteration cap" if st == QP_ITERLIM else "numerical breakdown"}')
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
        ok = (out['status'] == QP_OPTIMAL).cpu().numpy()
        seen, order = set(), []
        for a in self.active_sets(out['active'][torch.from_numpy(ok).to(self.eng.tdev)]):
            a = tuple(a)
            if a not in seen:
                seen.add(a)
                order.append(a)
        return order


def verify_solution(solution, thetas=None, num_samples: int = 100000, seed: int = 0, tol: float = 1e-5,
                    solver: Optional[ThetaSolver] = None) -> Dict:
    """Explicit against implicit: per point, the region the solution's own rule locates (K7, the solution's overlap rule
    and point_location_tolerance) and its law, against the QP solved at that point (K8).  Points: ``thetas`` or
    ``num_samples`` draws in Theta.  Report:
        n_points, n_feasible      points checked / QP feasible
        holes, hole_thetas        QP feasible but no region located
        spurious, spurious_thetas, spurious_regions   QP infeasible but a region located
        max_dx, worst_theta       largest |x_explicit - x_implicit|_inf / max(1, |x_implicit|_inf) over the feasible points
                                  whose located region contains them without the tolerance
        n_dx_over_tol             such points where that relative difference exceeds ``tol``
        n_band, max_dx_band       feasible points located only through the tolerance band (a region they lie outside of by
                                  less than point_location_tolerance: its law is extrapolated there, and the first-hit rule
                                  may pick it before the region that contains the point) and their largest difference
        n_failed                  points where the QP hit the iteration cap or broke down (excluded from the above)"""
    from .point_location import PointLocation
    own = solver is None
    solver = ThetaSolver(solution.program) if own else solver
    try:
        th = solver.sample_thetas(num_samples, seed) if thetas is None else numpy.asarray(thetas, dtype=numpy.float64).reshape(-1, solver.t)
        pl = PointLocation(solution, device=solver.eng.device)
        region, x_exp = pl.evaluate_batch(th, tol=float(getattr(solution, 'point_location_tolerance', 1e-5)))
        exact = pl.locate_batch(th)
        out = solver.solve_batch(th)
        status, x_imp = out['status'].cpu().numpy(), out['x'].cpu().numpy()
    finally:
        if own:
            solver.close()
    feas, inf = status == QP_OPTIMAL, status == QP_INFEASIBLE
    holes, spurious = feas & (region < 0), inf & (region >= 0)
    located = feas & (region >= 0)
    rel = numpy.zeros(len(th))
    if located.any():
        rel[located] = numpy.abs(x_exp[located] - x_imp[located]).max(1) / numpy.maximum(1.0, numpy.abs(x_imp[located]).max(1))
    band = located & (exact != region)
    both = located & ~band
    worst = int(numpy.argmax(numpy.where(both, rel, -1.0))) if both.any() else -1
    return dict(n_points=int(len(th)), n_feasible=int(feas.sum()), holes=int(holes.sum()), hole_thetas=th[holes],
                spurious=int(spurious.sum()), spurious_thetas=th[spurious], spurious_regions=region[spurious],
                max_dx=float(rel[both].max()) if both.any() else 0.0, worst_theta=th[worst] if worst >= 0 else None,
                n_dx_over_tol=int((rel[both] > tol).sum()), n_band=int(band.sum()),
                max_dx_band=float(rel[band].max()) if band.any() else 0.0, n_failed=int((~feas & ~inf).sum()))
