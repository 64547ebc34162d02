"""Fixed-parameter solves of a mixed-integer program (mpMILP / mpMIQP) on the GPU, by binary assignment.

For a fixed theta and a fixed assignment y the program is the continuous program on the continuous variables x, and y enters
it the way theta does: right-hand side b + F theta - A_y y, linear term c_x + H_x theta + Q_xy y (Q symmetrised; zero for an
mpMILP).  The handle (``engine.Engine``) holds the continuous program at y = 0, made of the rows that contain a continuous
variable; the y columns of its reduced maps come from ``ppgpu_program_param_maps`` (host_math.hpp::parameter_column_maps) and
give every assignment an additive term vector, computed once on the device (``ppgpu_mi_offsets``).  A batch then runs

    pass 1   K8 (mpMIQP) / K9 (mpMILP) in pair mode: one warp per (point, assignment), status and the continuous part of the
             objective only, over chunks of floor(PAIRS_PER_LAUNCH / points) assignments (at least one, so a launch holds
             at most max(PAIRS_PER_LAUNCH, points) pairs: points x assignments never sizes an allocation);
             after each chunk ``ppgpu_mi_select`` folds the chunk into a running best per point;
    pass 2   the winning pair of every point solved again with the full outputs (x, dual, active set, iterations).

The winner is the exact minimum of the full objective over the assignments whose pair is optimal and whose binary-only rows
hold (b_i + F_i theta - A_{i,y} y >= -1e-7 (1 + |.|)); exact ties go to the lowest assignment index, so the result does not
depend on the chunking.  ``gap`` = runner-up - best (inf with one candidate).  Status per point: infeasible when no pair is
feasible, unbounded (mpMILP) when a feasible pair is unbounded, failed when a pair hit the iteration cap or broke down (the
minimum is then not certified), optimal otherwise.

    solver = MixedIntegerThetaSolver(program)      # ppopt's MPMILP_Program / MPMIQP_Program or an object with their attributes
    out = solver.solve_batch(thetas)               # device tensors: status, x, assignment, obj, gap, dual, active, iters
    rec = solver.solve_theta(theta)                # SolverOutput or None, as ThetaSolver.solve_theta

The assignments are the leaves of the relaxation tree (K11, mp_solvers/mitree.py) unless given.  The rows of Theta are not
imposed (a point outside Theta is solved as given).  Not covered (NotImplementedError): a continuous Hessian that is not
positive definite on the reduced space, an mpLP part without a vertex.  No CPU fallback.
"""
import ctypes
from typing import Dict, List, Optional

import numpy
import torch

from . import _lib
from . import engine as _engine
from .solve_theta import SolverOutput, _attr, _solver_output_class, theta_box

MI_OPTIMAL, MI_INFEASIBLE, MI_FAILED, MI_UNBOUNDED = 0, 1, 2, 4   # PPG_MI_* of csrc/tolerances.h
PAIRS_PER_LAUNCH = 1 << 21
ROW_TOL = 1e-7


def _f64(a):
    return numpy.ascontiguousarray(numpy.asarray(a, dtype=numpy.float64))


class MixedIntegerThetaSolver:
    """Fixed-theta solves of a mixed-integer program over a list of binary assignments (see the module docstring)."""

    def __init__(self, program, assignments=None, device: Optional[int] = None, chunk: Optional[int] = None):
        A = _f64(program.A)
        m, n = A.shape
        F = _f64(program.F).reshape(m, -1)
        t = F.shape[1]
        b = _f64(program.b).reshape(-1)
        c = _f64(program.c).reshape(-1)
        H = _f64(program.H)
        if H.shape != (n, t):
            if H.shape == (t, n) and not H.any():
                H = numpy.zeros((n, t))
            else:
                raise ValueError(f'H must be num_x x num_t = {(n, t)}, got {H.shape}')
        Qp = getattr(program, 'Q', None)
        self.is_qp = Qp is not None and type(program).__name__ not in ('MPLP_Program', 'MPMILP_Program')
        Q = 0.5 * (_f64(Qp) + _f64(Qp).T) if self.is_qp else numpy.zeros((n, n))
        bins = [int(i) for i in program.binary_indices]
        cont = [int(i) for i in program.cont_indices]
        nb = len(bins)
        if nb < 1 or nb > 63:
            raise ValueError(f'{nb} binaries: 1 <= nb <= 63 are supported (an assignment is one uint64)')
        if sorted(bins + cont) != list(range(n)):
            raise ValueError('binary_indices and cont_indices must partition the variables')
        eq = set(int(i) for i in program.equality_indices)
        has_x = numpy.abs(A[:, cont]).max(1, initial=0.0) > 0.0
        crow = [i for i in range(m) if has_x[i] and i in eq] + [i for i in range(m) if has_x[i] and i not in eq]
        brow = [i for i in range(m) if not has_x[i]]
        self.n, self.t, self.nb, self.bins, self.cont = n, t, nb, bins, cont
        self.rows, self.binary_rows = numpy.array(crow, dtype=numpy.int64), numpy.array(brow, dtype=numpy.int64)
        self.program = program
        A_t, b_t = _f64(program.A_t).reshape(-1, t), _f64(program.b_t).reshape(-1)
        self.A_t, self.b_t = A_t, b_t
        arrays = dict(A=_f64(A[crow][:, cont]), b=_f64(b[crow]), F=_f64(F[crow]), A_t=A_t, b_t=b_t, c=_f64(c[cont]),
                      H=_f64(H[cont]), n_eq=sum(1 for i in crow if i in eq), is_qp=self.is_qp,
                      Q=_f64(Q[numpy.ix_(cont, cont)]) if self.is_qp else None)
        eng = _engine.Engine(arrays, device)
        self.eng = eng
        try:   # the handle holds device buffers: close it on any failure below
            Fy = _f64(-A[crow][:, bins])
            Hy = _f64(Q[numpy.ix_(cont, bins)]) if self.is_qp else None
            rows = ctypes.c_int32(0)
            rc = eng.lib.ppgpu_program_param_maps(eng.h, nb, Fy.ctypes.data, None if Hy is None else Hy.ctypes.data, None,
                                                  ctypes.byref(rows))
            if rc == -2:
                raise NotImplementedError(eng.lib.ppgpu_last_error().decode())
            _lib.check(rc, 'program_param_maps')
            maps = numpy.zeros((rows.value, nb))
            _lib.check(eng.lib.ppgpu_program_param_maps(eng.h, nb, Fy.ctypes.data, None if Hy is None else Hy.ctypes.data,
                                                        maps.ctypes.data, ctypes.byref(rows)), 'program_param_maps')
            self.seg, mb = rows.value, len(brow)
            # the offset vector of an assignment: [solver terms (seg) | b_i - A_{i,y} y (mb) | H_y' y (t) | c_y' y + 1/2 y'Qyy y]
            full = numpy.vstack([maps, -A[brow][:, bins].reshape(mb, nb), H[bins].T.reshape(t, nb), c[bins].reshape(1, nb)])
            base = numpy.concatenate([numpy.zeros(self.seg), b[brow], numpy.zeros(t + 1)])
            self.off_ld = full.shape[0]
            self.mb = mb
            if assignments is None:
                from .mp_solvers import mitree
                assignments = mitree.feasible_combinations(program).leaves
            self.assignments = numpy.array([[int(v) for v in y] for y in assignments], dtype=numpy.int64).reshape(-1, nb)
            if self.assignments.size and not numpy.isin(self.assignments, (0, 1)).all():
                raise ValueError('assignments must be 0/1 vectors')
            words = (self.assignments.astype(numpy.uint64) << numpy.arange(nb, dtype=numpy.uint64)).sum(1, dtype=numpy.uint64)
            dev = lambda a: torch.from_numpy(_f64(a)).to(eng.tdev)  # noqa: E731
            self.n_assign = len(self.assignments)
            self._assign = torch.from_numpy(words.view(numpy.int64).copy()).to(eng.tdev)
            self._off = torch.empty((max(self.n_assign, 1), self.off_ld), dtype=torch.float64, device=eng.tdev)
            self._maps, self._base = dev(full), dev(base)
            self._qyy = dev(Q[numpy.ix_(bins, bins)]) if self.is_qp else None
            with torch.cuda.device(eng.tdev):
                _lib.check(eng.lib.ppgpu_mi_offsets(self._maps.data_ptr(), self._base.data_ptr(), self.off_ld, nb,
                                                    self._assign.data_ptr(), self.n_assign,
                                                    None if self._qyy is None else self._qyy.data_ptr(), self.off_ld - 1,
                                                    self._off.data_ptr(), eng._stream()), 'mi_offsets')
            self._Fb = dev(F[brow].reshape(mb, t))
            self._beq = torch.tensor([1 if i in eq else 0 for i in brow], dtype=torch.uint8, device=eng.tdev)
            self._bins = torch.tensor(bins, dtype=torch.int64, device=eng.tdev)
            self._cont = torch.tensor(cont, dtype=torch.int64, device=eng.tdev)
            self._rows = torch.from_numpy(self.rows).to(eng.tdev)
            self._ybits = torch.from_numpy(self.assignments.astype(numpy.float64)).to(eng.tdev)
            self._A, self._b, self._F = dev(A), dev(b), dev(F)
            self._Q = dev(Q) if self.is_qp else None
            self._H, self._c = dev(H), dev(c)
            self._c_c = float(_attr(program, 'c_c', (1,))[0])
            self._c_t = dev(_attr(program, 'c_t', (t,)))
            self._Q_t = dev(_attr(program, 'Q_t', (t, t)))
            self.m = m
            self.W = eng.W
            self.chunk = chunk
        except Exception:
            eng.close()
            raise
        self._entry = 'ppgpu_solve_pairs_qp' if self.is_qp else 'ppgpu_solve_pairs_lp'
        self._out_cls = _solver_output_class(program)

    def close(self):
        self.eng.close()

    def _thetas(self, thetas) -> torch.Tensor:
        if torch.is_tensor(thetas):
            th = thetas.to(self.eng.tdev, dtype=torch.float64)
        else:
            th = torch.from_numpy(numpy.ascontiguousarray(thetas, dtype=numpy.float64)).to(self.eng.tdev)
        return th.reshape(-1, self.t).contiguous()

    def _theta_terms(self, th: torch.Tensor) -> torch.Tensor:
        return self._c_c + th @ self._c_t + 0.5 * ((th @ self._Q_t) * th).sum(1)

    def objective(self, thetas: torch.Tensor, x: torch.Tensor) -> torch.Tensor:
        """evaluate_objective(x, theta) of the full program for every row (device tensors; x the full variable vector)"""
        obj = ((thetas @ self._H.T) * x).sum(1) + x @ self._c
        if self._Q is not None:
            obj = obj + 0.5 * ((x @ self._Q) * x).sum(1)
        return obj + self._theta_terms(thetas)

    def _pairs(self, pairs: torch.Tensor, th: torch.Tensor, status, obj=None, x=None, dual=None, active=None, iters=None):
        e = self.eng
        ptr = lambda v: None if v is None else v.data_ptr()  # noqa: E731
        if pairs.shape[0]:
            with torch.cuda.device(e.tdev):
                _lib.check(getattr(e.lib, self._entry)(e.h, th.data_ptr(), pairs.data_ptr(), pairs.shape[0], self._off.data_ptr(),
                                                       self.off_ld, status.data_ptr(), ptr(obj), ptr(x), ptr(dual), ptr(active),
                                                       ptr(iters), e._stream()), self._entry[6:])

    def _chunk(self, k: int) -> int:
        if self.chunk is not None:
            return max(1, min(int(self.chunk), self.n_assign))
        return max(1, min(self.n_assign, PAIRS_PER_LAUNCH // max(k, 1)))

    def _chunk_pairs(self, k: int, a0: int, na: int) -> torch.Tensor:
        dev = self.eng.tdev
        pt = torch.arange(k, dtype=torch.int32, device=dev).repeat_interleave(na)
        asg = (a0 + torch.arange(na, dtype=torch.int32, device=dev)).repeat(k)
        return torch.stack([pt, asg], 1).contiguous()

    def solve_pairs(self, thetas, full: bool = False) -> Dict[str, torch.Tensor]:
        """every (point, assignment) pair (for tests and small batches): device tensors status (n_points x n_assign uint8,
        the K8 / K9 status of the continuous program), obj (the full objective, NaN unless optimal) and rows_hold (whether
        the binary-only rows hold at that theta and assignment); full: also x (n_points x n_assign x the continuous
        variables) and dual (... x the handle's rows ``rows``)"""
        e = self.eng
        th = self._thetas(thetas)
        k, na = th.shape[0], self.n_assign
        status, obj = e.empty((k * na,), torch.uint8), e.empty((k * na,), torch.float64)
        x = e.empty((k * na, len(self.cont)), torch.float64) if full else None
        dual = e.empty((k * na, len(self.rows)), torch.float64) if full else None
        self._pairs(self._chunk_pairs(k, 0, na), th, status, obj, x, dual)
        off = self._off[:na]
        const = off[:, -1][None, :] + th @ off[:, self.seg + self.mb:self.seg + self.mb + self.t].T
        obj_full = obj.reshape(k, na) + const + self._theta_terms(th)[:, None]
        s = off[None, :, self.seg:self.seg + self.mb] + (th @ self._Fb.T)[:, None, :]
        tol = ROW_TOL * (1.0 + s.abs())
        hold = torch.where(self._beq.bool()[None, None, :], s.abs() <= tol, s >= -tol).all(2)
        out = dict(status=status.reshape(k, na), obj=obj_full, rows_hold=hold)
        if full:
            out.update(x=x.reshape(k, na, len(self.cont)), dual=dual.reshape(k, na, len(self.rows)))
        return out

    def solve_batch(self, thetas) -> Dict[str, torch.Tensor]:
        """thetas (n_points x t, host or device) -> device tensors: status (uint8, MI_*), x (n_points x n: the full variable
        vector, binaries in place; NaN unless optimal), assignment (int64 index into ``assignments``, -1 unless optimal),
        obj (evaluate_objective of the full program), gap (runner-up objective - best, inf with one candidate), dual
        (n_points x m in the program's row numbering: Q x + H theta + c + A' dual = 0 on the continuous variables, zero on
        the binary-only rows), active (n_points x words, the candidate mask of the continuous handle's rows ``rows``), iters
        (the winning pair's, as ThetaSolver / ThetaLPSolver report them)"""
        e = self.eng
        th = self._thetas(thetas)
        k = th.shape[0]
        best = torch.full((k,), float('inf'), dtype=torch.float64, device=e.tdev)
        second, idx = best.clone(), torch.full((k,), -1, dtype=torch.int32, device=e.tdev)
        flags, status = torch.zeros((k,), dtype=torch.uint8, device=e.tdev), torch.full((k,), MI_INFEASIBLE, dtype=torch.uint8,
                                                                                          device=e.tdev)
        step = self._chunk(k)
        for a0 in range(0, self.n_assign if k else 0, step):
            na = min(step, self.n_assign - a0)
            pst, pobj = e.empty((k * na,), torch.uint8), e.empty((k * na,), torch.float64)
            self._pairs(self._chunk_pairs(k, a0, na), th, pst, pobj)
            with torch.cuda.device(e.tdev):
                _lib.check(e.lib.ppgpu_mi_select(th.data_ptr(), k, self.t, pst.data_ptr(), pobj.data_ptr(), a0, na,
                                                 self._off.data_ptr(), self.off_ld, self.seg, self.mb,
                                                 self._Fb.data_ptr() if self.mb else None,
                                                 self._beq.data_ptr() if self.mb else None, best.data_ptr(), second.data_ptr(),
                                                 idx.data_ptr(), flags.data_ptr(), status.data_ptr(), e._stream()), 'mi_select')
        ok = status == MI_OPTIMAL
        win = torch.nonzero(ok).reshape(-1)
        nw, nc = win.shape[0], len(self.cont)
        pairs = torch.stack([win.to(torch.int32), idx[win]], 1).contiguous()
        wst = e.empty((nw,), torch.uint8)
        xc, dc = e.empty((nw, nc), torch.float64), e.empty((nw, len(self.rows)), torch.float64)
        act = torch.zeros((nw, self.W), dtype=torch.int64, device=e.tdev)
        it = e.empty((nw,) if self.is_qp else (nw, 2), torch.int32)
        self._pairs(pairs, th, wst, None, xc, dc, act, it)
        # the same pair gives the same result, so pass 2 is optimal wherever pass 1 was; a point where it is not is reported
        # failed, with no x or dual, rather than optimal with NaN
        lost = wst != MI_OPTIMAL
        status[win[lost]] = MI_FAILED
        ok = status == MI_OPTIMAL
        nan = float('nan')
        x = torch.full((k, self.n), nan, dtype=torch.float64, device=e.tdev)
        xw = torch.empty((nw, self.n), dtype=torch.float64, device=e.tdev)
        xw[:, self._cont] = xc
        xw[:, self._bins] = self._ybits[idx[win].long()]
        xw[lost] = nan
        x[win] = xw
        dual = torch.full((k, self.m), nan, dtype=torch.float64, device=e.tdev)
        dw = torch.zeros((nw, self.m), dtype=torch.float64, device=e.tdev)
        dw[:, self._rows] = dc
        dw[lost] = nan
        dual[win] = dw
        active = torch.zeros((k, self.W), dtype=torch.int64, device=e.tdev)
        active[win] = act
        iters = torch.zeros((k,) + tuple(it.shape[1:]), dtype=torch.int32, device=e.tdev)
        iters[win] = it
        obj = torch.where(ok, best + self._theta_terms(th), torch.full_like(best, nan))
        gap = torch.where(ok, second - best, torch.full_like(best, nan))
        assignment = torch.where(ok, idx.long(), torch.full_like(idx, -1).long())
        return dict(status=status, x=x, assignment=assignment, obj=obj, gap=gap, dual=dual, active=active, iters=iters)

    def active_sets(self, active: torch.Tensor) -> List[List[int]]:
        """working-set / basis masks -> active rows in the program's row numbering (the continuous equality rows first)"""
        return [[int(self.rows[i]) for i in a] for a in self.eng.lists_from_masks(active.cpu().numpy())]

    def solve_theta(self, theta_point):
        """the reference's solve_theta of a mixed-integer program: SolverOutput(obj, sol, slack, active_set, dual) at one
        theta (sol the full variable vector), None when no assignment is feasible or the program is unbounded there;
        RuntimeError when a pair hit the iteration cap or broke down"""
        th = numpy.asarray(theta_point, dtype=numpy.float64).reshape(1, -1)
        out = self.solve_batch(th)
        st = int(out['status'][0])
        if st in (MI_INFEASIBLE, MI_UNBOUNDED):
            return None
        if st != MI_OPTIMAL:
            raise RuntimeError('fixed-theta mixed-integer solve failed: a pair hit the iteration cap or broke down')
        x = out['x'][:1]
        slack = self._b + self._thetas(th) @ self._F.T - x @ self._A.T
        return self._out_cls(obj=float(out['obj'][0]), sol=x[0].cpu().numpy(), slack=slack[0].cpu().numpy(),
                             active_set=numpy.array(self.active_sets(out['active'][:1])[0], dtype=numpy.int64),
                             dual=out['dual'][0].cpu().numpy())

    def sample_thetas(self, num_samples: int, seed: int = 0) -> numpy.ndarray:
        """uniform draws in theta_box(A_t, b_t), kept where every row of A_t theta <= b_t holds"""
        lo, hi = theta_box(self.A_t, self.b_t)
        th = numpy.random.default_rng(seed).uniform(lo, hi, size=(int(num_samples), self.t))
        return th[(th @ self.A_t.T <= self.b_t[None, :]).all(1)]


__all__ = ['MixedIntegerThetaSolver', 'SolverOutput', 'MI_OPTIMAL', 'MI_INFEASIBLE', 'MI_FAILED', 'MI_UNBOUNDED']


def verify_mixed_integer_solution(solution, thetas=None, num_samples: int = 100000, seed: int = 0, tol: float = 1e-5,
                                  solver: Optional[MixedIntegerThetaSolver] = None) -> Dict:
    """verify_solution for a solution whose regions carry y_fixation (solve_mpmiqp): per point the region the solution's own
    rule locates (K7 over the full variable vector, the overlap rule) against the fixed-theta minimum over the assignments
    of the solver - by default the relaxation tree's leaves, not ``solution.feasible_combinations``, so that an assignment
    the solution misses shows up as holes or dx.  The report of verify_solution (holes, spurious, max_dx, the band,
    n_failed; spurious counts the points without an optimum that a region contains), and
        n_spurious_band           points without an optimum located only through the tolerance band (outside every region
                                  by less than point_location_tolerance: the band reaches across the feasible set's edge)
        max_dobj                  largest |obj_explicit - obj_implicit| / max(1, |obj_implicit|) over the points of max_dx
        n_unbounded               points where the program is unbounded (an mpMILP)
        n_ties                    feasible points whose gap <= 1e-7 (1 + |obj|): two assignments are equally good there, x
                                  need not agree, and they are left out of max_dx / n_dx_over_tol
        n_assignment_mismatch     points of max_dx whose located region fixes another assignment than the winner's"""
    from .point_location import PointLocation
    own = solver is None
    solver = MixedIntegerThetaSolver(solution.program) if own else solver
    try:
        th = solver.sample_thetas(num_samples, seed) if thetas is None else numpy.asarray(thetas, dtype=numpy.float64).reshape(-1, solver.t)
        pl = PointLocation(solution, device=solver.eng.device)
        region, x_exp = pl.evaluate_batch(th, tol=float(getattr(solution, 'point_location_tolerance', 1e-5)))
        exact = pl.locate_batch(th)
        out = solver.solve_batch(th)
        status, x_imp = out['status'].cpu().numpy(), out['x'].cpu().numpy()
        obj_imp, gap, win = out['obj'].cpu().numpy(), out['gap'].cpu().numpy(), out['assignment'].cpu().numpy()
        x_dev = torch.from_numpy(numpy.ascontiguousarray(x_exp, dtype=numpy.float64)).to(solver.eng.tdev)
        obj_exp = solver.objective(solver._thetas(th), x_dev).cpu().numpy()
    finally:
        if own:
            solver.close()
    feas, inf, unb = status == MI_OPTIMAL, status == MI_INFEASIBLE, status == MI_UNBOUNDED
    # no optimum but a region: spurious where a region contains the point, a band point where it is only located through
    # the tolerance band (the band reaches across the feasible set's edge, where the program has no optimum)
    holes, spurious, spurious_band = feas & (region < 0), (inf | unb) & (exact >= 0), (inf | unb) & (region >= 0) & (exact < 0)
    located = feas & (region >= 0)
    rel = numpy.zeros(len(th))
    if located.any():
        rel[located] = numpy.abs(x_exp[located] - x_imp[located]).max(1) / numpy.maximum(1.0, numpy.abs(x_imp[located]).max(1))
    band = located & (exact != region)
    both = located & ~band
    dobj = numpy.zeros(len(th))
    dobj[both] = numpy.abs(obj_exp[both] - obj_imp[both]) / numpy.maximum(1.0, numpy.abs(obj_imp[both]))
    ties = feas & (gap <= 1e-7 * (1.0 + numpy.abs(numpy.where(feas, obj_imp, 0.0))))
    regions = solution.critical_regions
    fixed = numpy.array([[int(v) for v in r.y_fixation] for r in regions], dtype=numpy.int64).reshape(len(regions), -1)
    # the region's binaries in the order of the solver's binary_indices
    order = [list(regions[0].y_indices).index(i) for i in solver.bins] if regions else []
    mismatch = numpy.zeros(len(th), dtype=bool)
    chk = both & ~ties
    if chk.any():
        mismatch[chk] = (fixed[region[chk]][:, order] != solver.assignments[win[chk]]).any(1)
    both_dx = both & ~ties
    worst = int(numpy.argmax(numpy.where(both_dx, rel, -1.0))) if both_dx.any() else -1
    return dict(n_points=int(len(th)), n_feasible=int(feas.sum()), holes=int(holes.sum()), hole_thetas=th[holes],
                spurious=int(spurious.sum()), spurious_thetas=th[spurious], spurious_regions=region[spurious],
                n_spurious_band=int(spurious_band.sum()),
                max_dx=float(rel[both_dx].max()) if both_dx.any() else 0.0, worst_theta=th[worst] if worst >= 0 else None,
                n_dx_over_tol=int((rel[both_dx] > tol).sum()), n_band=int(band.sum()),
                max_dx_band=float(rel[band].max()) if band.any() else 0.0, n_failed=int((status == MI_FAILED).sum()),
                max_dobj=float(dobj[both].max()) if both.any() else 0.0, n_unbounded=int(unb.sum()), n_ties=int(ties.sum()),
                n_assignment_mismatch=int(mismatch.sum()))
