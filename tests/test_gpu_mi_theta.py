"""Fixed-theta solves of mixed-integer programs on the GPU (ppopt_b200.MixedIntegerThetaSolver: K8 / K9 in pair mode and the
winner of csrc/mi_theta.cu), point location of solutions with fixed binaries (K7) and verify_solution on them.

1. Pairs, checked without the solver's own logic: KKT of every optimal mpMIQP pair in numpy, HiGHS on every infeasible pair,
   and the pair objectives against ThetaSolver / ThetaLPSolver on the substituted program (a separate handle and reduction).
2. Winner: scipy.optimize.milp on the full mpMILP, the numpy minimum over the pairs of an mpMIQP; identical outputs for any
   chunking, batch order and batch size; points outside Theta, points without a feasible assignment and assignments that
   are infeasible everywhere.
3. Point location of solve_mpmiqp's solutions against the mirror Solution.get_region / evaluate.
4. verify_solution end to end; the envelope (nb = 63 / 64) and the refusals.
"""
import numpy
import pytest
from scipy.optimize import Bounds, LinearConstraint, linprog, milp

from mi_programs import MixedIntegerObjectiveProgram, objective_program
from mitree_programs import MixedIntegerProgram

pytestmark = pytest.mark.gpu

MIQP = [dict(nb=4, seed=0), dict(nb=4, seed=7, couple=True), dict(nb=6, seed=6)]
MILP = [dict(nb=5, seed=4), dict(nb=5, seed=8, couple=True)]
MILP_SOLVED = dict(nb=3, seed=3)   # an mpMILP whose solve_mpmiqp solution the point location and verify tests use


def _solver(prog, **kw):
    from ppopt_b200 import MixedIntegerThetaSolver
    return MixedIntegerThetaSolver(prog, **kw)


def _np(out):
    return {k: v.cpu().numpy() for k, v in out.items()}


def _thetas(prog, k, seed, scale=1.0):
    rng = numpy.random.default_rng(seed)
    return rng.uniform(-scale, scale, size=(k, prog.F.shape[1]))


def _continuous_rows(prog, solver, th, y):
    """(A, h, eq) of the solver's continuous rows at (theta, y), in the handle's order"""
    rows = solver.rows
    A = prog.A[rows][:, prog.cont_indices]
    h = prog.b.ravel()[rows] + prog.F[rows] @ th - prog.A[rows][:, prog.binary_indices] @ y
    eq = numpy.isin(rows, prog.equality_indices)
    return A, h, eq


def _margin(A, h, eq):
    """min over x of the largest scaled violation (HiGHS); <= 0: feasible"""
    sc = 1.0 + numpy.abs(h)
    n = A.shape[1]
    G = numpy.vstack([numpy.hstack([A, -sc[:, None]]), numpy.hstack([-A[eq], -sc[eq][:, None]])])
    hh = numpy.concatenate([h, -h[eq]])
    c = numpy.zeros(n + 1)
    c[-1] = 1.0
    res = linprog(c, A_ub=G, b_ub=hh, bounds=[(None, None)] * n + [(-1.0, None)], method='highs')
    assert res.status == 0, res.message
    return float(res.x[-1])


@pytest.mark.parametrize('kind,spec', [('qp', s) for s in MIQP] + [('lp', s) for s in MILP],
                         ids=lambda v: v if isinstance(v, str) else f"nb{v['nb']}s{v['seed']}")
def test_pairs_kkt_and_highs(kind, spec):
    """every optimal pair (K8 for an mpMIQP, K9 for an mpMILP) satisfies KKT, every infeasible pair is infeasible for HiGHS
    outside the 1e-7 band"""
    prog = objective_program(kind=kind, **spec)
    s = _solver(prog)
    th = _thetas(prog, 40, spec['seed'], scale=1.3)
    out = _np(s.solve_pairs(th, full=True))
    n = prog.A.shape[1]
    Qs = numpy.zeros((n, n)) if prog.Q is None else 0.5 * (prog.Q + prog.Q.T)
    xi, bi = prog.cont_indices, prog.binary_indices
    n_opt = n_inf = 0
    for p in range(len(th)):
        for a, y in enumerate(s.assignments):
            A, h, eq = _continuous_rows(prog, s, th[p], y)
            st = out['status'][p, a]
            if st == 0:
                n_opt += 1
                x, lam = out['x'][p, a], out['dual'][p, a]
                slack = h - A @ x
                scale = 1.0 + numpy.abs(h)
                assert (slack >= -1e-7 * scale).all() and (numpy.abs(slack[eq]) <= 1e-7 * scale[eq]).all()
                assert (lam[~eq] >= -1e-9).all()
                assert (numpy.abs(lam[~eq] * slack[~eq]) <= 1e-7 * (1.0 + numpy.abs(lam[~eq])) * scale[~eq]).all()
                g = Qs[numpy.ix_(xi, xi)] @ x + prog.c.ravel()[xi] + prog.H[xi] @ th[p] + Qs[numpy.ix_(xi, bi)] @ y + A.T @ lam
                assert numpy.abs(g).max() <= 1e-8 * (1.0 + numpy.abs(x).max()), (p, a, numpy.abs(g).max())
            elif st == 1:
                n_inf += 1
                assert _margin(A, h, eq) > -1e-7, (p, a)
            else:
                raise AssertionError(f'pair ({p}, {a}) status {st}')
    assert n_opt > 0 and n_inf > 0
    s.close()


@pytest.mark.parametrize('kind,spec', [('qp', s) for s in MIQP] + [('lp', s) for s in MILP],
                         ids=lambda v: v if isinstance(v, str) else f"nb{v['nb']}s{v['seed']}")
def test_pair_objectives_match_substituted_program(kind, spec):
    """an assignment is skipped only where the substituted mpQP leaves no free direction after its presolve (n - n_eq = 0,
    outside ThetaSolver); every other assignment is compared"""
    from ppopt_b200.solve_theta import solver_for
    prog = objective_program(kind=kind, **spec)
    s = _solver(prog)
    th = s.sample_thetas(400, seed=spec['seed'])
    out = _np(s.solve_pairs(th))
    compared, skipped, checked = 0, [], 0
    for a, y in enumerate(s.assignments):
        sub = prog.generate_substituted_problem(y)
        if kind == 'qp' and sub.A.shape[1] - len(sub.equality_indices) < 1:
            skipped.append(a)
            continue
        ref = solver_for(sub)
        try:
            r = _np(ref.solve_batch(th))
        finally:
            ref.close()
        checked += 1
        both = (out['status'][:, a] == 0) & out['rows_hold'][:, a] & (r['status'] == 0)
        got, want = out['obj'][both, a], r['obj'][both]
        assert (numpy.abs(got - want) <= 1e-9 * (1.0 + numpy.abs(want))).all(), (a, numpy.abs(got - want).max())
        compared += int(both.sum())
    assert compared > 0 and checked >= max(1, s.n_assign // 2), (checked, skipped, s.n_assign)
    s.close()


def _milp(prog, th, shrink=0.0):
    """scipy.optimize.milp on the full program at theta: (status 0 optimal / 1 infeasible, objective, z).  The objective is
    taken from HiGHS' LP at the rounded assignment: the MIP's integrality tolerance lets a big-M row open a little.
    shrink: every inequality row tightened to A_i z <= h_i - shrink (1 + |h_i|)."""
    n = prog.A.shape[1]
    c = prog.c.ravel() + prog.H @ th
    h = prog.b.ravel() + prog.F @ th
    eq = numpy.zeros(len(h), bool)
    eq[list(prog.equality_indices)] = True
    h = numpy.where(eq, h, h - shrink * (1.0 + numpy.abs(h)))
    lo = numpy.where(eq, h, -numpy.inf)
    integrality = numpy.zeros(n)
    integrality[prog.binary_indices] = 1
    lb, ub = numpy.full(n, -numpy.inf), numpy.full(n, numpy.inf)
    lb[prog.binary_indices], ub[prog.binary_indices] = 0.0, 1.0
    res = milp(c, constraints=LinearConstraint(prog.A, lo, h), integrality=integrality, bounds=Bounds(lb, ub),
               options=dict(mip_rel_gap=0.0))
    if res.status != 0:
        return 1, numpy.nan, None
    y = numpy.round(res.x[prog.binary_indices])
    lb[prog.binary_indices], ub[prog.binary_indices] = y, y
    lp = linprog(c, A_ub=prog.A[~eq], b_ub=h[~eq], A_eq=prog.A[eq] if eq.any() else None, b_eq=h[eq] if eq.any() else None,
                 bounds=list(zip(lb, ub)), method='highs')
    if lp.status == 0:
        res = lp
    const = float(prog.c_c[0, 0] + prog.c_t.ravel() @ th + 0.5 * th @ prog.Q_t @ th)
    return 0, float(res.fun) + const, res.x


@pytest.mark.parametrize('spec', MILP, ids=lambda s: f"nb{s['nb']}s{s['seed']}")
def test_milp_winner_matches_scipy_milp(spec):
    prog = objective_program(kind='lp', **spec)
    s = _solver(prog)
    th = s.sample_thetas(300, seed=7)
    out = _np(s.solve_batch(th))
    agree = 0
    for p in range(len(th)):
        st, obj, z = _milp(prog, th[p])
        if out['status'][p] == 0 and st == 0:
            assert abs(out['obj'][p] - obj) <= 1e-7 * (1.0 + abs(obj)), (p, out['obj'][p], obj)
            agree += 1
        elif out['status'][p] == 0:
            # HiGHS finds no point, the solver does: its point lies inside the tolerance band
            h = prog.b.ravel() + prog.F @ th[p]
            viol = (prog.A @ out['x'][p] - h) / (1.0 + numpy.abs(h))
            viol[prog.equality_indices] = numpy.abs(viol[prog.equality_indices])
            assert viol.max() <= 1e-6, (p, st, viol.max())
        elif st == 0:
            # HiGHS finds an optimum, the solver does not: it must say infeasible, and the program must be infeasible
            # once every inequality row is tightened by the band
            assert out['status'][p] == 1, (p, out['status'][p])
            assert _milp(prog, th[p], shrink=1e-7)[0] == 1, p
        else:
            assert out['status'][p] == 1, (p, out['status'][p])   # HiGHS: infeasible
    assert agree > 0
    s.close()


@pytest.mark.parametrize('spec', MIQP, ids=lambda s: f"nb{s['nb']}s{s['seed']}")
def test_miqp_winner_is_the_pair_minimum(spec):
    prog = objective_program(kind='qp', **spec)
    s = _solver(prog)
    th = s.sample_thetas(500, seed=8)
    pairs, out = _np(s.solve_pairs(th)), _np(s.solve_batch(th))
    cand = (pairs['status'] == 0) & pairs['rows_hold']
    val = numpy.where(cand, pairs['obj'], numpy.inf)
    has = cand.any(1)
    assert numpy.array_equal(out['status'] == 0, has)
    best = val.min(1)
    assert numpy.allclose(out['obj'][has], best[has], rtol=1e-12, atol=1e-12)
    # the winner: the lowest index among the assignments within rounding of the minimum
    w = out['assignment'][has]
    assert (val[has, w] <= best[has] + 1e-12 * (1.0 + numpy.abs(best[has]))).all()
    x = out['x'][has]
    assert numpy.array_equal(x[:, prog.binary_indices], s.assignments[w].astype(float))
    # obj is evaluate_objective of the full x
    for p in numpy.nonzero(has)[0][:50]:
        assert abs(prog.evaluate_objective(out['x'][p], th[p]) - out['obj'][p]) <= 1e-9 * (1.0 + abs(out['obj'][p]))
    srt = numpy.sort(val[has], 1)
    gap = numpy.where(numpy.isfinite(srt[:, 1]), srt[:, 1] - srt[:, 0], numpy.inf) if srt.shape[1] > 1 else numpy.inf
    assert numpy.allclose(out['gap'][has], gap, rtol=1e-9, atol=1e-9)
    s.close()


def _same(a, b):
    for k in a:
        assert numpy.array_equal(a[k], b[k], equal_nan=True), k


@pytest.mark.parametrize('kind', ['qp', 'lp'])
def test_chunking_order_and_batch_size_do_not_matter(kind):
    prog = objective_program(4, 7, kind=kind, couple=True)
    th = _thetas(prog, 700, 3, scale=1.3)
    s1, s2 = _solver(prog, chunk=1), _solver(prog)
    assert s2._chunk(len(th)) == s2.n_assign > 1
    ref = _np(s2.solve_batch(th))
    _same(_np(s1.solve_batch(th)), ref)
    perm = numpy.random.default_rng(0).permutation(len(th))
    got = _np(s2.solve_batch(th[perm]))
    _same(got, {k: v[perm] for k, v in ref.items()})
    _same(_np(s1.solve_batch(th[:37])), {k: v[:37] for k, v in ref.items()})
    s1.close(), s2.close()


def test_outside_theta_no_feasible_assignment_and_infeasible_assignments():
    prog = objective_program(4, 5, kind='qp')
    s = _solver(prog)
    # far outside Theta: solved as given; the winner is still the pair minimum
    th = numpy.vstack([_thetas(prog, 200, 1, scale=4.0), numpy.full((3, prog.F.shape[1]), 1e3)])
    pairs, out = _np(s.solve_pairs(th)), _np(s.solve_batch(th))
    cand = (pairs['status'] == 0) & pairs['rows_hold']
    assert numpy.array_equal(out['status'] == 0, cand.any(1))
    none = ~cand.any(1)
    assert none.any()
    assert (out['status'][none] == 1).all() and numpy.isnan(out['x'][none]).all() and (out['assignment'][none] == -1).all()
    # assignments that break a binary-only row everywhere never win and change nothing else
    allone = numpy.ones(len(prog.binary_indices), dtype=int)
    bad = [list(allone)] if not any((allone == a).all() for a in s.assignments) else []
    assert bad, 'the test needs an assignment outside the feasible list'
    s2 = _solver(prog, assignments=bad + [list(a) for a in s.assignments] + bad)
    out2 = _np(s2.solve_batch(th))
    for k in ('status', 'x', 'obj', 'gap', 'dual'):
        assert numpy.array_equal(out2[k], out[k], equal_nan=True), k
    ok = out['status'] == 0
    assert numpy.array_equal(out2['assignment'][ok] - 1, out['assignment'][ok])
    s.close(), s2.close()


def test_solve_theta_record():
    prog = objective_program(3, 0, kind='qp')
    s = _solver(prog)
    th = s.sample_thetas(50, seed=2)
    out = _np(s.solve_batch(th))
    p = int(numpy.nonzero(out['status'] == 0)[0][0])
    rec = s.solve_theta(th[p])
    assert numpy.array_equal(rec.sol, out['x'][p]) and rec.obj == out['obj'][p]
    assert numpy.allclose(rec.slack, prog.b.ravel() + prog.F @ th[p] - prog.A @ rec.sol)
    assert set(rec.active_set) <= set(s.rows.tolist())
    far = numpy.full(prog.F.shape[1], 1e3)
    if int(s.solve_batch(far[None])['status'][0]) == 1:
        assert s.solve_theta(far) is None
    s.close()


def _solution(prog):
    from ppopt_b200.mp_solvers.solve_mpmiqp import solve_mpmiqp
    return solve_mpmiqp(prog)


@pytest.mark.parametrize('kind,spec', [('qp', MIQP[0]), ('qp', MIQP[1]), ('lp', MILP_SOLVED)],
                         ids=lambda v: v if isinstance(v, str) else f"nb{v['nb']}s{v['seed']}")
def test_point_location_of_fixed_binaries_matches_mirror(kind, spec):
    from ppopt_b200 import PointLocation
    prog = objective_program(kind=kind, **spec)
    sol = _solution(prog)
    assert sol.critical_regions and sol.is_overlapping
    th = _thetas(prog, 10000, 9, scale=1.05)
    pl = PointLocation(sol)
    assert pl.n_x == prog.A.shape[1]
    region, x = pl.evaluate_batch(th, tol=sol.point_location_tolerance)
    regs = sol.critical_regions
    idx = {id(r): i for i, r in enumerate(regs)}
    n_tie = 0
    for p in range(len(th)):
        r = sol.get_region(th[p].reshape(-1, 1))
        want = -1 if r is None else idx[id(r)]
        if want < 0 or region[p] < 0:
            assert want == region[p], p
            continue
        xe = sol.evaluate(th[p].reshape(-1, 1)).ravel()
        if region[p] != want:
            n_tie += 1
            o1 = prog.evaluate_objective(x[p], th[p])
            o2 = prog.evaluate_objective(xe, th[p])
            assert abs(o1 - o2) <= 1e-9 * (1.0 + abs(o2)), p
        else:
            assert numpy.allclose(x[p], xe, rtol=1e-12, atol=1e-12)
    assert n_tie <= len(th) // 100
    assert (region >= 0).sum() > 0


def test_point_location_refuses_more_than_128_variables():
    from ppopt_b200 import PointLocation
    from ppopt_b200.critical_region import CriticalRegion
    from ppopt_b200.solution import Solution
    r = CriticalRegion(numpy.zeros((100, 1)), numpy.zeros((100, 1)), None, None, numpy.ones((1, 1)), numpy.ones((1, 1)), [],
                       y_fixation=[0] * 40, y_indices=list(range(100, 140)), x_indices=list(range(100)))
    with pytest.raises(NotImplementedError, match='128'):
        PointLocation(Solution(None, [r], is_overlapping=True))


VERIFY = [('qp', MIQP[0]), ('qp', MIQP[1]), ('qp', MIQP[2]), ('lp', MILP_SOLVED), ('lp', dict(nb=22, seed=6, at_most=1))]


@pytest.mark.parametrize('kind,spec', VERIFY, ids=lambda v: v if isinstance(v, str) else f"nb{v['nb']}s{v['seed']}")
def test_verify_solution_of_mixed_integer_solutions(kind, spec):
    from ppopt_b200 import verify_solution
    prog = objective_program(kind=kind, **spec)
    sol = _solution(prog)
    rep = verify_solution(sol, num_samples=20000, seed=1)
    assert rep['n_feasible'] > 0
    assert rep['holes'] == 0 and rep['spurious'] == 0, rep
    assert rep['max_dobj'] <= 1e-7 and rep['max_dx'] <= 1e-6, rep
    assert rep['n_assignment_mismatch'] == 0 and rep['n_failed'] == 0, rep


def test_63_binaries_work_and_64_are_refused():
    # (the relaxation tree holds at most 64 free variables, so the assignments are given: none or one binary set)
    prog = objective_program(63, 0, kind='lp', at_most=1)
    s = _solver(prog, assignments=numpy.vstack([numpy.zeros((1, 63), int), numpy.eye(63, dtype=int)]))
    assert s.nb == 63 and s.n_assign == 64
    out = _np(s.solve_batch(s.sample_thetas(200, seed=0)))
    assert (out['status'] == 0).any()
    opt = out['status'] == 0
    assert numpy.array_equal(out['x'][opt][:, prog.binary_indices], s.assignments[out['assignment'][opt]].astype(float))
    s.close()
    with pytest.raises(ValueError, match='nb <= 63'):
        _solver(objective_program(64, 0, kind='lp', at_most=1), assignments=[[0] * 64])


def test_programs_outside_k8_k9_are_refused_and_failures_raise():
    from ppopt_b200 import _lib
    prog = objective_program(3, 0, kind='qp')
    Q = prog.Q.copy()
    Q[numpy.ix_(prog.cont_indices, prog.cont_indices)] = 0.0
    semi = MixedIntegerObjectiveProgram(prog, Q, prog.H, prog.c)
    with pytest.raises(NotImplementedError):
        _solver(semi, assignments=[[0, 0, 1]])
    # a continuous variable in no row: the mpLP part has no vertex
    lp = objective_program(3, 0, kind='lp')
    nc = len(lp.cont_indices)
    A = numpy.hstack([lp.A[:, :nc], numpy.zeros((lp.A.shape[0], 1)), lp.A[:, nc:]])
    base = MixedIntegerProgram(A, lp.b, lp.F, lp.A_t, lp.b_t, [i + 1 for i in lp.binary_indices], lp.equality_indices)
    free = MixedIntegerObjectiveProgram(base, None, numpy.vstack([lp.H[:nc], numpy.zeros((1, lp.H.shape[1])), lp.H[nc:]]),
                                        numpy.concatenate([lp.c.ravel()[:nc], [1.0], lp.c.ravel()[nc:]]))
    with pytest.raises(NotImplementedError):
        _solver(free, assignments=[[0, 0, 1]])
    s = _solver(prog)
    with pytest.raises(RuntimeError, match='null argument'):
        _lib.check(s.eng.lib.ppgpu_solve_pairs_qp(s.eng.h, None, None, 5, None, s.off_ld, None, None, None, None, None, None,
                                                  s.eng._stream()), 'solve_pairs_qp')
    s.close()
