"""The geometric mpQP algorithm (ppopt_b200.mp_solvers.mpqp_geometric) and its facet Chebyshev balls (K10,
chebyshev.facet_balls).

1. K10 against HiGHS on the facet LP written directly in theta (equality row, |P a_j|): every facet of every region of the
   full-solution goldens and of ctrl_alloc_n5, and random polytopes with redundant rows, unbounded polytopes and t = 1.
2. Every region the geometric algorithm finds is a golden region (laws, half-spaces); no facet stays unresolved.
3. Coverage: at every golden region's Chebyshev centre the solution evaluates to the golden law; verify_solution holds.
4. Where the golden is a partition (no two regions overlap), the region sets are equal; the same for the graph goldens.
5. mpc_n10 against the combinatorial solve.  6. Seed independence.  7. Variants and determinism.  8. The retry path.
9. Refusals, a program infeasible on all of Theta, and an mpMIQP sub-problem loop.
"""
import os

import numpy
import pytest
import scipy.optimize

from conftest import GOLDEN
from parity import REL_TOL, golden_regions, rel_err, rows_match_as_sets

pytestmark = pytest.mark.gpu

FULL = ['ctrl_alloc_n1', 'ctrl_alloc_n2', 'doc_portfolio', 'factory_mpqp', 'mpc_n3', 'mpc_n5', 'mpc_n7', 'portfolio_analog',
        'rand_5_3_10_s2', 'rand_6_3_12_s1', 'simple_mpqp_1d']
GRAPH = sorted(f[:-4] for f in os.listdir(os.path.join(GOLDEN, 'graph')) if f.endswith('.npz'))
_solutions = {}


def _load(name):
    from ppopt_b200.mplp_program import load_presolved
    return load_presolved(os.path.join(GOLDEN, name + '.npz'))


def _geometric(name):
    if name not in _solutions:
        from ppopt_b200 import mpqp_algorithm, solve_mpqp
        _solutions[name] = solve_mpqp(_load(name), mpqp_algorithm.geometric)
    return _solutions[name]


def _key(r):
    return tuple(int(i) for i in (r['active_set'] if isinstance(r, dict) else r.active_set))


# ---- 1. K10 -------------------------------------------------------------------------------------------------------------
def _facet_reference(E, f, i):
    """HiGHS on max r s.t. E_j theta + |P E_j| r <= f_j (j != i), E_i theta = f_i -> (code, radius, centre or None)"""
    t = E.shape[1]
    n = E[i] / numpy.linalg.norm(E[i])
    others = [j for j in range(E.shape[0]) if j != i]
    PE = E[others] - numpy.outer(E[others] @ n, n)
    A_ub = numpy.hstack([E[others], numpy.linalg.norm(PE, axis=1)[:, None]]) if others else None
    res = scipy.optimize.linprog(numpy.r_[numpy.zeros(t), -1.0], A_ub=A_ub, b_ub=f[others] if others else None,
                                 A_eq=numpy.r_[E[i], 0.0][None, :], b_eq=[f[i]], bounds=[(None, None)] * (t + 1), method='highs',
                                 options=dict(primal_feasibility_tolerance=1e-10, dual_feasibility_tolerance=1e-10))
    if res.status == 0:
        return 0, -res.fun, res.x[:t]
    # 3: infeasible, 2: unbounded; HiGHS's other statuses (4: numerical difficulties) as -100 - status
    return {2: 3, 3: 2}.get(res.status, -100 - res.status), (numpy.inf if res.status == 3 else -numpy.inf), None


def _supported_radius(E, f, i, x):
    """the largest r for which the ball of radius r at x (projected on the facet's hyperplane) fits the facet:
    min_j (f_j - E_j x) / |P E_j| over the rows not parallel to the facet, with a rounding allowance of 4 ulp of the row's
    terms in favour of x"""
    nrm = numpy.linalg.norm(E, axis=1)
    n = E[i] / nrm[i]
    x = x - (E[i] @ x - f[i]) / nrm[i] * n
    o = numpy.arange(len(f)) != i
    pn = numpy.linalg.norm(E[o] - numpy.outer(E[o] @ n, n), axis=1)
    eps = 4e-16 * (numpy.abs(f[o]) + nrm[o] * numpy.abs(x).max())
    par = pn <= 1e-9 * nrm[o]      # K10's rule for rows parallel to the facet
    return ((f[o] - E[o] @ x + eps)[~par] / pn[~par]).min(initial=numpy.inf)


def _run_k10(polys, facets, t):
    import torch
    from ppopt_b200.chebyshev import facet_balls
    rows = numpy.vstack([numpy.hstack([f[:, None], E]) for E, f in polys])
    off = numpy.concatenate([[0], numpy.cumsum([len(f) for _, f in polys])])
    dev = torch.device('cuda', torch.cuda.current_device())
    c, r, code = facet_balls(torch.from_numpy(rows).to(dev), torch.from_numpy(off).to(dev),
                             torch.tensor(facets, dtype=torch.int64, device=dev), t)
    return c.cpu().numpy(), r.cpu().numpy(), code.cpu().numpy()


def _check_k10(polys, t):
    """K10 against HiGHS on every facet of ``polys``; returns the (polytope, row) pairs where the two disagree (code, or radius
    by more than 1e-9 (1 + |r|)) and those of them where HiGHS's centre supports a larger radius than K10's (K10 the wrong
    side; the 1e-8 decision must then agree outside the 1e-7 band).  K10's own ball is always checked: its centre lies on the hyperplane and supports
    its radius (every other row's slack >= |P a_j| r - 1e-9, rows scaled to unit length), and HiGHS's centre supports no larger
    radius: min_j slack_j / |P a_j| over the rows not parallel to the facet (or HiGHS reports no optimum where K10's centre is
    a feasible certificate).  Everywhere else the two agree within 1e-9 (1 + |r|)."""
    facets = [(p, i) for p, (E, f) in enumerate(polys) for i in range(len(f))]
    c, r, code = _run_k10(polys, facets, t)
    differ, short, same_side = [], [], []
    for k, (p, i) in enumerate(facets):
        E, f = polys[p]
        rc, rr, x = _facet_reference(E, f, i)
        tol = 1e-9 * (1 + abs(r[k]))
        if code[k] == 0:
            nrm = numpy.linalg.norm(E, axis=1)
            assert abs(E[i] @ c[k] - f[i]) / nrm[i] <= 1e-10 * max(1.0, numpy.abs(c[k]).max()), (t, p, i)
            n = E[i] / nrm[i]
            o = numpy.arange(len(f)) != i
            PE = E[o] - numpy.outer(E[o] @ n, n)
            slack = (f[o] - E[o] @ c[k]) / nrm[o]
            assert (slack >= numpy.linalg.norm(PE, axis=1) / nrm[o] * r[k] - 1e-9).all(), (t, p, i)
        elif t == 1 and code[k] == 2:
            assert abs(E[i, 0] * c[k, 0] - f[i]) <= 1e-12 * max(1.0, abs(f[i]))
        if code[k] == rc and (rc != 0 or abs(r[k] - rr) <= 1e-9 * (1 + abs(rr))):
            continue
        differ.append((p, i))
        assert code[k] == 0, (t, p, i, code[k], rc, r[k], rr)     # only a K10 optimum with its certificate may disagree
        if rc == 0:
            rho_h = _supported_radius(E, f, i, x)
            if rho_h > r[k] + tol:
                # K10 is the wrong side: its ball fits (asserted above) but is not the largest.  The centre is still a
                # point inside the facet, and the 1e-8 full-dimension decision must come out the same
                short.append((p, i))
                # (inside the 1e-7 band the engine itself reports full-dimension decisions as thin)
                same_side.append((rho_h > 1e-8) == (r[k] > 1e-8) or max(abs(rho_h), abs(r[k])) <= 1e-7)
        else:
            assert rc == 3 or rc <= -100, (t, p, i, rc)
    # permuting or splitting the facet list changes nothing
    perm = numpy.random.default_rng(1).permutation(len(facets))
    c2, r2, code2 = _run_k10(polys, [facets[j] for j in perm], t)
    assert numpy.array_equal(code2, code[perm]) and numpy.array_equal(r2, r[perm], equal_nan=True)
    assert numpy.array_equal(c2, c[perm], equal_nan=True)
    h = len(facets) // 2
    parts = [_run_k10(polys, facets[:h], t), _run_k10(polys, facets[h:], t)] if h else []
    if parts:
        assert numpy.array_equal(numpy.concatenate([parts[0][1], parts[1][1]]), r, equal_nan=True)
        assert numpy.array_equal(numpy.concatenate([parts[0][0], parts[1][0]]), c, equal_nan=True)
    print('K10 off HiGHS:', differ)
    print('K10 radius below a point HiGHS found:', short)
    assert all(same_side), [x for x, ok in zip(short, same_side) if not ok]
    return differ, short


def _random_polys(t, rng):
    polys = []
    for rows in (t + 1, 2 * t + 3, 40, 255):            # (+1 redundant row: 256, the envelope)
        # a bounded polytope around a random point; then a redundant copy of a row pushed outwards
        E = rng.standard_normal((rows, t)) * rng.uniform(0.5, 3.0, (rows, 1))
        x0 = rng.standard_normal(t)
        f = E @ x0 + rng.uniform(0.1, 2.0, rows)
        E = numpy.vstack([E, 2.0 * E[0]])
        f = numpy.r_[f, 2.0 * f[0] + 5.0]
        polys.append((E, f))
    if t > 1:
        E = numpy.vstack([numpy.eye(t)[:1], -numpy.eye(t)[:1]])      # a slab: unbounded facets
        polys.append((E, numpy.array([1.0, 1.0])))
    return polys


@pytest.mark.parametrize('t', [1, 2, 3, 8, 14])
def test_k10_random_polytopes_match_highs(t):
    assert _check_k10(_random_polys(t, numpy.random.default_rng(100 + t)), t) == ([], [])


def test_k10_t1_point_facets():
    E = numpy.array([[1.0], [-2.0], [1.0], [3.0]])
    f = numpy.array([1.0, 0.0, 0.5, 9.0])   # theta <= 1, theta >= 0, theta <= 0.5 (makes the facet theta = 1 empty), theta <= 3
    assert _check_k10([(E, f)], 1) == ([], [])


# Facets of ctrl_alloc_n5 (golden polytope: rows) where K10 and HiGHS disagree: in code, or in radius by more than
# 1e-9 (1 + |r|).  These are nearly degenerate facets of its thin regions.  Outside K10_SHORT, HiGHS is the wrong side: K10's
# centre supports K10's radius and HiGHS's centre no larger one, or HiGHS reports no optimum (or fails) where K10's centre
# is a feasible certificate.  None of the other goldens has such a facet.
K10_DIFFER = {'ctrl_alloc_n5': {
    8: (0, 6, 9), 9: (0, 7, 10), 10: (0, 7, 10), 11: (0, 7, 10), 12: (0, 10), 13: (0, 13), 14: (0, 14), 15: (0, 13),
    32: (8,), 35: (9,), 38: (9,), 41: (10,), 44: (0, 1), 45: (0, 1, 12), 46: (0, 1, 12), 47: (0, 1, 13), 50: (5,),
    51: (3,), 52: (3,), 53: (5,), 92: (7, 8), 93: (6, 7), 97: (6, 7), 98: (8, 9), 102: (8, 9), 103: (7, 8),
    107: (5, 6), 108: (7, 8), 118: (0, 6), 119: (0, 7, 11, 12), 120: (11,), 121: (10, 11), 126: (6, 7, 8, 10, 13),
    129: (6, 7, 8, 11, 14), 132: (6, 7, 8, 9, 12), 133: (10,), 135: (6, 7, 8, 10, 13), 138: (7, 9, 10, 11),
    140: (6, 7), 142: (5, 6, 7), 144: (7, 9, 11, 13), 146: (7, 9), 152: (7, 8), 158: (14,), 159: (6, 7), 165: (7, 9),
    171: (13,), 195: (13, 15), 196: (13, 15), 197: (4, 11), 198: (9,), 199: (2, 3, 8), 200: (2, 3, 8), 203: (7,),
    204: (4, 10), 205: (2, 3, 8), 206: (2, 3, 8), 209: (4, 12), 210: (11,), 211: (2, 3, 9), 212: (2, 3, 9),
    213: (12, 14), 214: (12, 14), 216: (4, 9), 217: (2, 3, 7), 218: (2, 3, 7), 221: (12, 13, 14, 15, 18, 20),
    222: (2, 6, 7), 223: (2, 6, 7), 224: (1, 3), 225: (2, 7), 226: (1, 3), 227: (12, 13, 14, 15, 16, 18, 19),
    228: (2, 7), 230: (2, 6, 7), 232: (12, 13, 14, 16, 17, 19, 20), 233: (2, 6, 7), 234: (1, 3), 235: (2, 6, 7),
    236: (1, 3), 237: (2, 6, 7), 238: (12, 13, 14, 15, 17, 18, 20)}}

# facets of K10_DIFFER where K10 is the wrong side: HiGHS's centre supports a larger radius than K10 reports.  K10's ball
# still fits the facet, so its centre is a valid probe origin, and the 1e-8 full-dimension decision agrees outside the 1e-7
# band in which the engine reports such decisions as thin (both asserted).
K10_SHORT = {'ctrl_alloc_n5': {
    119: (12,), 120: (11,), 126: (6, 8), 129: (6, 7, 8), 132: (6, 7, 8), 135: (6,), 142: (5,), 197: (11,), 198: (9,),
    203: (7,), 204: (4,), 209: (4, 12), 210: (11,), 216: (4,), 221: (12, 15), 222: (6,), 223: (6,),
    227: (12, 13, 14, 15, 18), 230: (6,), 232: (12, 13, 17, 20), 233: (6,), 238: (13, 14, 15, 18)}}


@pytest.mark.parametrize('name', FULL + ['ctrl_alloc_n5'])
def test_k10_golden_facets_match_highs(name):
    g = numpy.load(os.path.join(GOLDEN, name + '.npz'))
    regs = golden_regions(g)
    t = numpy.asarray(regs[0]['E']).reshape(len(regs[0]['f']), -1).shape[1]
    polys = [(numpy.asarray(r['E'], float).reshape(len(r['f']), t), numpy.asarray(r['f'], float).ravel()) for r in regs]
    differ, short = _check_k10(polys, t)
    pinned = lambda d: sorted((p, i) for p, rows in d.get(name, {}).items() for i in rows)   # noqa: E731
    assert sorted(differ) == pinned(K10_DIFFER)
    assert sorted(short) == pinned(K10_SHORT)


# ---- 2.-4. regions against the goldens ------------------------------------------------------------------------------
def _chebyshev_centre(E, f):
    E, f = numpy.asarray(E, float), numpy.asarray(f, float).ravel()
    t = E.shape[1]
    res = scipy.optimize.linprog(numpy.r_[numpy.zeros(t), -1.0], A_ub=numpy.hstack([E, numpy.linalg.norm(E, axis=1)[:, None]]),
                                 b_ub=f, bounds=[(None, None)] * t + [(0, None)], method='highs')
    return res.x[:t]


def _overlapping_pairs(regs):
    """pairs of regions that intersect with a Chebyshev radius above 1e-8 (chebyshev_radii on stacked pairs)"""
    from ppopt_b200.chebyshev import chebyshev_radii
    pairs = [(i, j) for i in range(len(regs)) for j in range(i + 1, len(regs))]
    if not pairs:
        return []
    P = [(numpy.vstack([numpy.asarray(regs[i]['E'], float), numpy.asarray(regs[j]['E'], float)]),
          numpy.vstack([numpy.asarray(regs[i]['f'], float).reshape(-1, 1), numpy.asarray(regs[j]['f'], float).reshape(-1, 1)]))
         for i, j in pairs]
    rad = chebyshev_radii(P)
    return [p for p, r in zip(pairs, rad) if r > 1e-8]


@pytest.mark.parametrize('name', FULL)
def test_regions_are_golden_regions(name):
    g = numpy.load(os.path.join(GOLDEN, name + '.npz'))
    ref = {_key(r): r for r in golden_regions(g)}
    sol = _geometric(name)
    assert sol.unresolved == [], (name, sol.unresolved)
    mine = [_key(r) for r in sol.critical_regions]
    assert len(set(mine)) == len(mine)
    for r in sol.critical_regions:
        b = ref.get(_key(r))
        assert b is not None, (name, _key(r))
        for fld in 'AbCd':
            assert rel_err(getattr(r, fld), b[fld]) <= 1e-8, (name, _key(r), fld)
        u1, u2 = rows_match_as_sets(r.E, r.f, b['E'], b['f'])
        assert not u1 and not u2, (name, _key(r))


# golden regions smaller than the point-location tolerance (1e-5) at whose Chebyshev centre Solution.evaluate picks a
# neighbour's law through that tolerance band (it takes the lowest objective among the regions it locates); the region
# itself is in the solution and is the only one that contains the centre exactly
BAND_LOCATED = {'rand_6_3_12_s1': [(0, 2, 3, 5, 7, 9), (1, 3, 4, 5, 8, 9), (1, 3, 4, 5, 9, 11)]}

# goldens where two regions overlap with a Chebyshev radius above 1e-8: none of the full-solution goldens
OVERLAPPING = []


@pytest.mark.parametrize('name', FULL)
def test_coverage_and_partition_equality(name):
    from ppopt_b200 import verify_solution
    g = numpy.load(os.path.join(GOLDEN, name + '.npz'))
    regs = golden_regions(g)
    sol = _geometric(name)
    mine = {_key(r): r for r in sol.critical_regions}
    banded = []
    for r in regs:
        th = _chebyshev_centre(r['E'], r['f'])
        x = sol.evaluate(th.reshape(-1, 1))
        want = (numpy.asarray(r['A'], float) @ th.reshape(-1, 1) + numpy.asarray(r['b'], float).reshape(-1, 1)).ravel()
        scale = 1e-6 * max(1.0, numpy.abs(want).max())
        if x is not None and numpy.abs(numpy.asarray(x, float).ravel() - want).max() <= scale:
            continue
        banded.append(_key(r))
        exact = [k for k, s_ in mine.items() if (numpy.asarray(s_.E) @ th - numpy.asarray(s_.f).ravel()).max() <= 0]
        assert exact == [_key(r)], (name, _key(r), exact)
        assert numpy.abs(mine[_key(r)].evaluate(th.reshape(-1, 1)).ravel() - want).max() <= scale, (name, _key(r))
    assert banded == BAND_LOCATED.get(name, []), (name, banded)
    rep = verify_solution(sol, num_samples=100000, seed=3)
    assert rep['n_points'] > 50000 and rep['n_failed'] == 0, rep
    assert rep['holes'] == 0, (name, rep['hole_thetas'][:5])
    assert rep['max_dx'] <= 1e-6, (name, rep['max_dx'], rep['worst_theta'])
    assert rep['n_band'] < 0.01 * rep['n_points'], rep['n_band']
    for th, ri in zip(rep['spurious_thetas'], rep['spurious_regions']):
        cr = sol.critical_regions[int(ri)]
        E, f = numpy.asarray(cr.E, dtype=float), numpy.asarray(cr.f, dtype=float).ravel()
        assert ((E @ th - f) / numpy.linalg.norm(E, axis=1)).max() >= -1e-5, (name, th)
    over = _overlapping_pairs(regs)
    assert bool(over) == (name in OVERLAPPING), (name, over[:5])
    if not over:
        assert {_key(r) for r in sol.critical_regions} == {_key(r) for r in regs}, name


@pytest.mark.parametrize('name', GRAPH)
def test_graph_golden_region_sets(name):
    g = numpy.load(os.path.join(GOLDEN, 'graph', name + '.npz'))
    regs = golden_regions(g)
    if _overlapping_pairs(regs):
        pytest.skip(f'{name}: the golden regions overlap')
    assert {_key(r) for r in _geometric(name).critical_regions} == {_key(r) for r in regs}


def test_mpc_n10_matches_combinatorial():
    import time
    from ppopt_b200 import mpqp_algorithm, solve_mpqp
    prog = _load('mpc_n10')
    t0 = time.perf_counter()
    ref = solve_mpqp(prog, mpqp_algorithm.combinatorial)
    print('mpc_n10 combinatorial solve', time.perf_counter() - t0, 's')
    sol = solve_mpqp(prog, mpqp_algorithm.geometric)
    assert sol.unresolved == []
    refs = [dict(active_set=r.active_set, E=r.E, f=r.f) for r in ref.critical_regions]
    mine, want = {_key(r) for r in sol.critical_regions}, {_key(r) for r in refs}
    assert mine <= want
    if not _overlapping_pairs(refs):
        assert mine == want


# ---- 6.-8. ------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize('name', FULL)
def test_seed_independence(name):
    from ppopt_b200.mp_solvers import mpqp_geometric
    regs = golden_regions(numpy.load(os.path.join(GOLDEN, name + '.npz')))
    want = {_key(r) for r in _geometric(name).critical_regions}
    for k in {0, len(regs) // 2, len(regs) - 1}:
        sol = mpqp_geometric.solve(_load(name), initial_active_sets=[list(_key(regs[k]))])
        assert {_key(r) for r in sol.critical_regions} == want, (name, k)


@pytest.mark.parametrize('name', ['ctrl_alloc_n2', 'mpc_n5', 'rand_6_3_12_s1'])
def test_variants_and_determinism(name):
    from ppopt_b200 import mpqp_algorithm, solve_mpqp
    runs = [solve_mpqp(_load(name), a) for a in (mpqp_algorithm.geometric, mpqp_algorithm.geometric,
                                                 mpqp_algorithm.geometric_parallel, mpqp_algorithm.geometric_parallel_exp)]
    for s in runs[1:]:
        assert [_key(r) for r in s.critical_regions] == [_key(r) for r in runs[0].critical_regions]
        for a, b in zip(s.critical_regions, runs[0].critical_regions):
            for fld in ('A', 'b', 'C', 'd', 'E', 'f'):
                assert numpy.array_equal(numpy.asarray(getattr(a, fld)), numpy.asarray(getattr(b, fld))), (name, fld)


@pytest.mark.parametrize('name', ['rand_6_3_12_s1', 'ctrl_alloc_n2'])
def test_retry_path(name, monkeypatch):
    """PROBE_STEP = 1e-10: first probes that K8 still answers with the source's own set (or no region) are retried further
    out, and the retries recover the whole partition"""
    from ppopt_b200.mp_solvers import mpqp_geometric
    want = {_key(r) for r in _geometric(name).critical_regions}
    monkeypatch.setattr(mpqp_geometric, 'PROBE_STEP', 1e-10)
    sol = mpqp_geometric.solve(_load(name))
    assert sol.retries > 0
    assert sol.unresolved == []
    assert {_key(r) for r in sol.critical_regions} == want


@pytest.mark.parametrize('name', ['rand_6_3_12_s1', 'ctrl_alloc_n2'])
def test_retry_limit(name, monkeypatch):
    """the documented limit: at PROBE_STEP = 1e-14 even delta x 100 stays inside K8's tolerances, the retries do not
    recover the facets, and the search stops early with them recorded as unresolved (pinned exactly)"""
    from ppopt_b200.mp_solvers import mpqp_geometric
    want = {_key(r) for r in _geometric(name).critical_regions}
    monkeypatch.setattr(mpqp_geometric, 'PROBE_STEP', 1e-14)
    sol = mpqp_geometric.solve(_load(name))
    got = {_key(r) for r in sol.critical_regions}
    assert sol.retries > 0 and got <= want
    print(name, 'retries', sol.retries, 'regions', len(got), 'of', len(want), 'unresolved', len(sol.unresolved))
    assert (len(got), len(sol.unresolved) > 0) == RETRY_LIMIT[name], (len(got), len(sol.unresolved))


RETRY_LIMIT = {'rand_6_3_12_s1': (3, True), 'ctrl_alloc_n2': (1, True)}


def test_refusals_and_infeasible_program():
    from ppopt_b200 import mpqp_algorithm, solve_mpqp
    from ppopt_b200.mplp_program import MPQP_Program
    from test_solve_theta_twin import _program
    lp = [f[:-4] for f in sorted(os.listdir(GOLDEN)) if f.endswith('.npz') and _program(f[:-4]) is None]
    assert lp
    with pytest.raises(NotImplementedError):
        solve_mpqp(_load(lp[0]), mpqp_algorithm.geometric)
    A = numpy.array([[1.0, 0.0], [0.0, 1.0], [-1.0, 0.0], [0.0, -1.0]])
    semi = MPQP_Program(A, numpy.ones((4, 1)), numpy.zeros((2, 1)), numpy.zeros((2, 1)), numpy.diag([1.0, 0.0]),
                        numpy.array([[1.0], [-1.0]]), numpy.ones((2, 1)), numpy.zeros((4, 1)), presolved=True)
    with pytest.raises(NotImplementedError):
        solve_mpqp(semi, mpqp_algorithm.geometric)
    # x <= -1 - theta and x >= 0 with theta in [0, 1]: no theta has a feasible QP
    infeas = MPQP_Program(numpy.array([[1.0], [-1.0]]), numpy.array([[-1.0], [0.0]]), numpy.zeros((1, 1)), numpy.zeros((1, 1)),
                          numpy.eye(1), numpy.array([[1.0], [-1.0]]), numpy.array([[1.0], [0.0]]), numpy.array([[-1.0], [0.0]]),
                          presolved=True)
    sol = solve_mpqp(infeas, mpqp_algorithm.geometric)
    assert len(sol.critical_regions) == 0 and sol.unresolved == []


def test_mpmiqp_with_geometric():
    from test_gpu_mpmiqp import MI, StoredMixedIntegerProgram
    from ppopt_b200 import mpqp_algorithm
    from ppopt_b200.mp_solvers import mpmiqp_enumeration
    g = numpy.load(os.path.join(MI, 'random_mpmiqp_5_4.npz'))
    prog = StoredMixedIntegerProgram(g)
    combos = [list(c) for c in g['combinations'].tolist()]
    per = {}
    for algo in (mpqp_algorithm.geometric, mpqp_algorithm.combinatorial):
        sol = mpmiqp_enumeration.solve_mpmiqp_enumeration(prog, cont_algorithm=algo, feasible_combinations=combos, streams=1)
        d = {}
        for r in sol.critical_regions:
            d.setdefault(tuple(numpy.asarray(r.y_fixation).ravel().tolist()), set()).add(_key(r))
        per[algo] = d
    assert per[mpqp_algorithm.geometric] == per[mpqp_algorithm.combinatorial]
