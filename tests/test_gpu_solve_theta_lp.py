"""Fixed-theta LP solves on the GPU (K9, csrc/k9_theta_lp.cu) through the C ABI, ppopt_b200.ThetaLPSolver and
MPLP_Program.

1. At the Chebyshev centre of every golden mpLP region (intersected with Theta, radius >= 1e-6) the status is optimal, the
   basis is the region's active set, x its law and the basis multipliers its C theta + d.  Centres where HiGHS finds the LP
   degenerate may pick another optimal basis; they are listed and counted.
2. Against HiGHS on 2,000 seeded points per program: status outside the feasibility band, objective within 1e-9; KKT
   within 1e-9 on every optimal point of 100k.
3. Hand-made LPs reach the infeasible and unbounded branches; an LP without a vertex and a QP handle are refused.
4. The dispatch envelope: mi = 256 with n' = 60, and a dictionary just above 48 KB, against HiGHS and from a fresh process.
5. A point's result does not depend on its batch.
6. The public API (SolverOutput, None without an optimum, sample_theta_space).
7. Explicit against implicit: verify_solution on the combinatorial solution of the complete mpLP goldens.
"""
import ctypes
import os
import subprocess
import sys

import numpy
import pytest
from scipy.optimize import linprog

from conftest import GOLDEN, ROOT
from parity import golden_regions
from test_gpu_solve_theta import kkt_batch
from test_solve_theta_twin import random_thetas, region_centres
from test_theta_lp_dict import LP_GOLDEN, program, seeded_eq_mplp

pytestmark = pytest.mark.gpu

LP_OPTIMAL, LP_INFEASIBLE, LP_ITERLIM, LP_NUMERIC, LP_UNBOUNDED = 0, 1, 2, 3, 4
COMPLETE = ['simple_mplp', 'transport_mplp', 'rand_lp_4_2_8_s3']
RANDOM = LP_GOLDEN + ['seeded_eq', 'bench_mplp']
KKT_TOL = 1e-9


def mplp(g):
    from ppopt_b200.mplp_program import MPLP_Program
    return MPLP_Program(g['A'], g['b'], g['c'], g['H'], g['A_t'], g['b_t'], g['F'], equality_indices=range(int(g['n_eq'])),
                        presolved=True)


def gpu_solve(solver, thetas):
    out = solver.solve_batch(thetas)
    return dict(status=out['status'].cpu().numpy(), x=out['x'].cpu().numpy(), dual=out['dual'].cpu().numpy(),
                mask=out['active'].cpu().numpy().view(numpy.uint64), iters=out['iters'].cpu().numpy(),
                obj=out['obj'].cpu().numpy())


def basis_lists(masks, n_eq, m):
    from ppopt_b200.solve_theta import _mask_bits
    bits = _mask_bits(masks, m - n_eq)
    return [tuple(range(n_eq)) + tuple(n_eq + numpy.nonzero(b)[0]) for b in bits]


def highs(g, th):
    """HiGHS at one theta: the linprog result (status 0 optimal, 2 infeasible, 3 unbounded)"""
    A, b, F = g['A'], g['b'].ravel(), g['F']
    ne = int(g['n_eq'])
    rhs = b + F @ th
    cost = g['c'].ravel() + g['H'] @ th
    return linprog(cost, A_ub=A[ne:], b_ub=rhs[ne:], A_eq=A[:ne] if ne else None, b_eq=rhs[:ne] if ne else None,
                   bounds=[(None, None)] * A.shape[1], method='highs')


def highs_margin(g, th):
    """the largest s with A_in x + s (1 + |rhs|) <= rhs, A_eq x = rhs_eq (s <= 1): the point is feasible iff s >= 0"""
    A, b, F = g['A'], g['b'].ravel(), g['F']
    ne, n = int(g['n_eq']), A.shape[1]
    rhs = b + F @ th
    A_ub = numpy.c_[A[ne:], 1.0 + numpy.abs(rhs[ne:])]
    r = linprog(numpy.r_[numpy.zeros(n), -1.0], A_ub=A_ub, b_ub=rhs[ne:],
                A_eq=numpy.c_[A[:ne], numpy.zeros(ne)] if ne else None, b_eq=rhs[:ne] if ne else None,
                bounds=[(None, None)] * n + [(None, 1.0)], method='highs')
    return -r.fun if r.status == 0 else -numpy.inf


def highs_degenerate(g, th, res):
    """more rows active than n - n_eq (primal) or an active row with a zero multiplier (dual) at HiGHS' optimum"""
    A, b, F = g['A'], g['b'].ravel(), g['F']
    ne, n = int(g['n_eq']), A.shape[1]
    rhs = b + F @ th
    s = (rhs - A @ res.x)[ne:]
    act = s <= 1e-9 * (1.0 + numpy.abs(rhs[ne:]) + numpy.abs(A[ne:]) @ numpy.abs(res.x))
    lam = -res.ineqlin.marginals
    return act.sum() > n - ne or (lam[act] <= 1e-9 * (1.0 + numpy.abs(lam).max(initial=0.0))).any()


def lp_solver(g):
    from ppopt_b200.solve_theta import ThetaLPSolver
    return ThetaLPSolver(mplp(g))


def kkt_lp(g, thetas, x, dual):
    return kkt_batch(dict(g, Q=numpy.zeros((g['A'].shape[1],) * 2)), thetas, x, dual)


@pytest.mark.parametrize('name', LP_GOLDEN)
def test_region_centres(name):
    g = program(name)
    pairs = region_centres(g, golden_regions(numpy.load(os.path.join(GOLDEN, name + '.npz'))))
    assert pairs, name
    thetas = numpy.array([c for _, c in pairs])
    out = gpu_solve(lp_solver(g), thetas)
    ne, m = int(g['n_eq']), g['A'].shape[0]
    got = basis_lists(out['mask'], ne, m)
    skipped = []
    for p, (r, th) in enumerate(pairs):
        aset = tuple(int(i) for i in r['active_set'])
        assert out['status'][p] == LP_OPTIMAL, (name, aset)
        if got[p] != aset:
            res = highs(g, th)
            assert res.status == 0 and highs_degenerate(g, th, res), (name, aset, got[p])
            skipped.append(aset)
            continue
        x_law = r['A'] @ th + r['b'].ravel()
        assert numpy.abs(out['x'][p] - x_law).max() <= 1e-8 * max(1.0, numpy.abs(x_law).max()), (name, aset)
        lam_law = r['C'] @ th + r['d'].ravel()
        lam = out['dual'][p][list(aset)]
        assert numpy.abs(lam - lam_law).max(initial=0.0) <= 1e-8 * max(1.0, numpy.abs(lam_law).max(initial=0.0)), \
            (name, aset, lam, lam_law)
    print(f'{name}: {len(pairs)} centres, {len(skipped)} degenerate skipped: {skipped}')
    assert len(skipped) < len(pairs), (name, skipped)


def check_against_highs(g, thetas, out, label):
    """status outside the feasibility band, objective within 1e-9, KKT on the optimal points"""
    n_band = 0
    for p, th in enumerate(thetas):
        res = highs(g, th)
        want = {0: LP_OPTIMAL, 2: LP_INFEASIBLE, 3: LP_UNBOUNDED}.get(res.status, -1)
        if want != out['status'][p]:
            assert abs(highs_margin(g, th)) <= 1e-7, (label, th, out['status'][p], res.status)
            n_band += 1
            continue
        if want == LP_OPTIMAL:
            assert abs(out['obj'][p] - res.fun) <= 1e-9 * max(1.0, abs(res.fun)), (label, th, out['obj'][p], res.fun)
    opt = out['status'] == LP_OPTIMAL
    k = kkt_lp(g, thetas[opt], out['x'][opt], out['dual'][opt])
    assert k.max(initial=0.0) <= KKT_TOL, (label, k.max(), thetas[opt][numpy.argmax(k)])
    return n_band


@pytest.mark.parametrize('name', RANDOM)
def test_against_highs(name):
    g = program(name)
    solver = lp_solver(g)
    thetas = random_thetas(g, 2000, seed=5)
    out = gpu_solve(solver, thetas)
    assert set(numpy.unique(out['status']).tolist()) <= {LP_OPTIMAL, LP_INFEASIBLE, LP_UNBOUNDED}, name
    n_band = check_against_highs(g, thetas, out, name)
    print(f'{name}: statuses {numpy.bincount(out["status"], minlength=5).tolist()}, band {n_band}, '
          f'pivots mean {out["iters"][:, 0].mean():.1f} max {out["iters"][:, 0].max()}')
    thetas = random_thetas(g, 100000, seed=6)
    out = gpu_solve(solver, thetas)
    assert set(numpy.unique(out['status']).tolist()) <= {LP_OPTIMAL, LP_INFEASIBLE, LP_UNBOUNDED}, name
    opt = out['status'] == LP_OPTIMAL
    assert opt.any(), name
    k = kkt_lp(g, thetas[opt], out['x'][opt], out['dual'][opt])
    assert k.max(initial=0.0) <= KKT_TOL, (name, k.max(), thetas[opt][numpy.argmax(k)])
    assert (out['iters'][:, 1] <= out['iters'][:, 0]).all()


def _tiny(A, b, F, c, H=None):
    A = numpy.asarray(A, dtype=float)
    n = A.shape[1]
    return dict(A=A, b=numpy.asarray(b, dtype=float).reshape(-1, 1), F=numpy.asarray(F, dtype=float).reshape(len(A), 1),
                A_t=numpy.array([[1.0], [-1.0]]), b_t=10.0 * numpy.ones((2, 1)), c=numpy.asarray(c, dtype=float).reshape(-1, 1),
                H=numpy.zeros((n, 1)) if H is None else numpy.asarray(H, dtype=float), n_eq=0)


def test_infeasible_unbounded_and_refusals():
    import torch
    from ppopt_b200 import _lib, engine
    from ppopt_b200.mplp_program import load_presolved
    from ppopt_b200.solve_theta import ThetaLPSolver
    # x1 <= theta, -x1 <= -1, x2 <= 1, -x2 <= 1: empty for theta < 1;  min x1 + x2
    g = _tiny([[1, 0], [-1, 0], [0, 1], [0, -1]], [0, -1, 1, 1], [1, 0, 0, 0], [1, 1])
    out = gpu_solve(lp_solver(g), numpy.array([[0.0], [2.0]]))
    assert out['status'].tolist() == [LP_INFEASIBLE, LP_OPTIMAL]
    assert numpy.isnan(out['x'][0]).all() and numpy.isnan(out['dual'][0]).all()
    numpy.testing.assert_allclose(out['x'][1], [1.0, -1.0], atol=1e-12)
    numpy.testing.assert_allclose(out['dual'][1], [0.0, 1.0, 0.0, 1.0], atol=1e-12)
    # x1 <= 1, x2 <= 1: min x1 is unbounded below, min -x1 - x2 + theta x1 is not for theta < 1
    g = _tiny([[1, 0], [0, 1]], [1, 1], [0, 0], [-1, -1], H=[[1.0], [0.0]])
    out = gpu_solve(lp_solver(g), numpy.array([[0.0], [2.0]]))
    assert out['status'].tolist() == [LP_OPTIMAL, LP_UNBOUNDED]
    numpy.testing.assert_allclose(out['x'][0], [1.0, 1.0], atol=1e-12)
    # no vertex: the rows only see x1 + x2
    flat = _tiny([[1, 1], [-1, -1]], [1, 1], [0, 0], [1, 1])
    with pytest.raises(NotImplementedError):
        ThetaLPSolver(mplp(flat))
    with pytest.raises(NotImplementedError):
        ThetaLPSolver(load_presolved(os.path.join(GOLDEN, 'factory_mpqp.npz')))
    lib = _lib.load()
    for prog, what in ((mplp(flat), b'no vertex'), (load_presolved(os.path.join(GOLDEN, 'factory_mpqp.npz')), b'mpQP')):
        eng = engine.Engine(engine.program_arrays(prog))
        th = torch.zeros((1, eng.t), dtype=torch.float64, device=eng.tdev)
        st = torch.zeros((1,), dtype=torch.uint8, device=eng.tdev)
        rc = lib.ppgpu_solve_theta_lp_batch(eng.h, th.data_ptr(), 1, st.data_ptr(), None, None, None, None,
                                            ctypes.c_void_p(torch.cuda.current_stream().cuda_stream))
        assert rc == -2 and what in lib.ppgpu_last_error(), lib.ppgpu_last_error()
        eng.close()


# (mi, n', t): the largest dictionary the engine admits (256 rows, n' + t + 2 = 64), and one whose per-warp scratch is just
# above the 48 KB a block gets without opting in (187 x 31 doubles of dictionary)
ENVELOPE = [(256, 60, 2), (186, 29, 3)]


def envelope_mplp(mi, n, t, seed=3):
    """n box pairs |x_i| <= 50 plus mi - 2n random rows; Theta = [-2, 2]^t, given as rows where mi + 2t fits the 256 region
    rows, else left to the sampling box of theta_box (no rows: +-10, with the parameter columns scaled to match)"""
    rng = numpy.random.default_rng(seed)
    k = mi - 2 * n
    rows = mi + 2 * t <= 256
    A = numpy.vstack([rng.standard_normal((k, n)), numpy.eye(n), -numpy.eye(n)])
    b = numpy.r_[rng.uniform(1.0, 4.0, k), 50.0 * numpy.ones(2 * n)].reshape(-1, 1)
    F = numpy.vstack([(1.0 if rows else 0.2) * rng.standard_normal((k, t)), numpy.zeros((2 * n, t))])
    A_t = numpy.vstack([numpy.eye(t), -numpy.eye(t)]) if rows else numpy.zeros((0, t))
    return dict(A=A, b=b, F=F, A_t=A_t, b_t=2.0 * numpy.ones((len(A_t), 1)), c=rng.standard_normal((n, 1)),
                H=rng.standard_normal((n, t)), n_eq=0)


@pytest.mark.parametrize('mi,n,t', ENVELOPE)
def test_envelope_against_highs(mi, n, t):
    g = envelope_mplp(mi, n, t)
    thetas = random_thetas(g, 500, seed=1)
    out = gpu_solve(lp_solver(g), thetas)
    assert (out['status'] == LP_OPTIMAL).sum() > 100, numpy.bincount(out['status'])
    check_against_highs(g, thetas, out, (mi, n, t))


@pytest.mark.parametrize('mi,n,t', ENVELOPE)
def test_envelope_first_launch_in_fresh_process(mi, n, t):
    code = ('import sys, numpy; sys.path[:0] = [{root!r}, {tests!r}]; '
            'from test_gpu_solve_theta_lp import envelope_mplp, lp_solver; '
            'from test_solve_theta_twin import random_thetas; '
            'g = envelope_mplp({mi}, {n}, {t}); out = lp_solver(g).solve_batch(random_thetas(g, 64, seed=2)); '
            'st = out["status"].cpu().numpy(); assert (st == 0).any() and (st <= 4).all(), st; print("ok")')
    code = code.format(root=ROOT, tests=os.path.join(ROOT, 'tests'), mi=mi, n=n, t=t)
    r = subprocess.run([sys.executable, '-c', code], capture_output=True, text=True, timeout=600)
    assert r.returncode == 0 and 'ok' in r.stdout, r.stderr[-2000:]


def test_point_result_does_not_depend_on_batch():
    g = program('bench_mplp')
    solver = lp_solver(g)
    thetas = random_thetas(g, 100000, seed=9)
    perm = numpy.random.default_rng(4).permutation(len(thetas))
    full = gpu_solve(solver, thetas[perm])
    where = numpy.argsort(perm)
    for p in (0, 1, 17, 4242, 99999):
        one = gpu_solve(solver, thetas[p:p + 1])
        q = where[p]
        assert one['status'][0] == full['status'][q]
        for f in ('x', 'dual', 'mask', 'iters'):
            assert numpy.array_equal(one[f][0], full[f][q], equal_nan=f in ('x', 'dual')), (p, f)


def test_solve_theta_record():
    g = program('seeded_eq')
    prog = mplp(g)
    thetas = random_thetas(g, 400, seed=2)
    out = gpu_solve(prog._theta_solver(), thetas)
    st = out['status']
    assert (st == LP_OPTIMAL).any() and (st == LP_INFEASIBLE).any(), numpy.bincount(st)
    p_opt, p_inf = int(numpy.argmax(st == LP_OPTIMAL)), int(numpy.argmax(st == LP_INFEASIBLE))
    assert prog.solve_theta(thetas[p_inf].reshape(-1, 1)) is None
    rec = prog.solve_theta(thetas[p_opt].reshape(-1, 1))
    (m, n), ne = g['A'].shape, int(g['n_eq'])
    assert rec.sol.shape == (n,) and rec.slack.shape == (m,) and rec.dual.shape == (m,)
    assert rec.active_set.ndim == 1 and rec.active_set.dtype.kind == 'i' and len(rec.active_set) == n
    assert rec.active_set[:ne].tolist() == list(range(ne))
    x, th = rec.sol.reshape(-1, 1), thetas[p_opt].reshape(-1, 1)
    assert abs(rec.obj - prog.evaluate_objective(x, th)) <= 1e-9 * max(1.0, abs(rec.obj))
    numpy.testing.assert_allclose(rec.slack, (g['b'] + g['F'] @ th - g['A'] @ x).ravel(), atol=1e-12)
    assert numpy.all(rec.slack[rec.active_set] <= 1e-8) and numpy.all(rec.dual[numpy.setdiff1d(numpy.arange(m), rec.active_set)] == 0)
    unb = mplp(_tiny([[1, 0], [0, 1]], [1, 1], [0, 0], [1, 0]))
    assert unb.solve_theta(numpy.zeros((1, 1))) is None
    seeds = prog.sample_theta_space(200)
    assert seeds and all(isinstance(a, tuple) for a in seeds) and len(set(seeds)) == len(seeds)


@pytest.mark.parametrize('name', COMPLETE)
def test_sampled_bases_are_golden_regions(name):
    from ppopt_b200.mplp_program import load_presolved
    prog = load_presolved(os.path.join(GOLDEN, name + '.npz'))
    g = program(name)
    want = {tuple(int(i) for i in r['active_set']) for r in golden_regions(numpy.load(os.path.join(GOLDEN, name + '.npz')))}
    seeds = prog.sample_theta_space(2000)
    solver = prog._theta_solver()
    thetas = solver.sample_thetas(2000, 0)
    out = gpu_solve(solver, thetas)
    ne, m = int(g['n_eq']), g['A'].shape[0]
    bases = basis_lists(out['mask'], ne, m)
    opt = numpy.nonzero(out['status'] == LP_OPTIMAL)[0]
    assert list(dict.fromkeys(bases[p] for p in opt)) == seeds
    for p in opt:
        if bases[p] in want:
            continue
        res = highs(g, thetas[p])
        assert res.status == 0 and highs_degenerate(g, thetas[p], res), (name, bases[p], thetas[p])


@pytest.mark.parametrize('name', COMPLETE)
def test_explicit_matches_implicit(name):
    from ppopt_b200 import mpqp_algorithm, solve_mpqp, verify_solution
    from ppopt_b200.mplp_program import load_presolved
    prog = load_presolved(os.path.join(GOLDEN, name + '.npz'))
    sol = solve_mpqp(prog, mpqp_algorithm.combinatorial)
    rep = verify_solution(sol, num_samples=100000, seed=3)
    print(name, {k: v for k, v in rep.items() if not k.endswith('thetas') and k not in ('spurious_regions', 'worst_theta')})
    assert rep['n_points'] > 50000 and rep['n_failed'] == 0, rep
    assert rep['holes'] == 0, (name, rep['hole_thetas'][:5])
    assert rep['max_dobj'] <= 1e-9, (name, rep['max_dobj'])
    assert rep['max_dx'] <= 1e-6, (name, rep['max_dx'], rep['worst_theta'])
    assert rep['n_band'] < 0.01 * rep['n_points'], rep['n_band']
    for th, r in zip(rep['spurious_thetas'], rep['spurious_regions']):
        cr = sol.critical_regions[int(r)]
        E, f = numpy.asarray(cr.E, dtype=float), numpy.asarray(cr.f, dtype=float).ravel()
        assert ((E @ th - f) / numpy.linalg.norm(E, axis=1)).max() >= -1e-5, (name, th)
