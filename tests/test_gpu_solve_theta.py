"""Fixed-theta QP solves on the GPU (K8, csrc/k8_theta_qp.cu) through the C ABI and ppopt_b200.ThetaSolver.

4. Against the CPU twin on every use_gram golden (the bench program included): at region centres and on 100k random
   points of Theta, status, working set and step count agree wherever the twin's smallest decision margin exceeds 1e-9;
   x within 1e-10 relative; KKT on every optimal point.
5. The public API repeats the CPU checks (region centres, KKT, HiGHS on infeasible points); solve_theta returns the
   SolverOutput fields or None; mpLPs and Hessians that are not positive definite on the reduced space are refused.
6. Explicit against implicit: verify_solution on the combinatorial solution of every full-solution mpQP golden.
7. Seeding the combinatorial graph search with sample_theta_space gives the golden region set.
"""
import ctypes
import os

import numpy
import pytest

from conftest import GOLDEN
from parity import golden_regions
from test_solve_theta_twin import (GRAM, QP_INFEASIBLE, QP_OPTIMAL, REGION_SETS, _program, check_random,
                                   check_region_centres, random_thetas, region_centres, twin_for)

pytestmark = pytest.mark.gpu

FULL = ['ctrl_alloc_n1', 'ctrl_alloc_n2', 'doc_portfolio', 'factory_mpqp', 'mpc_n3', 'mpc_n5', 'mpc_n7', 'portfolio_analog',
        'rand_5_3_10_s2', 'rand_6_3_12_s1', 'simple_mpqp_1d']
GRAPH = sorted(f[:-4] for f in os.listdir(os.path.join(GOLDEN, 'graph')) if f.endswith('.npz'))
KKT_TOL = 1e-9


def solver_for(name):
    from ppopt_b200.mplp_program import load_presolved
    from ppopt_b200.solve_theta import ThetaSolver
    return ThetaSolver(load_presolved(os.path.join(GOLDEN, name + '.npz')))


def gpu_solve(solver):
    def run(thetas):
        out = solver.solve_batch(thetas)
        return dict(status=out['status'].cpu().numpy(), x=out['x'].cpu().numpy(), dual=out['dual'].cpu().numpy(),
                    mask=out['active'].cpu().numpy().view(numpy.uint64), iters=out['iters'].cpu().numpy())
    return run


def kkt_batch(g, thetas, x, dual):
    """per-point max of the scaled KKT residuals (as test_solve_theta_twin.kkt_residuals, vectorised)"""
    A, b, F, Q, H, c = g['A'], g['b'].ravel(), g['F'], g['Q'], g['H'], g['c'].ravel()
    ne = int(g['n_eq'])
    rhs = b[None, :] + thetas @ F.T
    s = rhs - x @ A.T
    scale = 1.0 + numpy.abs(rhs) + numpy.abs(x) @ numpy.abs(A).T
    lam = dual[:, ne:]
    lmax = 1.0 + numpy.abs(lam).max(1, initial=0.0)
    primal = numpy.maximum(numpy.abs(s[:, :ne] / scale[:, :ne]).max(1, initial=0.0), (-s[:, ne:] / scale[:, ne:]).max(1, initial=0.0))
    dual_inf = numpy.maximum(0.0, -lam.min(1, initial=0.0)) / lmax
    compl = numpy.abs(lam * s[:, ne:] / scale[:, ne:]).max(1, initial=0.0) / lmax
    grad = x @ Q.T + thetas @ H.T + c[None, :]
    at = dual @ A
    stat = numpy.abs(grad + at).max(1) / (1.0 + numpy.abs(grad).max(1) + numpy.abs(at).max(1))
    return numpy.maximum.reduce([primal, dual_inf, compl, stat])


def compare_with_twin(name, thetas, require_all=False):
    g = _program(name)
    ref = twin_for(name).theta_qp(thetas)
    got = gpu_solve(solver_for(name))(thetas)
    sure = ref['margin'] > 1e-9
    if require_all:
        # (the control-allocation programs are symmetric: many points see exactly tied slacks or step ratios)
        assert sure.mean() > 0.25, (name, sure.mean())
    for f in ('status', 'iters'):
        bad = numpy.nonzero(sure & (got[f] != ref[f]))[0]
        assert not len(bad), (name, f, thetas[bad[:3]], got[f][bad[:3]], ref[f][bad[:3]])
    bad = numpy.nonzero(sure & (got['mask'] != ref['mask']).any(1))[0]
    assert not len(bad), (name, 'mask', thetas[bad[:3]])
    both = (got['status'] == QP_OPTIMAL) & (ref['status'] == QP_OPTIMAL) & sure
    dx = numpy.abs(got['x'][both] - ref['x'][both]).max(1, initial=0.0) / numpy.maximum(1.0, numpy.abs(ref['x'][both]).max(1, initial=0.0))
    assert dx.max(initial=0.0) <= 1e-10, (name, dx.max())
    opt = got['status'] == QP_OPTIMAL
    assert set(numpy.unique(got['status']).tolist()) <= {QP_OPTIMAL, QP_INFEASIBLE}, name
    k = kkt_batch(g, thetas[opt], got['x'][opt], got['dual'][opt])
    assert k.max(initial=0.0) <= KKT_TOL, (name, k.max(), thetas[opt][numpy.argmax(k)])
    return sure.mean()


@pytest.mark.parametrize('name,sampled', REGION_SETS)
def test_kernel_matches_twin_at_region_centres(name, sampled):
    g = _program(name)
    rg = numpy.load(os.path.join(GOLDEN, 'sampled', name + '.npz')) if sampled else g
    thetas = numpy.array([c for _, c in region_centres(g, golden_regions(rg))])
    compare_with_twin(name, thetas)


@pytest.mark.parametrize('name', GRAM)
def test_kernel_matches_twin_on_random_thetas(name):
    compare_with_twin(name, random_thetas(_program(name), 100000, seed=1), require_all=True)


@pytest.mark.parametrize('name,sampled', REGION_SETS)
def test_api_region_centres(name, sampled):
    check_region_centres(name, sampled, gpu_solve(solver_for(name)))


@pytest.mark.parametrize('name', GRAM)
def test_api_random_thetas_kkt(name):
    check_random(name, gpu_solve(solver_for(name)))


def test_solve_theta_record():
    from ppopt_b200.mplp_program import load_presolved
    prog = load_presolved(os.path.join(GOLDEN, 'mpc_n10.npz'))
    g = _program('mpc_n10')
    thetas = random_thetas(g, 400, seed=2)
    out = prog._theta_solver().solve_batch(thetas)
    st = out['status'].cpu().numpy()
    assert (st == QP_OPTIMAL).any() and (st == QP_INFEASIBLE).any()   # mpc_n10 is infeasible on part of Theta
    p_opt, p_inf = int(numpy.argmax(st == QP_OPTIMAL)), int(numpy.argmax(st == QP_INFEASIBLE))
    assert prog.solve_theta(thetas[p_inf].reshape(-1, 1)) is None
    rec = prog.solve_theta(thetas[p_opt].reshape(-1, 1))
    n, m = g['A'].shape[1], g['A'].shape[0]
    assert rec.sol.shape == (n,) and rec.slack.shape == (m,) and rec.dual.shape == (m,)
    assert rec.active_set.ndim == 1 and rec.active_set.dtype.kind == 'i'
    x, th = rec.sol.reshape(-1, 1), thetas[p_opt].reshape(-1, 1)
    assert abs(rec.obj - prog.evaluate_objective(x, th)) <= 1e-9 * max(1.0, abs(rec.obj))
    numpy.testing.assert_allclose(rec.slack, (g['b'] + g['F'] @ th - g['A'] @ x).ravel(), atol=1e-12)
    assert numpy.all(rec.slack[rec.active_set] <= 1e-8) and numpy.all(rec.dual[numpy.setdiff1d(numpy.arange(m), rec.active_set)] == 0)
    seeds = prog.sample_theta_space(200)
    assert seeds and all(isinstance(a, tuple) for a in seeds) and len(set(seeds)) == len(seeds)


def test_refuses_mplp_and_semidefinite_hessian():
    import torch
    from ppopt_b200 import _lib, engine
    from ppopt_b200.mplp_program import MPQP_Program, load_presolved
    from ppopt_b200.solve_theta import ThetaSolver
    lp_names = [f[:-4] for f in sorted(os.listdir(GOLDEN)) if f.endswith('.npz') and _program(f[:-4]) is None]
    assert lp_names
    for name in lp_names:
        with pytest.raises(NotImplementedError):
            ThetaSolver(load_presolved(os.path.join(GOLDEN, name + '.npz')))
    # Q = diag(1, 0): not positive definite on the reduced space
    A = numpy.array([[1.0, 0.0], [0.0, 1.0], [-1.0, 0.0], [0.0, -1.0]])
    semi = MPQP_Program(A, numpy.ones((4, 1)), numpy.zeros((2, 1)), numpy.zeros((2, 1)), numpy.diag([1.0, 0.0]),
                        numpy.array([[1.0], [-1.0]]), numpy.ones((2, 1)), numpy.zeros((4, 1)), presolved=True)
    with pytest.raises(NotImplementedError):
        ThetaSolver(semi)
    lib = _lib.load()
    for prog in (semi, load_presolved(os.path.join(GOLDEN, lp_names[0] + '.npz'))):
        eng = engine.Engine(engine.program_arrays(prog))
        th = torch.zeros((1, eng.t), dtype=torch.float64, device=eng.tdev)
        st = torch.zeros((1,), dtype=torch.uint8, device=eng.tdev)
        rc = lib.ppgpu_solve_theta_batch(eng.h, th.data_ptr(), 1, st.data_ptr(), None, None, None, None,
                                         ctypes.c_void_p(torch.cuda.current_stream().cuda_stream))
        assert rc == -2 and b'use_gram' in lib.ppgpu_last_error()
        eng.close()


@pytest.mark.parametrize('name', FULL)
def test_explicit_matches_implicit(name):
    from ppopt_b200 import mpqp_algorithm, solve_mpqp, verify_solution
    from ppopt_b200.mplp_program import load_presolved
    prog = load_presolved(os.path.join(GOLDEN, name + '.npz'))
    sol = solve_mpqp(prog, mpqp_algorithm.combinatorial)
    rep = verify_solution(sol, num_samples=100000, seed=3)
    assert rep['n_points'] > 50000 and rep['n_failed'] == 0, rep
    assert rep['holes'] == 0, (name, rep['hole_thetas'][:5])
    assert rep['max_dx'] <= 1e-6, (name, rep['max_dx'], rep['worst_theta'])
    assert rep['n_band'] < 0.01 * rep['n_points'], rep['n_band']
    # a point the QP calls infeasible may only be located within the location tolerance of a region's boundary
    for th, r in zip(rep['spurious_thetas'], rep['spurious_regions']):
        cr = sol.critical_regions[int(r)]
        E, f = numpy.asarray(cr.E, dtype=float), numpy.asarray(cr.f, dtype=float).ravel()
        assert ((E @ th - f) / numpy.linalg.norm(E, axis=1)).max() >= -1e-5, (name, th)


@pytest.mark.parametrize('name', GRAPH)
def test_sampled_seeds_give_graph_region_set(name):
    from ppopt_b200.mp_solvers import mpqp_combi_graph
    from ppopt_b200.mplp_program import load_presolved
    from ppopt_b200.solve_theta import ThetaSolver
    prog = load_presolved(os.path.join(GOLDEN, name + '.npz'))
    seeds = ThetaSolver(prog).sample_theta_space()
    assert seeds
    sol = mpqp_combi_graph.solve(prog, initial_active_sets=seeds)
    g = numpy.load(os.path.join(GOLDEN, 'graph', name + '.npz'))
    want = {tuple(int(i) for i in r['active_set']) for r in golden_regions(g)}
    assert {tuple(int(i) for i in r.active_set) for r in sol.critical_regions} == want
