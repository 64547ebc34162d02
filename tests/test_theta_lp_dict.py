"""Start dictionary of the fixed-theta LP kernel (K9, host_math.hpp::build_lp_dictionary), read through
tests/lp_dict_export.py and checked against numpy.  No GPU needed.

For every mpLP golden, a seeded mpLP with equality rows and the bench-shaped synthetic mpLP:
1. the np inequality rows the dictionary holds nonbasic, with the equality rows, form a nonsingular system;
2. at 100 seeded theta the dictionary's D, beta(theta), rows of v (mapped to x through X0t and Q2) and objective row d(theta)
   equal what numpy derives from that basis, within 1e-9 scaled.
3. A program whose reduced rows have rank below n - n_eq has no dictionary.
"""
import os
import sys

import numpy
import pytest

from conftest import GOLDEN, ROOT

sys.path.insert(0, os.path.join(ROOT, 'oracle'))
import problems  # noqa: E402
from lp_dict_export import lp_dict  # noqa: E402

LP_GOLDEN = ['simple_mplp', 'transport_mplp', 'rand_lp_4_2_8_s3', 'envelope/env_lp_w3']


def seeded_eq_mplp(seed=7, n=6, t=3, ne=2, m_rand=14):
    """a bounded mpLP with equality rows: random rows, a box |x_i| <= 10 and Theta = [-2, 2]^t (presolved layout);
    infeasible on part of Theta"""
    rng = numpy.random.default_rng(seed)
    A = numpy.vstack([rng.standard_normal((ne + m_rand, n)), numpy.eye(n), -numpy.eye(n)])
    b = numpy.r_[rng.uniform(-0.5, 0.5, ne), rng.uniform(1.0, 3.0, m_rand), 10.0 * numpy.ones(2 * n)].reshape(-1, 1)
    F = numpy.vstack([1.5 * rng.standard_normal((ne + m_rand, t)), numpy.zeros((2 * n, t))])
    return dict(kind='lp', A=A, b=b, F=F, A_t=numpy.vstack([numpy.eye(t), -numpy.eye(t)]), b_t=2.0 * numpy.ones((2 * t, 1)),
                c=rng.standard_normal((n, 1)), H=0.3 * rng.standard_normal((n, t)), n_eq=ne)


def bench_mplp():
    """the shape of bench.py's program as an mpLP: 30 variables, 6 parameters, 100 random rows plus a box of 1e7"""
    g = problems.random_mpqp(30, 6, 100, 0, kind='lp')
    return dict(g, n_eq=0)


def program(name):
    if name == 'seeded_eq':
        return seeded_eq_mplp()
    if name == 'bench_mplp':
        return bench_mplp()
    g = numpy.load(os.path.join(GOLDEN, name + '.npz'))
    return {k: g[k] for k in ('A', 'b', 'F', 'A_t', 'b_t', 'c', 'H')} | dict(kind='lp', n_eq=int(g['n_eq']))


def start_dict(g):
    return lp_dict(g['A'], g['b'], g['F'], g['A_t'], g['b_t'], None, g['c'], g['H'], int(g['n_eq']))


@pytest.mark.parametrize('name', LP_GOLDEN + ['seeded_eq', 'bench_mplp'])
def test_start_dictionary_matches_numpy(name):
    g = program(name)
    d = start_dict(g)
    assert d is not None, name
    A, b, F, c, H = g['A'], g['b'].ravel(), g['F'], g['c'].ravel(), g['H']
    ne, (m, n), t = int(g['n_eq']), g['A'].shape, g['F'].shape[1]
    mi, npr = m - ne, n - ne
    D0, bvar, nvar = d['D0'], d['bvar'], d['nvar']
    assert D0.shape == (mi, 1 + npr + t)
    # every slack is basic in one row or nonbasic in one column, every v_c sits in one row
    assert sorted(nvar.tolist() + bvar[bvar >= 0].tolist()) == list(range(mi))
    assert sorted((-1 - bvar[bvar < 0]).tolist()) == list(range(npr))
    rows = numpy.r_[numpy.arange(ne), ne + nvar].astype(int)
    M = A[rows]
    assert numpy.linalg.cond(M) < 1e12, (name, numpy.linalg.cond(M))
    Minv = numpy.linalg.inv(M)
    dx_ds = -Minv[:, ne:]                         # d x / d s_N
    B = D0[:, 1:1 + npr]
    rng = numpy.random.default_rng(11)
    from ppopt_b200.solve_theta import theta_box
    lo, hi = theta_box(g['A_t'], g['b_t'].ravel())
    for th in rng.uniform(lo, hi, size=(100, t)):
        rhs = b + F @ th
        x = Minv @ rhs[rows]                      # the vertex at s_N = 0
        beta = D0[:, 0] - D0[:, 1 + npr:] @ th
        for r in range(mi):
            if bvar[r] >= 0:                      # s = rhs - A x, and D = -d s / d s_N
                i = ne + bvar[r]
                s, ds = rhs[i] - A[i] @ x, -A[i] @ dx_ds
                sc = 1.0 + abs(rhs[i]) + numpy.abs(A[i]) @ numpy.abs(x)
                assert abs(beta[r] - s) <= 1e-9 * sc, (name, r, beta[r], s)
                assert numpy.abs(B[r] + ds).max() <= 1e-9 * (1.0 + numpy.abs(ds).max()), (name, r)
        vrow = numpy.zeros(npr, dtype=int)
        vrow[-1 - bvar[bvar < 0]] = numpy.nonzero(bvar < 0)[0]
        x_dict = d['X0t'] @ numpy.r_[1.0, th] + d['Q2'] @ beta[vrow]
        assert numpy.abs(x_dict - x).max() <= 1e-9 * (1.0 + numpy.abs(x).max()), (name, x_dict, x)
        assert numpy.abs(-d['Q2'] @ B[vrow] - dx_ds).max() <= 1e-9 * (1.0 + numpy.abs(dx_ds).max()), name
        # z = zeta - d' s_N:  d = -(c + H theta)' dx/ds_N
        want = -(c + H @ th) @ dx_ds
        got = d['obj'][:, 0] + d['obj'][:, 1:] @ th
        assert numpy.abs(got - want).max() <= 1e-9 * (1.0 + numpy.abs(want).max()), (name, got, want)


def test_rank_deficient_rows_have_no_vertex():
    # x1 + x2 is all the rows see: the reduced rows have rank 1 < 2
    A = numpy.array([[1.0, 1.0], [-1.0, -1.0], [2.0, 2.0]])
    g = dict(A=A, b=numpy.ones((3, 1)), F=numpy.zeros((3, 1)), A_t=numpy.array([[1.0], [-1.0]]), b_t=numpy.ones((2, 1)),
             c=numpy.array([[1.0], [0.0]]), H=numpy.zeros((2, 1)), n_eq=0)
    assert start_dict(g) is None
    # the same with an equality row that leaves one direction the inequalities do not see
    A = numpy.array([[1.0, -1.0, 0.0], [1.0, 1.0, 0.0], [-1.0, -1.0, 0.0]])
    g = dict(g, A=A, b=numpy.ones((3, 1)), F=numpy.zeros((3, 1)), c=numpy.ones((3, 1)), H=numpy.zeros((3, 1)), n_eq=1)
    assert start_dict(g) is None
    assert start_dict(seeded_eq_mplp()) is not None


def test_qp_handles_have_no_lp_dictionary():
    g = numpy.load(os.path.join(GOLDEN, 'factory_mpqp.npz'))
    assert lp_dict(g['A'], g['b'], g['F'], g['A_t'], g['b_t'], g['Q'], g['c'], g['H'], int(g['n_eq']), is_qp=True) is None
