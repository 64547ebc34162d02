"""CPU tests of the relaxation tree of a mixed-integer program (K11): the lifted system that build_tree_dictionary builds
(host_math.hpp), and a HiGHS model of the breadth-first tree whose ordering and pruning the GPU tree must reproduce."""
import numpy
import pytest

from mitree_programs import MixedIntegerProgram, brute_force, random_program, tree_model
from tree_dict_export import tree_dict

_SEEDS = [(nb, s) for nb in (3, 5, 7) for s in range(3)]


def _lifted(prog):
    from ppopt_b200.mp_solvers.mitree import lifted_arrays
    return lifted_arrays(prog)


@pytest.mark.parametrize('nb,seed', _SEEDS)
def test_dictionary_slacks_equal_lifted_rows(nb, seed):
    prog = random_program(nb, seed)
    A, b, F, A_t, b_t, ne, bins = _lifted(prog)
    T = tree_dict(A, b, F, A_t, b_t, ne, bins)
    n, t = A.shape[1], F.shape[1]
    nv, rows, cols, rb0 = T['nv'], T['rows'], T['cols'], T['rb0']
    assert (nv, rows, cols) == (n + t, A.shape[0] - ne + A_t.shape[0] + 2 * nb, n + t - ne)
    # lifted rows, equalities first
    G = numpy.vstack([numpy.hstack([A, -F]), numpy.hstack([numpy.zeros((A_t.shape[0], n)), A_t])])
    for k, i in enumerate(bins):
        e = numpy.zeros(nv)
        e[i] = 1.0
        G = numpy.vstack([G, e, -e])
    rng = numpy.random.default_rng(100 + seed)
    D0, ld = T['D0'], T['D0'].shape[1]
    for _ in range(5):
        v = rng.normal(size=cols)
        z = T['z0'] + T['Q2'] @ v
        assert numpy.allclose(G[:ne] @ z, b[:ne], atol=1e-10)          # the equalities are eliminated
        u, l = rng.normal(size=nb), rng.normal(size=nb)
        h = numpy.concatenate([b[ne:], b_t, numpy.ravel(numpy.column_stack([u, -l]))])
        s = h - G[ne:] @ z                                            # slacks of the inequality rows at these bounds
        p = numpy.ravel(numpy.column_stack([u - 1.0, -l])) if nb else numpy.zeros(1)
        sN = s[T['nvar']]
        for r in range(rows):
            val = D0[r, 0] - D0[r, 1:1 + cols] @ sN - D0[r, 1 + cols:] @ p
            want = s[T['bvar'][r]] if T['bvar'][r] >= 0 else v[-1 - T['bvar'][r]]
            assert abs(val - want) <= 1e-8 * (1 + abs(want)), (r, val, want)
    assert numpy.allclose(T['hs'], 1.0 + numpy.abs(numpy.concatenate([b[ne:], b_t, numpy.tile([1.0, 0.0], nb)])))


def test_dictionary_refuses_a_system_without_vertex():
    # x_1 appears in no row: the lifted rows have rank below the free variables
    prog = MixedIntegerProgram(numpy.array([[1.0, 0.0, 1.0], [-1.0, 0.0, 0.0]]), [1.0, 0.0], numpy.zeros((2, 1)),
                               numpy.array([[1.0], [-1.0]]), [1.0, 1.0], [2])
    with pytest.raises(ValueError, match='no vertex'):
        tree_dict(*_lifted(prog))


@pytest.mark.parametrize('nb,seed', _SEEDS)
def test_tree_model_leaves_equal_brute_force(nb, seed):
    prog = random_program(nb, seed)
    feas, near = brute_force(prog)
    leaves = [y for y in tree_model(prog) if y not in near]
    assert leaves == feas
    assert leaves == sorted(leaves)   # lexicographic: y_0 is the leading key
