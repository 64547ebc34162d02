"""GPU tests of the relaxation tree of a mixed-integer program (K11, ppopt_b200.mp_solvers.mitree): leaves against the
mpMIQP goldens, against HiGHS on every assignment and against the 2^nb screen; programs beyond that screen's 20 binaries;
node-level statuses, points and inheritance; the limits of the handle."""
import os

import numpy
import pytest
import torch

from conftest import GOLDEN
from mitree_programs import MixedIntegerProgram, brute_force, random_program, relaxation_margin
from parity import REL_TOL, rel_err, rows_match_as_sets

pytestmark = pytest.mark.gpu
MI = os.path.join(GOLDEN, 'mpmiqp')


# ---- the programs of oracle/gen_mpmiqp_golden.py (arrays copied)
def simple_mpmiqp():
    A = numpy.array([[0, 1, 1], [1, 0, 0], [-1, 0, 0], [1, -1, 0], [1, 0, -1]], float)
    b = numpy.array([1, 0, 0, 0, 0], float)
    F = numpy.array([0, 1, 0, 0, 0], float).reshape(-1, 1)
    return MixedIntegerProgram(A, b, F, numpy.array([[1.0], [1.0]]), [2.0, 2.0], [1, 2])


def market_mpmiqp():
    A = numpy.array(
        [[1, 1, 0, 0, 0], [0, 0, 1, 1, 0], [-1, 0, -1, 0, 0], [0, -1, 0, -1, -500], [-1, 0, 0, 0, 0], [0, -1, 0, 0, 0],
         [0, 0, -1, 0, 0], [0, 0, 0, -1, 0], [0, 0, 0, 0, -1], [0, 0, 0, 0, 1]], float)
    b = numpy.array([350, 600, 0, 0, 0, 0, 0, 0, 0, 1], float)
    F = numpy.array([[0, 0], [0, 0], [-1, 0], [0, -1], [0, 0], [0, 0], [0, 0], [0, 0], [0, 0], [0, 0]], float)
    A_t = numpy.array([[1.0, 0.0], [0.0, 1.0], [-1.0, 0.0], [0.0, -1.0]])
    return MixedIntegerProgram(A, b, F, A_t, [1000.0, 1000.0, 0.0, 0.0], [4])


def random_mpmiqp_5_4(seed=7, n_cont=5, n_bin=4, t=2, m=10):
    rng = numpy.random.default_rng(seed)
    n = n_cont + n_bin
    A = numpy.vstack([rng.normal(size=(m, n)), numpy.hstack([numpy.eye(n_cont), numpy.zeros((n_cont, n_bin))]),
                      numpy.hstack([-numpy.eye(n_cont), numpy.zeros((n_cont, n_bin))])])
    A[:m, n_cont:] *= 0.5
    b = numpy.vstack([rng.uniform(1.0, 3.0, size=(m, 1)), 2.0 * numpy.ones((2 * n_cont, 1))])
    F = numpy.vstack([rng.normal(size=(m, t)) * 0.5, numpy.zeros((2 * n_cont, t))])
    return MixedIntegerProgram(A, b, F, numpy.vstack([numpy.eye(t), -numpy.eye(t)]), numpy.ones(2 * t),
                               list(range(n_cont, n)))


FIXTURES = {'simple_mpmiqp': simple_mpmiqp, 'market_mpmiqp': market_mpmiqp, 'random_mpmiqp_5_4': random_mpmiqp_5_4}


class StoredTreeProgram(MixedIntegerProgram):
    """the real arrays (for the tree) and the reference's stored sub-problems (for the solves)"""

    def __init__(self, name):
        p = FIXTURES[name]()
        super().__init__(p.A, p.b, p.F, p.A_t, p.b_t, p.binary_indices, p.equality_indices)
        from test_gpu_mpmiqp import StoredMixedIntegerProgram
        self.stored = StoredMixedIntegerProgram(numpy.load(os.path.join(MI, name + '.npz')))

    def generate_substituted_problem(self, y):
        return self.stored.generate_substituted_problem(y)


def _leaves(prog, **kw):
    from ppopt_b200.mp_solvers.mitree import feasible_combinations
    return feasible_combinations(prog, **kw)


@pytest.mark.parametrize('name', sorted(FIXTURES))
def test_fixture_leaves_equal_golden(name):
    g = numpy.load(os.path.join(MI, name + '.npz'))
    assert _leaves(FIXTURES[name]()).leaves == g['combinations'].tolist()


@pytest.mark.parametrize('name', sorted(FIXTURES))
def test_fixture_solve_with_tree_screen(name):
    from ppopt_b200.mp_solvers.solve_mpmiqp import solve_mpmiqp
    from test_gpu_mpmiqp import _ref_regions
    g = numpy.load(os.path.join(MI, name + '.npz'))
    prog = StoredTreeProgram(name)
    combos = g['combinations'].tolist()
    sol = solve_mpmiqp(prog, screen='tree')
    assert sol.feasible_combinations == combos and sol.is_overlapping
    want = [(c, r) for k, c in enumerate(combos) for r in _ref_regions(g, k)]
    assert len(sol.critical_regions) == len(want)
    for a, (c, b) in zip(sol.critical_regions, want):
        assert list(a.active_set) == b['active_set'].tolist() and a.y_fixation == c
        assert a.y_indices == prog.binary_indices and a.x_indices == prog.cont_indices
        for fld in 'AbCd':
            assert rel_err(getattr(a, fld), b[fld]) <= REL_TOL, (name, c, a.active_set, fld)
        u1, u2 = rows_match_as_sets(a.E, a.f, b['E'], b['f'])
        assert not u1 and not u2, (name, c, a.active_set)


_RANDOM = [(nb, s) for nb in (4, 6, 8, 10, 12) for s in (0, 1)]


@pytest.mark.parametrize('nb,seed', _RANDOM)
def test_random_leaves_equal_highs(nb, seed):
    prog = random_program(nb, seed)
    feas, near = brute_force(prog)
    res = _leaves(prog)
    assert [y for y in res.leaves if y not in near] == feas, f'{len(near)} assignments in the band'
    assert res.leaves == sorted(res.leaves)


def _without_theta_rows(prog):
    q = MixedIntegerProgram(prog.A, prog.b, prog.F, numpy.zeros((0, prog.F.shape[1])), numpy.zeros(0), prog.binary_indices,
                            prog.equality_indices)
    return q


@pytest.mark.parametrize('nb,seed', [(4, 0), (5, 1), (6, 2)])
def test_random_leaves_equal_enumerate_screen(nb, seed):
    """Outside the tolerance band the tree and the 2^nb screen agree wherever the screen agrees with HiGHS on the lifted
    LP.  The screen also keeps assignments that HiGHS rejects (all of them because of Theta's rows A_t theta <= b_t but one,
    [0, 0, 0, 1, 0] of seed 1); the tree rejects every one of them, as HiGHS does."""
    import itertools
    from ppopt_b200.mp_solvers.mpmiqp_enumeration import solve_mpmiqp_enumeration
    prog = random_program(nb, seed)
    got = solve_mpmiqp_enumeration(prog, screen='tree').feasible_combinations
    want = solve_mpmiqp_enumeration(prog, screen='enumerate').feasible_combinations
    margin = {y: relaxation_margin(prog, y) for y in itertools.product((0, 1), repeat=nb)}
    band = [list(y) for y, mg in margin.items() if abs(mg) <= 1e-6]
    screen_only = [y for y in want if margin[tuple(y)] > 1e-6]
    assert len(screen_only) <= {4: 0, 5: 2, 6: 7}[nb]
    assert all(y not in got for y in screen_only)
    assert [y for y in want if y not in band and y not in screen_only] == [y for y in got if y not in band]


def _sum_program(nb, nc, t, k, equality):
    """sum(y) <= k (or == k), couplings x_j <= 10 y_j, x in [0, 10], one theta row, theta in [-1, 1]^t"""
    n = nc + nb
    rows, rhs = [numpy.r_[numpy.zeros(nc), numpy.ones(nb)]], [float(k)]
    for j in range(nc):
        a = numpy.zeros(n)
        a[j], a[nc + (7 * j) % nb] = 1.0, -10.0
        rows.append(a)
        rhs.append(0.0)
        rows += [numpy.eye(n)[j], -numpy.eye(n)[j]]
        rhs += [10.0, 0.0]
    rows.append(numpy.r_[numpy.ones(nc), numpy.zeros(nb)])
    rhs.append(5.0)
    F = numpy.zeros((len(rows), t))
    F[-1, 0] = 1.0
    return MixedIntegerProgram(numpy.array(rows), rhs, F, numpy.vstack([numpy.eye(t), -numpy.eye(t)]), numpy.ones(2 * t),
                               list(range(nc, n)), [0] if equality else [])


def _lex(nb, max_ones):
    import itertools
    return [list(y) for y in itertools.product((0, 1), repeat=nb) if sum(y) <= max_ones] if nb <= 16 else None


def test_nb40_at_most_two():
    prog = _sum_program(40, 2, 1, 2, equality=False)
    res = _leaves(prog)
    assert len(res.leaves) == 1 + 40 + 780
    assert res.leaves == sorted(res.leaves) and all(sum(y) <= 2 for y in res.leaves)
    for y in res.leaves[::20]:
        assert relaxation_margin(prog, y) <= 1e-9


def test_nb40_solve_mpmiqp():
    from ppopt_b200.mp_solvers.mpmiqp_enumeration import solve_mpmiqp_enumeration
    from ppopt_b200.mp_solvers.solve_mpmiqp import solve_mpmiqp
    prog = _sum_program(40, 2, 1, 2, equality=False)
    with pytest.raises(ValueError, match='more than 20 binaries'):
        solve_mpmiqp_enumeration(prog, screen='enumerate')
    sol = solve_mpmiqp(prog)
    assert len(sol.feasible_combinations) == 821 and len(sol.critical_regions) > 0


def test_nb56_exactly_one():
    prog = _sum_program(56, 3, 2, 1, equality=True)
    res = _leaves(prog)
    assert res.leaves == [[int(j == i) for j in range(56)] for i in range(55, -1, -1)]
    for y in res.leaves:
        assert relaxation_margin(prog, y) <= 1e-9


def _tree(prog, inherit=True):
    from ppopt_b200.mp_solvers.mitree import RelaxationTree
    return RelaxationTree(prog, inherit=inherit)


def _lifted_rows(prog, y_fixed, nb):
    A, b, F = prog.A, prog.b.ravel(), prog.F
    n, t = A.shape[1], F.shape[1]
    G = [numpy.hstack([A, -F]), numpy.hstack([numpy.zeros((prog.A_t.shape[0], n)), prog.A_t])]
    h = [b, prog.b_t.ravel()]
    for k, i in enumerate(prog.binary_indices):
        lo, hi = (y_fixed[k], y_fixed[k]) if k < len(y_fixed) else (0.0, 1.0)
        e = numpy.zeros(n + t)
        e[i] = 1.0
        G += [e[None], -e[None]]
        h += [numpy.array([hi]), numpy.array([-lo])]
    eq = numpy.zeros(sum(len(x) for x in h), bool)
    eq[list(prog.equality_indices)] = True
    return numpy.vstack(G), numpy.concatenate(h), eq


@pytest.mark.parametrize('seed', [0, 1, 2])
def test_node_status_points_and_batch_independence(seed):
    prog = random_program(10, 20 + seed)
    tree = _tree(prog, inherit=False)
    rng = numpy.random.default_rng(seed)
    try:
        for depth in (0, 3, 7, 10):
            vals = rng.integers(0, 1 << depth, size=48) if depth else numpy.zeros(48, dtype=numpy.int64)
            nodes = torch.tensor(vals, dtype=torch.int64, device='cuda')
            st, pt, it = tree.eval(nodes, depth)
            st, pt = st.cpu().numpy(), pt.cpu().numpy()
            assert set(st.tolist()) <= {0, 1}
            for j, v in enumerate(vals):
                y = [int(v >> k) & 1 for k in range(depth)]
                mg = relaxation_margin(prog, y)
                if abs(mg) > 1e-6:
                    assert (st[j] == 0) == (mg < 0), (depth, y, mg)
                if st[j] == 0:
                    G, h, eq = _lifted_rows(prog, y, 10)
                    r = G @ pt[j] - h
                    r[eq] = numpy.abs(r[eq])
                    assert numpy.all(r <= 1e-7 * (1 + numpy.abs(h))), (depth, y, r.max())
                else:
                    assert numpy.isnan(pt[j]).all()
            # the same nodes alone, and inside a larger shuffled batch
            single = [int(tree.eval(nodes[j:j + 1], depth)[0].item()) for j in range(0, 48, 7)]
            assert single == st[::7].tolist()
            perm = rng.permutation(48)
            big = torch.cat([nodes[perm], nodes[perm]])
            st2 = tree.eval(big, depth, points=False)[0].cpu().numpy()
            assert numpy.array_equal(st2[:48], st[perm]) and numpy.array_equal(st2[48:], st[perm])
    finally:
        tree.close()


def _walk(prog, inherit):
    tree = _tree(prog, inherit=inherit)
    out = []
    try:
        nodes = torch.zeros(1, dtype=torch.int64, device='cuda')
        pp = po = None
        for d in range(tree.nb + 1):
            st, pt, it = tree.eval(nodes, d, points=True, parent_point=pp, parent_of=po)
            out.append((nodes.cpu().numpy(), st.cpu().numpy(), it.cpu().numpy()))
            if d < tree.nb:
                nodes, po = tree.children(nodes, st, d)
                pp = pt
    finally:
        tree.close()
    return out


@pytest.mark.parametrize('nb,seed', [(8, 3), (12, 4)])
def test_inheritance_on_off_identical_status(nb, seed):
    on, off = _walk(random_program(nb, seed), True), _walk(random_program(nb, seed), False)
    inherited = 0
    for (n1, s1, i1), (n2, s2, i2) in zip(on, off):
        assert numpy.array_equal(n1, n2) and numpy.array_equal(s1, s2)
        assert (i2 >= 0).all()
        inherited += int((i1 < 0).sum())
    assert inherited > 0


def test_no_binaries_gives_the_root():
    box = numpy.vstack([numpy.eye(2), -numpy.eye(2)])
    prog = MixedIntegerProgram(box, [1.0, 1.0, 0.0, 0.0], numpy.zeros((4, 1)), numpy.array([[1.0], [-1.0]]), [1.0, 1.0], [])
    res = _leaves(prog)
    assert res.leaves == [[]] and res.stats['nodes'] == [1]


def _envelope_program(nb, nc, extra_rows, equality):
    p = _sum_program(nb, nc, 2, 1, equality)
    n = p.A.shape[1]
    fill = numpy.zeros((extra_rows, n))
    fill[:, 0] = 1.0
    A = numpy.vstack([p.A, fill])
    b = numpy.r_[p.b.ravel(), 20.0 + numpy.arange(extra_rows)]
    F = numpy.vstack([p.F, numpy.zeros((extra_rows, 2))])
    return MixedIntegerProgram(A, b, F, p.A_t, p.b_t, p.binary_indices, p.equality_indices)


def test_envelope_rows_and_columns():
    # 60 binaries + 3 continuous + 2 parameters: 65 free variables without the equality, 64 with it
    with pytest.raises(RuntimeError, match='at most 64'):
        _tree(_envelope_program(60, 3, 0, equality=False))
    base = _envelope_program(60, 3, 0, equality=True)
    rows = base.A.shape[0] - 1 + base.A_t.shape[0] + 2 * 60
    with pytest.raises(RuntimeError, match='at most 256'):
        _tree(_envelope_program(60, 3, 257 - rows, equality=True))
    res = _leaves(_envelope_program(60, 3, 256 - rows, equality=True))
    assert len(res.leaves) == 60


def test_max_leaves_raises():
    prog = random_program(10, 0, eq=False)
    prog.A, prog.b, prog.F = prog.A[-6:], prog.b[-6:], prog.F[-6:]   # the box rows only: every assignment is feasible
    prog.equality_indices = []
    with pytest.raises(ValueError, match='max_leaves'):
        _leaves(prog, max_leaves=100)
    assert len(_leaves(prog).leaves) == 1024


def test_library_errors_are_runtime_errors():
    # a continuous variable in no row: the relaxation has no vertex
    prog = MixedIntegerProgram(numpy.array([[1.0, 0.0, 1.0], [-1.0, 0.0, 0.0]]), [1.0, 0.0], numpy.zeros((2, 1)),
                               numpy.array([[1.0], [-1.0]]), [1.0, 1.0], [2])
    with pytest.raises(RuntimeError, match='no vertex'):
        _leaves(prog)
