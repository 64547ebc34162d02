"""Mixed-integer test programs built with numpy, and HiGHS (scipy) answers about their relaxations.  TEST INFRASTRUCTURE
for test_mitree_host.py / test_gpu_mitree.py.

A program object carries the attributes the relaxation tree reads (A, b, F, A_t, b_t, equality_indices, binary_indices,
cont_indices) and builds its substituted sub-problems the way ppopt's MPMIQP_Program does: the binaries moved to the
right-hand side, the rows without continuous variables and parameters dropped."""
import itertools

import numpy
from scipy.optimize import linprog


class MixedIntegerProgram:
    def __init__(self, A, b, F, A_t, b_t, binary_indices, equality_indices=()):
        self.A, self.F, self.A_t = (numpy.asarray(x, dtype=float) for x in (A, F, A_t))
        self.b = numpy.asarray(b, dtype=float).reshape(-1, 1)
        self.b_t = numpy.asarray(b_t, dtype=float).reshape(-1, 1)
        self.binary_indices = list(binary_indices)
        self.cont_indices = [i for i in range(self.A.shape[1]) if i not in set(self.binary_indices)]
        self.equality_indices = list(equality_indices)

    def generate_substituted_problem(self, y):
        from ppopt_b200.mplp_program import MPQP_Program
        yv = numpy.asarray(y, dtype=float)
        Ac, Ay = self.A[:, self.cont_indices], self.A[:, self.binary_indices]
        keep = [i for i in range(self.A.shape[0]) if not (numpy.allclose(Ac[i], 0) and numpy.allclose(self.F[i], 0))]
        eq = [k for k, i in enumerate(keep) if i in set(self.equality_indices)]
        b = self.b.ravel()[keep] - Ay[keep] @ yv
        nc, t = len(self.cont_indices), self.F.shape[1]
        return MPQP_Program(Ac[keep], b.reshape(-1, 1), numpy.zeros((nc, 1)), numpy.zeros((nc, t)), numpy.eye(nc), self.A_t,
                            self.b_t, self.F[keep], equality_indices=eq)


def random_program(nb, seed, nc=3, t=2, eq=True, big_m=10.0):
    """binaries with equality rows over binaries, binary-only rows, big-M couplings x <= M y, and theta-dependent rows;
    every continuous variable in [0, 10], theta in [-1, 1]^t"""
    rng = numpy.random.default_rng(seed)
    n = nc + nb
    rows, rhs, frows = [], [], []
    eqs = []

    def add(a, b, f=None, equality=False):
        if equality:
            eqs.append(len(rows))
        rows.append(a)
        rhs.append(b)
        frows.append(numpy.zeros(t) if f is None else f)

    if eq and nb >= 3:   # exactly one of three binaries
        a = numpy.zeros(n)
        a[nc + rng.choice(nb, 3, replace=False)] = 1.0
        add(a, 1.0, equality=True)
    for _ in range(max(1, nb // 3)):   # binary-only rows: at most k of a handful
        a = numpy.zeros(n)
        a[nc + rng.choice(nb, min(nb, 4), replace=False)] = 1.0
        add(a, float(rng.integers(1, 3)))
    for j in range(nc):   # x_j <= M y_k
        a = numpy.zeros(n)
        a[j], a[nc + rng.integers(nb)] = 1.0, -big_m
        add(a, 0.0)
    for _ in range(nc + 2):   # theta-dependent rows over x and y
        a = numpy.zeros(n)
        a[:nc] = rng.normal(size=nc)
        a[nc:] = rng.normal(size=nb) * (rng.random(nb) < 0.3)
        add(a, float(rng.uniform(-1.0, 2.0)), rng.normal(size=t) * 0.5)
    for j in range(nc):   # 0 <= x_j <= 10
        a = numpy.zeros(n)
        a[j] = 1.0
        add(a, 10.0)
        add(-a, 0.0)
    A_t = numpy.vstack([numpy.eye(t), -numpy.eye(t)])
    return MixedIntegerProgram(numpy.array(rows), numpy.array(rhs), numpy.array(frows), A_t, numpy.ones(2 * t),
                               list(range(nc, n)), eqs)


def relaxation_margin(prog, fixed):
    """min over (x, theta) of the largest scaled violation  max_i (a_i z - h_i) / (1 + |h_i|)  (|.| on equality rows) of the
    lifted rows, with y_k = fixed[k] for k < len(fixed) and the other binaries in [0, 1]: <= 0 iff the relaxation is
    feasible.  Clipped below at -1."""
    A, b, F = prog.A, prog.b.ravel(), prog.F
    n, t = A.shape[1], F.shape[1]
    rows = [numpy.hstack([A, -F])]
    rhs = [b]
    rows.append(numpy.hstack([numpy.zeros((prog.A_t.shape[0], n)), prog.A_t]))
    rhs.append(prog.b_t.ravel())
    for k, i in enumerate(prog.binary_indices):
        lo, hi = (fixed[k], fixed[k]) if k < len(fixed) else (0.0, 1.0)
        e = numpy.zeros(n + t)
        e[i] = 1.0
        rows += [e[None], -e[None]]
        rhs += [numpy.array([hi]), numpy.array([-lo])]
    G, h = numpy.vstack(rows), numpy.concatenate(rhs)
    eq = numpy.zeros(len(h), bool)
    eq[list(prog.equality_indices)] = True
    sc = 1.0 + numpy.abs(h)
    # variables (z, s): G z - s sc <= h, and for equalities also -G z - s sc <= -h
    Gi = numpy.vstack([numpy.hstack([G, -sc[:, None]]), numpy.hstack([-G[eq], -sc[eq][:, None]])])
    hi = numpy.concatenate([h, -h[eq]])
    c = numpy.zeros(n + t + 1)
    c[-1] = 1.0
    res = linprog(c, A_ub=Gi, b_ub=hi, bounds=[(None, None)] * (n + t) + [(-1.0, None)], method='highs')
    assert res.status == 0, res.message
    return float(res.x[-1])


def brute_force(prog, band=1e-6):
    """(feasible assignments in lexicographic order, assignments within +-band of the threshold)"""
    feas, near = [], []
    for y in itertools.product((0, 1), repeat=len(prog.binary_indices)):
        mg = relaxation_margin(prog, y)
        if abs(mg) <= band:
            near.append(list(y))
        elif mg < 0:
            feas.append(list(y))
    return feas, near


def tree_model(prog):
    """breadth-first relaxation tree with HiGHS: children of feasible nodes in parent order, y_d = 0 first"""
    nb = len(prog.binary_indices)
    level = [()]
    for d in range(nb + 1):
        feas = [y for y in level if relaxation_margin(prog, y) <= 0.0]
        if d == nb:
            return [list(y) for y in feas]
        level = [y + (v,) for y in feas for v in (0, 1)]
