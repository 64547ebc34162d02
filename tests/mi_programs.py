"""Mixed-integer test programs WITH an objective (mpMIQP / mpMILP), built on mitree_programs.random_program.  TEST
INFRASTRUCTURE for test_mi_host.py / test_gpu_mi_theta.py.

The objective is  1/2 z'Qz + theta'H'z + c'z + c_c + c_t'theta + 1/2 theta'Q_t theta  over z = (x, y) in program order
(Q = 0 for an mpMILP).  Q is positive definite with a nonzero x-y block.  generate_substituted_problem(y) substitutes the
objective consistently: c_x + Q_xy y (Q symmetrised), c_c + c_y'y + 1/2 y'Q_yy y, c_t + H_y'y."""
import numpy

from mitree_programs import MixedIntegerProgram, random_program


class MixedIntegerObjectiveProgram(MixedIntegerProgram):
    def __init__(self, base: MixedIntegerProgram, Q, H, c, c_c=0.0, c_t=None, Q_t=None):
        super().__init__(base.A, base.b, base.F, base.A_t, base.b_t, base.binary_indices, base.equality_indices)
        t = self.F.shape[1]
        self.Q = None if Q is None else numpy.asarray(Q, dtype=float)
        self.H, self.c = numpy.asarray(H, dtype=float), numpy.asarray(c, dtype=float).reshape(-1, 1)
        self.c_c = numpy.array([[float(c_c)]])
        self.c_t = numpy.zeros((t, 1)) if c_t is None else numpy.asarray(c_t, dtype=float).reshape(-1, 1)
        self.Q_t = numpy.zeros((t, t)) if Q_t is None else numpy.asarray(Q_t, dtype=float)

    def num_x(self):
        return self.A.shape[1]

    def num_t(self):
        return self.F.shape[1]

    def evaluate_objective(self, x, theta_point) -> float:
        x, th = numpy.asarray(x, dtype=float).reshape(-1, 1), numpy.asarray(theta_point, dtype=float).reshape(-1, 1)
        v = th.T @ self.H.T @ x + self.c.T @ x + self.c_c + self.c_t.T @ th + 0.5 * th.T @ self.Q_t @ th
        if self.Q is not None:
            v = v + 0.5 * x.T @ self.Q @ x
        return float(v[0, 0])

    def substituted_objective(self, y):
        """(Q_xx or None, c, H, c_c, c_t) of the continuous program at the assignment y"""
        yv = numpy.asarray(y, dtype=float)
        xi, bi = self.cont_indices, self.binary_indices
        c, H = self.c.ravel(), self.H
        Qs = None if self.Q is None else 0.5 * (self.Q + self.Q.T)
        cx = c[xi] + (Qs[numpy.ix_(xi, bi)] @ yv if Qs is not None else 0.0)
        cc = float(self.c_c[0, 0] + c[bi] @ yv + (0.5 * yv @ Qs[numpy.ix_(bi, bi)] @ yv if Qs is not None else 0.0))
        ct = self.c_t.ravel() + H[bi].T @ yv
        return (None if Qs is None else Qs[numpy.ix_(xi, xi)]), cx, H[xi], cc, ct

    def generate_substituted_problem(self, y):
        from ppopt_b200.mplp_program import MPLP_Program, MPQP_Program
        yv = numpy.asarray(y, dtype=float)
        Ac, Ay = self.A[:, self.cont_indices], self.A[:, self.binary_indices]
        keep = [i for i in range(self.A.shape[0]) if not (numpy.allclose(Ac[i], 0) and numpy.allclose(self.F[i], 0))]
        eq = [k for k, i in enumerate(keep) if i in set(self.equality_indices)]
        b = (self.b.ravel()[keep] - Ay[keep] @ yv).reshape(-1, 1)
        Qx, cx, Hx, cc, ct = self.substituted_objective(y)
        if Qx is None:
            return MPLP_Program(Ac[keep], b, cx.reshape(-1, 1), Hx, self.A_t, self.b_t, self.F[keep], c_c=cc, c_t=ct,
                                Q_t=self.Q_t, equality_indices=eq)
        return MPQP_Program(Ac[keep], b, cx.reshape(-1, 1), Hx, Qx, self.A_t, self.b_t, self.F[keep], c_c=cc, c_t=ct,
                            Q_t=self.Q_t, equality_indices=eq)


def _feasible_point(prog):
    """a point (z, theta) of the program with theta in Theta (HiGHS MIP, zero objective)"""
    from scipy.optimize import Bounds, LinearConstraint, milp
    n, t = prog.A.shape[1], prog.F.shape[1]
    h = prog.b.ravel()
    eq = numpy.zeros(len(h), bool)
    eq[list(prog.equality_indices)] = True
    G = numpy.vstack([numpy.hstack([prog.A, -prog.F]), numpy.hstack([numpy.zeros((prog.A_t.shape[0], n)), prog.A_t])])
    hi = numpy.concatenate([h, prog.b_t.ravel()])
    lo = numpy.concatenate([numpy.where(eq, h, -numpy.inf), numpy.full(prog.A_t.shape[0], -numpy.inf)])
    integ = numpy.zeros(n + t)
    integ[prog.binary_indices] = 1
    lb, ub = numpy.full(n + t, -numpy.inf), numpy.full(n + t, numpy.inf)
    lb[prog.binary_indices], ub[prog.binary_indices] = 0.0, 1.0
    res = milp(numpy.zeros(n + t), constraints=LinearConstraint(G, lo, hi), integrality=integ, bounds=Bounds(lb, ub))
    assert res.status == 0, 'the program has no point'
    return res.x[:n], res.x[n:]


def objective_program(nb, seed, kind='qp', nc=3, t=2, couple=False, at_most=None):
    """random_program(nb, seed, nc, t) with an objective.  couple: an equality row x_0 + x_1 + 2 y_k = r + 0.2 theta_0 that
    couples x and y (r from a point of the program); at_most: a binary-only row sum(y) <= at_most (keeps the
    number of feasible assignments small)."""
    base = random_program(nb, seed, nc=nc, t=t)
    rng = numpy.random.default_rng(1000 + seed)
    n = nc + nb
    A, b, F, eqs = list(base.A), list(base.b.ravel()), list(base.F), list(base.equality_indices)
    if couple:   # through a point of the program, so that its assignment stays feasible near there
        a = numpy.zeros(n)
        a[0], a[1], a[nc + int(rng.integers(nb))] = 1.0, 1.0, 2.0
        f = numpy.zeros(t)
        f[0] = 0.2
        eqs.append(len(A))
        z, th = _feasible_point(base)
        A.append(a), b.append(float(a @ z - f @ th)), F.append(f)
    if at_most is not None:
        a = numpy.zeros(n)
        a[nc:] = 1.0
        A.append(a), b.append(float(at_most)), F.append(numpy.zeros(t))
    base = MixedIntegerProgram(numpy.array(A), numpy.array(b), numpy.array(F), base.A_t, base.b_t, base.binary_indices, eqs)
    H = rng.normal(size=(n, t)) * 0.5
    c = rng.normal(size=n)
    if kind == 'lp':
        return MixedIntegerObjectiveProgram(base, None, H, c, c_c=0.3, c_t=rng.normal(size=t))
    M = rng.normal(size=(n, n))
    Q = M @ M.T / n + 0.5 * numpy.eye(n)
    return MixedIntegerObjectiveProgram(base, Q, H, c, c_c=0.3, c_t=rng.normal(size=t), Q_t=numpy.eye(t) * 0.1)
