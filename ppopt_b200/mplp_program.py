"""Program containers with the constructor signature and attribute surface of the reference's MPLP_Program /
MPQP_Program (/root/reference/src/ppopt/mplp_program.py:45-134,140-156; mpqp_program.py:15-42).

``MPQP_Program(A, b, c, H, Q, A_t, b_t, F, equality_indices=..., post_process=True)`` runs the reference's presolve
(presolve.py: host numpy steps + one GPU batch of redundancy LPs).  ``presolved=True`` skips all processing for data that
already went through a program constructor (tests/golden fixtures, genuine ppopt objects' arrays).
"""
from typing import List, Optional

import numpy


def _f64(a, cols=None):
    a = numpy.ascontiguousarray(numpy.asarray(a, dtype=numpy.float64))
    if a.ndim == 1:
        a = a.reshape(-1, 1) if cols is None else a.reshape(-1, cols)
    return a


class MPLP_Program:
    r"""min theta'H'x + c'x  s.t.  A x <= b + F theta (first n_eq rows equalities),  A_t theta <= b_t."""

    def __init__(self, A, b, c, H, A_t, b_t, F, c_c=None, c_t=None, Q_t=None, equality_indices=None, solver=None,
                 post_process=True, presolved=False):
        self.A, self.b, self.c, self.H = _f64(A), _f64(b), _f64(c), _f64(H)
        self.A_t, self.b_t, self.F = _f64(A_t), _f64(b_t), _f64(F)
        if not presolved:
            from . import presolve
            self.A, self.b, self.F, self.A_t, self.b_t, equality_indices = presolve.base_processing(
                self.A, self.b, self.F, self.A_t, self.b_t, [] if equality_indices is None else list(equality_indices))
            if post_process and type(self) is MPLP_Program:
                self.process_constraints(len(equality_indices))
        t = self.F.shape[1]
        self.c_c = numpy.array([[0.0]]) if c_c is None else _f64(c_c)
        self.c_t = numpy.zeros((t, 1)) if c_t is None else _f64(c_t)
        self.Q_t = numpy.zeros((t, t)) if Q_t is None else _f64(Q_t)
        eq = [] if equality_indices is None else [int(i) for i in equality_indices]
        if eq != list(range(len(eq))):
            raise ValueError('presolved programs have their equality rows first: equality_indices must be range(n_eq)')
        self.equality_indices: List[int] = eq
        self.solver = solver

    def process_constraints(self, n_eq=None) -> None:
        """Removes redundant constraints (mplp_program.py:285-306); the per-row LPs run as one GPU batch."""
        from . import presolve
        n_eq = len(self.equality_indices) if n_eq is None else n_eq
        self.A, self.b, self.F, self.A_t, self.b_t = [numpy.ascontiguousarray(x) for x in presolve.remove_redundant(
            self.A, self.b, self.F, self.A_t, self.b_t, n_eq)]

    def warnings(self):
        """The two numerical checks of the reference constructor's warnings() (mplp_program.py:204-215) on the GPU: the
        Chebyshev ball of the (x, theta) feasible space and the feasibility of the program as stated.  (The shape checks of
        :166-202 are raised as errors by this constructor.)"""
        from .chebyshev import chebyshev_radii
        out = []
        n, t = self.A.shape[1], self.F.shape[1]
        ne = len(self.equality_indices)
        if ne == 0:
            # (with equality rows the ball lives in their affine hull: chebyshev_ball gives those rows no radius term, the
            # batched kernel has no equality rows, so that variant is only covered by the feasibility check below)
            A_xt = numpy.vstack([numpy.hstack([self.A, -self.F]), numpy.hstack([numpy.zeros((self.A_t.shape[0], n)), self.A_t])])
            b_xt = numpy.vstack([self.b.reshape(-1, 1), self.b_t.reshape(-1, 1)])
            rad = chebyshev_radii([(A_xt, b_xt)])[0]
            if not (rad > 0.0):
                out.append('The chebychev ball has either a radius of zero, or the problem is not feasible!')
        from . import engine as _engine
        import torch
        eng = _engine.Engine(_engine.program_arrays(self))
        try:
            m0 = torch.zeros((1, eng.W), dtype=torch.int64, device=eng.tdev)
            if not (int(eng.level_eval(m0, 0, stages=3).cpu()[0]) & 2):
                out.append('The multiparametric program, as stated, is not feasible!')
        finally:
            eng.close()
        return out

    def num_x(self) -> int:
        return self.A.shape[1]

    def num_t(self) -> int:
        return self.F.shape[1]

    def num_constraints(self) -> int:
        return self.A.shape[0]

    def num_inequality_constraints(self) -> int:
        return self.A.shape[0] - len(self.equality_indices)

    def num_equality_constraints(self) -> int:
        return len(self.equality_indices)

    def evaluate_objective(self, x, theta_point) -> float:
        v = theta_point.T @ self.H.T @ x + self.c.T @ x + self.c_c + self.c_t.T @ theta_point \
            + 0.5 * theta_point.T @ self.Q_t @ theta_point
        return float(v[0, 0])

    def _theta_solver(self):
        if getattr(self, '_theta_solver_cache', None) is None:
            from .solve_theta import ThetaLPSolver
            self._theta_solver_cache = ThetaLPSolver(self)
        return self._theta_solver_cache

    def solve_theta(self, theta_point, deterministic_solver=None):
        """LP at a fixed theta (mplp_program.py solve_theta) on the GPU (ppopt_b200.solve_theta.ThetaLPSolver): a
        SolverOutput(obj, sol, slack, active_set, dual), or None when infeasible or unbounded.  ``deterministic_solver`` is
        accepted for the reference's signature and ignored.  The solver is built on first use and caches the program data:
        call again after changing the arrays of this object only on a new object."""
        return self._theta_solver().solve_theta(theta_point)

    def sample_theta_space(self, num_samples: int = 100):
        """distinct optimal bases (equality rows first) of LPs solved at points sampled in Theta (mplp_program.py
        sample_theta_space)"""
        return self._theta_solver().sample_theta_space(num_samples)


class MPQP_Program(MPLP_Program):
    r"""min 1/2 x'Qx + theta'H'x + c'x  with the constraints of MPLP_Program."""

    def __init__(self, A, b, c, H, Q, A_t, b_t, F, c_c=None, c_t=None, Q_t=None, equality_indices=None, solver=None,
                 post_process=True, presolved=False):
        self.Q = _f64(Q)
        super().__init__(A, b, c, H, A_t, b_t, F, c_c, c_t, Q_t, equality_indices, solver, post_process=False,
                         presolved=presolved)
        if post_process and not presolved:  # same order as the reference: base processing first, then redundancy
            self.process_constraints()

    def evaluate_objective(self, x, theta_point) -> float:
        v = 0.5 * x.T @ self.Q @ x + theta_point.T @ self.H.T @ x + self.c.T @ x + self.c_c \
            + self.c_t.T @ theta_point + 0.5 * theta_point.T @ self.Q_t @ theta_point
        return float(v[0, 0])

    def _theta_solver(self):
        if getattr(self, '_theta_solver_cache', None) is None:
            from .solve_theta import ThetaSolver
            self._theta_solver_cache = ThetaSolver(self)
        return self._theta_solver_cache

    def solve_theta(self, theta_point, deterministic_solver=None):
        """QP at a fixed theta (mpqp_program.py solve_theta) on the GPU (ppopt_b200.solve_theta.ThetaSolver): a
        SolverOutput(obj, sol, slack, active_set, dual), or None when infeasible.  ``deterministic_solver`` is accepted for
        the reference's signature and ignored.  The solver is built on first use and caches the program data: call
        again after changing the arrays of this object only on a new object."""
        return self._theta_solver().solve_theta(theta_point)

    def sample_theta_space(self, num_samples: int = 100):
        """distinct optimal active sets of QPs solved at points sampled in Theta (mpqp_program.py sample_theta_space)"""
        return self._theta_solver().sample_theta_space(num_samples)


def load_presolved(path: str):
    """Program object from a tests/golden/*.npz fixture (post-presolve arrays written by oracle/gen_golden.py)."""
    g = numpy.load(path)
    eq = list(range(int(g['n_eq'])))
    if str(g['kind']) == 'qp':
        return MPQP_Program(g['A'], g['b'], g['c'], g['H'], g['Q'], g['A_t'], g['b_t'], g['F'], equality_indices=eq,
                            presolved=True)
    return MPLP_Program(g['A'], g['b'], g['c'], g['H'], g['A_t'], g['b_t'], g['F'], equality_indices=eq, presolved=True)
