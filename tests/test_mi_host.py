"""CPU tests of the y maps of a mixed-integer program's continuous part (host_math.hpp::parameter_column_maps, read by the
pair mode of K8 / K9): every map equals a numpy reduction of the program with parameters (theta, y), solved directly."""
import numpy
import pytest

from mi_maps_export import param_maps
from mi_programs import objective_program

CASES = [(kind, nb, seed, couple) for kind in ('qp', 'lp') for nb in (3, 6) for seed in range(2) for couple in (False, True)]
REL = 1e-12


def continuous_part(prog):
    """the rows that contain a continuous variable (equalities first) on the continuous variables, and the y columns"""
    A, b, F = prog.A, prog.b.ravel(), prog.F
    xi, bi = prog.cont_indices, prog.binary_indices
    eq = set(prog.equality_indices)
    has_x = numpy.abs(A[:, xi]).max(1) > 0
    rows = [i for i in range(len(b)) if has_x[i] and i in eq] + [i for i in range(len(b)) if has_x[i] and i not in eq]
    ne = sum(1 for i in rows if i in eq)
    Q = None if prog.Q is None else 0.5 * (prog.Q + prog.Q.T)
    return dict(A=A[rows][:, xi], b=b[rows], F=F[rows], ne=ne, Fy=-A[rows][:, bi], c=prog.c.ravel()[xi], H=prog.H[xi],
                Q=None if Q is None else Q[numpy.ix_(xi, xi)], Hy=None if Q is None else Q[numpy.ix_(xi, bi)])


def _close(got, want):
    scale = max(1.0, float(numpy.abs(want).max(initial=0.0)))
    return float(numpy.abs(got - want).max(initial=0.0)) <= REL * scale


@pytest.mark.parametrize('kind,nb,seed,couple', CASES)
def test_maps_equal_numpy_reduction(kind, nb, seed, couple):
    prog = objective_program(nb, seed, kind=kind, couple=couple)
    P = continuous_part(prog)
    A, F, ne, Fy = P['A'], P['F'], P['ne'], P['Fy']
    m, n = A.shape
    maps, bvar, nvar, Q2 = param_maps(A, P['b'], F, prog.A_t, prog.b_t, ne, P['c'], P['H'], P['Q'], Fy, P['Hy'])
    mi = m - ne
    Aeq, Ain = A[:ne], A[ne:]
    if kind == 'qp':
        assert maps.shape == (mi + 2 * n, nb)
        # x at lambda = 0: the minimiser on the equality rows; its derivative in y_k, and the slacks' (V_y)
        K = numpy.block([[P['Q'], Aeq.T], [Aeq, numpy.zeros((ne, ne))]])
        dx = numpy.linalg.solve(K, numpy.vstack([-P['Hy'], Fy[:ne]]))[:n]
        assert _close(maps[mi:mi + n], dx)
        assert _close(maps[:mi], Fy[ne:] - Ain @ dx)
        assert _close(maps[mi + n:], P['Hy'])
    else:
        assert maps.shape == (2 * mi + n, nb)
        # the dictionary's vertex: equalities and the nonbasic rows tight; its basic entries are beta0 - Dth theta - Dth_y y
        tight = numpy.vstack([Aeq, Ain[nvar]])
        dx = numpy.linalg.solve(tight, numpy.vstack([Fy[:ne], Fy[ne:][nvar]]))
        dslack = Fy[ne:] - Ain @ dx
        dv = Q2.T @ dx
        want = numpy.array([dslack[r] if r >= 0 else dv[-1 - r] for r in bvar])
        assert _close(maps[:mi], -want)
        # the reduced rows' right-hand side bti + Ft theta + Ft_y y and the particular solution x0 (minimum norm)
        x0 = numpy.linalg.pinv(Aeq) @ Fy[:ne] if ne else numpy.zeros((n, nb))
        assert _close(maps[mi:2 * mi], Fy[ne:] - Ain @ x0)
        assert _close(maps[2 * mi:], x0)


def test_maps_refuse_a_semidefinite_hessian():
    prog = objective_program(3, 0, kind='qp')
    P = continuous_part(prog)
    with pytest.raises(ValueError, match='outside the fixed-theta solves'):
        param_maps(P['A'], P['b'], P['F'], prog.A_t, prog.b_t, P['ne'], P['c'], P['H'], numpy.zeros_like(P['Q']), P['Fy'], P['Hy'])
