"""ppopt_b200 - B200-native engine for PPOPT's combinatorial mpQP/mpLP critical-region enumeration.

    from ppopt_b200 import solve_mpqp, mpqp_algorithm
    solution = solve_mpqp(program, mpqp_algorithm.combinatorial)     # program: ppopt or ppopt_b200 program object

    ThetaSolver(program).solve_batch(thetas)    # fixed-theta QPs, one batch (ThetaLPSolver: mpLPs)
    verify_solution(solution)                   # explicit vs implicit

    import ppopt_b200; ppopt_b200.install()      # or: make ppopt.solve_mpqp(..., combinatorial) run on the GPU
"""
from .mp_solvers.solve_mpqp import mpqp_algorithm, solve_mpqp  # noqa: F401
from .mplp_program import MPLP_Program, MPQP_Program  # noqa: F401
from .point_location import PointLocation  # noqa: F401
from .solve_theta import ThetaLPSolver, ThetaSolver, verify_solution  # noqa: F401


def install(ppopt_package=None):
    """Replaces ``<ppopt>.mp_solvers.mpqp_combinatorial.solve`` with the GPU engine.  solve_mpqp looks the attribute up
    at call time (solve_mpqp.py:70-71), so user code and solve_mpmiqp are untouched.  Returns the original function."""
    import importlib
    if ppopt_package is None:
        ppopt_package = importlib.import_module('ppopt')
    mod = importlib.import_module(ppopt_package.__name__ + '.mp_solvers.mpqp_combinatorial')
    original = mod.solve
    from .mp_solvers import mpqp_combinatorial as mine
    mod.solve = mine.solve
    return original
