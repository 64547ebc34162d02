"""Dispatch with the reference's surface (/root/reference/src/ppopt/mp_solvers/solve_mpqp.py:23-114).

The combinatorial algorithm is the scope (BASELINE.json north_star), the two connected-graph algorithms ride on the same
kernels (SURVEY.md 8f row 2), and the geometric algorithm steps across facets with K10 and K8 (mpqp_geometric); the enum keeps the reference's member names so
that calling code type-checks, and every other member raises NotImplementedError instead of silently returning an
empty solution."""
from enum import Enum

import numpy

from . import mpqp_combi_graph, mpqp_combinatorial, mpqp_geometric, mpqp_graph


class mpqp_algorithm(Enum):
    combinatorial = 'combinatorial'
    combinatorial_parallel = 'p combinatorial'
    combinatorial_parallel_exp = 'p combinatorial exp'
    graph = 'graph'
    graph_exp = 'graph exp'
    graph_parallel = 'p graph'
    graph_parallel_exp = 'p graph exp'
    geometric = 'geometric'
    geometric_parallel = 'p geometric'
    geometric_parallel_exp = 'p geometric exp'
    combinatorial_graph = 'combinatorial graph'

    def __str__(self):
        return self.name

    @staticmethod
    def all_algos():
        return ''.join(f'mpqp_algorithm.{a}\n' for a in mpqp_algorithm)


def solve_mpqp(problem, algorithm: mpqp_algorithm = mpqp_algorithm.combinatorial):
    """Solves an mpQP or mpLP; same argument meaning and TypeError as the reference (solve_mpqp.py:52-66)."""
    if not isinstance(algorithm, mpqp_algorithm):
        raise TypeError("You must pass an algorithm from mpqp_algorithm as the continuous algorithm. These can be found "
                        "by importing the following \n\nfrom ppopt_b200.mp_solvers.solve_mpqp import mpqp_algorithm\n\n"
                        f"With the following choices\n{mpqp_algorithm.all_algos()}")
    if algorithm is mpqp_algorithm.combinatorial_graph:
        solution = mpqp_combi_graph.solve(problem)          # solve_mpqp.py:100-101
    elif algorithm in (mpqp_algorithm.combinatorial, mpqp_algorithm.combinatorial_parallel,
                       mpqp_algorithm.combinatorial_parallel_exp):
        # solve_mpqp.py:70-77: the reference's pool-parallel variants enumerate the same levels with the same per-candidate
        # work (mpqp_parrallel_combinatorial.py:67-150); here every level is one GPU batch anyway
        solution = mpqp_combinatorial.solve(problem)
    elif algorithm is mpqp_algorithm.graph:
        solution = mpqp_graph.solve(problem)                # solve_mpqp.py:79-80
    elif algorithm is mpqp_algorithm.graph_exp:
        solution = mpqp_graph.solve(problem, use_pruning=False)   # solve_mpqp.py:82-83
    elif algorithm in (mpqp_algorithm.geometric, mpqp_algorithm.geometric_parallel, mpqp_algorithm.geometric_parallel_exp):
        # the reference's pool variants do the same work per facet; here every wave of facets is one GPU batch anyway
        solution = mpqp_geometric.solve(problem)
    else:
        raise NotImplementedError(f'{algorithm} is outside the scope of the B200 engine (combinatorial*, combinatorial_graph, '
                                  'graph, graph_exp, geometric*)')
    # overlap flags exactly as the reference sets them (solve_mpqp.py:105-112)
    if hasattr(problem, 'Q') and problem.Q is not None:
        if min(numpy.linalg.eigvalsh(problem.Q)) <= 0:
            solution.is_overlapping = True
    solution.is_overlapping = True  # isinstance(problem, MPLP_Program) holds for both program types in the reference
    return solution
