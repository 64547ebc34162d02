"""Dispatch with the reference's surface (/root/reference/src/ppopt/mp_solvers/solve_mpmiqp.py:13-66): the enumeration
algorithm over the GPU engine (mpmiqp_enumeration.py).  The 1-D overlap reduction of mpMILP solutions (:57-63,
utils/region_overlap_utils.py) is post-processing outside the hot path and is not provided: such solutions are returned
overlapping, which Solution.get_region handles by comparing objectives.  ``screen`` ('auto' / 'tree' / 'enumerate'):
how the feasible binary combinations are found when ``feasible_combinations`` is not given (mpmiqp_enumeration)."""
from enum import Enum

from .mpmiqp_enumeration import solve_mpmiqp_enumeration
from .solve_mpqp import mpqp_algorithm, solve_mpqp


class mpmiqp_algorithm(Enum):
    enumerate = 'enumerate'

    def __str__(self):
        return self.name

    @staticmethod
    def all_algos():
        return ''.join(f'mpmiqp_algorithm.{a}\n' for a in mpmiqp_algorithm)


def solve_mpmiqp(problem, mpmiqp_algo: mpmiqp_algorithm = mpmiqp_algorithm.enumerate,
                 cont_algo: mpqp_algorithm = mpqp_algorithm.combinatorial, num_cores=-1, reduce_overlap=True,
                 feasible_combinations=None, screen='auto'):
    if len(problem.binary_indices) == 0:
        return solve_mpqp(problem, cont_algo)
    if not isinstance(mpmiqp_algo, mpmiqp_algorithm):
        raise TypeError("You must pass an algorithm from mpmiqp_algorithm as the continuous algorithm. These can be found by "
                        "importing the following \n\nfrom ppopt_b200.mp_solvers.solve_mpmiqp import mpmiqp_algorithm\n\nWith "
                        f"the following choices\n{mpmiqp_algorithm.all_algos()}")
    return solve_mpmiqp_enumeration(problem, num_cores, cont_algo, feasible_combinations=feasible_combinations,
                                    screen=screen)
