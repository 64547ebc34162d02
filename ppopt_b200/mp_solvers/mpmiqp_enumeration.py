"""Drop-in for ppopt.mp_solvers.mpmiqp_enumeration (/root/reference/src/ppopt/mp_solvers/mpmiqp_enumeration.py:12-64), the
caller above the combinatorial path (SURVEY.md section 8f row 3): one continuous mpQP/mpLP per feasible binary
combination, merged into one overlapping Solution.

What runs where
  * the binary tree (``MITree`` / ``check_bin_feasibility``, mitree.py, mpmilp_program.py:206-246) needs a MILP solver
    (the reference only has a Gurobi binding, solver.py:278-281).  Here the feasible combinations come from one of
      - ``feasible_combinations`` passed by the caller (what the reference's tree returns), which wins over ``screen``;
      - ``screen='tree'``: the relaxation tree on the GPU (K11, mitree.py): breadth first, one batch per depth, an inner
        node answers the LP relaxation of its partial assignment, a leaf the LP the MILP reduces to;
      - ``screen='enumerate'``: all 2^nb combinations on the host, keeping the ones whose substituted problem is feasible -
        for a LEAF the MILP feasibility question is an LP (every binary is fixed), and that LP is the base-set feasibility
        test of the engine (K2 on the empty active set); at most 20 binaries;
      - ``screen='auto'`` (default): 'enumerate' up to 20 binaries, 'tree' beyond;
  * the sub-problems are built by the program's own ``generate_substituted_problem`` (mpmilp_program.py:150-195,
    mpmiqp_program.py:71-116: numpy + the constructor's presolve);
  * every sub-problem is solved by the GPU engine.  A sub-problem is small (the binaries are gone), so one solve cannot fill
    148 SMs: the sub-problems are BATCHED ACROSS - a pool of host threads, one CUDA stream each, drives several engines at
    once (the reference maps them over a pathos process pool, :47-50); kernels of different sub-problems overlap on the
    device and the per-level host synchronisations of one solve hide behind the kernels of the others.
"""
import itertools
import threading
from concurrent.futures import ThreadPoolExecutor
from typing import Iterable, List, Optional

import numpy
import torch

from .. import engine as _engine
from . import mitree
from .._lib import ST_FEAS
from .solve_mpqp import mpqp_algorithm, solve_mpqp


def binary_rows_hold(program, y) -> bool:
    """rows that involve neither continuous variables nor parameters are dropped by generate_substituted_problem
    (mpmilp_program.py:161-170); for a full binary assignment they are plain arithmetic"""
    A, F, b = numpy.asarray(program.A, float), numpy.asarray(program.F, float), numpy.asarray(program.b, float).reshape(-1)
    yv = numpy.asarray(y, float)
    eq = set(int(i) for i in program.equality_indices)
    for i in range(A.shape[0]):
        if numpy.allclose(A[i, program.cont_indices], 0) and numpy.allclose(F[i], 0):
            v = float(A[i, program.binary_indices] @ yv) - b[i]
            if (abs(v) > 1e-9) if i in eq else (v > 1e-9):
                return False
    return True


def leaf_is_feasible(sub_problem) -> bool:
    """check_bin_feasibility for a full binary assignment = feasibility of the substituted constraint set (an LP): the
    engine's feasibility stage on the base (equality-only) active set"""
    eng = _engine.Engine(_engine.program_arrays(sub_problem))
    try:
        m0 = torch.zeros((1, eng.W), dtype=torch.int64, device=eng.tdev)
        return bool(int(eng.level_eval(m0, 0, stages=3).cpu()[0]) & ST_FEAS)
    finally:
        eng.close()


def solve_mpmiqp_enumeration(program, num_cores: int = -1, cont_algorithm: mpqp_algorithm = mpqp_algorithm.combinatorial,
                             feasible_combinations: Optional[Iterable[List[int]]] = None, streams: int = 4,
                             screen: str = 'auto'):
    """Same arguments and result as the reference's solve_mpmiqp_enumeration (``num_cores`` is accepted for signature
    parity; the GPU replaces the process pool).  ``feasible_combinations``: the leaves of the reference's MITree, when the
    caller has them; otherwise ``screen`` selects how they are found: 'tree' (the relaxation tree on the GPU), 'enumerate'
    (all 2^nb assignments, at most 20 binaries) or 'auto' ('enumerate' up to 20 binaries, 'tree' beyond).
    ``streams``: sub-problems in flight."""
    if screen not in ('auto', 'tree', 'enumerate'):
        raise ValueError(f"screen must be 'auto', 'tree' or 'enumerate', not {screen!r}")
    nb = len(program.binary_indices)
    subs = {}
    if feasible_combinations is None and (screen == 'tree' or (screen == 'auto' and nb > 20)):
        combos = []
        for y in mitree.feasible_combinations(program).leaves:
            try:
                sub = program.generate_substituted_problem(list(y))
            except Exception:   # the constructor's presolve found the substituted constraint set infeasible (tolerance band)
                continue
            combos.append(list(y))
            subs[tuple(y)] = sub
    elif feasible_combinations is None:
        if nb > 20:
            raise ValueError("more than 20 binaries: use screen='tree' or pass feasible_combinations")
        combos = []
        for y in itertools.product((0, 1), repeat=nb):
            if not binary_rows_hold(program, y):
                continue
            try:
                sub = program.generate_substituted_problem(list(y))
            except Exception:   # the constructor's presolve found the substituted constraint set infeasible
                continue
            if leaf_is_feasible(sub):
                combos.append(list(y))
                subs[tuple(y)] = sub
        # the reference's tree visits y = 0 before y = 1 at every depth (mitree.py:49-50, get_full_leafs: right child first)
    else:
        combos = [list(int(v) for v in y) for y in feasible_combinations]
    for y in combos:
        if tuple(y) not in subs:
            subs[tuple(y)] = program.generate_substituted_problem(list(y))

    device = torch.cuda.current_device()
    local = threading.local()

    def work(y):
        # one CUDA stream per worker thread: the launches of concurrent sub-problems interleave on the device
        if not hasattr(local, 'stream'):
            local.stream = torch.cuda.Stream(device=device)
        torch.cuda.set_device(device)
        with torch.cuda.stream(local.stream):
            sol = solve_mpqp(subs[tuple(y)], cont_algorithm)
            local.stream.synchronize()
        return sol

    if streams <= 1 or len(combos) <= 1:
        sols = [work(y) for y in combos]
    else:
        with ThreadPoolExecutor(max_workers=min(streams, len(combos))) as pool:
            sols = list(pool.map(work, combos))

    cont_indices = getattr(program, 'cont_indices', None)
    regions = []
    for y, sol in zip(combos, sols):
        for r in sol.critical_regions:
            # the fixed binary combination, the binary indices and the continuous variable indices (:54-59)
            r.y_fixation = y
            r.y_indices = program.binary_indices
            r.x_indices = cont_indices
            regions.append(r)
    _, sol_cls = _engine._region_classes(program)
    try:
        out = sol_cls(program, regions, is_overlapping=True)
    except TypeError:
        out = sol_cls(program, regions)
        out.is_overlapping = True
    out.feasible_combinations = combos
    out.sub_solutions = sols
    return out
