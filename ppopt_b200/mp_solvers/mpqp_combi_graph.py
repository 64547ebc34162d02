"""Drop-in for ppopt.mp_solvers.mpqp_combi_graph (/root/reference/src/ppopt/mp_solvers/mpqp_combi_graph.py:69-145), the
combinatorial connected-graph algorithm of Arnstrom et al. (SURVEY.md section 8f row 2), on the same kernels as the
combinatorial solver.

The reference pops one active set at a time from a Python set and, per set, runs is_full_rank (SVD), the theta-space
non-emptiness LP ``feasability_check`` (:48-66) and gen_cr_from_active_set.  Here the FRONTIER of the graph search is the
batch: every wave groups the frontier by cardinality and sends each group through
    K1  (LICQ rank screen, csrc/k1_rank.cu)                     <- is_full_rank
    K3/K4 (KKT by Schur complement + theta-space polytope LP)    <- feasability_check: non-empty  <=>  radius >= -1e-7
    K5  (LU-accurate rows, full-dimension test, redundancy)      <- gen_cr_from_active_set
and the host only does what the reference does with Python sets: neighbours (drop one inequality / add one constraint),
the visited set E, the next frontier.  The visited closure does not depend on the order in which sets are popped, so
the region SET equals the reference's (its list order is the arbitrary order of ``set.pop()``).

Seeding.  The reference samples one theta and solves a QP for its active set (``program.sample_theta_space(1)``); the
default seed here is the first optimal active set the level-wise enumeration meets (any optimal active set will do: the
graph of optimal active sets is connected - the premise of the algorithm).  ``initial_active_sets`` overrides it, as in
``combinatorial_graph_initialization`` (:10-29): ``initial_active_sets=ThetaSolver(program).sample_theta_space()``
(ppopt_b200.solve_theta, batched QP solves on the GPU) gives reference-style seeding.
"""
from typing import Iterable, List, Optional

import numpy
import torch

from .. import engine as _engine
from .._lib import ST_FEAS, ST_OPT, ST_RANK, ST_REGION, ST_THIN


def _seed(program, eng) -> List[tuple]:
    """first optimal active set of the level-wise enumeration (base set first)"""
    m0 = torch.zeros((1, eng.W), dtype=torch.int64, device=eng.tdev)
    if int(eng.level_eval(m0, 0).cpu()[0]) & ST_OPT:
        return [tuple(range(eng.n_eq))]
    masks = eng.root_level()
    for lvl in range(eng.max_depth):
        if masks.shape[0] == 0:
            break
        status = eng.level_eval(masks, lvl + 1)
        opt = eng.select(status, ST_OPT, ST_OPT)
        if opt.shape[0]:
            return [tuple(eng.lists_from_masks(masks[opt[:1]].cpu().numpy())[0])]
        masks = eng.children(masks, eng.select(status, ST_FEAS, ST_FEAS), lvl + 1)
    raise RuntimeError('no optimal active set found to seed the graph search')


def solve(program, initial_active_sets: Optional[Iterable] = None, return_trace: bool = False):
    """Solves the mpQP with the combinatorial connected-graph algorithm; Solution as the reference's (region order is
    arbitrary there).  ``return_trace``: also return {active set: (full_rank, non_empty, region, thin_only)} for every visited set."""
    eng = _engine.Engine(_engine.program_arrays(program))
    try:
        if not (eng.is_qp and eng.use_gram):
            raise NotImplementedError('combinatorial_graph on the GPU needs an mpQP with a positive definite reduced Hessian')
        cr_cls, sol_cls = _engine._region_classes(program)
        n_eq, m = eng.n_eq, eng.m
        eq = set(range(n_eq))
        seeds = [tuple(sorted(int(i) for i in a)) for a in initial_active_sets] if initial_active_sets is not None \
            else _seed(program, eng)
        visited = set(seeds)             # E of the reference
        frontier = list(dict.fromkeys(seeds))
        regions, trace = [], {}
        while frontier:
            by_k = {}
            for a in frontier:
                by_k.setdefault(len(a) - n_eq, []).append(a)
            nxt = []

            def push(a_):
                if a_ not in visited:
                    visited.add(a_)
                    nxt.append(a_)
            for k_act in sorted(by_k):
                sets = by_k[k_act]
                if k_act > eng.n - n_eq:
                    # more active rows than variables: rank deficient by counting (is_full_rank compares rank with len(A))
                    for a in sets:
                        trace[a] = (False, False, False, False)
                        for i in a:
                            if i not in eq:
                                push(tuple(x for x in a if x != i))
                    continue
                masks = eng.masks_from_lists(sets)
                status = eng.level_eval(masks, k_act, stages=1)                       # is_full_rank
                full = (status & ST_RANK) != 0
                # feasability_check works in theta space and needs no primal feasibility LP: hand every full-rank set to K3/K4
                status = torch.where(full, status | ST_FEAS, status)
                eng.level_eval(masks, k_act, status, stages=4)
                opt = eng.select(status, ST_OPT, ST_OPT)
                built = {}
                if opt.shape[0]:
                    laws, rows, flags, info = [x.cpu().numpy() for x in eng.emit(masks, opt, k_act, status)]
                    if numpy.any(info[:, 0] < 0):
                        raise numpy.linalg.LinAlgError('Singular matrix')
                    asets = [list(sets[i]) for i in opt.cpu().tolist()]
                    for a_, r in zip(asets, _engine.build_regions(eng, cr_cls, asets, k_act, laws, rows, flags, info)):
                        if r is not None:
                            built[tuple(a_)] = r
                st = status.cpu().numpy()
                for a, s_ in zip(sets, st):
                    rank_ok = bool(s_ & ST_RANK)
                    nonempty = rank_ok and bool(s_ & (ST_OPT | ST_THIN))
                    # 4th entry: non-empty only by the LP tolerance band (radius in [-1e-7, 0.5e-8)): the reference's LP, run on
                    # UN-normalised rows, may call such a polytope empty
                    trace[a] = (rank_ok, nonempty, a in built, bool(s_ & ST_THIN) and not bool(s_ & ST_OPT))
                    if a in built:
                        regions.append(built[a])
                    if (not rank_ok) or nonempty:
                        for i in a:                                        # explore_subset (:88-98)
                            if i not in eq:
                                push(tuple(x for x in a if x != i))
                    if nonempty:
                        present = set(a)
                        for i in range(m):                                 # explore_superset (:100-110)
                            if i not in present:
                                push(tuple(sorted(present | {i})))
            frontier = nxt
        solution = sol_cls(program, regions)
        solution.gpu_launches = eng.launch_count()
        solution.visited = len(visited)
        return (solution, trace) if return_trace else solution
    finally:
        eng.close()
