"""Drop-in for ppopt.mp_solvers.mpqp_graph (/root/reference/src/ppopt/mp_solvers/mpqp_graph.py:38-103), the connected-graph
algorithm of Oberdieck et al. 2016 (SURVEY.md section 8f row 2), on the kernels of the combinatorial path.

The reference pops ONE active set at a time (lowest cardinality first, stable order), and per set runs is_full_rank,
check_feasibility, check_optimality, gen_cr_from_active_set and CriticalRegion.is_full_dimension; what it attempts next
depends on the order of those pops (its pruning list filters neighbours at generation time).  To return exactly the
reference's solution the host replays that loop verbatim - same list, same sort, same pruning list - but never evaluates a
single set: whenever the loop needs a decision that is not cached, EVERY set waiting in the list is evaluated in one batch
on the GPU (speculative frontier batching; grouped by cardinality):
    K1     LICQ rank screen                                   <- is_full_rank
    K2w/K2a/K2  feasibility                                    <- program.check_feasibility
    K3/K4  KKT + theta-space polytope LP                       <- program.check_optimality  (non-empty  <=>  radius >= -1e-7)
    K5     LU-accurate rows, full-dimension test, redundancy   <- gen_cr_from_active_set + region.is_full_dimension
A few speculatively evaluated sets are never popped by the reference (their results are simply not used).

Seeding.  The reference samples theta and solves QPs (``program.sample_theta_space()``); the default seed here is the
first optimal active set of the level-wise enumeration (mpqp_combi_graph._seed).  ``initial_active_sets`` overrides it,
as in the reference (``graph_initialization``, :10-35): ``initial_active_sets=ThetaSolver(program).sample_theta_space()``
(ppopt_b200.solve_theta, batched QP solves on the GPU) gives reference-style seeding.
"""
from typing import Dict, Iterable, List, Optional, Tuple

import numpy
import torch

from .. import engine as _engine
from .._lib import ST_FEAS, ST_OPT, ST_RANK, ST_REGION, ST_THIN
from .mpqp_combi_graph import _seed
from .solver_utils import CombinationTester


def _evaluate(eng, cr_cls, sets: List[Tuple[int, ...]], cache: Dict, keep: Optional[list] = None):
    """cache[a] = (full_rank, feasible, optimal, region or None) for every active set in ``sets``.  ``keep`` (list): receives,
    per cardinality group that emitted regions, (active sets, regions or None, K5's device buffers laws / rows / flags / info)
    in the order of the sets handed to K5"""
    n_eq = eng.n_eq
    by_k: Dict[int, List[Tuple[int, ...]]] = {}
    for a in sets:
        by_k.setdefault(len(a) - n_eq, []).append(a)
    for k_act, group in sorted(by_k.items()):
        if k_act > eng.n - n_eq or k_act < 0:
            for a in group:     # more active rows than variables: rank deficient by counting
                cache[a] = (False, False, False, None)
            continue
        masks = eng.masks_from_lists(group)
        status = eng.level_eval(masks, k_act, stages=7)
        opt = eng.select(status, ST_OPT, ST_OPT)
        built = {}
        if opt.shape[0]:
            bufs = eng.emit(masks, opt, k_act, status)
            laws, rows, flags, info = [x.cpu().numpy() for x in bufs]
            if numpy.any(info[:, 0] < 0):
                raise numpy.linalg.LinAlgError('Singular matrix')
            asets = [list(group[i]) for i in opt.cpu().tolist()]
            regs = _engine.build_regions(eng, cr_cls, asets, k_act, laws, rows, flags, info)
            for a_, r in zip(asets, regs):
                if r is not None:
                    built[tuple(a_)] = r
            if keep is not None:
                keep.append(([tuple(a_) for a_ in asets], regs, bufs))
        for a, s_ in zip(group, status.cpu().numpy()):
            rank_ok = bool(s_ & ST_RANK)
            feas = rank_ok and bool(s_ & ST_FEAS)
            optimal = feas and bool(s_ & (ST_OPT | ST_THIN))
            cache[a] = (rank_ok, feas, optimal, built.get(a))


def solve(program, initial_active_sets: Optional[Iterable] = None, use_pruning: bool = True):
    """Solves the mpQP with the graph algorithm; returns the reference's Solution (same regions, same order)."""
    from .solver_utils import generate_extra, generate_reduce
    eng = _engine.Engine(_engine.program_arrays(program))
    try:
        if not (eng.is_qp and eng.use_gram):
            raise NotImplementedError('the graph algorithm on the GPU needs an mpQP with a positive definite reduced Hessian')
        cr_cls, sol_cls = _engine._region_classes(program)
        seeds = [tuple(int(i) for i in a) for a in initial_active_sets] if initial_active_sets is not None \
            else _seed(program, eng)
        attempted = set()
        murder = CombinationTester() if use_pruning else None
        to_attempt = list(seeds)
        regions = []
        cache: Dict = {}
        eqs = set(range(eng.n_eq))
        batches = 0
        while to_attempt:
            to_attempt.sort(key=len)                       # lowest cardinality first (mpqp_graph.py:60)
            candidate = to_attempt.pop(0)
            if candidate in attempted:
                continue
            attempted.add(candidate)
            if candidate not in cache:
                pending = [candidate] + [a for a in dict.fromkeys(to_attempt) if a not in cache and a not in attempted]
                _evaluate(eng, cr_cls, pending, cache)
                batches += 1
            rank_ok, feas, optimal, region = cache[candidate]
            if not rank_ok or not feas:                    # :72-85
                to_attempt.extend(generate_reduce(candidate, murder, attempted, eqs))
                if murder is not None:
                    murder.add_combo(candidate)
                continue
            if not optimal:                                # :87-90
                to_attempt.extend(generate_reduce(candidate, murder, attempted, eqs))
                continue
            if region is None:                             # optimal but not full dimensional: nothing to do (:92-97)
                continue
            regions.append(region)                         # :98-103
            to_attempt.extend(generate_reduce(candidate, murder, attempted, eqs))
            to_attempt.extend(generate_extra(candidate, region.regular_set[1], murder, attempted))
        solution = sol_cls(program, regions)
        solution.gpu_launches = eng.launch_count()
        solution.attempted = len(attempted)
        solution.gpu_batches = batches
        return solution
    finally:
        eng.close()
