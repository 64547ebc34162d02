"""K2w's deferred dictionary updates (csrc/k2w_walk.cu, K2wDeferDict) against the policy that applies every pivot to the
whole dictionary (K2wSmemDict, selected per handle with PPGPU_OPT_K2W_REF).  The deferred policy performs the same FMAs in
the same order, so the walk must take the same pivots everywhere: two handles of the same program, one per policy, the walk
forced on at every level (PPGPU_OPT_K2W_MIN = 0), run level by level in lockstep and must agree on
  * every status byte,
  * every witness byte,
  * the walk's counters: pivots, certificates, drives given up and counted work.
Inputs: every golden program at its golden depth, and levels 1..5 of the bench program in full (74.5 M candidates), with
and without witness inheritance.  The bench levels also reload the dictionary after K2W_RESET pivots while deferred pivots
are pending (counter k2w_drop_reset).  A reload after a vertex left the certification band with pivots pending
(k2w_drop_giveup) does not occur on these inputs; it runs the same reload, which discards whatever is pending."""
import os

import pytest

from conftest import GOLDEN, golden_names

pytestmark = pytest.mark.gpu

WALK_COUNTERS = ('k2w_pivots', 'k2w_certified', 'k2w_giveup', 'k2w_work')


def _engines(name):
    from ppopt_b200 import engine
    from ppopt_b200._lib import OPT_K2W_MIN, OPT_K2W_REF
    from ppopt_b200.mplp_program import load_presolved
    prog = load_presolved(os.path.join(GOLDEN, name + '.npz'))
    engs = []
    for ref in (0, 1):
        eng = engine.Engine(engine.program_arrays(prog))
        eng.set_option(OPT_K2W_MIN, 0)
        eng.set_option(OPT_K2W_REF, ref)
        engs.append(eng)
    return engine, engs


def _levels(engine, eng, depth, witnesses):
    """level loop through the C ABI; yields (masks, status, witness, counters of the level)"""
    import torch
    from ppopt_b200._lib import ST_FEAS, WITNESS_SLOTS
    masks, parent = eng.root_level(), None
    for lvl in range(depth):
        n = masks.shape[0]
        if n == 0:
            return
        wit = torch.zeros((n, WITNESS_SLOTS, eng.W), dtype=torch.int64, device=eng.tdev) if witnesses else None
        c0 = eng.counters()
        st = eng.level_eval(masks, lvl + 1, witness=wit, parent=parent)
        c1 = eng.counters()
        yield masks, st, wit, {k: c1[k] - c0[k] for k in c1}
        if lvl + 1 == depth:
            return
        feas = eng.select(st, ST_FEAS, ST_FEAS)
        keep = {}
        masks = eng.children(masks, feas, lvl + 1, keep=keep)
        parent = engine.ParentLevel(keep['feas_masks'], keep['ws'], keep['nf'], wit[feas].contiguous()) if (witnesses and keep) else None


def _compare(name, depth, witnesses):
    """runs both policies in lockstep; returns the deferred policy's counters summed over the levels"""
    import torch
    engine, (eng, ref) = _engines(name)
    if not eng.has_walk_vertex:
        eng.close()
        ref.close()
        pytest.skip('feasibility polyhedron without a vertex: no walk')
    depth = min(depth, eng.max_depth)
    total = {}
    levels = 0
    for lv, (a, b) in enumerate(zip(_levels(engine, eng, depth, witnesses), _levels(engine, ref, depth, witnesses))):
        (m1, s1, w1, c1), (m0, s0, w0, c0) = a, b
        where = f'{name} level {lv + 1} (witnesses {witnesses})'
        assert torch.equal(m1, m0), f'{where}: different candidates'
        assert torch.equal(s1, s0), f'{where}: status bytes differ'
        if witnesses:
            assert torch.equal(w1, w0), f'{where}: witnesses differ'
        for k in WALK_COUNTERS:
            assert c1[k] == c0[k], (where, k, c1[k], c0[k])
        assert c0['k2w_drop_reset'] == 0 and c0['k2w_drop_giveup'] == 0, 'the reference policy has nothing to defer'
        for k, v in c1.items():
            total[k] = total.get(k, 0) + v
        levels += 1
    assert levels > 0
    print(name, 'witnesses' if witnesses else 'no witnesses', {k: total[k] for k in WALK_COUNTERS + ('k2w_drop_reset', 'k2w_drop_giveup')})
    eng.close()
    ref.close()
    return total


@pytest.mark.parametrize('witnesses', [True, False])
@pytest.mark.parametrize('name', golden_names())
def test_deferred_walk_matches_reference_on_goldens(name, witnesses):
    import numpy
    g = numpy.load(os.path.join(GOLDEN, name + '.npz'))
    _compare(name, int(g['n_levels']), witnesses)


@pytest.mark.parametrize('witnesses', [True, False])
def test_deferred_walk_matches_reference_at_the_benchmarked_depth(witnesses):
    import torch
    total = _compare('synthetic_30_6_40_s0', 5, witnesses)
    torch.cuda.empty_cache()
    assert total['k2w_pivots'] > 0
    # reloads after K2W_RESET pivots with deferred pivots pending
    assert total['k2w_drop_reset'] > 0, total
