"""K2w's infeasibility certificate (csrc/k2w_walk.cu, k2w_infeasible_verdict): a drive of a candidate's last row that ends
at the optimum of that row proves the candidate infeasible when the bound it gives on K2's LP clears the feasibility
tolerance by PPG_WALK_INF_MARGIN.  Such candidates are decided by the walk and skipped by K2a and K2; everything else
(bounds inside the band, drives ended by the iteration cap, a vertex out of the certification band, degenerate targets,
small positive coefficients) goes to K2a and K2 as before.  The certificate must never change a decision.

Two handles of the same program, the walk forced on at every level (PPGPU_OPT_K2W_MIN = 0), one with the certificate
(the default) and one without (PPGPU_OPT_K2W_INFEAS = 0), run level by level in lockstep and must agree on every status
byte and witness, and take the same pivots.  The walk's give-ups are the same drives in both runs; the certified ones are
exactly the LPs K2 and the relaxation no longer see.  Inputs: every golden program at its golden depth, levels 1..5 of the
bench program in full, and a hand-built program with one candidate far from feasible and one infeasible by less than the
margin."""
import os

import numpy
import pytest

from conftest import GOLDEN, golden_names

pytestmark = pytest.mark.gpu


def _pair(arrays):
    from ppopt_b200 import engine
    from ppopt_b200._lib import OPT_K2W_INFEAS, OPT_K2W_MIN
    engs = []
    for infeas in (1, 0):
        eng = engine.Engine(arrays)
        eng.set_option(OPT_K2W_MIN, 0)
        eng.set_option(OPT_K2W_INFEAS, infeas)
        engs.append(eng)
    return engs


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


def _check_counters(where, c1, c0):
    """c1: certificate on, c0: off (one level)"""
    assert c0['k2w_infeasible'] == 0 and c0['k2w_inf_band'] == 0, (where, 'the reference run proved something')
    for k in ('k2w_pivots', 'k2w_certified', 'k2w_giveup', 'k2w_work'):
        assert c1[k] == c0[k], (where, k, c1[k], c0[k])
    # every certificate and every band case is a drive the reference run gave up as well
    assert c1['k2w_infeasible'] + c1['k2w_inf_band'] <= c1['k2w_giveup'], (where, c1)
    # the candidates the walk proved infeasible are exactly the ones K2a and K2 no longer try
    assert c1['k2a_tried'] == c0['k2a_tried'] - c1['k2w_infeasible'], (where, c1['k2a_tried'], c0['k2a_tried'])
    assert c1['k2_lps'] == c0['k2_lps'] - c1['k2w_infeasible'], (where, c1['k2_lps'], c0['k2_lps'])
    assert c1['k2a_certified'] == c0['k2a_certified'], where


def _compare(name, depth, witnesses):
    """runs both handles in lockstep; returns the certificate run's counters summed over the levels"""
    import torch
    from ppopt_b200 import engine
    from ppopt_b200._lib import ST_FEAS, ST_RANK
    from ppopt_b200.mplp_program import load_presolved
    eng, ref = _pair(engine.program_arrays(load_presolved(os.path.join(GOLDEN, name + '.npz'))))
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
        assert int(((s1 & 128) != 0).sum().item()) == 0, f'{where}: a transient mark was left in the status bytes'
        if witnesses:
            assert torch.equal(w1, w0), f'{where}: witnesses differ'
        _check_counters(where, c1, c0)
        # a proof is never given for a candidate the reference calls feasible
        infeasible = int(((s1 & (ST_RANK | ST_FEAS)) == ST_RANK).sum().item())
        assert c1['k2w_infeasible'] <= infeasible, (where, c1['k2w_infeasible'], infeasible)
        for k, v in c1.items():
            total[k] = total.get(k, 0) + v
        levels += 1
    assert levels > 0
    print(name, {k: total[k] for k in ('k2w_infeasible', 'k2w_inf_band', 'k2w_giveup', 'k2w_pivots', 'k2a_tried', 'k2_lps')})
    eng.close()
    ref.close()
    return total


@pytest.mark.parametrize('name', golden_names())
def test_certificate_never_changes_a_decision_on_goldens(name):
    g = numpy.load(os.path.join(GOLDEN, name + '.npz'))
    _compare(name, int(g['n_levels']), True)


def test_certificate_never_changes_a_decision_at_the_benchmarked_depth():
    import torch
    total = _compare('synthetic_30_6_40_s0', 5, True)
    torch.cuda.empty_cache()
    assert total['k2w_infeasible'] > 0, total


def _two_corners(delta):
    """x in R^2, theta in [-1, 1] (no coupling): rows
         0: x1 >= 0   1: x2 >= 0   2: x1 + x2 >= 1   3: x1 <= 10   4: x2 <= 10   5: x1 + x2 <= 20 - delta
    {0, 1} misses row 2 by 1 (far from feasible), {3, 4} misses row 5 by delta (infeasible for K2 when delta is a few
    1e-7, but the walk's bound stays inside PPG_WALK_INF_MARGIN's band)."""
    A = numpy.array([[-1., 0.], [0., -1.], [-1., -1.], [1., 0.], [0., 1.], [1., 1.]])
    b = numpy.array([0., 0., -1., 10., 10., 20. - delta])
    return dict(A=A, b=b, F=numpy.zeros((6, 1)), A_t=numpy.array([[1.], [-1.]]), b_t=numpy.array([1., 1.]),
                c=numpy.zeros(2), H=numpy.zeros((2, 1)), n_eq=0, is_qp=True, Q=numpy.eye(2))


def test_clear_and_marginal_infeasibility():
    from ppopt_b200._lib import ST_FEAS, ST_RANK
    eng, ref = _pair(_two_corners(4e-7))
    assert eng.has_walk_vertex
    for rows, proved in (([0, 1], True), ([3, 4], False)):
        masks = eng.masks_from_lists([rows])
        c0 = eng.counters()
        st = eng.level_eval(masks, 2, stages=3)
        c1 = eng.counters()
        r0 = ref.counters()
        st_ref = ref.level_eval(masks, 2, stages=3)
        r1 = ref.counters()
        c = {k: c1[k] - c0[k] for k in c1}
        r = {k: r1[k] - r0[k] for k in r1}
        assert int(st[0]) == ST_RANK and int(st_ref[0]) == ST_RANK, (rows, int(st[0]), int(st_ref[0]))
        assert r['k2_lps'] == 1 and r['k2w_infeasible'] == 0, (rows, r)
        if proved:
            # decided by the walk: neither the relaxation nor the simplex looked at it
            assert c['k2w_infeasible'] == 1 and c['k2a_tried'] == 0 and c['k2_lps'] == 0, c
        else:
            # the bound (about -4e-7) is inside the band: K2 decides it
            assert c['k2w_infeasible'] == 0 and c['k2w_inf_band'] == 1 and c['k2_lps'] == 1, c
    # the whole second level: both corners among 15 candidates, same bytes either way
    import torch
    from itertools import combinations
    masks = eng.masks_from_lists([list(p) for p in combinations(range(6), 2)])
    st, st_ref = eng.level_eval(masks, 2, stages=3), ref.level_eval(masks, 2, stages=3)
    assert torch.equal(st, st_ref)
    assert int(((st & (ST_RANK | ST_FEAS)) == ST_RANK).sum().item()) >= 2
    eng.close()
    ref.close()
