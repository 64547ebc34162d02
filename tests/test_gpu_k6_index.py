"""K6's prefix-group index (csrc/k6_children.cu) against plain Python sets.

children_count_kernel decides a parent's children by intersecting the bitmaps E_Q of the groups Q = P \\ {j}, and
inherit_kernel finds a parent as start(Q) + |E_Q below h|.  Both are checked here, through the C ABI, against the
definitions they replace:
  * a child P + {i} survives iff every k-subset is in the feasible list (the mpLP cardinality filter drops or waives the
    rows at its limit), compared bit for bit in d_survive and d_counts, with the parents split into two ranges;
  * inheritance tries the parents C \\ {b} from the highest b down, finds each by binary search in the sorted feasible
    list and takes the first witness slot that holds C: the chosen witness, the certified candidates and the number of
    parents tried must all agree.
Inputs: random sorted feasible lists (W = 1..4, mpQP and mpLP, levels with a single group, prefixes without a group) and
the real levels of golden programs."""
import bisect
import ctypes
import itertools
import os
import zlib

import numpy
import pytest

from conftest import GOLDEN

pytestmark = pytest.mark.gpu

SLOTS = 2   # PPGPU_WITNESS_SLOTS


def make_engine(path):
    from ppopt_b200 import engine
    from ppopt_b200.mplp_program import load_presolved
    prog = load_presolved(path)
    return prog, engine.Engine(engine.program_arrays(prog))


@pytest.fixture(scope='module')
def engines():
    made = {}

    def get(name):
        if name not in made:
            path = os.path.join(GOLDEN, name + '.npz')
            made[name] = make_engine(path if os.path.exists(path) else os.path.join(GOLDEN, 'envelope', name + '.npz'))
        return made[name]
    yield get
    for _, eng in made.values():
        eng.close()


def limits(prog):
    """(mi, ne, child_limit(k), sub_limit(k)) in inequality-row space; the limits are None for an mpQP"""
    m, n, ne = prog.num_constraints(), prog.num_x(), len(prog.equality_indices)
    if type(prog).__name__ != 'MPLP_Program':
        return m - ne, ne, None, None
    # a list of length L whose last element g is dropped iff g >= L + m - n (mpqp_combinatorial.py:40-42)
    return m - ne, ne, (lambda k: k + 1 + m - n), (lambda k: k + m - n)


def ref_children(feas, k, prog):
    """rows i of the surviving children of every parent, and whether a waived row occurred"""
    mi, _, child_limit, sub_limit = limits(prog)
    present = set(feas)
    out, waived_any = [], False
    for p in feas:
        rows = []
        for i in range((p[-1] if p else -1) + 1, mi):
            if child_limit is not None and i >= child_limit(k):
                continue
            waived = sub_limit is not None and i >= sub_limit(k)
            waived_any |= waived
            if waived or all(p[:j] + p[j + 1:] + (i,) in present for j in range(len(p))):
                rows.append(i)
        out.append(rows)
    return out, waived_any


def to_masks(eng, sets, ne):
    return eng.masks_from_lists([[ne + r for r in s] for s in sets])


def bits_of(row_words):
    """row indices set in one mask row (int64 words)"""
    return [w * 64 + b for w, x in enumerate(row_words.view(numpy.uint64).tolist()) for b in range(64) if (x >> b) & 1]


def prepare(eng, level_masks, feas_idx):
    import torch
    from ppopt_b200 import _lib
    nf = int(feas_idx.shape[0])
    feas_masks = eng.empty((nf, eng.W), torch.int64)
    ws_bytes = eng.lib.ppgpu_scan_workspace_bytes(nf)
    ws = eng.empty(((ws_bytes + 7) // 8,), torch.int64)
    _lib.check(eng.lib.ppgpu_children_prepare(eng.h, level_masks.data_ptr(), feas_idx.data_ptr(), nf, feas_masks.data_ptr(),
                                              ws.data_ptr(), ws_bytes, eng._stream()), 'prepare')
    return feas_masks, ws, ws_bytes


def check_k6(eng, prog, level, feas, k):
    """K6 through prepare / count_range (two ranges) / scan on a level whose feasible members are `feas`"""
    import torch
    from ppopt_b200 import _lib
    mi, ne, _, _ = limits(prog)
    pos = {s: i for i, s in enumerate(level)}
    feas_idx = torch.tensor([pos[s] for s in feas], dtype=torch.int64, device=eng.tdev)
    feas_masks, ws, ws_bytes = prepare(eng, to_masks(eng, level, ne), feas_idx)
    nf = len(feas)
    survive = torch.zeros((nf, eng.W), dtype=torch.int64, device=eng.tdev)
    counts = torch.zeros((nf + 1,), dtype=torch.int64, device=eng.tdev)
    eng.counters(reset=True)
    for lo, hi in ((0, nf // 3), (nf // 3, nf)):
        _lib.check(eng.lib.ppgpu_children_count_range(eng.h, feas_masks.data_ptr(), nf, k, survive.data_ptr(),
                                                      counts.data_ptr(), lo, hi, ws.data_ptr(), ws_bytes, eng._stream()),
                   'count_range')
    lookups = eng.counters()['k6_lookups']
    want, waived = ref_children(feas, k, prog)
    sv = survive.cpu().numpy()
    got = [bits_of(sv[p]) for p in range(nf)]
    assert got == want
    assert counts.cpu().tolist() == [len(r) for r in want] + [0]
    assert lookups <= k * nf   # one group probe per parent row at most
    tot = ctypes.c_int64(0)
    _lib.check(eng.lib.ppgpu_children_scan(eng.h, counts.data_ptr(), nf, ctypes.byref(tot), ws.data_ptr(), ws_bytes,
                                           eng._stream()), 'scan')
    assert tot.value == sum(len(r) for r in want)
    return feas_masks, ws, want, waived


def random_level(rng, mi, k, universe, drop):
    """all k-subsets of a random row universe less a fraction `drop`, plus as many random k-sets: sorted, so that many
    prefixes of size k - 1 have no group"""
    rows = sorted(rng.choice(mi, size=universe, replace=False).tolist())
    dense = [c for c in itertools.combinations(rows, k) if rng.random() >= drop]
    sparse = {tuple(sorted(rng.choice(mi, size=k, replace=False).tolist())) for _ in range(len(dense) + 1)}
    return sorted(set(dense) | sparse)


CASES = [   # (program, parent size k, rows in the universe)
    ('factory_mpqp', 1, 8), ('factory_mpqp', 3, 8),
    ('synthetic_30_6_40_s0', 1, 100), ('synthetic_30_6_40_s0', 2, 24), ('synthetic_30_6_40_s0', 4, 14),
    ('env_w3', 2, 30), ('env_w3', 5, 12),
    ('env_w4_r256', 3, 22), ('env_w4_r256', 6, 12),
    ('transport_mplp', 2, 8), ('rand_lp_4_2_8_s3', 3, 10),
    ('env_lp_w3', 1, 150), ('env_lp_w3', 3, 20),
]


@pytest.mark.parametrize('name,k,universe', CASES)
def test_k6_random_sorted_levels(engines, name, k, universe):
    prog, eng = engines(name)
    mi, _, child_limit, _ = limits(prog)
    rng = numpy.random.default_rng(zlib.crc32(f'{name} {k}'.encode()))
    level = random_level(rng, mi, k, min(universe, mi), 0.15)
    feas = [s for s in level if rng.random() < 0.9] or level[:1]
    _, _, want, waived = check_k6(eng, prog, level, feas, k)
    assert any(want), 'no parent has a surviving child: the case tests nothing'
    if child_limit is not None and k == 1:
        assert waived


@pytest.mark.parametrize('name', ['synthetic_30_6_40_s0', 'env_w4_r256', 'env_lp_w3'])
def test_k6_single_group_levels(engines, name):
    """level 1 (one group: the empty prefix) and a level-3 list whose members all share one prefix"""
    prog, eng = engines(name)
    mi = limits(prog)[0]
    rows = list(range(mi))
    check_k6(eng, prog, [(r,) for r in rows], [(r,) for r in rows if r % 7 != 3], 1)
    one = [(0, mi // 2, x) for x in range(mi // 2 + 1, mi)]
    check_k6(eng, prog, one, one[::2], 3)


@pytest.mark.parametrize('order', ['swapped', 'duplicate', 'mixed_cardinality'])
def test_k6_rejects_parents_out_of_level_order(engines, order):
    """the group index needs the level's lexicographic order: a selection that breaks it is an error, not wrong children"""
    import torch
    from ppopt_b200 import _lib
    prog, eng = engines('synthetic_30_6_40_s0')
    level = [(a, b) for a in range(12) for b in range(a + 1, 12)]
    sets = {'swapped': level[:40] + [level[41], level[40]] + level[42:], 'duplicate': level[:30] + level[29:],
            'mixed_cardinality': level[:20] + [(20,)] + level[20:]}[order]
    masks = to_masks(eng, sets, 0)
    feas_idx = torch.arange(len(sets), dtype=torch.int64, device=eng.tdev)
    with pytest.raises(RuntimeError, match='lexicographic order'):
        eng.children(masks, feas_idx, 2)
    # the split form reports it at the scan
    nf = len(sets)
    feas_masks, ws, ws_bytes = prepare(eng, masks, feas_idx)
    counts = torch.zeros((nf + 1,), dtype=torch.int64, device=eng.tdev)
    survive = torch.zeros((nf, eng.W), dtype=torch.int64, device=eng.tdev)
    _lib.check(eng.lib.ppgpu_children_count_range(eng.h, feas_masks.data_ptr(), nf, 2, survive.data_ptr(), counts.data_ptr(),
                                                  0, nf, ws.data_ptr(), ws_bytes, eng._stream()), 'count_range')
    tot = ctypes.c_int64(0)
    with pytest.raises(RuntimeError, match='lexicographic order'):
        _lib.check(eng.lib.ppgpu_children_scan(eng.h, counts.data_ptr(), nf, ctypes.byref(tot), ws.data_ptr(), ws_bytes,
                                               eng._stream()), 'scan')
    # the same level in order is accepted
    check_k6(eng, prog, level, level, 2)


@pytest.mark.parametrize('name', ['synthetic_30_6_40_s0', 'transport_mplp', 'env_lp_w3'])
def test_k6_real_levels(engines, name):
    """the levels a solve generates, with the feasibility the engine decides: K6 through the ABI against the sets"""
    from ppopt_b200._lib import ST_FEAS
    prog, eng = engines(name)
    mi, ne, _, _ = limits(prog)
    masks = eng.root_level()
    for k in range(1, 4):
        status = eng.level_eval(masks, k)
        level = [tuple(r - ne for r in s[ne:]) for s in eng.lists_from_masks(masks.cpu().numpy())]
        feas = [level[i] for i in eng.select(status, ST_FEAS, ST_FEAS).cpu().tolist()]
        if not feas:
            break
        check_k6(eng, prog, level, feas, k)
        masks = eng.children(masks, eng.select(status, ST_FEAS, ST_FEAS), k)


def ref_inherit(feas, wit_rows, cands, status):
    """(chosen (parent, slot) or None, parents tried) per candidate: parents C \\ {b} from the highest b down, each found by
    binary search in the sorted feasible list; the first slot whose witness holds C"""
    out, tried = [], 0
    for c, st in zip(cands, status):
        pick = None
        if (st & 1) and not (st & 2):
            cs = set(c)
            for b in reversed(c):
                s = tuple(x for x in c if x != b)
                if not s:
                    continue
                tried += 1
                e = bisect.bisect_left(feas, s)
                if e == len(feas) or feas[e] != s:
                    continue
                pick = next(((e, sl) for sl in range(SLOTS) if cs <= wit_rows[e][sl]), None)
                if pick:
                    break
        out.append(pick)
    return out, tried


@pytest.mark.parametrize('name,k,universe', [c for c in CASES if c[1] >= 2] + [('synthetic_30_6_40_s0', 'real', 0)])
def test_inherit_picks_parent_by_lexicographic_rank(engines, name, k, universe):
    import torch
    from ppopt_b200 import engine
    from ppopt_b200._lib import ST_FEAS
    prog, eng = engines(name)
    mi, ne, _, _ = limits(prog)
    rng = numpy.random.default_rng(zlib.crc32(f'{name} {k} inherit'.encode()))
    if k == 'real':
        masks = eng.root_level()
        for k in (1, 2):
            status = eng.level_eval(masks, k)
            if k == 2:
                break
            masks = eng.children(masks, eng.select(status, ST_FEAS, ST_FEAS), k)
        level = [tuple(r - ne for r in s[ne:]) for s in eng.lists_from_masks(masks.cpu().numpy())]
        feas = [level[i] for i in eng.select(status, ST_FEAS, ST_FEAS).cpu().tolist()]
    else:
        level = random_level(rng, mi, k, min(universe, mi), 0.15)
        feas = [s for s in level if rng.random() < 0.9]
    feas_masks, ws, want, _ = check_k6(eng, prog, level, feas, k)
    # candidates: every child K6 lets through, and (k+1)-sets with missing parents or parents outside every group
    cands = [p + (i,) for p, rows in zip(feas, want) for i in rows]
    rows_used = sorted({r for s in feas for r in s})
    extra = {tuple(sorted(rng.choice(rows_used, size=k + 1, replace=False).tolist())) for _ in range(len(cands) // 2 + 50)}
    cands += sorted(extra)
    # shuffled, and few enough that the vertex walk (which writes witnesses of its own) does not run
    cands = [cands[i] for i in rng.permutation(len(cands))[:20000]]
    # witnesses: each slot holds the parent and ~60 % of the other rows, or is empty (certified without a vertex)
    nf = len(feas)
    wit_rows = []
    for s in feas:
        wit_rows.append([set() if rng.random() < 0.25 else set(s) | {r for r in range(mi) if rng.random() < 0.6}
                         for _ in range(SLOTS)])
    pwit = to_masks(eng, [sorted(w) for ws_ in wit_rows for w in ws_], ne).reshape(nf, SLOTS, eng.W).contiguous()
    status_np = rng.choice(numpy.array([1, 1, 1, 1, 1, 1, 3, 0], dtype=numpy.uint8), size=len(cands))
    status = torch.from_numpy(status_np).to(eng.tdev)
    wout = torch.zeros((len(cands), SLOTS, eng.W), dtype=torch.int64, device=eng.tdev)
    pick, tried = ref_inherit(feas, wit_rows, cands, status_np.tolist())
    eng.counters(reset=True)
    eng.level_eval(to_masks(eng, cands, ne), k + 1, status, stages=2, witness=wout,
                   parent=engine.ParentLevel(feas_masks, ws, nf, pwit))
    c = eng.counters()
    assert c['inherited'] == sum(p is not None for p in pick)
    assert c['inherit_lookups'] == tried
    st, wo, pw = status.cpu().numpy(), wout.cpu().numpy(), pwit.cpu().numpy()
    for i, p in enumerate(pick):
        if p is None:
            assert not wo[i].any(), cands[i]
        else:
            assert st[i] & ST_FEAS, cands[i]
            assert numpy.array_equal(wo[i, 0], pw[p[0], p[1]]), (cands[i], p)
            assert not wo[i, 1].any()
    assert any(p is not None for p in pick) and any(p is None for p in pick)
