"""The engine's kernels across their whole dispatch envelope (tests/golden/envelope, table in tests/test_envelope.py): active
sets deeper than 8, 129-256 region rows, up to 14 parameters, four mask words, working sets of more than 32 rows.

1. Each program selects the instantiation the table says (ppgpu_program_info), and the counters show which certificate
   kernels ran: the vertex walk K2w wherever k' - 2 <= 30, the relaxation K2a wherever k' <= 32, the simplex K2 always.
2. Status bits of every stored candidate: the rank bit equals numpy's matrix_rank, dependent-row decisions inside the QR
   band are flagged ST_BORDER, bits & 11 equal the CPU twin's, and all bits equal the oracle's stored verdicts.
3. Certificates never change a decision: walk forced on, default, and simplex only give identical status bytes.
4. K5 on every candidate the oracle calls a region: laws, [E|f] as row sets and kept-index lists against the oracle.
5. K6 with 3 and 4 mask words against the reference's set arithmetic under arbitrary feasibility patterns.
6. K8 against the CPU twin at seeded theta, including working sets of more than 32 rows and a G too large to stage.
7. One complete enumeration to depth 9 (env_full_np9) against the oracle's."""
import os
import sys

import numpy
import pytest

from conftest import ROOT
from parity import (MARGIN_BAND, REL_TOL, check_status_bits, golden_regions, index_lists_match, masks_to_lists, rel_err,
                    rows_match_as_sets)
from test_envelope import BANDS, ENVELOPE, NAMES, TABLE, candidates, load, rank_band, twin
from test_gpu_solve_theta import kkt_batch
from test_solve_theta_twin import QP_INFEASIBLE, QP_OPTIMAL

pytestmark = pytest.mark.gpu
sys.path.insert(0, os.path.join(ROOT, 'oracle'))

QP_NAMES = [n for n in NAMES if str(numpy.load(os.path.join(ENVELOPE, n + '.npz'))['kind']) == 'qp']
RANK_BORDER = (1e-14, 1e-9)   # noise levels whose rank decision falls inside the QR band (csrc/tolerances.h, PPG_RANK_*)


def engine_for(name):
    from ppopt_b200 import engine
    from ppopt_b200.mplp_program import load_presolved
    prog = load_presolved(os.path.join(ENVELOPE, name + '.npz'))
    return engine, prog, engine.Engine(engine.program_arrays(prog))


def eval_all(eng, g, stages=7):
    """{k': status bytes of every stored candidate of that cardinality}, K5 run on the optimal ones (region bit)"""
    from ppopt_b200._lib import ST_OPT
    out = {}
    for k, (c, _) in candidates(g).items():
        masks = eng.masks_from_lists(c.tolist())
        status = eng.level_eval(masks, k, stages=stages)
        opt = eng.select(status, ST_OPT, ST_OPT)
        if opt.shape[0]:
            eng.emit(masks, opt, k, status)
        out[k] = status.cpu().numpy()
    return out


@pytest.mark.parametrize('name', NAMES)
def test_intended_instantiation_runs(name):
    from ppopt_b200._lib import OPT_K2W_MIN
    g = load(name)
    npr, R0, W, cols, _, _, _ = TABLE[name]
    engine, prog, eng = engine_for(name)
    assert (eng.W, eng.R0, eng.lp_columns, eng.use_gram) == (W, R0, cols, str(g['kind']) == 'qp')
    report = {}
    for walk in (False, True):
        if walk:
            eng.set_option(OPT_K2W_MIN, 0)
        for k, (c, _) in candidates(g).items():
            eng.counters(reset=True)
            eng.level_eval(eng.masks_from_lists(c.tolist()), k)
            report[(walk, k)] = eng.counters()
    has_walk = eng.has_walk_vertex
    eng.close()
    # per band of k': K2 solves LPs, K2a is tried up to k' = 32, the walk (given a start vertex) pivots while its prefix of
    # k' - 2 rows fits in 30; counted over the cardinalities that hold full-rank candidates
    full_rank = [k for k, (_, st) in candidates(g).items() if (st & 1).any()]
    assert sum(report[(False, k)]['k2_lps'] for k in full_rank) > 0, name
    for lo, hi in BANDS:
        ks = [k for k in full_rank if lo <= k <= hi]
        if not ks or hi > 32:
            continue
        assert sum(report[(False, k)]['k2a_tried'] for k in ks) > 0, (name, (lo, hi))
        if has_walk:
            assert sum(report[(True, k)]['k2w_pivots'] for k in ks) > 0, (name, (lo, hi))


@pytest.mark.parametrize('name', NAMES)
def test_status_bits_match_numpy_twin_and_oracle(name):
    from ppopt_b200._lib import ST_BORDER, ST_RANK
    g = load(name)
    engine, prog, eng = engine_for(name)
    tw = twin(name)
    A, ne = g['A'], int(g['n_eq'])
    dep = {int(r): ([int(p) for p in par if p >= 0], float(d)) for r, par, d in zip(g['dep_rows'], g['dep_parents'], g['dep_delta'])}
    got = eval_all(eng, g)
    for k, (c, ref) in candidates(g).items():
        st = got[k]
        want = numpy.array([numpy.linalg.matrix_rank(A[a]) == len(a) for a in c])
        bad = numpy.nonzero(((st & ST_RANK) != 0) != want)[0]
        assert not len(bad), (name, k, [c[i].tolist() for i in bad[:3]])
        for i, a in enumerate(c.tolist()):
            for r, (par, d) in dep.items():
                if r in a and set(par) <= set(a) and RANK_BORDER[0] < d <= RANK_BORDER[1] and k <= eng.n - ne:
                    assert st[i] & ST_BORDER, (name, a, r, d)
        # the twin keeps the QR verdict inside the rank band; the kernel re-decides by singular values (checked above)
        tst, aux = tw.eval(tw.masks(c.tolist()), aux=True)
        bad = numpy.nonzero(((st & 11) != (tst & 11)) & ~(rank_band(aux) & ((st & 1) != (tst & 1))))[0]
        assert not len(bad), (name, k, 'twin', [(c[i].tolist(), int(st[i]), int(tst[i])) for i in bad[:3]])
        check_status_bits(st, ref, f'{name} k={k}')
    eng.close()


@pytest.mark.parametrize('name', NAMES)
def test_certificate_kernels_never_change_a_decision(name):
    from ppopt_b200._lib import OPT_K2W_MIN
    g = load(name)
    engine, prog, eng = engine_for(name)
    default = eval_all(eng, g)
    simplex = eval_all(eng, g, stages=7 | 8)
    eng.set_option(OPT_K2W_MIN, 0)
    walked = eval_all(eng, g)
    eng.close()
    for k in default:
        assert numpy.array_equal(default[k], walked[k]), (name, k, 'walk')
        assert numpy.array_equal(default[k], simplex[k]), (name, k, 'simplex only')


@pytest.mark.parametrize('name', NAMES)
def test_k5_regions_match_oracle(name):
    import torch
    from ppopt_b200.critical_region import CriticalRegion
    g = load(name)
    engine, prog, eng = engine_for(name)
    tw = twin(name)
    ne, m = eng.n_eq, prog.num_constraints()
    ref_by = {tuple(r['active_set'].tolist()): r for r in golden_regions(g)}
    n_cmp = 0
    for k, (c, st) in candidates(g).items():
        pick = numpy.nonzero(st & 8)[0]
        if not len(pick):
            continue
        asets = [c[i].tolist() for i in pick]
        masks = eng.masks_from_lists(asets)
        status = torch.full((len(asets),), 7, dtype=torch.uint8, device=eng.tdev)
        sel = torch.arange(len(asets), dtype=torch.int64, device=eng.tdev)
        laws, rows, flags, info = [x.cpu().numpy() for x in eng.emit(masks, sel, k, status)]
        regs = engine.build_regions(eng, CriticalRegion, asets, k, laws, rows, flags, info)
        for si, (a, reg) in enumerate(zip(asets, regs)):
            rc, _, trows, tflags, _, mg = tw.emit(tw.masks([a])[0], margins=True)
            assert (info[si, 0] == 1.0) == (rc == 1), (name, a, info[si, 0], rc)
            assert reg is not None, (name, a)
            b = ref_by[tuple(a)]
            for fld in 'AbCd':
                assert rel_err(getattr(reg, fld), b[fld]) <= REL_TOL, (name, a, fld)
            u1, u2 = rows_match_as_sets(reg.E, reg.f, b['E'], b['f'])
            band = trows[[i for i in range(len(tflags)) if (tflags[i] & 1) and abs(mg[i]) < MARGIN_BAND]]
            for r in u1 + u2:
                d = numpy.max(numpy.abs(band[:, 1:] - r[:-1]), axis=1) + numpy.abs(band[:, 0] - r[-1]) if len(band) else [1.0]
                assert numpy.min(d) <= 1e-7, (name, a, 'E/f row differs outside the margin band')
            bad = index_lists_match(reg, b, margins=mg, k_act=k, n_eq=ne, m=m)
            assert not bad, (name, a, bad[:3])
            n_cmp += 1
    assert n_cmp == len(ref_by)
    eng.close()


class SubsetTester:
    """CombinationTester.check (a candidate is pruned iff it contains a stored combination) by hashing the candidate's
    subsets instead of scanning the combinations: the same set arithmetic, fast enough for 10^5 candidates.  Checked
    against CombinationTester itself on the first two levels below."""

    def __init__(self):
        self.combos, self.sizes = set(), set()

    def add_combo(self, c):
        self.combos.add(tuple(c))
        self.sizes.add(len(c))

    def check(self, c):
        import itertools
        return not any(s in self.combos for k in self.sizes if k <= len(c) for s in itertools.combinations(c, k))


@pytest.mark.parametrize('name', ['env_w3', 'env_w4_r256'])
def test_k6_three_and_four_words_match_reference_set_arithmetic(name):
    """next-level generation + superset pruning with W = 3 and 4 mask words under an arbitrary pseudo-random 'feasible'
    predicate, as test_gpu_properties.test_k6_matches_reference_set_arithmetic_for_arbitrary_feasibility does for W <= 2;
    the predicate is thinned at level 1 so that level 3 stays large and keeps rows of every word"""
    import torch
    from ppopt_b200.mp_solvers.solver_utils import CombinationTester, generate_children_sets
    engine, prog, eng = engine_for(name)
    m, ne = prog.num_constraints(), len(prog.equality_indices)
    assert eng.W == TABLE[name][2] >= 3
    rng = numpy.random.default_rng(5)
    tester, ref_tester = SubsetTester(), CombinationTester()
    to_check = generate_children_sets(prog.equality_indices, m, tester)
    masks = eng.root_level()
    for level in range(1, 4):
        assert masks_to_lists(masks.cpu().numpy(), ne) == to_check, f'{name} level {level}'
        keep_p = (0.4, 0.9, 0.2)[level - 1]   # 3,000-4,000 candidates at level 2, 50,000-90,000 at level 3
        feas = rng.random(len(to_check)) < keep_p
        status = torch.from_numpy(numpy.where(feas, 3, 1).astype(numpy.uint8)).to(eng.tdev)
        feasible = []
        for c, ok in zip(to_check, feas):
            if ok:
                feasible.append(c)
            else:
                tester.add_combo(c)
                if level == 1:
                    ref_tester.add_combo(c)
        nxt = []
        for c in feasible:
            nxt.extend(generate_children_sets(c, m, tester))
        if level == 1:
            assert nxt == [x for c in feasible for x in generate_children_sets(c, m, ref_tester)]
        idx = eng.select(status, 2, 2)
        assert idx.cpu().tolist() == numpy.nonzero(feas)[0].tolist()
        masks = eng.children(masks, idx, level)
        to_check = nxt
    # the children of level 3 as well; they hold rows of the last word
    last = masks.cpu().numpy()
    assert masks_to_lists(last, ne) == to_check and len(to_check) > 500
    assert numpy.any(last.view(numpy.uint64)[:, eng.W - 1] != 0)
    eng.close()


def k8_stage_g(mi):
    """csrc/k8_theta_qp.cu::launch_theta_qp stages G (mi x mi doubles) in shared memory only when it fits with four warps'
    scratch in the 227 KB a block may opt in to: never for mi >= 170"""
    return mi < 170


@pytest.mark.parametrize('name', QP_NAMES)
def test_k8_matches_twin(name):
    from gen_envelope_golden import theta_samples
    from ppopt_b200.mplp_program import load_presolved
    from ppopt_b200.solve_theta import ThetaSolver
    from twin_theta_qp import ThetaQpTwin
    g = load(name)
    path = os.path.join(ENVELOPE, name + '.npz')
    thetas = theta_samples(g['F'].shape[1], 20000, numpy.random.default_rng(17))
    ref = ThetaQpTwin.from_npz(path).theta_qp(thetas)
    out = ThetaSolver(load_presolved(path)).solve_batch(thetas)
    got = dict(status=out['status'].cpu().numpy(), x=out['x'].cpu().numpy(), dual=out['dual'].cpu().numpy(),
               mask=out['active'].cpu().numpy().view(numpy.uint64), iters=out['iters'].cpu().numpy())
    sure = ref['margin'] > 1e-9
    assert sure.mean() > 0.5, (name, sure.mean())
    for f in ('status', 'iters'):
        bad = numpy.nonzero(sure & (got[f] != ref[f]))[0]
        assert not len(bad), (name, f, thetas[bad[:3]], got[f][bad[:3]], ref[f][bad[:3]])
    bad = numpy.nonzero(sure & (got['mask'] != ref['mask']).any(1))[0]
    assert not len(bad), (name, 'mask', thetas[bad[:3]])
    both = (got['status'] == QP_OPTIMAL) & (ref['status'] == QP_OPTIMAL) & sure
    dx = numpy.abs(got['x'][both] - ref['x'][both]).max(1, initial=0.0) / numpy.maximum(1.0, numpy.abs(ref['x'][both]).max(1, initial=0.0))
    assert dx.max(initial=0.0) <= 1e-10, (name, dx.max())
    assert set(numpy.unique(got['status']).tolist()) <= {QP_OPTIMAL, QP_INFEASIBLE}, name
    opt = got['status'] == QP_OPTIMAL
    k = kkt_batch(g, thetas[opt], got['x'][opt], got['dual'][opt])
    assert k.max(initial=0.0) <= 1e-9, (name, k.max())
    sizes = numpy.unpackbits(got['mask'].view(numpy.uint8), axis=1).sum(1)
    if name in ('env_w4_r256', 'env_np60'):
        assert (sizes > 32).sum() >= 50, (name, sizes.max())   # the drop's second-lane branch (working set > 32 rows)
    assert k8_stage_g(g['A'].shape[0] - int(g['n_eq'])) == (name not in ('env_w3', 'env_w4_r256', 'env_np60'))


def test_complete_solve_past_depth_eight():
    """engine.solve to depth 9 on env_full_np9 against the oracle's complete enumeration: same regions in the same order"""
    from ppopt_b200 import engine
    from ppopt_b200.mplp_program import load_presolved
    g = load('env_full_np9')
    full = {k[5:]: g[k] for k in g.files if k.startswith('full_')}
    ref = golden_regions(full)
    prog = load_presolved(os.path.join(ENVELOPE, 'env_full_np9.npz'))
    sol = engine.solve(prog, max_levels=int(g['full_levels']), collect_status=True)
    for lv, (masks, st) in enumerate(sol.level_status):
        assert masks_to_lists(masks, 0) == g[f'full_level{lv}_candidates'].tolist(), f'level {lv + 1}'
        check_status_bits(st, g[f'full_level{lv}_status'], f'level {lv + 1}')
    got = sol.critical_regions
    assert [list(r.active_set) for r in got] == [r['active_set'].tolist() for r in ref]
    for a, b in zip(got, ref):
        for fld in 'AbCd':
            assert rel_err(getattr(a, fld), b[fld]) <= REL_TOL, (a.active_set, fld)
        u1, u2 = rows_match_as_sets(a.E, a.f, b['E'], b['f'])
        assert not u1 and not u2, a.active_set


def test_k5_first_launch_just_below_the_default_shared_memory():
    """env_w3 at k' = 6 asks K5 for 48,496 bytes of dynamic shared memory, less than the 49,152 a block gets without the
    opt-in; with the kernel's static arrays it is more.  The first emission in a fresh process (nothing opted the kernel in before) must
    succeed and agree with the oracle."""
    import subprocess
    code = f'''
import sys
sys.path[:0] = {[os.path.join(ROOT, 'tests'), ROOT]!r}
import numpy, torch
from test_envelope import ENVELOPE, candidates, load
from ppopt_b200 import engine
from ppopt_b200.mplp_program import load_presolved
g = load('env_w3')
c, ref = candidates(g)[6]
eng = engine.Engine(engine.program_arrays(load_presolved(ENVELOPE + '/env_w3.npz')))
masks = eng.masks_from_lists(c.tolist())
status = eng.level_eval(masks, 6)
eng.emit(masks, eng.select(status, 4, 4), 6, status)
st = status.cpu().numpy()
assert (st & 8).any() and numpy.array_equal(st & 11, ref & 11), (st, ref)
'''
    r = subprocess.run([sys.executable, '-c', code], capture_output=True, text=True, cwd=ROOT)
    assert r.returncode == 0, r.stderr[-2000:]
