"""Region emission as three launches (K5a / K5b / K5c, csrc/k5_emit.cu) against the fused one-CTA-per-region kernel that
PPGPU_K5_FUSED=1 selects.

The split moves the redundancy LPs of all regions of a call into one batch with a warp per LP, and the duplicate test into a
kernel of its own; every LP is the same routine on the same inputs.  So the outputs must be identical to the byte: laws (of
every non-singular candidate; K5 leaves the laws of a singular one unwritten), rows, flags, info, the status bytes after
emission, and the k5 LP / pivot / work counters.  The switch is read once per process, so each variant runs in a child
process of its own (this file as a script) over the same cases:
  * every main golden program that has a region, level by level to its golden depth, and its equality-only base set
    (mpQP, mpLP, t = 1);
  * the stored candidates of the envelope programs (129-256 region rows, up to 14 parameters);
  * the sampled deep levels of the goldens that have regions there; the bench program's hold every region of those levels (4,041 at
    level 5: some 450 k LPs in one batch, many times what the device holds at once);
  * a batch of a single region."""
import os
import subprocess
import sys

import numpy
import pytest

from conftest import GOLDEN, ROOT, golden_names

ENVELOPE = os.path.join(GOLDEN, 'envelope')
SAMPLED = os.path.join(GOLDEN, 'sampled')


def _names(d):
    return sorted(f[:-4] for f in os.listdir(d) if f.endswith('.npz')) if os.path.isdir(d) else []


def _with_regions(d, names):
    """the programs whose stored levels hold a region (none do in rand_wide_40_8_90_s5's two golden levels or in the sampled
    levels 6 and 7 of mpc_n10): elsewhere there is nothing to compare"""
    return [n for n in names if int(numpy.load(os.path.join(d, n + '.npz'))['n_regions']) > 0]


def _goldens():
    return _with_regions(GOLDEN, golden_names())


def _sampled():
    return _with_regions(SAMPLED, _names(SAMPLED))


CASES = (['golden/' + n for n in _goldens()] + ['envelope/' + n for n in _names(ENVELOPE)] +
         ['sampled/' + n for n in _sampled()] + ['single_region'])
BENCH = 'synthetic_30_6_40_s0'


def run_all(out_path):
    """emits every case with the kernel the environment selects and saves what came back to out_path"""
    import torch
    from ppopt_b200 import engine
    from ppopt_b200._lib import ST_FEAS, ST_OPT
    from ppopt_b200.mplp_program import load_presolved
    from test_envelope import candidates, load
    res = {}

    def emit(eng, key, masks, sel, k_act, status):
        eng.counters(reset=True)
        l0 = eng.launch_count()
        laws, rows, flags, info = [x.cpu().numpy() for x in eng.emit(masks, sel, k_act, status)]
        c = eng.counters()
        laws[info[:, 0] < 0] = 0.0
        res.update({key + '|laws': laws, key + '|rows': rows, key + '|flags': flags, key + '|info': info,
                    key + '|status': status.cpu().numpy(),
                    key + '|k5': numpy.array([c['k5_lps'], c['k5_pivots'], c['k5_work']], dtype=numpy.uint64),
                    key + '|launches': numpy.array([eng.launch_count() - l0, eng.t])})

    def make(path):
        return engine.Engine(engine.program_arrays(load_presolved(path)))

    for name in _goldens():
        path = os.path.join(GOLDEN, name + '.npz')
        cap = int(numpy.load(path)['level_cap'])
        eng = make(path)
        depth = eng.max_depth if cap < 0 else min(cap, eng.max_depth)
        masks = eng.root_level()
        for lvl in range(depth):
            if masks.shape[0] == 0:
                break
            status = eng.level_eval(masks, lvl + 1)
            sel = eng.select(status, ST_OPT, ST_OPT)
            if sel.shape[0]:
                emit(eng, f'golden/{name}|{lvl + 1}', masks, sel, lvl + 1, status)
            if lvl + 1 < depth:
                masks = eng.children(masks, eng.select(status, ST_FEAS, ST_FEAS), lvl + 1)
        if cap < 0:
            m0 = torch.zeros((1, eng.W), dtype=torch.int64, device=eng.tdev)
            st0 = eng.level_eval(m0, 0)
            sel0 = eng.select(st0, ST_OPT, ST_OPT)
            if sel0.shape[0]:
                emit(eng, f'golden/{name}|0', m0, sel0, 0, st0)
        eng.close()
    for name in _names(ENVELOPE):
        g = load(name)
        eng = make(os.path.join(ENVELOPE, name + '.npz'))
        for k, (c, _) in candidates(g).items():
            masks = eng.masks_from_lists(c.tolist())
            status = eng.level_eval(masks, k)
            sel = eng.select(status, ST_OPT, ST_OPT)
            if sel.shape[0]:
                emit(eng, f'envelope/{name}|{k}', masks, sel, k, status)
        eng.close()
    for name in _sampled():
        s = numpy.load(os.path.join(SAMPLED, name + '.npz'))
        eng = make(os.path.join(GOLDEN, name + '.npz'))
        for lvl in s['levels'].tolist():
            masks = eng.masks_from_lists(s[f'level{lvl}_candidates'].tolist())
            status = eng.level_eval(masks, lvl + 1)
            sel = eng.select(status, ST_OPT, ST_OPT)
            if name == BENCH and lvl == 3:
                emit(eng, f'single_region|{lvl + 1}', masks, sel[:1], lvl + 1, status.clone())
            if sel.shape[0]:
                emit(eng, f'sampled/{name}|{lvl + 1}', masks, sel, lvl + 1, status)
        eng.close()
    numpy.savez(out_path, **res)


@pytest.fixture(scope='module')
def variants(tmp_path_factory):
    d = tmp_path_factory.mktemp('k5_batch')
    out = {}
    for name, fused in (('fused', '1'), ('split', '0')):
        path = str(d / (name + '.npz'))
        env = dict(os.environ, PPGPU_K5_FUSED=fused)
        subprocess.run([sys.executable, os.path.abspath(__file__), path], env=env, cwd=ROOT, check=True, timeout=3600)
        out[name] = dict(numpy.load(path))
    return out


@pytest.mark.gpu
@pytest.mark.parametrize('case', CASES)
def test_split_emission_equals_fused(variants, case):
    fused, split = variants['fused'], variants['split']
    keys = sorted(k for k in fused if k.split('|')[0] == case)
    assert keys, f'{case}: no region was emitted'
    assert keys == sorted(k for k in split if k.split('|')[0] == case)
    for k in keys:
        if k.endswith('|launches'):
            n, t = fused[k].tolist()
            assert n == 1, (k, 'the fused kernel did not run')
            assert split[k].tolist() == [1 if t == 1 else 3, t], (k, 'the three-launch path did not run')
            continue
        a, b = fused[k], split[k]
        assert a.dtype == b.dtype and a.shape == b.shape, k
        assert a.tobytes() == b.tobytes(), (k, int(numpy.count_nonzero(a.view(numpy.uint8) != b.view(numpy.uint8))))


@pytest.mark.gpu
def test_bench_batch_spans_several_waves(variants):
    import torch
    sms = torch.cuda.get_device_properties(0).multi_processor_count
    lps = int(variants['split'][f'sampled/{BENCH}|5|k5'][0])
    assert lps > 8 * sms * 16, (lps, sms)


if __name__ == '__main__':
    run_all(sys.argv[1])
