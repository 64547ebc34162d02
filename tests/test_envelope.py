"""Envelope programs (tests/golden/envelope, oracle/gen_envelope_golden.py) on the CPU: each program sits where the dispatch
table below says, its candidates cover every outcome in every listed band of active-row counts, and the CPU twin of the
batched algorithms (oracle/twin.cpp) agrees with the oracle's stored verdicts and regions.  No GPU needed.

Dispatch table (what each program's sizes select; csrc/api.cu::ppgpu_program_create accepts m - n_eq <= 256,
(m - n_eq) + q <= 256, n - n_eq + t + 2 <= 64, t <= 14, n - n_eq <= 64):
  NP       K1 register width, the smallest of 8/16/32/64 >= n' = n - n_eq
  R0       region rows (m - n_eq) + q: K2 rows per warp, K3/K4/K5 rows per lane RPT = 1/2/4/8 for R0 <= 32/64/128/256
  W        mask words ceil((m - n_eq) / 64): K6 key width, K1..K5 mask decoding
  K2 cols  n' + t + 2 padded to 8/16/24/32/40/48/64 (feasibility tableau, K2 and K2w)
  DCV      K3/K4/K5 theta columns, 8 for t + 2 <= 8, else 16
and the bands of k' (active inequality rows) in which each program's golden holds rank-deficient, infeasible, feasible
and region candidates: k' <= 8 the K1 prefilters, 9-16 the K1 group-16 kernel, > 16 one warp per candidate; K2a's register
form up to 8, its generic form up to 32, nothing above; K2w's prefix k' - 2 <= 30."""
import os
import sys

import numpy
import pytest

from conftest import GOLDEN, ROOT
from parity import (MARGIN_BAND, REL_TOL, check_status_bits, golden_regions, index_lists_match, rel_err,
                    rows_match_as_sets)

sys.path.insert(0, os.path.join(ROOT, 'oracle'))
import twin_binding  # noqa: E402

ENVELOPE = os.path.join(GOLDEN, 'envelope')
BANDS = ((1, 2), (3, 4), (5, 6), (7, 8), (9, 16), (17, 30), (31, 32), (33, 64))
RADIUS, RADIUS_BAND, FEAS_BAND = 1e-8, 1e-7, 1e-7   # csrc/tolerances.h PPG_RADIUS, PPG_RADIUS_BAND, PPG_FEAS_TOL

# name: n', R0, W, K2 columns, DCV, NP, bands with all four outcomes
TABLE = {
    'env_np9_r33': (9, 33, 1, 16, 8, 16, [(3, 4), (5, 6), (7, 8), (9, 16)]),
    'env_np16_r64': (16, 64, 1, 24, 8, 16, [(3, 4), (5, 6), (7, 8), (9, 16)]),
    'env_np17_w2': (17, 79, 2, 32, 16, 32, [(3, 4), (5, 6), (7, 8), (9, 16)]),
    'env_np33_r129': (33, 129, 2, 40, 8, 64, [(7, 8), (9, 16), (17, 30)]),
    'env_w3': (32, 212, 3, 48, 16, 32, [(3, 4), (7, 8), (9, 16), (17, 30)]),
    'env_w4_r256': (48, 256, 4, 64, 16, 64, [(3, 4), (9, 16), (17, 30), (31, 32), (33, 64)]),
    'env_np60': (60, 254, 4, 64, 8, 64, [(3, 4), (9, 16), (17, 30), (33, 64)]),
    'env_eq35': (35, 100, 2, 48, 8, 64, [(3, 4), (7, 8), (9, 16), (17, 30)]),
    'env_lp_w3': (12, 160, 3, 24, 8, 16, [(9, 16)]),
    'env_full_np9': (9, 16, 1, 16, 8, 16, [(3, 4), (5, 6), (7, 8)]),
}
NAMES = sorted(TABLE)


def load(name):
    return numpy.load(os.path.join(ENVELOPE, name + '.npz'))


def candidates(g):
    """{k': (candidate index lists int32 array, oracle status bytes)}"""
    return {int(k): (g[f'k{k}_candidates'], g[f'k{k}_status']) for k in g['k_values']}


def band_of(k):
    return next(b for b in BANDS if b[0] <= k <= b[1])


def twin(name):
    return twin_binding.Twin.from_npz(os.path.join(ENVELOPE, name + '.npz'))


def rank_band(aux):
    """the twin's QR pivot ratio lies in the borderline band (PPG_RANK_BORDER_LO, PPG_RANK_BORDER_HI): the twin keeps the
    QR verdict there, the engine re-decides by singular values (csrc/k1_rank.cu) as numpy.linalg.matrix_rank does"""
    return (aux[:, 0] > 1e-15) & (aux[:, 0] < 1e-7)


def lp_band(st, aux):
    """the twin's feasibility margin (rank-full candidates) or Chebyshev radius (feasible ones) lies inside the documented
    tolerance band of its threshold"""
    return (((st & 1) != 0) & (numpy.abs(aux[:, 1]) < FEAS_BAND)) | \
        (((st & 2) != 0) & (numpy.abs(aux[:, 2] - RADIUS) < RADIUS_BAND))


def pad_columns(c):
    return next(o for o in (8, 16, 24, 32, 40, 48, 64) if c <= o)


@pytest.mark.parametrize('name', NAMES)
def test_program_lands_on_its_dispatch_cell(name):
    g = load(name)
    n, t, m, ne, q = g['A'].shape[1], g['F'].shape[1], g['A'].shape[0], int(g['n_eq']), g['A_t'].shape[0]
    npr, R0, W, cols, dcv, NP, _ = TABLE[name]
    assert n - ne == npr
    assert (m - ne) + q == R0
    assert -(-(m - ne) // 64) == W
    assert pad_columns(n - ne + t + 2) == cols
    assert (8 if t + 2 <= 8 else 16) == dcv
    assert next(p for p in (8, 16, 32, 64) if npr <= p) == NP
    assert numpy.all(numpy.linalg.eigvalsh(g['Q']) > 0.5) or str(g['kind']) == 'lp'
    # dependent rows sit at the word boundaries and really are combinations of their parents
    for r, par, delta in zip(g['dep_rows'], g['dep_parents'], g['dep_delta']):
        par = [p for p in par if p >= 0]
        assert (r - ne) in (63, 64, 127, 128, 191, 192, 255) or (r == len(g['A']) - 1 and r - ne < 63)
        resid = numpy.linalg.lstsq(g['A'][par].T, g['A'][r], rcond=None)[1]
        assert float(numpy.sqrt(resid.sum())) <= 10 * delta + 1e-14


@pytest.mark.parametrize('name', NAMES)
def test_bands_hold_every_outcome(name):
    g = load(name)
    seen = {}
    for k, (c, st) in candidates(g).items():
        kinds = seen.setdefault(band_of(k), set())
        for s in st:
            kinds.add('rank' if not s & 1 else 'infeasible' if not s & 2 else 'region' if s & 8 else 'feasible')
    for b in TABLE[name][6]:
        assert seen.get(b) == {'rank', 'infeasible', 'feasible', 'region'}, (name, b, seen.get(b))
    assert sum(len(c) for c, _ in candidates(g).values()) <= 160


@pytest.mark.parametrize('name', NAMES)
def test_twin_matches_oracle_verdicts(name):
    """bits & 11 agree except (a) rank decisions in the QR band, which the dependent rows with noise 1e-13 produce on
    purpose (the oracle, like the reference, decides by singular values), and (b) decisions inside the LP tolerance
    bands, which must stay rare"""
    g = load(name)
    tw = twin(name)
    n_band = n_all = 0
    for k, (c, ref) in candidates(g).items():
        st, aux = tw.eval(tw.masks(c.tolist()), aux=True)
        bad = numpy.nonzero((st & 11) != (ref & 11))[0]
        by_rank = rank_band(aux) & ((st & 1) != (ref & 1))
        by_lp = lp_band(st, aux)
        assert all(by_rank[i] or by_lp[i] for i in bad), \
            (name, k, [(c[i].tolist(), int(st[i]), int(ref[i])) for i in bad if not (by_rank[i] or by_lp[i])][:3])
        for i in bad:
            if by_rank[i]:
                assert any(r in c[i] and d == 1e-13 for r, d in zip(g['dep_rows'], g['dep_delta'])), (name, c[i].tolist())
            else:
                n_band += 1
        n_all += len(c)
    assert n_band <= 0.02 * n_all, (name, n_band, n_all)


@pytest.mark.parametrize('name', NAMES)
def test_twin_emit_matches_oracle_regions(name):
    g = load(name)
    tw = twin(name)
    n, ne, m = tw.n, tw.n_eq, tw.m
    regions = golden_regions(g)
    assert regions
    for r in regions:
        aset = r['active_set'].tolist()
        rc, laws, rows, flags, info, mg = tw.emit(tw.masks([aset])[0], margins=True)
        assert rc == 1, (name, aset)
        assert rel_err(laws[:n, 1:], r['A']) <= REL_TOL and rel_err(laws[:n, :1], r['b']) <= REL_TOL, (name, aset)
        assert rel_err(laws[n:, 1:], r['C']) <= REL_TOL and rel_err(laws[n:, :1], r['d']) <= REL_TOL, (name, aset)
        sel = [i for i in range(len(flags)) if (flags[i] & 3) == 3 and not (flags[i] & 4)]
        u1, u2 = rows_match_as_sets(rows[sel, 1:], rows[sel, :1], r['E'], r['f'])
        band = [i for i in range(len(flags)) if (flags[i] & 1) and abs(mg[i]) < MARGIN_BAND]
        assert all(numpy.min(numpy.abs(rows[band][:, 1:] - u[:-1]).max(1) + numpy.abs(rows[band][:, 0] - u[-1])) <= 1e-7
                   for u in u1 + u2) if band else not (u1 or u2), (name, aset)
        kept = [i for i in range(len(flags)) if (flags[i] & 1) and mg[i] >= -1e-9]
        k_act = len(aset) - ne
        n_inact = m - len(aset)
        inactive = [i for i in range(m) if i not in set(aset)]
        mine = type('R', (), dict(active_set=aset, omega_set=[i - k_act - n_inact for i in kept if i >= k_act + n_inact],
                                  lambda_set=[aset[ne + i] for i in kept if i < k_act],
                                  regular_set=[[i - k_act for i in kept if k_act <= i < k_act + n_inact],
                                               [inactive[i - k_act] for i in kept if k_act <= i < k_act + n_inact]]))
        bad = index_lists_match(mine, r, margins=mg, k_act=k_act, n_eq=ne, m=m)
        assert not bad, (name, aset, bad[:3])


def test_full_solve_is_stored_and_consistent():
    """env_full_np9 holds the oracle's complete enumeration to depth 9: every level's candidates in the reference's
    lexicographic order, and the region list equals the regions of its region-bit candidates"""
    g = load('env_full_np9')
    L = int(g['full_levels'])
    assert L == 9
    n_reg = 0
    for lv in range(L):
        c = g[f'full_level{lv}_candidates'].tolist()
        assert c == sorted(c) and all(len(x) == lv + 1 for x in c)
        n_reg += int((g[f'full_level{lv}_status'] & 8 != 0).sum())
    full = {k[5:]: g[k] for k in g.files if k.startswith('full_')}
    regions = golden_regions(full)
    # the equality-only active set is tested last, after the levels (mpqp_combinatorial.py:65-70)
    assert len(regions) == n_reg + 1 and len(regions[-1]['active_set']) == 0
    tw = twin('env_full_np9')
    for lv in range(L):
        st = tw.eval(tw.masks(g[f'full_level{lv}_candidates'].tolist()))
        check_status_bits(st, g[f'full_level{lv}_status'], f'env_full_np9 level {lv + 1}')
