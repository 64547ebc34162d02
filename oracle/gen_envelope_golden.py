"""Envelope golden vectors: seeded synthetic programs at the edges of the kernels' dispatch table, and the ORACLE's verdicts
on candidates of every active-set band they reach.

TEST INFRASTRUCTURE.  python oracle/gen_envelope_golden.py [name ...]   (GOLDEN_PROCS worker processes, default 8)

These goldens are the verdicts of oracle/ppopt_oracle.py (numpy + HiGHS), NOT of the unmodified reference: the reference
cannot be run at these sizes in useful time.  The oracle itself is pinned to the reference's own outputs by
tests/test_oracle.py.

Each program (PROGRAMS below) is built from its seed alone, presolved as given (no constructor presolve):
  * Q is SPD and well conditioned (eigenvalues in [1, 3]), Theta is the box |theta_j| <= 1 (q = 2 t);
  * b > |F| theta on Theta, so x = 0 is feasible everywhere, and H is scaled so that the optimal active sets of theta in
    Theta spread over the program's band of active-row counts k';
  * rows at the word boundaries 63/64, 127/128, 191/192 and 255 of the inequality rows are convex combinations of two or
    three earlier rows with relative noise delta in {0, 1e-13, 1e-9, 1e-4} (rank decisions at every noise level, masks
    whose bits straddle two words).
Candidates, per band of k' (BANDS), come from four sources: (a) optimal active sets of seeded theta (tests/twin_theta_qp.py
for an mpQP, HiGHS for an mpLP: used only to generate them), (b) one row added to, removed from and swapped in each of
those, (c) random subsets of every size, (d) a dependent row with its parents plus random rows.  The golden stores a
seeded sample of at most SAMPLE candidates per program (drawn from POOL evaluated ones, the four outcomes of a band in
turn, the region matrices within REGION_BYTES) with the oracle's status bits (1 rank, 2 feasible, 4 optimal,
8 region, as in the level goldens) and every region that sample produces, in the compact layout tests/parity.py reads.
env_full_np9 also stores oracle.solve(P) to depth 9: every level's candidates and status bytes and every region.

Deterministic: the same command rewrites byte-identical files (fixed seeds, sorted candidate lists, zip members without
time stamps)."""
import io
import os
import sys
import time
import zipfile

import numpy
from scipy.optimize import linprog

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
sys.path.insert(0, HERE)
sys.path.insert(0, os.path.join(ROOT, 'tests'))

import ppopt_oracle as oracle  # noqa: E402

OUT = os.path.join(ROOT, 'tests', 'golden', 'envelope')
BANDS = ((1, 2), (3, 4), (5, 6), (7, 8), (9, 16), (17, 30), (31, 32), (33, 64))
DELTAS = (0.0, 1e-13, 1e-9, 1e-4)
BOUNDARY_ROWS = (63, 64, 127, 128, 191, 192, 255)   # inequality-row indices (bit positions of the candidate masks)
SAMPLE = 150   # stored candidates per program
POOL = 480     # candidates evaluated by the oracle per program, the sample is drawn from them
REGION_BYTES = 240_000   # stored region matrices per program: keeps every golden file under half a megabyte

# name: n, n_eq, t, m - n_eq, H scale, seed, is_qp
PROGRAMS = {
    'env_np9_r33': (9, 0, 3, 27, 14.0, 101, True),
    'env_np16_r64': (16, 0, 6, 52, 8.0, 102, True),
    'env_np17_w2': (20, 3, 7, 65, 8.0, 103, True),
    'env_np33_r129': (33, 0, 4, 121, 16.0, 104, True),
    'env_w3': (40, 8, 10, 192, 10.0, 105, True),
    'env_w4_r256': (48, 0, 14, 228, 10.0, 106, True),
    'env_np60': (60, 0, 2, 250, 40.0, 107, True),
    'env_eq35': (45, 10, 5, 90, 12.0, 108, True),
    'env_lp_w3': (12, 0, 5, 150, 1.0, 109, False),
    'env_full_np9': (9, 0, 2, 12, 10.0, 110, True),
}
FULL_SOLVE = {'env_full_np9': 9}


def build_program(name):
    """the program's arrays (post-presolve layout of the level goldens) and the dependent rows: {row: (parents, delta)}"""
    n, ne, t, mi, hs, seed, is_qp = PROGRAMS[name]
    rng = numpy.random.default_rng(seed)
    m = ne + mi
    A = rng.normal(size=(m, n))
    A /= numpy.linalg.norm(A, axis=1, keepdims=True)
    F = 0.3 * rng.normal(size=(m, t)) / numpy.sqrt(t)
    b = numpy.abs(F).sum(1) + rng.uniform(0.2, 1.0, size=m)
    b[:ne] = rng.normal(size=ne) * 0.1
    dep = {}
    for k, p in enumerate([p for p in BOUNDARY_ROWS if p < mi] or [mi - 1]):
        r = ne + p
        parents = sorted(rng.choice(numpy.arange(ne, ne + min(p, 60)), size=2 + k % 2, replace=False).tolist())
        w = rng.uniform(0.3, 0.7, size=len(parents))
        w /= w.sum()
        delta = DELTAS[k % len(DELTAS)]
        A[r] = (w @ A[parents]) * (1.0 + delta * rng.normal(size=n))
        F[r] = w @ F[parents]
        b[r] = w @ b[parents] + 0.05
        dep[r] = (parents, delta)
    M = rng.normal(size=(n, n))
    U = numpy.linalg.qr(M)[0]
    Q = U @ numpy.diag(rng.uniform(1.0, 3.0, size=n)) @ U.T
    Q = 0.5 * (Q + Q.T)
    H = hs * rng.normal(size=(n, t)) / numpy.sqrt(t)
    c = 0.1 * rng.normal(size=n)
    if not is_qp:
        c = rng.normal(size=n)
        H = hs * rng.normal(size=(n, t))
    A_t = numpy.vstack([numpy.eye(t), -numpy.eye(t)])
    b_t = numpy.ones(2 * t)
    arrays = dict(A=A, b=b.reshape(-1, 1), F=F, A_t=A_t, b_t=b_t.reshape(-1, 1), c=c.reshape(-1, 1), H=H,
                  Q=Q if is_qp else numpy.zeros((n, n)), n_eq=numpy.int64(ne), kind=numpy.str_('qp' if is_qp else 'lp'))
    return arrays, dep


def theta_samples(t, k, rng):
    """points of Theta at radii from 1e-2 to 1 (log-uniform): small radii give shallow active sets, large ones deep"""
    u = rng.uniform(-1.0, 1.0, size=(k, t))
    u /= numpy.abs(u).max(1, keepdims=True)
    return u * numpy.exp(rng.uniform(numpy.log(1e-2), 0.0, size=(k, 1)))


def optimal_sets(g, rng, k=3000):
    """source (a): distinct optimal active sets (equality rows first) of seeded theta"""
    ne, t = int(g['n_eq']), g['F'].shape[1]
    th = theta_samples(t, k, rng)
    out = set()
    if str(g['kind']) == 'qp':
        from twin_theta_qp import ThetaQpTwin
        tw = ThetaQpTwin(g['A'], g['b'], g['F'], g['A_t'], g['b_t'], g['Q'], g['c'], g['H'], ne)
        res = tw.theta_qp(th)
        mi = g['A'].shape[0] - ne
        for st, mk in zip(res['status'], res['mask']):
            if st == 0:
                out.add(tuple(range(ne)) + tuple(ne + i for i in range(mi) if (int(mk[i >> 6]) >> (i & 63)) & 1))
    else:
        A, b, F, H, c = g['A'], g['b'].ravel(), g['F'], g['H'], g['c'].ravel()
        for p in th:
            r = linprog(c + H @ p, A_ub=A, b_ub=b + F @ p, bounds=[(None, None)] * A.shape[1], method='highs')
            if r.status == 0:
                s = b + F @ p - A @ r.x
                out.add(tuple(int(i) for i in numpy.nonzero(numpy.abs(s) <= 1e-9 * (1 + numpy.abs(b + F @ p)))[0]))
    return sorted(out)


def band_of(k):
    for j, (lo, hi) in enumerate(BANDS):
        if lo <= k <= hi:
            return j
    return None


def candidate_pools(g, dep, rng):
    """{band: {source: set of candidates}} (sources 'a'..'d')"""
    ne, m, n = int(g['n_eq']), g['A'].shape[0], g['A'].shape[1]
    top = min(n - ne + 2, m - ne)   # rank-deficient candidates one and two rows past n'
    pools = {}

    def put(src, c):
        c = tuple(sorted(set(c)))
        k = len(c) - ne
        if 1 <= k <= top and all(i >= ne for i in c[ne:]) and band_of(k) is not None:
            pools.setdefault(band_of(k), {}).setdefault(src, set()).add(c)

    eq = tuple(range(ne))
    ineq = numpy.arange(ne, m)
    opt = optimal_sets(g, rng)
    for c in opt:
        put('a', c)
    for c in opt[::max(1, len(opt) // 200)]:
        act = list(c[ne:])
        free = numpy.setdiff1d(ineq, act)
        if len(free):
            put('b', eq + tuple(act) + (int(rng.choice(free)),))
        if len(act) > 1:
            put('b', eq + tuple(a for a in act if a != act[rng.integers(len(act))]))
        if len(act) and len(free):
            drop = act[rng.integers(len(act))]
            put('b', eq + tuple(a for a in act if a != drop) + (int(rng.choice(free)),))
    for k in range(1, top + 1):
        for _ in range(6):
            put('c', eq + tuple(rng.choice(ineq, size=k, replace=False).tolist()))
    for r, (parents, _) in dep.items():
        base = [r] + parents
        for k in range(len(base), top + 1, max(1, (top - len(base)) // 6 or 1)):
            rest = numpy.setdiff1d(ineq, base)
            put('d', eq + tuple(base) + tuple(rng.choice(rest, size=k - len(base), replace=False).tolist()))
        put('d', eq + tuple(base))
    return pools


def sample(pools, rng, total):
    """seeded, stratified: the same share for every band, within a band the sources in turn"""
    picked = []
    per_band = max(8, total // max(1, len(pools)))
    for j in sorted(pools):
        srcs = {s: sorted(v) for s, v in sorted(pools[j].items())}
        for s in srcs:
            rng.shuffle(srcs[s])
        out = []
        while len(out) < per_band and any(srcs.values()):
            for s in list(srcs):
                if srcs[s] and len(out) < per_band:
                    out.append(srcs[s].pop())
        picked.extend(out)
    return sorted(set(picked))


def outcome(s):
    return 'rank' if not s & 1 else 'infeasible' if not s & 2 else 'region' if s & 8 else 'feasible'


def region_bytes(r):
    return 8 * sum(numpy.asarray(r[k]).size for k in ('A', 'b', 'C', 'd', 'E', 'f')) if r is not None else 0


def keep_sample(cands, status, sizes, ne, total=SAMPLE, budget=REGION_BYTES):
    """indices of the stored sample: the same share for every band, within a band the four outcomes in turn (the pool is
    evaluated first so that every outcome a band holds is represented).  Regions (sizes: their bytes) share `budget`
    equally between the bands; the first region of a band is kept whatever its size"""
    by_band = {}
    for i, (c, s) in enumerate(zip(cands, status)):
        by_band.setdefault(band_of(len(c) - ne), {}).setdefault(outcome(s), []).append(i)
    per_band = total // len(by_band)
    per_band_bytes = budget // len(by_band)
    keep = []
    for j in sorted(by_band):
        kinds = [by_band[j][o] for o in sorted(by_band[j])]
        out, used = [], 0
        while len(out) < per_band and any(kinds):
            for lst in kinds:
                while lst and sizes[lst[0]] and used and used + sizes[lst[0]] > per_band_bytes:
                    lst.pop(0)   # a region over the band's share of the budget
                if lst and len(out) < per_band:
                    used += sizes[lst[0]]
                    out.append(lst.pop(0))
        keep.extend(out)
    return sorted(keep)


def pack_regions(regions, out, prefix=''):
    """the compact layout of oracle/gen_sampled_golden.py::pack_regions_compact, for the oracle's region dicts"""
    def cat(get, dtype):
        parts = [numpy.asarray(get(r), dtype=dtype).reshape(-1) for r in regions]
        off = numpy.zeros(len(parts) + 1, dtype=numpy.int64)
        off[1:] = numpy.cumsum([len(x) for x in parts])
        return (numpy.concatenate(parts) if parts else numpy.zeros(0, dtype=dtype)), off
    out[prefix + 'n_regions'] = numpy.int64(len(regions))
    out[prefix + 'packed'] = numpy.bool_(True)
    f64, i32 = numpy.float64, numpy.int32
    for key, get, dt in (('active_set', lambda r: r['active_set'], i32), ('A', lambda r: r['A'], f64), ('b', lambda r: r['b'], f64),
                         ('C', lambda r: r['C'], f64), ('d', lambda r: r['d'], f64), ('E', lambda r: r['E'], f64),
                         ('f', lambda r: r['f'], f64), ('omega_set', lambda r: r['omega_set'], i32),
                         ('lambda_set', lambda r: r['lambda_set'], i32),
                         ('regular_pos', lambda r: r['regular_set'][0], i32),
                         ('regular_idx', lambda r: r['regular_set'][1], i32)):
        out[prefix + 'pk_' + key], out[prefix + 'pk_' + key + '_off'] = cat(get, dt)
    out[prefix + 'pk_E_int'] = numpy.array([numpy.asarray(r['E']).dtype.kind == 'i' for r in regions], dtype=numpy.bool_)


def save_deterministic(path, arrays):
    """numpy.savez_compressed, but with fixed zip time stamps and member order: reruns give byte-identical files"""
    buf = io.BytesIO()
    with zipfile.ZipFile(buf, 'w', compression=zipfile.ZIP_DEFLATED) as zf:
        for k in sorted(arrays):
            b = io.BytesIO()
            numpy.lib.format.write_array(b, numpy.asanyarray(arrays[k]), allow_pickle=False)
            info = zipfile.ZipInfo(k + '.npy', date_time=(1980, 1, 1, 0, 0, 0))
            info.compress_type = zipfile.ZIP_DEFLATED
            zf.writestr(info, b.getvalue())
    with open(path, 'wb') as f:
        f.write(buf.getvalue())


def generate(name, procs):
    t0 = time.time()
    g, dep = build_program(name)
    rng = numpy.random.default_rng(PROGRAMS[name][5] + 1000)
    ne = int(g['n_eq'])
    P = oracle.Program(g['A'], g['b'], g['c'], g['H'], g['A_t'], g['b_t'], g['F'], g['Q'] if str(g['kind']) == 'qp' else None, ne)
    out = dict(g)
    dep_rows = sorted(dep)
    out['dep_rows'] = numpy.array(dep_rows, dtype=numpy.int64)
    out['dep_parents'] = numpy.array([dep[r][0] + [-1] * (3 - len(dep[r][0])) for r in dep_rows], dtype=numpy.int64).reshape(-1, 3)
    out['dep_delta'] = numpy.array([dep[r][1] for r in dep_rows], dtype=numpy.float64)
    pool = sample(candidate_pools(g, dep, rng), rng, POOL)
    res = oracle.evaluate_many(P, [list(c) for c in pool], cores=procs)
    keep = keep_sample(pool, [s for s, _ in res], [region_bytes(r) for _, r in res], ne)
    cands, res = [pool[i] for i in keep], [res[i] for i in keep]
    status = numpy.array([s for s, _ in res], dtype=numpy.uint8)
    # candidates are stored one band per array: the same cardinality in each row
    by_k = {}
    for c, s in zip(cands, status):
        by_k.setdefault(len(c) - ne, []).append((c, s))
    out['k_values'] = numpy.array(sorted(by_k), dtype=numpy.int64)
    for k in sorted(by_k):
        out[f'k{k}_candidates'] = numpy.array([c for c, _ in by_k[k]], dtype=numpy.int32).reshape(len(by_k[k]), ne + k)
        out[f'k{k}_status'] = numpy.array([s for _, s in by_k[k]], dtype=numpy.uint8)
    pack_regions([r for _, r in res if r is not None], out)
    summary = {}
    for c, s in zip(cands, status):
        j = band_of(len(c) - ne)
        kind = outcome(s)
        summary.setdefault(BANDS[j], {}).setdefault(kind, 0)
        summary[BANDS[j]][kind] += 1
    if name in FULL_SOLVE:
        record = []
        regions = oracle.solve(P, max_levels=FULL_SOLVE[name], cores=procs, record=record)
        out['full_levels'] = numpy.int64(len(record))
        for lv, (cs, st) in enumerate(record):
            out[f'full_level{lv}_candidates'] = numpy.array(cs, dtype=numpy.int32).reshape(len(cs), ne + lv + 1)
            out[f'full_level{lv}_status'] = st
        pack_regions(regions, out, prefix='full_')
        print(f'[{name}] full solve: {len(record)} levels, {sum(len(c) for c, _ in record)} candidates, '
              f'{len(regions)} regions', flush=True)
    os.makedirs(OUT, exist_ok=True)
    save_deterministic(os.path.join(OUT, name + '.npz'), out)
    print(f'[{name}] {len(cands)} candidates, {int((status & 8 != 0).sum())} regions, {time.time() - t0:.1f}s: '
          + '; '.join(f'{lo}-{hi}: {d}' for (lo, hi), d in sorted(summary.items())), flush=True)


if __name__ == '__main__':
    procs = int(os.environ.get('GOLDEN_PROCS', '8'))
    for nm in sys.argv[1:] or list(PROGRAMS):
        generate(nm, procs)
