"""Comparison helpers shared by the parity tests (reference semantics: SURVEY.md 3.4 / 7.1)."""
import numpy

REL_TOL = 1e-8  # north_star: law / half-space matrices within 1e-8 relative after PPOPT's own row normalisation
ST_THIN = 64    # csrc/tolerances.h PPG_ST_THIN: full-dimension decision inside the LP backend's tolerance band


def check_status_bits(mine, ref, what=''):
    """rank (1) and feasible (2) must agree on every candidate.  The region bit (8) must agree too, except on candidates
    that the engine itself flagged PPG_ST_THIN: there the reference's answer is its LP backend's rounding (HiGHS reports a
    radius of 2.78e-8 for polytopes whose exact radius is -7.78e-9, DESIGN.md section 5), the engine answers with the
    accurate radius and says so.  Returns the indices of such tolerated candidates."""
    mine = numpy.asarray(mine)
    ref = numpy.asarray(ref)
    for bit, name in ((1, 'rank'), (2, 'feasible')):
        bad = numpy.nonzero((mine & bit) != (ref & bit))[0]
        assert bad.size == 0, f'{what}: {name} differs at {bad[:5].tolist()}'
    bad = numpy.nonzero((mine & 8) != (ref & 8))[0]
    untolerated = [int(i) for i in bad if not (mine[i] & ST_THIN)]
    assert not untolerated, f'{what}: region decision differs at {untolerated[:5]} (not flagged thin)'
    return bad


def rel_err(a, b):
    a = numpy.asarray(a, dtype=float)
    b = numpy.asarray(b, dtype=float)
    if a.shape != b.shape:
        return numpy.inf
    if a.size == 0:
        return 0.0
    scale = max(1.0, float(numpy.max(numpy.abs(b))))
    return float(numpy.max(numpy.abs(a - b))) / scale


def golden_regions(g):
    out = []
    if 'packed' in g:   # compact layout of the sampled goldens (oracle/gen_sampled_golden.py::pack_regions_compact)
        keys = ('active_set', 'A', 'b', 'C', 'd', 'E', 'f', 'omega_set', 'lambda_set', 'regular_pos', 'regular_idx')
        data = {k: (g['pk_' + k], g['pk_' + k + '_off']) for k in keys}
        t = None
        for i in range(int(g['n_regions'])):
            r = {k: data[k][0][data[k][1][i]:data[k][1][i + 1]] for k in keys}
            nb, nd, nf = len(r['b']), len(r['d']), len(r['f'])
            t = len(r['A']) // nb if nb else (len(r['C']) // nd if nd else t)
            r['A'], r['b'] = r['A'].reshape(nb, -1), r['b'].reshape(nb, 1)
            r['C'], r['d'] = r['C'].reshape(nd, t), r['d'].reshape(nd, 1)   # (nd = 0: the equality-only active set)
            r['E'], r['f'] = r['E'].reshape(nf, -1), r['f'].reshape(nf, 1)
            if g['pk_E_int'][i]:
                r['E'] = r['E'].astype(numpy.int64)
            out.append(r)
        return out
    for i in range(int(g['n_regions'])):
        out.append({k: g[f'r{i}_{k}'] for k in ('active_set', 'A', 'b', 'C', 'd', 'E', 'f', 'omega_set', 'lambda_set',
                                                  'regular_pos', 'regular_idx')})
    return out


def rows_match_as_sets(E1, f1, E2, f2, tol=REL_TOL):
    """every row of [E1|f1] has a partner in [E2|f2] within tol and vice versa; returns the unmatched rows"""
    R1 = numpy.hstack([numpy.asarray(E1, float), numpy.asarray(f1, float).reshape(-1, 1)])
    R2 = numpy.hstack([numpy.asarray(E2, float), numpy.asarray(f2, float).reshape(-1, 1)])

    def unmatched(X, Y):
        bad = []
        for r in X:
            if Y.shape[0] == 0:
                bad.append(r)
                continue
            d = numpy.max(numpy.abs(Y - r) / numpy.maximum(1.0, numpy.abs(r)), axis=1)
            if d.min() > tol:
                bad.append(r)
        return bad
    return unmatched(R1, R2), unmatched(R2, R1)


def masks_to_lists(masks, n_eq):
    m = numpy.ascontiguousarray(masks).view(numpy.uint64)
    if m.shape[0] == 0:
        return []
    m = m.reshape(m.shape[0], -1)
    bits = numpy.unpackbits(m.view(numpy.uint8).reshape(m.shape[0], -1), axis=1, bitorder='little')
    eq = list(range(n_eq))
    return [eq + (numpy.nonzero(r)[0] + n_eq).tolist() for r in bits]


MARGIN_BAND = 1e-7   # DESIGN.md section 5, deviation 1: the reference's keep/drop decisions are its LP backend's, whose
                     # feasibility tolerance is 1e-7 (observed: overlapping decisions for margins in [-6.7e-8, 5e-11])


def index_lists_match(region, ref, rows=None, flags=None, margins=None, k_act=0, n_eq=0, m=0, one_d=False):
    """kept-index lists of a region (omega_set, lambda_set, regular_set; mpqp_utils.py:181-184) against the golden ones.
    Returns the list of discrepancies that are NOT explained by the documented reference-side ambiguity:
      * a row whose redundancy margin (``margins``, from the CPU checker's emit with margins=True) lies inside
        +-MARGIN_BAND may be kept by one side and dropped by the other;
      * 1-D programs: the reference compares bitwise-rounded interval end points, so which of several rows attaining the
        end point is listed depends on the last ulp (DESIGN.md deviation 2) - the lists must then agree as sets of
        END-POINT VALUES, checked by the caller through f."""
    want = {'omega': ref['omega_set'].tolist(), 'lambda': ref['lambda_set'].tolist(),
            'regular_pos': ref['regular_pos'].tolist(), 'regular_idx': ref['regular_idx'].tolist()}
    got = {'omega': list(region.omega_set), 'lambda': list(region.lambda_set),
           'regular_pos': list(region.regular_set[0]), 'regular_idx': list(region.regular_set[1])}
    if got == want:
        return []
    if one_d:
        return []   # end-point ties; f is compared by the caller
    if margins is None:
        return [(k, got[k], want[k]) for k in got if got[k] != want[k]]
    aset = list(region.active_set)
    active = aset[n_eq:]
    n_inact = m - len(aset)
    bad = []
    pos_of = {}
    for j, a in enumerate(active):
        pos_of[('lambda', a)] = j
    for p_ in range(n_inact):
        pos_of[('regular_pos', p_)] = k_act + p_
    inactive = [i for i in range(m) if i not in set(aset)]
    for p_, i in enumerate(inactive):
        pos_of[('regular_idx', i)] = k_act + p_
    for key in ('omega', 'lambda', 'regular_pos', 'regular_idx'):
        for v in set(got[key]) ^ set(want[key]):
            row = pos_of.get((key, v), k_act + n_inact + v if key == 'omega' else None)
            mg = None if row is None else margins[row]
            if mg is None or not (abs(mg) < MARGIN_BAND):
                bad.append((key, v, mg))
        if not bad and [x for x in got[key] if x in want[key]] != [x for x in want[key] if x in got[key]]:
            bad.append((key, 'order', got[key], want[key]))
    return bad
