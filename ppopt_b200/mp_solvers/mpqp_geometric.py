"""The geometric mpQP algorithm (the reference's mpqp_geometric / mpqp_parallel_geometric*): grow the partition by stepping
across every facet of every region found and asking the QP which active set holds just beyond it.

Unlike the two graph drivers, which move from an active set to the sets with one row more or one row fewer (a rule that
rests on non-degeneracy), a probe names the region that is actually there.  The cost grows with the number of regions.
Every wave of the search is one batch on the GPU, with the frontier as the batch:

    regions    the wave's new active sets through the graph drivers' evaluation (K1..K5, mpqp_graph._evaluate)
    facets     every kept, non-duplicate row of each new region, gathered on the device from K5's buffers (t = 1: the two
               bounds of K5's interval); their Chebyshev balls by K10 (chebyshev.facet_balls); a facet whose radius is at most
               1e-8 (the full-dimension threshold) is skipped and counted
    probes     theta = c + delta n with delta = min(PROBE_STEP max(1, |c|_inf), r / 2), solved by K8 on the same handle
    resolve    outside Theta: no neighbour.  K8 infeasible: the facet lies on the boundary of the feasible parameter set.
               K8 optimal with a known set that has a region: resolved.  With a new set: it joins the next wave (if that
               evaluation gives no region, the probe has failed and is retried in that wave).  With the source's own set,
               a known set without a region, the iteration cap or a breakdown: failed.
    retries    failed probes again with delta x 100 (capped at r / 2), then as the two tangential probes
               c +- (r / 4) u + delta n, u a unit vector of the facet's hyperplane: a centre that lies exactly on the
               boundary between two neighbours (the symmetric control-allocation programs) resolves on either side; the
               facet is resolved when either tangential probe resolves.  A facet still unresolved after both rounds is
               recorded in ``solution.unresolved``, never dropped.

Regions appear in discovery order: by wave, then by source region, facet row and retry round.  That order does not depend on
batch sizes; it is not the reference's order, which depends on its process pool.
"""
from typing import Dict, Iterable, List, Optional, Tuple

import numpy
import torch

from .. import engine as _engine
from ..chebyshev import RADIUS_TOL, facet_balls
from ..solve_theta import QP_INFEASIBLE, QP_OPTIMAL, ThetaSolver, theta_box
from .mpqp_graph import _evaluate

# Probe distance beyond a facet, relative to max(1, |c|_inf).  Far enough that K8's decisions (1e-10 relative tolerances) are
# not taken on the facet itself, and small next to the regions of the goldens (widths down to ~1e-3), so that a probe lands
# in the neighbour across the facet and not beyond it.
PROBE_STEP = 1e-7
_RETRY_FACTOR = 100.0


def _facet_polytopes(eng, groups, t):
    """stacked [f | E] rows of the new regions (in the order of ``groups``: one (rows, flags, info, selection) per cardinality
    group) and the offsets of every region's block"""
    blocks, counts = [], []
    for rows, flags, info, sel in groups:
        if t == 1:
            lo, hi = info[sel, 2], info[sel, 3]
            one = torch.ones_like(lo)
            blk = torch.stack([torch.stack([hi, one], 1), torch.stack([-lo, -one], 1)], 1)   # E = [1; -1], f = [hi; -lo]
            blocks.append(blk.reshape(-1, 2))
            counts.append(torch.full((lo.shape[0],), 2, dtype=torch.int64, device=eng.tdev))
        else:
            r, fl = rows[sel], flags[sel]
            keep = (fl & 7) == 3                      # non-zero, non-redundant, not a duplicate: build_regions' rows
            blocks.append(r[keep])
            counts.append(keep.sum(1))
    rows = torch.cat(blocks) if blocks else torch.zeros((0, t + 1), dtype=torch.float64, device=eng.tdev)
    cnt = torch.cat(counts) if counts else torch.zeros((0,), dtype=torch.int64, device=eng.tdev)
    off = torch.zeros((cnt.shape[0] + 1,), dtype=torch.int64, device=eng.tdev)
    off[1:] = torch.cumsum(cnt, 0)
    return rows, off, cnt


def _in_plane_unit(n):
    """first column of N, the in-hyperplane columns of the Householder reflector K10 uses (unit, orthogonal to n)"""
    k = torch.argmax(n.abs(), 1)
    ar = torch.arange(n.shape[0], device=n.device)
    nk = n[ar, k]
    v = n.clone()
    v[ar, k] = nk + torch.where(nk >= 0, 1.0, -1.0).to(n.dtype)
    c0 = torch.where(k == 0, 1, 0)
    e = torch.zeros_like(n)
    e[ar, c0] = 1.0
    u = e - (2.0 * v[ar, c0] / (v * v).sum(1))[:, None] * v
    return u / u.norm(dim=1, keepdim=True)


def solve(program, initial_active_sets: Optional[Iterable] = None):
    """Solves the mpQP with the geometric algorithm; returns the Solution (regions in discovery order) with the counters
    gpu_launches, waves, facets, facets_thin, qp_solves, probes_outside_theta, probes_infeasible, retries and unresolved (a
    list of (region index, facet row) pairs)."""
    arrays = _engine.program_arrays(program)
    eng = _engine.Engine(arrays)
    try:
        if not (eng.is_qp and eng.use_gram):
            raise NotImplementedError('the geometric algorithm on the GPU needs an mpQP with a positive definite reduced Hessian')
        cr_cls, sol_cls = _engine._region_classes(program)
        qp = ThetaSolver.__new__(ThetaSolver)
        qp._setup(program, arrays, eng)
        return _Search(eng, qp, cr_cls, sol_cls, program).run(initial_active_sets)
    finally:
        eng.close()


class _Search:
    def __init__(self, eng, qp, cr_cls, sol_cls, program):
        self.eng, self.qp, self.cr_cls, self.sol_cls, self.program = eng, qp, cr_cls, sol_cls, program
        self.t = eng.t
        self.A_t = torch.from_numpy(numpy.ascontiguousarray(qp.A_t)).to(eng.tdev)
        self.b_t = torch.from_numpy(numpy.ascontiguousarray(qp.b_t)).to(eng.tdev)
        self.cache: Dict = {}
        self.regions: List = []
        self.region_of: Dict[Tuple[int, ...], int] = {}
        self.stats = dict(waves=0, facets=0, facets_thin=0, qp_solves=0, probes_outside_theta=0, probes_infeasible=0, retries=0)
        self.unresolved: List[Tuple[int, int]] = []

    # ---- seeding ---------------------------------------------------------------------------------------------------
    def _seeds(self):
        lo, hi = theta_box(self.qp.A_t, self.qp.b_t)
        mid = 0.5 * (lo + hi)
        pts = [mid[None, :]] if bool((self.qp.A_t @ mid <= self.qp.b_t).all()) else []
        pts.append(self.qp.sample_thetas(1000, seed=0))
        out = self.qp.solve_batch(numpy.vstack(pts))
        self.stats['qp_solves'] += int(out['status'].shape[0])
        ok = out['status'] == QP_OPTIMAL
        if not bool(ok.any()):
            return []
        seen = []
        for a in self.qp.active_sets(out['active'][ok]):
            a = tuple(a)
            if a not in seen:
                seen.append(a)
        return seen

    # ---- one evaluation of new active sets -------------------------------------------------------------------------
    def _evaluate(self, sets):
        """evaluates ``sets`` (discovery order); returns the new regions' indices and the stacked facet polytopes"""
        keep = []
        _evaluate(self.eng, self.cr_cls, [a for a in sets if a not in self.cache], self.cache, keep)
        where = {}
        for gi, (asets, regs, _) in enumerate(keep):
            for j, (a, r) in enumerate(zip(asets, regs)):
                if r is not None:
                    where[a] = (gi, j)
        new = [a for a in sets if a in where and a not in self.region_of]
        new = list(dict.fromkeys(new))
        for a in new:
            self.region_of[a] = len(self.regions)
            self.regions.append(self.cache[a][3])
        # facet polytopes in the order of ``new``: one gather per group, then a permutation of the region blocks
        groups, order = [], []
        for gi, (asets, regs, bufs) in enumerate(keep):
            sel = [j for j, a in enumerate(asets) if regs[j] is not None and a in self.region_of and a in new]
            if not sel:
                continue
            idx = torch.tensor(sel, dtype=torch.int64, device=self.eng.tdev)
            groups.append((bufs[1], bufs[2], bufs[3], idx))
            order.extend(asets[j] for j in sel)
        rows, off, cnt = _facet_polytopes(self.eng, groups, self.t)
        if order != new:      # region blocks into discovery order
            pos = {a: i for i, a in enumerate(order)}
            perm = torch.tensor([pos[a] for a in new], dtype=torch.int64, device=self.eng.tdev)
            cnt = cnt[perm]
            start = torch.repeat_interleave(off[:-1][perm], cnt)
            new_off = torch.zeros_like(off)
            new_off[1:] = torch.cumsum(cnt, 0)
            within = torch.arange(start.shape[0], device=self.eng.tdev) - torch.repeat_interleave(new_off[:-1], cnt)
            rows, off = rows[start + within], new_off
        return [self.region_of[a] for a in new], rows, off, cnt

    # ---- probes --------------------------------------------------------------------------------------------------
    def _resolve(self, theta, src):
        """K8 at the probes ``theta`` (k x t device) of facets of the regions ``src`` (host list of region indices); returns
        per probe ('out' | 'inf' | 'known' | 'new' | 'fail', active set or None)"""
        k = theta.shape[0]
        if k == 0:
            return []
        inside = (theta @ self.A_t.T <= self.b_t[None, :]).all(1)
        out = self.qp.solve_batch(theta)
        self.stats['qp_solves'] += k
        status = out['status']
        opt = inside & (status == QP_OPTIMAL)
        act = torch.where(opt[:, None], out['active'], torch.zeros_like(out['active']))
        uniq, inv = torch.unique(act, dim=0, return_inverse=True)
        sets = self.eng.lists_from_masks(uniq.cpu().numpy())
        st = torch.stack([inside.to(torch.int64), status.to(torch.int64), opt.to(torch.int64), inv], 1).cpu().numpy()
        res = []
        for (ins, s, o, u), r in zip(st.tolist(), src):
            if not ins:
                self.stats['probes_outside_theta'] += 1
                res.append(('out', None))
            elif s == QP_INFEASIBLE:
                self.stats['probes_infeasible'] += 1
                res.append(('inf', None))
            elif not o:
                res.append(('fail', None))
            else:
                a = tuple(sets[u])
                if a in self.region_of:
                    res.append(('fail', None) if self.region_of[a] == r else ('known', a))
                elif a in self.cache:
                    res.append(('fail', None))
                else:
                    res.append(('new', a))
        return res

    def _probe_points(self, F, rnd):
        """probe points of the facet records F (device tensors c, n, r, u per record) for retry round ``rnd``; round 2 gives
        two points per record"""
        c, n, r, u = F['c'], F['n'], F['r'], F['u']
        step = PROBE_STEP * (_RETRY_FACTOR if rnd >= 1 else 1.0)
        delta = torch.minimum(step * torch.clamp(c.abs().amax(1), min=1.0), 0.5 * r)
        th = c + delta[:, None] * n
        if rnd < 2:
            return th
        side = (0.25 * torch.where(torch.isfinite(r), r, torch.zeros_like(r)))[:, None] * u
        return torch.stack([th + side, th - side], 1).reshape(-1, self.t)

    def run(self, initial_active_sets):
        ev = None
        if initial_active_sets is not None:
            frontier = list(dict.fromkeys(tuple(sorted(int(i) for i in a)) for a in initial_active_sets))
        else:
            frontier = []
            for a in self._seeds():     # the first seed whose set gives a full-dimensional region
                ev = self._evaluate([a])
                if ev[0]:
                    frontier = [a]
                    break
        # finders[a]: the facet records whose probe found the new set a (retried if a gives no region)
        finders: Dict[Tuple[int, ...], list] = {}
        while frontier:
            self.stats['waves'] += 1
            new_ids, rows, off, cnt = self._evaluate(frontier) if ev is None else ev
            ev = None
            carried = []
            for a in frontier:
                if a not in self.region_of and a in finders:
                    carried.append(finders[a])
            finders = {}
            F0 = self._facets(new_ids, rows, off, cnt)
            found = []      # (source region, facet row, round, active set, (records, index of the finding record))
            failed = self._round(F0, 0, found)
            failed = self._cat(failed, carried)
            while failed is not None and failed['src'].shape[0]:
                rnd = failed['rnd'] + 1
                done = rnd > 2
                if bool(done.any()):
                    for s_, j_ in zip(failed['src'][done].tolist(), failed['row'][done].tolist()):
                        self.unresolved.append((s_, j_))
                    failed = self._take(failed, ~done)
                    rnd = rnd[~done]
                if not failed['src'].shape[0]:
                    break
                # one batch per round present among the failures
                nxt = None
                for r_ in sorted(set(rnd.tolist())):
                    part = self._take(failed, rnd == r_)
                    self.stats['retries'] += int(part['src'].shape[0])
                    nxt = self._cat(nxt, self._round(part, r_, found))
                failed = nxt
            found.sort(key=lambda x: x[:3])
            frontier = []
            for s_, j_, r_, a, rec in found:
                if a not in finders:
                    frontier.append(a)
                finders.setdefault(a, []).append(rec)
            for a in finders:
                finders[a] = self._gather(finders[a])
        sol = self.sol_cls(self.program, self.regions)
        sol.gpu_launches = self.eng.launch_count()
        for k, v in self.stats.items():
            setattr(sol, k, v)
        sol.unresolved = self.unresolved
        return sol

    # ---- facet records: device tensors src, row, rnd, c, n, r, u (one entry per facet) ------------------------------
    _FIELDS = ('src', 'row', 'rnd', 'c', 'n', 'r', 'u')

    def _facets(self, new_ids, rows, off, cnt):
        dev, t = self.eng.tdev, self.t
        nf = int(rows.shape[0])
        if nf == 0:
            return None
        poly = torch.repeat_interleave(torch.arange(cnt.shape[0], device=dev), cnt)
        row = torch.arange(nf, device=dev) - off[poly]
        c, r, code = facet_balls(rows, off, torch.stack([poly, row], 1), t)
        n = rows[:, 1:] / rows[:, 1:].norm(dim=1, keepdim=True)
        u = _in_plane_unit(n) if t > 1 else torch.zeros_like(n)
        src = torch.tensor(new_ids, dtype=torch.int64, device=dev)[poly]
        thin = r <= RADIUS_TOL
        usable = ~thin & torch.isfinite(c).all(1)
        stat = torch.stack([thin.sum(), (~thin & ~usable).sum()]).cpu().tolist()
        self.stats['facets'] += nf
        self.stats['facets_thin'] += stat[0]
        if stat[1]:      # an unbounded facet (t > 1) or an LP that hit its cap: no centre to probe from
            bad = ~thin & ~usable
            self.unresolved.extend(zip(src[bad].tolist(), row[bad].tolist()))
        F = dict(src=src, row=row, rnd=torch.zeros_like(src), c=c, n=n, r=r, u=u)
        return self._take(F, usable)

    @staticmethod
    def _take(F, sel):
        return None if F is None else {k: v[sel] for k, v in F.items()}

    def _gather(self, refs):
        """one record set from (records, index) references; one gather per distinct record set"""
        by = {}
        for F, i in refs:
            by.setdefault(id(F), (F, []))[1].append(i)
        return self._cat(None, [self._take(F, torch.tensor(ix, device=self.eng.tdev)) for F, ix in by.values()])

    @staticmethod
    def _cat(a, b):
        if isinstance(b, list):
            b = {k: torch.cat([x[k] for x in b]) for k in _Search._FIELDS} if b else None
        if a is None:
            return b
        if b is None:
            return a
        return {k: torch.cat([a[k], b[k]]) for k in _Search._FIELDS}

    def _round(self, F, rnd, found):
        """probes of the facet records F in round ``rnd``; appends (source, row, round, set, record) of new sets to ``found``
        and returns the records whose probes failed (None if none)"""
        if F is None or not F['src'].shape[0]:
            return None
        th = self._probe_points(F, rnd)
        per = 2 if rnd == 2 else 1
        src, row = F['src'].tolist(), F['row'].tolist()
        res = self._resolve(th, [s for s in src for _ in range(per)])
        F = dict(F, rnd=torch.full_like(F['rnd'], rnd))
        fail = []
        for i, (s_, j_) in enumerate(zip(src, row)):
            outs = res[i * per:(i + 1) * per]
            for a in dict.fromkeys(a for kind, a in outs if kind == 'new'):
                found.append((s_, j_, rnd, a, (F, i)))
            # the two tangential probes resolve their facet when either does (rather than counting a facet unresolved
            # whose other probe fell back into the source region)
            fail.append(all(kind == 'fail' for kind, _ in outs))
        sel = torch.tensor(fail, dtype=torch.bool, device=self.eng.tdev)
        if not bool(sel.any()):
            return None
        return self._take(F, sel)
