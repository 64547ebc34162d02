"""Level-synchronous GPU driver behind mpqp_combinatorial.solve.

Host mirror of the reference's level loop (/root/reference/src/ppopt/mp_solvers/mpqp_combinatorial.py:10-72):
every enumeration level is ONE batch of candidate bitmasks that stays in HBM; the host only learns counts
(feasible, optimal, children) and receives the matrices of the regions that were actually emitted.
torch is used for device buffers, streams and torch.distributed - all arithmetic is in libppgpu.so.
"""
import ctypes
import time
from typing import Dict, List, Optional

import numpy
import torch

from . import _lib, sharding
from ._lib import ST_BORDER, ST_FEAS, ST_NUMERIC, ST_OPT, ST_RANK, ST_REGION, ST_THIN


def _c(a):
    return numpy.ascontiguousarray(numpy.asarray(a, dtype=numpy.float64))


def program_arrays(program) -> Dict:
    """Reads the attributes the reference's solver reads (mplp_program.py:45-58) from a ppopt or ppopt_b200 program."""
    A = _c(program.A)
    n = A.shape[1]
    F = _c(program.F)
    t = F.shape[1]
    is_qp = hasattr(program, 'Q') and program.Q is not None and type(program).__name__ != 'MPLP_Program'
    H = _c(program.H)
    if H.shape != (n, t):
        # some reference fixtures pass an all-zero H with the transposed shape (tests/test_fixtures.py:60,104)
        if H.shape == (t, n) and not numpy.any(H):
            H = numpy.zeros((n, t))
        else:
            raise ValueError(f'H must be num_x x num_t = {(n, t)}, got {H.shape}')
    eq = [int(i) for i in program.equality_indices]
    if eq != list(range(len(eq))):
        raise ValueError('equality_indices must be range(n_eq) (the reference constructor guarantees it)')
    out = dict(A=A, b=_c(program.b).reshape(-1), F=F, A_t=_c(program.A_t).reshape(-1, t),
               b_t=_c(program.b_t).reshape(-1), c=_c(program.c).reshape(-1), H=H, n_eq=len(eq), is_qp=bool(is_qp))
    out['Q'] = _c(program.Q) if is_qp else None
    return out


class Engine:
    """Owns one ppgpu_program handle on one device."""

    def __init__(self, arrays: Dict, device: Optional[int] = None):
        if not torch.cuda.is_available():
            raise RuntimeError('ppopt_b200 needs a CUDA device (there is no CPU fallback)')
        self.lib = _lib.load()
        self.device = torch.cuda.current_device() if device is None else int(device)
        self.tdev = torch.device('cuda', self.device)
        a = arrays
        self.n, self.t = a['A'].shape[1], a['F'].shape[1]
        self.m, self.q, self.n_eq, self.is_qp = a['A'].shape[0], a['A_t'].shape[0], a['n_eq'], a['is_qp']
        dims = _lib.Dims(self.n, self.t, self.m, self.q, self.n_eq, int(self.is_qp))
        self._keep = a  # host arrays must outlive the create call only, kept for debugging
        h = ctypes.c_void_p()
        ptr = lambda x: None if x is None else x.ctypes.data
        with torch.cuda.device(self.device):
            rc = self.lib.ppgpu_program_create(ctypes.byref(dims), ptr(a['A']), ptr(a['b']), ptr(a['F']), ptr(a['A_t']),
                                               ptr(a['b_t']), ptr(a['Q']), ptr(a['c']), ptr(a['H']), self.device,
                                               ctypes.byref(h))
        _lib.check(rc, 'program_create')
        self.h = h
        info = _lib.Info()
        _lib.check(self.lib.ppgpu_program_info(self.h, ctypes.byref(info)), 'program_info')
        self.W, self.mi, self.R0 = info.words, info.n_ineq, info.region_rows
        self.use_gram, self.max_depth, self.sm_count = bool(info.use_gram), info.max_depth, info.sm_count
        self.lp_columns = info.lp_columns
        self.has_walk_vertex = bool(info.reserved)
        self.h2d_bytes = sum(v.nbytes for v in a.values() if isinstance(v, numpy.ndarray))
        self.d2h_bytes = 0

    def close(self):
        if getattr(self, 'h', None) is not None and self.h:
            self.lib.ppgpu_program_destroy(self.h)
            self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    # ---- thin wrappers -------------------------------------------------------------------------------------------
    def set_option(self, option: int, value: int):
        _lib.check(self.lib.ppgpu_set_option(self.h, int(option), int(value)), 'set_option')

    def _stream(self):
        return ctypes.c_void_p(torch.cuda.current_stream(self.tdev).cuda_stream)

    def empty(self, shape, dtype):
        return torch.empty(shape, dtype=dtype, device=self.tdev)

    def root_level(self) -> torch.Tensor:
        masks = self.empty((max(self.mi, 1), self.W), torch.int64)
        cnt = ctypes.c_int64(0)
        _lib.check(self.lib.ppgpu_root_level(self.h, masks.data_ptr(), ctypes.byref(cnt), self._stream()), 'root_level')
        return masks[:cnt.value]

    def level_eval(self, masks: torch.Tensor, k_act: int, status: Optional[torch.Tensor] = None, stages: int = 7,
                   lo: int = 0, hi: Optional[int] = None, witness: Optional[torch.Tensor] = None,
                   parent: Optional['ParentLevel'] = None) -> torch.Tensor:
        """status bytes of masks[lo:hi].  ``witness`` (n x WITNESS_SLOTS x W int64, zeros): receives the active-row masks of
        vertices that hold a candidate; ``parent``: the level the candidates were generated from (feasible masks, their hash
        set, their witnesses) - candidates covered by a parent's witness are certified without any LP work
        (ppgpu_level_eval_w)."""
        n = masks.shape[0]
        if status is None:
            status = torch.zeros((n,), dtype=torch.uint8, device=self.tdev)
        hi = n if hi is None else hi
        if hi > lo:
            if witness is None and parent is None:
                _lib.check(self.lib.ppgpu_level_eval(self.h, masks.data_ptr() + lo * self.W * 8, hi - lo, k_act,
                                                     status.data_ptr() + lo, stages, self._stream()), 'level_eval')
            else:
                pf, pnf, pws, pw = (parent.feas_masks.data_ptr(), parent.nf, parent.ws.data_ptr(), parent.wit.data_ptr()) \
                    if parent is not None else (None, 0, None, None)
                _lib.check(self.lib.ppgpu_level_eval_w(self.h, masks.data_ptr() + lo * self.W * 8, hi - lo, k_act,
                                                       status.data_ptr() + lo, stages,
                                                       None if witness is None else witness.data_ptr() + lo * _lib.WITNESS_SLOTS * self.W * 8,
                                                       pf, pnf, pws, pw, self._stream()), 'level_eval_w')
        return status

    def select(self, status: torch.Tensor, bits: int, value: int) -> torch.Tensor:
        n = status.shape[0]
        if n == 0:
            return self.empty((0,), torch.int64)
        ws_bytes = self.lib.ppgpu_select_workspace_bytes(n)
        ws = self.empty(((ws_bytes + 7) // 8,), torch.int64)
        idx = self.empty((n,), torch.int64)
        cnt = ctypes.c_int64(0)
        _lib.check(self.lib.ppgpu_level_select(self.h, status.data_ptr(), n, bits, value, idx.data_ptr(), ctypes.byref(cnt),
                                               ws.data_ptr(), ws_bytes, self._stream()), 'level_select')
        return idx[:cnt.value]

    def emit(self, masks: torch.Tensor, sel: torch.Tensor, k_act: int, status: torch.Tensor):
        ns = sel.shape[0]
        N = self.n + self.n_eq + k_act
        laws = self.empty((ns, N, self.t + 1), torch.float64)
        rows = self.empty((ns, self.R0, self.t + 1), torch.float64)
        flags = self.empty((ns, self.R0), torch.int32)
        info = self.empty((ns, 4), torch.float64)
        _lib.check(self.lib.ppgpu_regions_emit(self.h, masks.data_ptr(), sel.data_ptr(), ns, k_act, laws.data_ptr(),
                                               rows.data_ptr(), flags.data_ptr(), info.data_ptr(), status.data_ptr(),
                                               self._stream()), 'regions_emit')
        return laws, rows, flags, info

    def children(self, masks: torch.Tensor, feas_idx: torch.Tensor, k_act: int, dist=None, keep: Optional[dict] = None) -> torch.Tensor:
        """next level's candidates; with dist (torch.distributed, world > 1) the pruning look-ups of the parents are split
        between the ranks and the per-parent results summed (every rank ends up with the identical child array).
        ``keep`` (dict) receives the gathered feasible masks and the workspace holding their prefix-group index: what the next
        level needs to look its candidates' parents up (witness inheritance)"""
        nf = feas_idx.shape[0]
        if nf == 0:
            return self.empty((0, self.W), torch.int64)
        if dist is not None and dist.get_world_size() > 1 and nf >= 65536:
            return self._children_sharded(masks, feas_idx, k_act, dist, keep)
        feas_masks = self.empty((nf, self.W), torch.int64)
        survive = self.empty((nf, self.W), torch.int64)
        offsets = self.empty((nf + 1,), torch.int64)
        ws_bytes = self.lib.ppgpu_scan_workspace_bytes(nf)
        ws = self.empty(((ws_bytes + 7) // 8,), torch.int64)
        tot = ctypes.c_int64(0)
        _lib.check(self.lib.ppgpu_children_count(self.h, masks.data_ptr(), feas_idx.data_ptr(), nf, k_act,
                                                 feas_masks.data_ptr(), survive.data_ptr(), offsets.data_ptr(),
                                                 ctypes.byref(tot), ws.data_ptr(), ws_bytes, self._stream()),
                   'children_count')
        if keep is not None:
            keep.update(feas_masks=feas_masks, ws=ws, nf=nf)
        out = self.empty((tot.value, self.W), torch.int64)
        if tot.value:
            _lib.check(self.lib.ppgpu_children_write(self.h, feas_masks.data_ptr(), survive.data_ptr(), offsets.data_ptr(),
                                                     nf, out.data_ptr(), self._stream()), 'children_write')
        return out

    def _children_sharded(self, masks, feas_idx, k_act, dist, keep=None):
        from . import sharding
        nf = feas_idx.shape[0]
        feas_masks = self.empty((nf, self.W), torch.int64)
        survive = torch.zeros((nf, self.W), dtype=torch.int64, device=self.tdev)
        counts = torch.zeros((nf + 1,), dtype=torch.int64, device=self.tdev)
        ws_bytes = self.lib.ppgpu_scan_workspace_bytes(nf)
        ws = self.empty(((ws_bytes + 7) // 8,), torch.int64)
        _lib.check(self.lib.ppgpu_children_prepare(self.h, masks.data_ptr(), feas_idx.data_ptr(), nf, feas_masks.data_ptr(),
                                                   ws.data_ptr(), ws_bytes, self._stream()), 'children_prepare')
        if keep is not None:
            keep.update(feas_masks=feas_masks, ws=ws, nf=nf)
        for lo, hi in sharding.chunks(nf, dist.get_rank(), dist.get_world_size()):
            _lib.check(self.lib.ppgpu_children_count_range(self.h, feas_masks.data_ptr(), nf, k_act, survive.data_ptr(),
                                                           counts.data_ptr(), lo, hi, ws.data_ptr(), ws_bytes,
                                                           self._stream()), 'children_count_range')
        dist.all_reduce(survive, op=dist.ReduceOp.SUM)   # disjoint supports: the sum is the union
        dist.all_reduce(counts, op=dist.ReduceOp.SUM)
        tot = ctypes.c_int64(0)
        _lib.check(self.lib.ppgpu_children_scan(self.h, counts.data_ptr(), nf, ctypes.byref(tot), ws.data_ptr(), ws_bytes,
                                                self._stream()), 'children_scan')
        out = self.empty((tot.value, self.W), torch.int64)
        if tot.value:
            _lib.check(self.lib.ppgpu_children_write(self.h, feas_masks.data_ptr(), survive.data_ptr(), counts.data_ptr(),
                                                     nf, out.data_ptr(), self._stream()), 'children_write')
        return out

    def counters(self, reset: bool = False) -> Dict[str, int]:
        buf = (ctypes.c_uint64 * _lib.NUM_COUNTERS)()
        _lib.check(self.lib.ppgpu_counters(self.h, buf, int(reset), self._stream()), 'counters')
        return {name: int(buf[i]) for i, name in enumerate(_lib.COUNTER_NAMES)}

    def profile(self, on: bool):
        _lib.check(self.lib.ppgpu_profile_enable(self.h, int(on)), 'profile_enable')

    def profile_read(self, reset: bool = False) -> Dict[str, Dict]:
        ms = (ctypes.c_double * _lib.NUM_FAMILIES)()
        ln = (ctypes.c_int64 * _lib.NUM_FAMILIES)()
        _lib.check(self.lib.ppgpu_profile_read(self.h, ms, ln, int(reset)), 'profile_read')
        return {name: dict(ms=float(ms[i]), launches=int(ln[i])) for i, name in enumerate(_lib.FAMILY_NAMES)}

    def launch_count(self) -> int:
        return int(self.lib.ppgpu_launch_count(self.h))

    # ---- bitmask helpers (host side, small) ----------------------------------------------------------------------
    def masks_from_lists(self, active_sets) -> torch.Tensor:
        """uint64 bitmasks (as int64 tensor) for full active-set index lists [eq..., ineq...]."""
        out = numpy.zeros((len(active_sets), self.W), dtype=numpy.uint64)
        for ci, aset in enumerate(active_sets):
            for idx in aset:
                i = int(idx) - self.n_eq
                if i >= 0:
                    out[ci, i >> 6] |= numpy.uint64(1) << numpy.uint64(i & 63)
        return torch.from_numpy(out.view(numpy.int64)).to(self.tdev)

    def lists_from_masks(self, masks_np: numpy.ndarray) -> List[List[int]]:
        eq = list(range(self.n_eq))
        m = masks_np.view(numpy.uint64).reshape(-1, self.W)
        bits = numpy.unpackbits(m.view(numpy.uint8).reshape(m.shape[0], -1), axis=1, bitorder='little')
        per_row = bits.sum(1)
        if m.shape[0] and (per_row == per_row[0]).all():
            # one level: every set has the same cardinality - one nonzero for all of them
            cols = (numpy.nonzero(bits)[1] + self.n_eq).reshape(m.shape[0], int(per_row[0])).tolist()
            return [eq + c for c in cols] if eq else cols
        return [eq + (numpy.nonzero(r)[0] + self.n_eq).tolist() for r in bits]


def measure_fp64_peak(iters: int = 20000) -> float:
    lib = _lib.load()
    v = ctypes.c_double(0.0)
    _lib.check(lib.ppgpu_measure_fp64_peak(iters, ctypes.byref(v), ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)),
               'fp64 peak')
    return v.value


def _region_classes(program):
    """ppopt's own result classes when the program is a ppopt object, else this package's mirrors."""
    mod = type(program).__module__
    root = mod.split('.mpqp_program')[0].split('.mplp_program')[0]
    if root not in ('ppopt_b200',) and root.endswith('ppopt'):
        import importlib
        try:
            cr = importlib.import_module(root + '.critical_region').CriticalRegion
            sol = importlib.import_module(root + '.solution').Solution
            return cr, sol
        except Exception:
            pass
    from .critical_region import CriticalRegion
    from .solution import Solution
    return CriticalRegion, Solution


def _to_host(x):
    """device tensor -> numpy through a pinned staging buffer (torch caches pinned blocks); numpy arrays pass through"""
    if isinstance(x, torch.Tensor):
        if x.is_cuda:
            h = torch.empty(x.shape, dtype=x.dtype, pin_memory=True)
            h.copy_(x, non_blocking=True)
            torch.cuda.current_stream(x.device).synchronize()
            return h.numpy()
        return x.numpy()
    return numpy.asarray(x)


# Kept-index lists of every region of a level (mpqp_utils.py:181-195): of the R0 rows of a region, rows [0, k_act) are the
# multiplier rows (lambda_set: the constraint they belong to), [k_act, k_act + n_inact) the inactive constraints
# (regular_set: position, constraint), the rest the Theta rows (omega_set).  Returns, for the kept rows of all regions in
# row-major order: val (the index each list reports), pos (row - k_act: the "position" of regular_set), and cnt (3 x ns:
# kept rows per region, of which multiplier rows, of which multiplier + inactive rows).  Two statements of the same
# arithmetic: whole-array numpy for host buffers, whole-array torch for device buffers (5,570 regions x 112 rows at the
# bench workload: on the host this was the largest part of the region assembly).
# Measured on the B200 box (bench e2e, 5,570 regions per solve): with the torch statement on the device AND the collector
# paused the end-to-end step went from 268 to 331 ms although both are 2-3x faster on CPU tensors in isolation; both are
# therefore off by default (PPGPU_ASSEMBLY_DEVICE=1 / PPGPU_ASSEMBLY_PAUSE_GC=1 switch them on), the whole-array numpy
# statement runs on the host copy of the flags.
_INDEX_LISTS_ON_DEVICE = __import__('os').environ.get('PPGPU_ASSEMBLY_DEVICE', '0') == '1'
_PAUSE_GC = __import__('os').environ.get('PPGPU_ASSEMBLY_PAUSE_GC', '0') == '1'


def _kept_index_lists_numpy(kept_all, asets, k_act, n_inact, ne, m):
    ns = kept_all.shape[0]
    ri, ci = numpy.nonzero(kept_all)
    is_l, is_r = ci < k_act, (ci >= k_act) & (ci < k_act + n_inact)
    val = ci - (k_act + n_inact)
    if k_act > 0:
        val = numpy.where(is_l, asets[ri, numpy.minimum(ne + ci, ne + k_act - 1)], val)
    if n_inact > 0:
        act_bool = numpy.zeros((ns, m), dtype=bool)
        if asets.shape[1]:
            act_bool[numpy.arange(ns)[:, None], asets] = True
        inactive = numpy.nonzero(~act_bool)[1].reshape(ns, n_inact)
        val = numpy.where(is_r, inactive[ri, numpy.clip(ci - k_act, 0, n_inact - 1)], val)
    cnt = numpy.stack([kept_all.sum(1), kept_all[:, :k_act].sum(1), kept_all[:, :k_act + n_inact].sum(1)]).astype(numpy.int64)
    return val.astype(numpy.int64), (ci - k_act).astype(numpy.int64), cnt


def _kept_index_lists_torch(kept_all, asets, k_act, n_inact, ne, m):
    ns = kept_all.shape[0]
    nz = torch.nonzero(kept_all)                     # row-major, like numpy.nonzero
    ri, ci = nz[:, 0], nz[:, 1]
    val = ci - (k_act + n_inact)
    if k_act > 0:
        val = torch.where(ci < k_act, asets[ri, torch.clamp(ne + ci, max=ne + k_act - 1)], val)
    if n_inact > 0:
        act_bool = torch.zeros((ns, m), dtype=torch.bool, device=kept_all.device)
        if asets.shape[1]:
            act_bool.scatter_(1, asets, True)
        inactive = torch.nonzero(~act_bool)[:, 1].reshape(ns, n_inact)
        is_r = (ci >= k_act) & (ci < k_act + n_inact)
        val = torch.where(is_r, inactive[ri, torch.clamp(ci - k_act, 0, n_inact - 1)], val)
    cnt = torch.stack([kept_all.sum(1), kept_all[:, :k_act].sum(1), kept_all[:, :k_act + n_inact].sum(1)])
    return val, ci - k_act, cnt


def build_regions(eng: Engine, cr_cls, active_sets, k_act, laws, rows, flags, info, d2h: Optional[list] = None) -> list:
    """CriticalRegion objects from K5's buffers (field meaning: mpqp_utils.py:181-195).  The buffers may be device tensors
    (the solver's case) or numpy arrays.  Everything that can be done for the whole level at once is done on whole arrays -
    on the DEVICE when the buffers are there: the law blocks are split into contiguous A, b, C, d, the kept half-spaces of
    all regions are gathered with one boolean mask (only those rows cross PCIe: ~1/5 of the rows buffer), the kept-index
    lists of all regions come from one nonzero - and per region only views and list slices remain.  At the bench workload
    5,570 regions are assembled per solve; a Python loop over the constraints of every region cost more than the level-5
    kernels.  ``d2h``: optional list that receives the number of bytes copied device -> host."""
    n, t, ne, m = eng.n, eng.t, eng.n_eq, eng.m
    ns = len(active_sets)
    if ns == 0:
        return []
    n_inact = eng.mi - k_act
    on_dev = isinstance(laws, torch.Tensor)
    copied = 0

    def host(x):
        nonlocal copied
        h = _to_host(x.contiguous() if isinstance(x, torch.Tensor) else numpy.ascontiguousarray(x))
        copied += h.nbytes
        return h
    kept_all = (flags & 3) == 3                       # non-zero and non-redundant rows
    nodup_all = kept_all & ((flags & 4) == 0)         # ... that are not duplicates of an earlier row
    info = host(info)
    emitted = (info[:, 0] == 1.0).tolist()
    A_all, b_all = host(laws[:, :n, 1:]), host(laws[:, :n, :1])
    C_all, d_all = host(laws[:, n:, 1:]), host(laws[:, n:, :1])
    if t != 1:
        # kept, de-duplicated half-spaces of every region, stacked; a region's block is a contiguous slice of it
        E_cat, f_cat = host(rows[:, :, 1:][nodup_all]), host(rows[:, :, :1][nodup_all])
        e_off = numpy.concatenate([[0], numpy.cumsum(host(nodup_all.sum(1)))]).tolist()
    asets = numpy.asarray(active_sets, dtype=numpy.int64).reshape(ns, ne + k_act)
    aset_lists = asets.tolist()
    if on_dev and _INDEX_LISTS_ON_DEVICE:
        val, pos, cnt = _kept_index_lists_torch(kept_all, torch.from_numpy(asets).to(kept_all.device), k_act, n_inact, ne, m)
        val, pos, cnt = host(val), host(pos), host(cnt)
    else:
        val, pos, cnt = _kept_index_lists_numpy(host(kept_all) if on_dev else numpy.asarray(kept_all), asets, k_act, n_inact, ne, m)
    bounds = numpy.concatenate([[0], numpy.cumsum(cnt[0])]).tolist()
    n_l, n_lr = cnt[1].tolist(), cnt[2].tolist()
    val_list, pos_list = val.tolist(), pos.tolist()
    # per region only views and list slices remain; the views of a whole array come from ONE iteration over its first axis
    # (list(array)), not from ns index operations
    import gc
    gc_was_on = gc.isenabled() and _PAUSE_GC
    if gc_was_on:
        gc.disable()   # thousands of small objects in one go: a generation-2 collection in the middle costs more than the assembly
    try:
        lo_l, hi_l = bounds[:-1], bounds[1:]
        le_l = [lo + x for lo, x in zip(lo_l, n_l)]
        re_l = [lo + x for lo, x in zip(lo_l, n_lr)]
        if t == 1:
            E_l = [numpy.array([[1], [-1]]) for _ in range(ns)]
            f_l = [numpy.array([[hi_], [-lo_]]) for lo_, hi_ in zip(info[:, 2].tolist(), info[:, 3].tolist())]
        else:
            E_l = [E_cat[a:b] for a, b in zip(e_off[:-1], e_off[1:])]
            f_l = [f_cat[a:b] for a, b in zip(e_off[:-1], e_off[1:])]
        out = [cr_cls(A, b, C, d, E, f, aset, val_list[re:hi], val_list[lo:le], [pos_list[le:re], val_list[le:re]]) if em else None
               for A, b, C, d, E, f, aset, lo, le, re, hi, em in zip(list(A_all), list(b_all), list(C_all), list(d_all), E_l, f_l,
                                                                     aset_lists, lo_l, le_l, re_l, hi_l, emitted)]
    finally:
        if gc_was_on:
            gc.enable()
    if d2h is not None:
        d2h.append(copied if on_dev else 0)
    return out


class ParentLevel:
    """What a level leaves behind for the next one (witness inheritance): its feasible masks in K6's order, the K6 workspace
    holding their prefix-group index, and the witnesses (active-row masks of the certifying vertices) in the same order."""
    __slots__ = ('feas_masks', 'ws', 'nf', 'wit')

    def __init__(self, feas_masks, ws, nf, wit):
        self.feas_masks, self.ws, self.nf, self.wit = feas_masks, ws, int(nf), wit


# levels below this size are neither walked nor worth a witness array (PPGPU_OPT_K2W_MIN's default)
WITNESS_MIN_LEVEL = 100000


def _inherit_on() -> bool:
    import os
    return os.environ.get('PPGPU_INHERIT', '1') != '0'


def _dist():
    import torch.distributed as dist
    if dist.is_available() and dist.is_initialized() and dist.get_world_size() > 1:
        return dist
    return None


class NumericalFailure(RuntimeError):
    """A candidate could not be decided (LP iteration limit / non-finite values) even after the cold re-evaluation.
    Raised instead of silently treating the candidate as infeasible, which would prune every superset of it."""


def _checksum(status: torch.Tensor) -> int:
    """order-sensitive checksum of the decision bits of a level (device side, one number crosses PCIe)"""
    n = status.shape[0]
    if n == 0:
        return 0
    w = (torch.arange(n, device=status.device, dtype=torch.int64) * 2654435761 + 12345) & 0x7fffffff
    return int((((status & 15).to(torch.int64) + 1) * w).sum().item() & 0x7fffffffffffffff)


def _eval_level(eng: Engine, masks: torch.Tensor, k_act: int, dist, rank: int, world: int,
                wit: Optional[torch.Tensor] = None, parent: Optional['ParentLevel'] = None) -> torch.Tensor:
    """status bytes of one level.  Multi-GPU: this rank's chunks (sharding.py) are packed into ONE contiguous array, so
    that every stage is one launch per rank (16 chunk-wise calls x 7 launches paid 16 kernel tails each), evaluated, and
    the bytes scattered back; one NCCL all-reduce(SUM) of the byte vector then gives every rank all statuses (and, when
    witnesses are collected, one more of the witness words: disjoint supports, the sum is the union)."""
    n = masks.shape[0]
    status = torch.zeros((n,), dtype=torch.uint8, device=eng.tdev)
    if world <= 1:
        eng.level_eval(masks, k_act, status, 7, witness=wit, parent=parent)
        return status
    mine = sharding.chunks(n, rank, world)
    if mine:
        if len(mine) == 1:
            lo, hi = mine[0]
            eng.level_eval(masks, k_act, status, 7, lo, hi, witness=wit, parent=parent)
        else:
            packed = torch.cat([masks[lo:hi] for lo, hi in mine])
            wp = torch.zeros((packed.shape[0],) + tuple(wit.shape[1:]), dtype=torch.int64, device=eng.tdev) if wit is not None else None
            st = eng.level_eval(packed, k_act, None, 7, witness=wp, parent=parent)
            off = 0
            for lo, hi in mine:
                status[lo:hi] = st[off:off + hi - lo]
                if wit is not None:
                    wit[lo:hi] = wp[off:off + hi - lo]
                off += hi - lo
    if wit is not None:
        dist.all_reduce(wit, op=dist.ReduceOp.SUM)
    return sharding.gather_status(status, dist)


def _escalate_numeric(eng: Engine, masks: torch.Tensor, status: torch.Tensor, k_act: int, flagged: Dict, level: int):
    """Never prune on a numerical failure (VERDICT r01 item 6).  Candidates whose feasibility LP hit the iteration limit
    (NUMERIC set, FEAS clear) are re-evaluated by the cold simplex - no relaxation, no warm origin: a genuinely different
    computation; if that does not decide them either the solve stops with NumericalFailure.  Candidates on which the
    Gram/Cholesky optimality screen failed (NUMERIC and FEAS set) go to K5, whose LU of the KKT matrix decides."""
    num = eng.select(status, ST_NUMERIC | ST_FEAS, ST_NUMERIC)
    if num.shape[0]:
        sub = masks[num].contiguous()
        st2 = torch.full((sub.shape[0],), ST_RANK, dtype=torch.uint8, device=eng.tdev)
        eng.level_eval(sub, k_act, st2, 2 | 4 | 8)     # stage bit 8: cold simplex only
        still = (st2 & (ST_NUMERIC | ST_FEAS)) == ST_NUMERIC
        if bool(still.any().item()):
            bad = eng.lists_from_masks(sub[still][:8].cpu().numpy())
            raise NumericalFailure(f'level {level}: {int(still.sum().item())} candidate(s) undecided after the cold '
                                   f're-evaluation, e.g. {bad}')
        status[num] = st2
        flagged['numeric_recovered'] += int(num.shape[0])
    scr = eng.select(status, ST_NUMERIC | ST_FEAS | ST_OPT, ST_NUMERIC | ST_FEAS)
    if scr.shape[0]:
        status[scr] = (status[scr] & ~ST_NUMERIC) | ST_OPT
        flagged['screen_failed'] += int(scr.shape[0])


def _collect_flags(eng: Engine, masks: torch.Tensor, status: torch.Tensor, flagged: Dict):
    """rank decisions inside the borderline band and full-dimension decisions inside the LP tolerance band are REPORTED
    (solution.flagged: counts, and the first 4096 active sets of each kind), never silent"""
    for name, bit in (('border', ST_BORDER), ('thin', ST_THIN)):
        idx = eng.select(status, bit, bit)
        if idx.shape[0]:
            flagged[name + '_count'] += int(idx.shape[0])
            room = 4096 - len(flagged[name])
            if room > 0:
                flagged[name].extend(eng.lists_from_masks(masks[idx[:room]].cpu().numpy()))


def solve(program, max_levels: Optional[int] = None, collect_status: bool = False, engine: Optional[Engine] = None,
          emit_regions: bool = True, distributed: bool = True, expand_last: bool = False,
          materialize: bool = True, digest: bool = False):
    """GPU replacement for mpqp_combinatorial.solve(program) (mpqp_combinatorial.py:10-72).

    Returns the Solution; per-level statistics are attached as ``solution.level_stats`` (candidates, feasible,
    optimal-screen, regions, seconds) - the counters the reference's parallel solvers print
    (mpqp_parrallel_combinatorial.py:103-104).  ``max_levels`` caps the depth for programs nobody can finish
    (applied identically to the CPU baselines in bench.py).  ``solution.flagged`` lists the candidates whose decision
    fell inside a documented tolerance band (rank: 'border', full dimension: 'thin'); a candidate that cannot be decided
    at all raises NumericalFailure.  ``digest=True`` adds ``solution.digest``, a hash of every level's decision bits and of
    the region list, used to prove that N-GPU runs decide exactly like the 1-GPU run (bench.py).

    Under torch.distributed (world size G > 1) every level's candidate array is cut into chunks dealt to the ranks in
    snake order (sharding.py), each rank evaluates its share as one contiguous batch, the status bytes are combined by one
    NCCL all-reduce, every rank generates the identical next level, and the raw region buffers of the owning ranks are
    all-gathered (NCCL) so that every rank builds the same Solution.
    """
    own = engine is None
    eng = Engine(program_arrays(program)) if own else engine
    cr_cls, sol_cls = _region_classes(program)
    dist = _dist() if distributed else None
    rank, world = (dist.get_rank(), dist.get_world_size()) if dist is not None else (0, 1)
    regions: list = []
    stats = []
    statuses = []
    sums = []
    flagged = {'border': [], 'thin': [], 'border_count': 0, 'thin_count': 0, 'numeric_recovered': 0, 'screen_failed': 0,
               'singular_skipped': []}
    depth = eng.max_depth if max_levels is None else min(eng.max_depth, max_levels)
    complete = max_levels is None or max_levels >= eng.max_depth
    masks = eng.root_level() if depth > 0 else eng.empty((0, eng.W), torch.int64)
    total = 0
    inherit = _inherit_on() and eng.has_walk_vertex
    parent = None
    for lvl in range(depth):
        n = masks.shape[0]
        if n == 0:
            break
        t0 = time.perf_counter()
        k_act = lvl + 1
        last = lvl + 1 == eng.max_depth or (lvl + 1 == depth and not expand_last)
        # witnesses: the rows active at the vertex that certified a candidate; the next level inherits them
        wit = torch.zeros((n, _lib.WITNESS_SLOTS, eng.W), dtype=torch.int64, device=eng.tdev) \
            if (inherit and not last and n >= WITNESS_MIN_LEVEL) else None
        status = _eval_level(eng, masks, k_act, dist, rank, world, wit, parent)
        parent = None
        # one device reduction answers "is any candidate flagged at all" for the three report bits (a sync per question
        # is what the small levels and the sharded runs pay for)
        any_flag = int((status & (ST_NUMERIC | ST_THIN | ST_BORDER)).max().item()) if n else 0
        if any_flag & ST_NUMERIC:
            _escalate_numeric(eng, masks, status, k_act, flagged, lvl + 1)
        n_reg = 0
        opt_idx = eng.select(status, ST_OPT, ST_OPT)
        n_opt = int(opt_idx.shape[0])
        if n_opt and emit_regions:
            # regions are emitted by the rank that owns the candidate
            mine = sharding.owned(opt_idx, n, rank, world) if world > 1 else opt_idx
            if not materialize:
                if mine.shape[0]:
                    eng.emit(masks, mine, k_act, status)  # results stay in HBM (device-resident throughput runs)
                if world > 1 and (digest or collect_status):
                    status = sharding.gather_region_bits(status, mine, dist)
            else:
                bufs = eng.emit(masks, mine, k_act, status) if mine.shape[0] else None
                if world > 1:
                    mine, bufs = sharding.gather_regions(eng, mine, bufs, k_act, dist)
                    status = sharding.gather_region_bits(status, mine, dist, already_global=True, bufs=bufs)
                if bufs is not None and mine.shape[0]:
                    laws, rows, flags, info = bufs
                    sel_masks = masks[mine].cpu().numpy()
                    eng.d2h_bytes += sel_masks.nbytes
                    asets = eng.lists_from_masks(sel_masks)
                    sing = torch.nonzero(info[:, 0] < 0).reshape(-1).cpu().numpy()
                    if sing.size:
                        if eng.use_gram or not eng.is_qp:
                            # passed the optimality screen and the KKT system is singular: what the reference raises
                            # (mpqp_program.py:187)
                            raise numpy.linalg.LinAlgError('Singular matrix')
                        # general path (reduced Hessian not positive definite): K5's LU is also the optimality test here;
                        # the reference only solves the KKT system of sets that passed check_optimality, so a singular
                        # system of an arbitrary feasible set is skipped and reported, not raised (ADVICE r01)
                        flagged['singular_skipped'].extend(asets[i] for i in sing[:256])
                    copied = []
                    built = build_regions(eng, cr_cls, asets, k_act, laws, rows, flags, info, d2h=copied)
                    eng.d2h_bytes += sum(copied)
                    regions.extend(r for r in built if r is not None)
            # (K5 decides full dimension with the accurate radius and may raise the THIN bit itself)
            after = torch.stack([((status & ST_REGION) != 0).sum(), (status & (ST_THIN | ST_BORDER)).max().to(torch.int64)]).cpu()
            n_reg = int(after[0])
            any_flag |= int(after[1])
        if last:
            # no next level: only the count is needed, not the ordered index list
            feas_idx = None
            n_feas = int(((status & ST_FEAS) != 0).sum().item())
        else:
            feas_idx = eng.select(status, ST_FEAS, ST_FEAS)
            n_feas = int(feas_idx.shape[0])
        if any_flag & (ST_THIN | ST_BORDER):
            _collect_flags(eng, masks, status, flagged)
        if collect_status:
            statuses.append((masks.cpu().numpy(), status.cpu().numpy()))
        if digest:
            sums.append((n, _checksum(status)))
        keep = {} if wit is not None else None
        nxt = eng.children(masks, feas_idx, k_act, dist if world > 1 else None, keep) if not last else eng.empty((0, eng.W), torch.int64)
        if keep:
            parent = ParentLevel(keep['feas_masks'], keep['ws'], keep['nf'], wit[feas_idx].contiguous())
        torch.cuda.synchronize(eng.tdev)
        total += n
        stats.append(dict(level=lvl + 1, candidates=n, feasible=n_feas, optimal=n_opt, regions=n_reg,
                          seconds=time.perf_counter() - t0))
        masks = nxt
    frontier = int(masks.shape[0])
    # base (equality-only) active set, tested last (mpqp_combinatorial.py:65-70)
    base_status = 0
    if complete:
        m0 = torch.zeros((1, eng.W), dtype=torch.int64, device=eng.tdev)
        st0 = eng.level_eval(m0, 0)
        sel0 = eng.select(st0, ST_OPT, ST_OPT)
        if sel0.shape[0] and emit_regions:
            laws, rows, flags, info = [x.cpu().numpy() for x in eng.emit(m0, sel0, 0, st0)]
            if info[0, 0] < 0:
                raise numpy.linalg.LinAlgError('Singular matrix')
            reg = build_regions(eng, cr_cls, [list(range(eng.n_eq))], 0, laws, rows, flags, info)[0]
            # region.is_full_dimension(): Chebyshev radius of (E, f) > 1e-8 (critical_region.py:89-105)
            if reg is not None and info[0, 1] > 1e-8:
                regions.append(reg)
        base_status = int(st0.cpu().numpy()[0])
    solution = sol_cls(program, regions)
    solution.level_stats = stats
    solution.total_candidates = total
    solution.frontier = frontier
    solution.base_status = base_status
    solution.engine_counters = eng.counters()
    solution.gpu_launches = eng.launch_count()
    solution.h2d_bytes, solution.d2h_bytes = eng.h2d_bytes, eng.d2h_bytes
    solution.flagged = flagged
    if collect_status:
        solution.level_status = statuses
    if digest:
        import hashlib
        hh = hashlib.sha256(repr(sums).encode())
        if materialize:
            hh.update(repr([tuple(r.active_set) for r in regions]).encode())
        solution.digest = hh.hexdigest()
    if own:
        eng.close()
    return solution
