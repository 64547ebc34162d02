"""Which binary assignments of a mixed-integer program are feasible: a breadth-first relaxation tree on the GPU (K11,
csrc/k11_mitree.cu), without a MILP solver.

The reference finds them with ``MITree`` (mitree.py) and ``check_bin_feasibility`` (mpmilp_program.py), one Gurobi MILP per
node.  Here a node at depth d fixes y_0..y_{d-1} and answers the LP RELAXATION of the lifted system

    z = (x, theta),   A x - F theta <= b  (= b on the equality rows),   A_t theta <= b_t,   l_k <= y_k <= u_k,

with the unfixed binaries relaxed to [0, 1].  An inner node therefore answers its relaxation, not the reference's MILP:
pruning an infeasible relaxation is sound (no leaf below it is feasible), and a leaf, where every binary is fixed, answers
exactly the LP the MILP reduces to, Theta's rows included.  So the leaves equal those of the reference's tree, except for
assignments whose margin lies within the feasibility tolerance (PPG_FEAS_TOL (1 + |rhs|) per row).  The 2^nb screen of
mpmiqp_enumeration (``leaf_is_feasible``) keeps a few assignments more: on the random test programs, assignments that HiGHS
rejects on the lifted LP, nearly all of them ruled out by Theta's rows alone (tests/test_gpu_mitree.py).

One depth is one batch in device memory: the nodes are evaluated one warp each (Phase 1 of the lifted LP), the feasible
ones are compacted in order and each writes its two children, y_d = 0 before y_d = 1, so that the leaves come out in
lexicographic order of (y_0, y_1, ...) - the order of ``itertools.product((0, 1), repeat=nb)``.  The host reads one count
per depth.  With ``inherit``, a feasible node keeps its Phase-1 point, and a child whose parent's point, with the new
binary snapped to the child's value, still satisfies every row is feasible without an LP (never used to decide
infeasibility).  Off by default: a depth of a few thousand nodes does not fill the GPU, so its time is the latency of its
longest LP, which inheritance does not shorten, while the point writes and the check cost extra (8.3-11.6 against
7.3-8.8 ms for nb = 16, 33.8-33.9 against 23.0-23.4 ms for nb = 40 on a B200, profiles/r07_mitree_bench.txt).  The points of a depth are kept only
while they fit ``point_budget`` bytes: a wider depth hands its children to the LP.

    res = feasible_combinations(program)     # res.leaves: [[y_0, ..., y_{nb-1}], ...];  res.stats: per depth
"""
import ctypes
import os
from dataclasses import dataclass, field
from typing import Dict, List, Optional

import numpy
import torch

from .. import _lib

TREE_FEASIBLE, TREE_INFEASIBLE, TREE_ITERLIM, TREE_NUMERIC = 0, 1, 2, 3   # PPG_TREE_* / PPG_TLP_* (csrc/tolerances.h)


def _f64(a, rows, cols):
    a = numpy.asarray(a if a is not None else numpy.zeros((rows, cols)), dtype=numpy.float64)
    return numpy.ascontiguousarray(a.reshape(rows, cols))


def lifted_arrays(program):
    """(A, b, F, A_t, b_t, n_eq, binary_indices) of a program with its equality rows moved to the front.  Reads the
    attributes of a ppopt MPMILP_Program / MPMIQP_Program (or any object with A, b, F, A_t, b_t, equality_indices,
    binary_indices)."""
    A = numpy.asarray(program.A, dtype=numpy.float64)
    A = A.reshape(-1, A.shape[-1])
    m = A.shape[0]
    A_t = numpy.asarray(program.A_t, dtype=numpy.float64)
    t = A_t.shape[-1]
    A_t = A_t.reshape(-1, t)
    F = _f64(program.F, m, t)
    b = _f64(program.b, m, 1).ravel()
    b_t = _f64(program.b_t, A_t.shape[0], 1).ravel()
    eq = sorted(int(i) for i in (getattr(program, 'equality_indices', None) or []))
    order = eq + [i for i in range(m) if i not in set(eq)]
    return (numpy.ascontiguousarray(A[order]), numpy.ascontiguousarray(b[order]), numpy.ascontiguousarray(F[order]),
            numpy.ascontiguousarray(A_t), numpy.ascontiguousarray(b_t), len(eq), [int(i) for i in program.binary_indices])


class RelaxationTree:
    """The device handle of one program's tree (``ppgpu_tree_*``).  Nodes are int64 tensors on the device: bit k = y_k for
    k < depth."""

    def __init__(self, program, inherit: bool = False, device=None):
        self.lib = _lib.load()
        A, b, F, A_t, b_t, ne, binary = lifted_arrays(program)
        self.nb, self.n, self.t = len(binary), A.shape[1], F.shape[1]
        self.nv = self.n + self.t
        self.device = torch.cuda.current_device() if device is None else int(device)
        self.tdev = torch.device('cuda', self.device)
        dims = _lib.Dims(n=self.n, t=self.t, m=A.shape[0], q=A_t.shape[0], n_eq=ne, is_qp=0)
        bins = numpy.ascontiguousarray(binary, dtype=numpy.int32)
        self._keep = (A, b, F, A_t, b_t, bins)
        h = ctypes.c_void_p()
        _lib.check(self.lib.ppgpu_tree_create(dims, bins.ctypes.data, self.nb, A.ctypes.data, b.ctypes.data, F.ctypes.data,
                                              A_t.ctypes.data, b_t.ctypes.data, self.device, h), 'ppgpu_tree_create')
        self.h = h.value
        self.inherit = bool(inherit)
        _lib.check(self.lib.ppgpu_tree_set_option(self.h, _lib.TREE_OPT_INHERIT, int(self.inherit)), 'ppgpu_tree_set_option')

    def close(self):
        if getattr(self, 'h', None):
            self.lib.ppgpu_tree_destroy(self.h)
            self.h = None

    def __del__(self):
        self.close()

    def _stream(self):
        return torch.cuda.current_stream(self.tdev).cuda_stream

    @staticmethod
    def _ptr(x):
        return None if x is None else x.data_ptr()

    def eval(self, nodes, depth: int, points: bool = True, parent_point=None, parent_of=None):
        """(status uint8, point float64 n x (n + t) or None, iters int32: pivots, -1 where the node inherited its point)"""
        n = nodes.numel()
        status = torch.empty(n, dtype=torch.uint8, device=self.tdev)
        iters = torch.empty(n, dtype=torch.int32, device=self.tdev)
        point = torch.empty((n, self.nv), dtype=torch.float64, device=self.tdev) if points else None
        _lib.check(self.lib.ppgpu_tree_eval(self.h, nodes.data_ptr(), n, int(depth), status.data_ptr(), self._ptr(point),
                                            self._ptr(parent_point), self._ptr(parent_of), iters.data_ptr(), self._stream()),
                   'ppgpu_tree_eval')
        return status, point, iters

    def children(self, nodes, status, depth: int):
        """(children int64 2 nf, parent_of int64 2 nf): the nodes with status 0 in order, each followed by its children"""
        n = nodes.numel()
        idx = torch.empty(n, dtype=torch.int64, device=self.tdev)
        ch = torch.empty(2 * n, dtype=torch.int64, device=self.tdev)
        po = torch.empty(2 * n, dtype=torch.int64, device=self.tdev)
        wsb = int(self.lib.ppgpu_select_workspace_bytes(n))
        ws = torch.empty(max(wsb, 8), dtype=torch.uint8, device=self.tdev)
        cnt = ctypes.c_int64(0)
        _lib.check(self.lib.ppgpu_tree_children(self.h, nodes.data_ptr(), status.data_ptr(), n, int(depth), idx.data_ptr(),
                                                ch.data_ptr(), po.data_ptr(), ctypes.byref(cnt), ws.data_ptr(), wsb,
                                                self._stream()), 'ppgpu_tree_children')
        k = 2 * cnt.value
        return ch[:k], po[:k]


@dataclass
class TreeResult:
    leaves: List[List[int]]
    # per depth 0..nb: nodes evaluated, feasible nodes, LPs solved, nodes that inherited their parent's point, pivots
    stats: Dict[str, List[int]] = field(default_factory=dict)


def feasible_combinations(program, max_leaves: int = 1 << 22, inherit: Optional[bool] = None, point_budget: int = 1 << 30,
                          device=None) -> TreeResult:
    """The binary assignments whose relaxation is feasible, in tree (lexicographic) order, and statistics per depth.
    ``max_leaves``: more feasible nodes than this at any depth (the leaves included) raise ValueError before the next depth
    is allocated.  ``inherit``: point inheritance (None: the environment's PPGPU_TREE_INHERIT, off unless it is 1).
    ``point_budget``: bytes of Phase-1 points kept per depth for the children's inheritance."""
    if inherit is None:
        inherit = os.environ.get('PPGPU_TREE_INHERIT', '0') == '1'
    tree = RelaxationTree(program, inherit=inherit, device=device)
    try:
        stats = {k: [] for k in ('nodes', 'feasible', 'lps', 'inherited', 'pivots')}
        nodes = torch.zeros(1, dtype=torch.int64, device=tree.tdev)
        parent_point = parent_of = None
        leaves = []
        for d in range(tree.nb + 1):
            n = nodes.numel()
            keep = d < tree.nb and inherit and n * tree.nv * 8 <= point_budget
            status, point, iters = tree.eval(nodes, d, points=keep, parent_point=parent_point, parent_of=parent_of)
            counts = torch.stack([(status == TREE_FEASIBLE).sum(), (iters >= 0).sum(), (iters < 0).sum(),
                                  iters.clamp(min=0).sum(dtype=torch.int64), (status > TREE_INFEASIBLE).sum()]).tolist()
            for k, v in zip(('nodes', 'feasible', 'lps', 'inherited', 'pivots'), [n] + counts[:4]):
                stats[k].append(int(v))
            if counts[4]:
                raise RuntimeError(f'relaxation tree: {counts[4]} node LPs at depth {d} hit the iteration cap or broke down '
                                   'numerically; their feasibility is undecided')
            if counts[0] > max_leaves:
                raise ValueError(f'relaxation tree: {counts[0]} feasible nodes at depth {d} exceed max_leaves = {max_leaves}')
            if d == tree.nb:
                v = nodes[status == TREE_FEASIBLE].cpu().numpy()
                bits = (v[:, None] >> numpy.arange(tree.nb, dtype=numpy.int64)[None, :]) & 1
                leaves = bits.astype(int).tolist()
                break
            nodes, parent_of = tree.children(nodes, status, d)
            parent_point = point
        return TreeResult(leaves, stats)
    finally:
        tree.close()
