"""Batched Chebyshev balls on the GPU (csrc/k34c_compact.cu::cheb_batch_kernel through ppgpu_chebyshev_batch).

Reference: chebyshev_ball (/root/reference/src/ppopt/utils/chebyshev_ball.py:10-63), used by
CriticalRegion.is_full_dimension (critical_region.py:89-105) and by the program constructor's warnings()
(mplp_program.py:204-215, feasible_space_chebychev_ball).  One call answers any number of polytopes."""
import ctypes
from typing import List, Sequence, Tuple

import numpy
import torch

from . import _lib

RADIUS_TOL = 1e-8   # full dimensional iff radius > 1e-8 (critical_region.py:105, mpqp_utils.py:343)


def chebyshev_radii(polytopes: Sequence[Tuple[numpy.ndarray, numpy.ndarray]], device=None) -> numpy.ndarray:
    """radius of the largest ball inside {theta : E theta <= f} for every (E, f); +inf unbounded, negative/-inf empty"""
    if not torch.cuda.is_available():
        raise RuntimeError('ppopt_b200 needs a CUDA device (there is no CPU fallback)')
    lib = _lib.load()
    if len(polytopes) == 0:
        return numpy.zeros(0)
    t = int(numpy.asarray(polytopes[0][0]).reshape(len(numpy.asarray(polytopes[0][1]).reshape(-1)), -1).shape[1])
    blocks, off = [], [0]
    for E, f in polytopes:
        f = numpy.asarray(f, dtype=numpy.float64).reshape(-1, 1)
        E = numpy.asarray(E, dtype=numpy.float64).reshape(f.shape[0], -1)
        if E.shape[1] != t:
            raise ValueError('all polytopes of a batch must live in the same parameter space')
        blocks.append(numpy.hstack([f, E]))
        off.append(off[-1] + f.shape[0])
    rows = numpy.ascontiguousarray(numpy.vstack(blocks)) if off[-1] else numpy.zeros((1, t + 1))
    max_rows = max(1, max(b.shape[0] for b in blocks))
    dev = torch.device('cuda', torch.cuda.current_device() if device is None else device)
    d_rows = torch.from_numpy(rows).to(dev)
    d_off = torch.tensor(off, dtype=torch.int64, device=dev)
    d_rad = torch.empty(len(polytopes), dtype=torch.float64, device=dev)
    d_code = torch.empty(len(polytopes), dtype=torch.int32, device=dev)
    with torch.cuda.device(dev):
        rc = lib.ppgpu_chebyshev_batch(d_rows.data_ptr(), d_off.data_ptr(), len(polytopes), t, max_rows, d_rad.data_ptr(),
                                       d_code.data_ptr(), ctypes.c_void_p(torch.cuda.current_stream(dev).cuda_stream))
    _lib.check(rc, 'chebyshev_batch')
    return d_rad.cpu().numpy()


def facet_balls(rows: torch.Tensor, row_off: torch.Tensor, facets: torch.Tensor, t: int):
    """Chebyshev balls of facets (K10, ppgpu_facet_chebyshev_batch) on device tensors: rows (total x (t + 1), [f | E] of the
    stacked polytopes), row_off (n_polytopes + 1, int64), facets (n_facets x 2 int64: polytope, row of that polytope).
    Returns device tensors (centre n_facets x t, radius n_facets, code n_facets int32); the ball lies in the facet's hyperplane
    E_i theta = f_i.  radius +inf unbounded, negative / -inf empty; centre NaN unless code is 0 (optimal), except for t = 1
    where it is the facet's point whenever the facet is not empty."""
    lib = _lib.load()
    dev = rows.device
    rows = rows.to(torch.float64).contiguous()
    row_off = row_off.to(torch.int64).contiguous()
    facets = facets.to(torch.int64).reshape(-1, 2).contiguous()
    nf, n_poly = facets.shape[0], row_off.shape[0] - 1
    center = torch.empty((nf, t), dtype=torch.float64, device=dev)
    radius = torch.empty((nf,), dtype=torch.float64, device=dev)
    code = torch.empty((nf,), dtype=torch.int32, device=dev)
    if nf:
        max_rows = max(1, int((row_off[1:] - row_off[:-1]).max().item())) if n_poly > 0 else 1
        with torch.cuda.device(dev):
            rc = lib.ppgpu_facet_chebyshev_batch(rows.data_ptr(), row_off.data_ptr(), n_poly, t, max_rows, facets.data_ptr(), nf,
                                                 center.data_ptr(), radius.data_ptr(), code.data_ptr(),
                                                 ctypes.c_void_p(torch.cuda.current_stream(dev).cuda_stream))
        _lib.check(rc, 'facet_chebyshev_batch')
    return center, radius, code


def full_dimensional(regions: List) -> List[bool]:
    """CriticalRegion.is_full_dimension() for a list of regions in one launch"""
    rad = chebyshev_radii([(r.E, r.f) for r in regions])
    return [bool(x > RADIUS_TOL) for x in rad]
