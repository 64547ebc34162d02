"""Batched point location and law evaluation on the GPU (SURVEY.md section 8f row 4 - the step right after the hot path).

Mirrors the reference's `upop.PointLocation` (/root/reference/src/ppopt/upop/point_location.py:10-133: same constructor,
`locate`, `evaluate`, `is_inside`) and adds the batched forms `locate_batch` / `evaluate_batch`, which run as ONE launch of
the K7 kernel (csrc/k7_locate.cu) through `ppgpu_locate_points`.  Region matrices are stacked once at construction, the
way the reference stacks `E` / `f` (`point_location.py:27-38`), and stay in HBM.

Acceptance rule: `tol=None` reproduces PointLocation (inside iff all(E theta <= f)); a number reproduces
`Solution.get_region_no_overlap` with that `point_location_tolerance` (all(E theta - f < tol), solution.py:75-88,
critical_region.py:81-84).  Overlapping solutions (the flag `solve_mpqp` leaves on its results, solve_mpqp.py:105-112)
use the reference's rule as well: among the containing regions the one with the lowest objective, ties to the later
region (solution.py:90-112, upop/point_location.py:68-84).  On a facet shared by two regions the two objectives agree to
rounding, so which of the two is reported is noise in the reference too; the objective of the reported region is what
is comparable.  Regions with fixed binaries (``y_fixation``, from solve_mpmiqp) are located the same way: their laws are
stacked over the full variable vector (``x_indices`` rows from A / b, ``y_indices`` rows the constant assignment), and the
overlap rule compares the full program's objective (Q, H, c), as Solution.get_region does; at most 128 variables.  No CPU
fallback.
"""
import ctypes
from typing import Optional, Tuple

import numpy
import torch

from . import _lib


class PointLocation:
    def __init__(self, solution, device: int = 0):
        if not torch.cuda.is_available():
            raise RuntimeError('ppopt_b200 needs a CUDA device (there is no CPU fallback)')
        self.solution = solution
        self.lib = _lib.load()
        regions = solution.critical_regions
        self.num_regions = len(regions)
        self.t = int(regions[0].E.shape[1]) if regions else int(solution.program.num_t())
        # regions with fixed binaries (solve_mpmiqp): laws over the full variable vector, binary rows constant y
        fixed = [getattr(r, 'y_fixation', None) is not None for r in regions]
        if any(fixed) and not all(fixed):
            raise ValueError('either every region or none fixes binaries')
        self.mixed_integer = bool(fixed) and all(fixed)
        if self.mixed_integer:
            self.n_x = len(regions[0].x_indices) + len(regions[0].y_indices)
            if self.n_x > 128:
                raise NotImplementedError(f'point location of regions with fixed binaries supports at most 128 variables '
                                          f'(continuous + binary), not {self.n_x}')
        else:
            self.n_x = int(regions[0].A.shape[0]) if regions else int(solution.program.num_x())
        off = numpy.zeros(self.num_regions + 1, dtype=numpy.int64)
        for i, r in enumerate(regions):
            off[i + 1] = off[i] + r.E.shape[0]
        self.region_constraints = off
        rows = numpy.zeros((int(off[-1]), self.t + 1))
        laws = numpy.zeros((self.num_regions, self.n_x, self.t + 1))
        for i, r in enumerate(regions):
            rows[off[i]:off[i + 1], 0] = numpy.asarray(r.f, dtype=float).ravel()
            rows[off[i]:off[i + 1], 1:] = numpy.asarray(r.E, dtype=float)
            if self.mixed_integer:
                xi, yi = list(r.x_indices), list(r.y_indices)
                laws[i, xi, 0] = numpy.asarray(r.b, dtype=float).ravel()
                laws[i, xi, 1:] = numpy.asarray(r.A, dtype=float)
                laws[i, yi, 0] = numpy.asarray(r.y_fixation, dtype=float).ravel()
            else:
                laws[i, :, 0] = numpy.asarray(r.b, dtype=float).ravel()
                laws[i, :, 1:] = numpy.asarray(r.A, dtype=float)
        self.tdev = torch.device('cuda', device)
        self._rows = torch.from_numpy(rows).to(self.tdev)
        self._laws = torch.from_numpy(laws).to(self.tdev)
        self._off = torch.from_numpy(off).to(self.tdev)
        # objective data for the overlapping rule (program.evaluate_objective, mpqp_program.py:44-57 / mplp_program.py:158-160)
        self.overlapping = bool(getattr(solution, 'is_overlapping', False))
        self._Q = self._H = self._c = None
        if self.overlapping:
            prog = solution.program
            if prog is None:
                raise ValueError('an overlapping solution needs its program (objective comparison)')
            if self.n_x > 128:
                raise NotImplementedError('the overlapping rule supports at most 128 variables')
            f64 = lambda a: torch.from_numpy(numpy.ascontiguousarray(a, dtype=numpy.float64)).to(self.tdev)  # noqa: E731
            H = numpy.asarray(prog.H, dtype=float)
            if H.shape != (self.n_x, self.t):
                if H.shape == (self.t, self.n_x) and not H.any():
                    H = numpy.zeros((self.n_x, self.t))   # all-zero H of either orientation (SURVEY.md 8b)
                else:
                    raise ValueError(f'H must be {self.n_x} x {self.t}')
            self._H, self._c = f64(H), f64(numpy.asarray(prog.c, dtype=float).reshape(-1))
            if getattr(prog, 'Q', None) is not None:
                self._Q = f64(prog.Q)

    # ---- batched forms -----------------------------------------------------------------------------------------------
    def _run(self, thetas, tol: Optional[float], want_x: bool) -> Tuple[torch.Tensor, Optional[torch.Tensor]]:
        if torch.is_tensor(thetas):
            th = thetas.to(self.tdev, dtype=torch.float64)
        else:
            th = torch.from_numpy(numpy.ascontiguousarray(thetas, dtype=numpy.float64)).to(self.tdev)
        th = th.reshape(-1, self.t).contiguous()
        n = th.shape[0]
        region = torch.empty((n,), dtype=torch.int32, device=self.tdev)
        x = torch.empty((n, self.n_x), dtype=torch.float64, device=self.tdev) if want_x else None
        with torch.cuda.device(self.tdev):
            stream = ctypes.c_void_p(torch.cuda.current_stream(self.tdev).cuda_stream)
            _lib.check(self.lib.ppgpu_locate_points(th.data_ptr(), n, self.t, self._rows.data_ptr(), self._off.data_ptr(),
                                                    self.num_regions, self._laws.data_ptr(), self.n_x if (want_x or self.overlapping) else 0,
                                                    0 if tol is None else 1, 0.0 if tol is None else float(tol),
                                                    1 if self.overlapping else 0,
                                                    self._Q.data_ptr() if self._Q is not None else None,
                                                    self._H.data_ptr() if self._H is not None else None,
                                                    self._c.data_ptr() if self._c is not None else None,
                                                    region.data_ptr(), x.data_ptr() if want_x else None, stream),
                       'locate_points')
        return region, x

    def locate_batch(self, thetas, tol: Optional[float] = None) -> numpy.ndarray:
        """index of the first containing region per row of thetas (n_points x t), -1 where there is none"""
        return self._run(thetas, tol, False)[0].cpu().numpy()

    def evaluate_batch(self, thetas, tol: Optional[float] = None) -> Tuple[numpy.ndarray, numpy.ndarray]:
        """(region index, x*(theta)) per point; rows of x are NaN where no region contains the point"""
        region, x = self._run(thetas, tol, True)
        return region.cpu().numpy(), x.cpu().numpy()

    # ---- the reference's single-point interface ----------------------------------------------------------------------
    def locate(self, theta) -> int:
        return int(self.locate_batch(numpy.asarray(theta, dtype=float).reshape(1, -1))[0])

    def is_inside(self, theta) -> bool:
        return self.locate(theta) != -1

    def evaluate(self, theta) -> Optional[numpy.ndarray]:
        idx, x = self.evaluate_batch(numpy.asarray(theta, dtype=float).reshape(1, -1))
        if idx[0] < 0:
            return None
        return x[0].reshape(-1, 1)
