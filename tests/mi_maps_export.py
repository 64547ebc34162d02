"""ctypes binding of tests/mi_maps_export.cpp: the y maps of a mixed-integer program's continuous part, as
host_math.hpp::parameter_column_maps builds them.  TEST INFRASTRUCTURE.

The library is compiled on first use into a directory under the system temporary directory, named by a hash of its
sources, so the repository tree is never written to."""
import ctypes
import hashlib
import os
import subprocess
import tempfile

import numpy

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
SOURCES = [os.path.join(HERE, 'mi_maps_export.cpp'), os.path.join(ROOT, 'ppopt_b200', 'csrc', 'host_math.hpp')]
_lib = None


def lib():
    global _lib
    if _lib is None:
        h = hashlib.sha256()
        for p in SOURCES:
            with open(p, 'rb') as f:
                h.update(f.read())
        out_dir = os.path.join(tempfile.gettempdir(), 'ppopt_b200_mi_maps_export')
        os.makedirs(out_dir, exist_ok=True)
        path = os.path.join(out_dir, f'libmi_maps_export_{h.hexdigest()[:16]}.so')
        if not os.path.exists(path):
            tmp = f'{path}.{os.getpid()}.tmp'
            subprocess.check_call([os.environ.get('CXX', 'g++'), '-O2', '-std=c++17', '-fPIC', '-shared', '-o', tmp, SOURCES[0]])
            os.replace(tmp, path)
        l = ctypes.CDLL(path)
        l.mimaps_build.restype = ctypes.c_int
        l.mimaps_build.argtypes = [ctypes.c_int] * 6 + [ctypes.c_void_p] * 8 + [ctypes.c_int] + [ctypes.c_void_p] * 3 + \
            [ctypes.c_int] + [ctypes.c_void_p] * 4 + [ctypes.c_char_p, ctypes.c_int]
        _lib = l
    return _lib


def _c(a, dtype=numpy.float64):
    return numpy.ascontiguousarray(numpy.asarray(a, dtype=dtype))


def param_maps(A, b, F, A_t, b_t, n_eq, c, H, Q, Fy, Hy=None):
    """(maps (rows x ny), lp_bvar, lp_nvar, Q2) of the continuous program (equality rows 0..n_eq-1) with the extra parameter
    columns Fy (m x ny) on the right-hand side and Hy (n x ny) on the linear term; ValueError with the builder's message"""
    A, F = _c(A), _c(F)
    m, n = A.shape
    t = F.shape[1]
    Fy = _c(Fy).reshape(m, -1)
    ny = Fy.shape[1]
    keep = [A, _c(b).ravel(), F, _c(A_t).reshape(-1, t), _c(b_t).ravel(), None if Q is None else _c(Q), _c(c).ravel(), _c(H),
            Fy, None if Hy is None else _c(Hy)]
    max_rows = 2 * m + 2 * n
    maps = numpy.zeros((max_rows, ny))
    rows = ctypes.c_int(0)
    bvar, nvar = numpy.zeros(max(m, 1), numpy.int32), numpy.zeros(max(n, 1), numpy.int32)
    q2 = numpy.zeros((n, max(n - n_eq, 1)))
    err = ctypes.create_string_buffer(512)
    ptr = lambda x: None if x is None else x.ctypes.data  # noqa: E731
    rc = lib().mimaps_build(n, t, m, keep[3].shape[0], int(n_eq), int(Q is not None), *[ptr(x) for x in keep[:8]], ny, ptr(Fy),
                            ptr(keep[9]), maps.ctypes.data, max_rows, ctypes.byref(rows), bvar.ctypes.data, nvar.ctypes.data, q2.ctypes.data,
                            err, 512)
    if rc:
        raise ValueError(err.value.decode())
    return maps[:rows.value], bvar[:m - n_eq], nvar[:n - n_eq], q2[:, :n - n_eq]
