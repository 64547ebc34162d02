"""ctypes binding of tests/lp_dict_export.cpp: the K9 start dictionary of a program, as reduce_program builds it.
TEST INFRASTRUCTURE.

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
SOURCES = [os.path.join(HERE, 'lp_dict_export.cpp'), os.path.join(ROOT, 'ppopt_b200', 'csrc', 'host_math.hpp'),
           os.path.join(ROOT, 'ppopt_b200', 'csrc', 'tolerances.h')]
_lib = None


def lib():
    global _lib
    if _lib is None:
        h = hashlib.sha256()
        for p in SOURCES:
            with open(p, 'rb') as f:
                h.update(f.read())
        out_dir = os.path.join(tempfile.gettempdir(), 'ppopt_b200_lp_dict_export')
        os.makedirs(out_dir, exist_ok=True)
        path = os.path.join(out_dir, f'liblp_dict_export_{h.hexdigest()[:16]}.so')
        if not os.path.exists(path):
            tmp = f'{path}.{os.getpid()}.tmp'
            subprocess.check_call([os.environ.get('CXX', 'g++'), '-O2', '-std=c++17', '-fPIC', '-shared', '-o', tmp, SOURCES[0]])
            os.replace(tmp, path)
        l = ctypes.CDLL(path)
        l.lpdict_create.restype = ctypes.c_void_p
        l.lpdict_create.argtypes = [ctypes.c_int] * 6 + [ctypes.c_void_p] * 8
        l.lpdict_destroy.argtypes = [ctypes.c_void_p]
        l.lpdict_get.argtypes = [ctypes.c_void_p] * 8
        _lib = l
    return _lib


def _c(a):
    return numpy.ascontiguousarray(numpy.asarray(a, dtype=numpy.float64))


def lp_dict(A, b, F, A_t, b_t, Q, c, H, n_eq, is_qp=False):
    """start dictionary of K9: dict(D0 [beta0 | D | Dth], bvar, nvar, obj [d0 | dth], X0t [x0 | Xt], Q2), or None when the
    reduced rows have no vertex or the program is a QP"""
    A, F = _c(A), _c(F)
    n, t, m = A.shape[1], F.shape[1], A.shape[0]
    A_t = _c(A_t).reshape(-1, t)
    Q = _c(Q) if is_qp else numpy.zeros((n, n))
    keep = [A, _c(b).ravel(), F, A_t, _c(b_t).ravel(), Q, _c(c).ravel(), _c(H)]
    h = lib().lpdict_create(n, t, m, A_t.shape[0], int(n_eq), int(is_qp), *[x.ctypes.data for x in keep])
    if not h:
        raise RuntimeError('reduce_program failed')
    try:
        ld = ctypes.c_int(0)
        if not lib().lpdict_get(h, ctypes.byref(ld), None, None, None, None, None, None):
            return None
        mi, npr = m - int(n_eq), n - int(n_eq)
        out = dict(D0=numpy.zeros((mi, ld.value)), bvar=numpy.zeros(mi, dtype=numpy.int32), nvar=numpy.zeros(npr, dtype=numpy.int32),
                   obj=numpy.zeros((npr, t + 1)), X0t=numpy.zeros((n, t + 1)), Q2=numpy.zeros((n, npr)))
        lib().lpdict_get(h, ctypes.byref(ld), *[out[k].ctypes.data for k in ('D0', 'bvar', 'nvar', 'obj', 'X0t', 'Q2')])
        return out
    finally:
        lib().lpdict_destroy(h)
