"""ctypes binding of tests/tree_dict_export.cpp: the K11 lifted system of a mixed-integer program, as build_tree_dictionary
builds it.  TEST INFRASTRUCTURE.

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
SOURCES = [os.path.join(HERE, 'tree_dict_export.cpp'), os.path.join(ROOT, 'ppopt_b200', 'csrc', 'host_math.hpp')]
_lib = None


def lib():
    global _lib
    if _lib is None:
        h = hashlib.sha256()
        for p in SOURCES:
            with open(p, 'rb') as f:
                h.update(f.read())
        out_dir = os.path.join(tempfile.gettempdir(), 'ppopt_b200_tree_dict_export')
        os.makedirs(out_dir, exist_ok=True)
        path = os.path.join(out_dir, f'libtree_dict_export_{h.hexdigest()[:16]}.so')
        if not os.path.exists(path):
            tmp = f'{path}.{os.getpid()}.tmp'
            subprocess.check_call([os.environ.get('CXX', 'g++'), '-O2', '-std=c++17', '-fPIC', '-shared', '-o', tmp, SOURCES[0]])
            os.replace(tmp, path)
        l = ctypes.CDLL(path)
        l.treedict_create.restype = ctypes.c_void_p
        l.treedict_create.argtypes = [ctypes.c_int] * 6 + [ctypes.c_void_p] * 6 + [ctypes.c_char_p, ctypes.c_int]
        l.treedict_destroy.argtypes = [ctypes.c_void_p]
        l.treedict_dims.argtypes = [ctypes.c_void_p, ctypes.c_void_p]
        l.treedict_get.argtypes = [ctypes.c_void_p] * 7
        _lib = l
    return _lib


def _c(a, dtype=numpy.float64):
    return numpy.ascontiguousarray(numpy.asarray(a, dtype=dtype))


def tree_dict(A, b, F, A_t, b_t, n_eq, binary_indices):
    """the lifted system of K11 (equality rows 0..n_eq-1): dict(nv, rows, cols, rb0, tp, D0 [beta0 | D | Dbnd], bvar, nvar,
    hs, z0, Q2); raises ValueError with the builder's message when it refuses the program"""
    A, F = _c(A), _c(F)
    n, t, m = A.shape[1], F.shape[1], A.shape[0]
    A_t = _c(A_t).reshape(-1, t)
    bins = _c(binary_indices, numpy.int32)
    keep = [bins, A, _c(b).ravel(), F, A_t, _c(b_t).ravel()]
    err = ctypes.create_string_buffer(512)
    h = lib().treedict_create(n, t, m, A_t.shape[0], int(n_eq), len(bins), *[x.ctypes.data for x in keep], err, 512)
    if not h:
        raise ValueError(err.value.decode())
    try:
        dims = numpy.zeros(6, dtype=numpy.int32)
        lib().treedict_dims(h, dims.ctypes.data)
        nv, rows, cols, rb0, tp, ld = (int(x) for x in dims)
        out = dict(nv=nv, rows=rows, cols=cols, rb0=rb0, tp=tp, D0=numpy.zeros((rows, ld)), bvar=numpy.zeros(rows, numpy.int32),
                   nvar=numpy.zeros(cols, numpy.int32), hs=numpy.zeros(rows), z0=numpy.zeros(nv), Q2=numpy.zeros((nv, cols)))
        lib().treedict_get(h, *[out[k].ctypes.data for k in ('D0', 'bvar', 'nvar', 'hs', 'z0', 'Q2')])
        return out
    finally:
        lib().treedict_destroy(h)
