"""ctypes binding of the CPU twin of the K8 fixed-theta QP kernel (tests/twin_theta_qp.cpp).  TEST INFRASTRUCTURE.

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
SOURCES = [os.path.join(HERE, 'twin_theta_qp.cpp'), os.path.join(ROOT, 'ppopt_b200', 'csrc', 'host_math.hpp'),
           os.path.join(ROOT, 'ppopt_b200', 'csrc', 'tolerances.h')]
_lib = None


def lib():
    global _lib
    if _lib is None:
        h = hashlib.sha256()
        for p in SOURCES:
            with open(p, 'rb') as f:
                h.update(f.read())
        out_dir = os.path.join(tempfile.gettempdir(), 'ppopt_b200_twin_theta_qp')
        os.makedirs(out_dir, exist_ok=True)
        path = os.path.join(out_dir, f'libtwin_theta_qp_{h.hexdigest()[:16]}.so')
        if not os.path.exists(path):
            tmp = f'{path}.{os.getpid()}.tmp'
            subprocess.check_call([os.environ.get('CXX', 'g++'), '-O2', '-std=c++17', '-fPIC', '-shared', '-o', tmp, SOURCES[0]])
            os.replace(tmp, path)
        l = ctypes.CDLL(path)
        l.k8twin_create.restype = ctypes.c_void_p
        l.k8twin_create.argtypes = [ctypes.c_int] * 6 + [ctypes.c_void_p] * 8
        l.k8twin_destroy.argtypes = [ctypes.c_void_p]
        l.k8twin_words.argtypes = [ctypes.c_void_p]
        l.k8twin_use_gram.argtypes = [ctypes.c_void_p]
        l.k8twin_theta_qp.argtypes = [ctypes.c_void_p, ctypes.c_void_p, ctypes.c_long] + [ctypes.c_void_p] * 6
        _lib = l
    return _lib


def _c(a):
    return numpy.ascontiguousarray(numpy.asarray(a, dtype=numpy.float64))


class ThetaQpTwin:
    """Sequential restatement of K8 on one program (same reduction, rules, tie-breaks and constants as the kernel)."""

    def __init__(self, A, b, F, A_t, b_t, Q, c, H, n_eq, is_qp=True):
        A, F = _c(A), _c(F)
        self.n, self.t, self.m = A.shape[1], F.shape[1], A.shape[0]
        A_t = _c(A_t).reshape(-1, self.t)
        self.q, self.n_eq, self.is_qp = A_t.shape[0], int(n_eq), bool(is_qp)
        Q = _c(Q) if is_qp else numpy.zeros((self.n, self.n))
        self._keep = [A, _c(b).ravel(), F, A_t, _c(b_t).ravel(), Q, _c(c).ravel(), _c(H)]
        self.h = lib().k8twin_create(self.n, self.t, self.m, self.q, self.n_eq, int(self.is_qp), *[x.ctypes.data for x in self._keep])
        if not self.h:
            raise RuntimeError('program reduction failed')
        self.W = lib().k8twin_words(self.h)
        self.use_gram = bool(lib().k8twin_use_gram(self.h))

    @classmethod
    def from_npz(cls, path):
        g = numpy.load(path)
        is_qp = str(g['kind']) == 'qp'
        return cls(g['A'], g['b'], g['F'], g['A_t'], g['b_t'], g['Q'] if is_qp else None, g['c'], g['H'], int(g['n_eq']), is_qp)

    def theta_qp(self, thetas):
        """thetas (n x t) -> dict of status (uint8), x (n x num_x), dual (n x m: equality multipliers, then lambda), mask
        (n x W uint64 working sets), iters (int32) and margin (smallest distance of any decision from its threshold or
        runner-up).  Raises NotImplementedError without Gram data."""
        th = _c(thetas).reshape(-1, self.t)
        k = th.shape[0]
        out = dict(status=numpy.zeros(k, dtype=numpy.uint8), x=numpy.zeros((k, self.n)), dual=numpy.zeros((k, self.m)),
                   mask=numpy.zeros((k, self.W), dtype=numpy.uint64), iters=numpy.zeros(k, dtype=numpy.int32),
                   margin=numpy.zeros(k))
        rc = lib().k8twin_theta_qp(self.h, th.ctypes.data, k,
                                   *[out[f].ctypes.data for f in ('status', 'x', 'dual', 'mask', 'iters', 'margin')])
        if rc == -2:
            raise NotImplementedError('fixed-theta QP needs a positive definite reduced Hessian (use_gram)')
        return out

    def __del__(self):
        try:
            if self.h:
                lib().k8twin_destroy(self.h)
        except Exception:
            pass
