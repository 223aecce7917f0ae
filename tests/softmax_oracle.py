"""ctypes access to tests/softmax_oracle.c — TEST INFRASTRUCTURE ONLY (the CPU restatement of spmm_b200_edge_softmax and
its backward).

The shared object is compiled on first use into the system's temporary directory, keyed by the source's hash, so the
repository tree is never written to.
"""
from __future__ import annotations

import ctypes as C
import hashlib
import os
import subprocess
import tempfile

import numpy as np

_SRC = os.path.join(os.path.dirname(os.path.abspath(__file__)), "softmax_oracle.c")


def _load():
    src = open(_SRC, "rb").read()
    tag = hashlib.sha1(src).hexdigest()[:16]
    so = os.path.join(tempfile.gettempdir(), f"hpc_b200_softmax_oracle_{os.getuid()}_{tag}.so")
    if not os.path.exists(so):
        tmp = f"{so}.{os.getpid()}.tmp"
        subprocess.run(["gcc", "-O3", "-mavx2", "-mfma", "-ffp-contract=off", "-fopenmp", "-fPIC", "-shared", "-o", tmp,
                        _SRC, "-lm"], check=True, capture_output=True)
        os.replace(tmp, so)
    lib = C.CDLL(so)
    P, I, LL = C.c_void_p, C.c_int, C.c_longlong
    lib.oracle_edge_softmax_f32.argtypes = [P, P, P, I, I, I]
    lib.oracle_edge_softmax_f32.restype = None
    lib.oracle_edge_softmax_backward_f32.argtypes = [P, P, P, P, I, I, I]
    lib.oracle_edge_softmax_backward_f32.restype = None
    lib.oracle_softmax_exp_array.argtypes = [P, P, LL, I]
    lib.oracle_softmax_exp_array.restype = None
    lib.oracle_softmax_exp_check.argtypes = [I, I, P]
    lib.oracle_softmax_exp_check.restype = None
    return lib


_lib = _load()


def _p(a):
    return a.ctypes.data_as(C.c_void_p)


def edge_softmax_f32(ptr, s, ftz=True, nthreads=0):
    """out = row softmax of s over the CSR rows of ptr, in the engine's order (edge_softmax.cu)."""
    ptr = np.ascontiguousarray(ptr, np.int32)
    s = np.ascontiguousarray(s, np.float32)
    out = np.empty(int(ptr[-1]), np.float32)
    _lib.oracle_edge_softmax_f32(_p(ptr), _p(s), _p(out), len(ptr) - 1, int(bool(ftz)), int(nthreads))
    return out


def edge_softmax_backward_f32(ptr, p, dp, ftz=True, nthreads=0):
    """ds = p * (dp - rowsum(p * dp)) in the engine's order."""
    ptr = np.ascontiguousarray(ptr, np.int32)
    p = np.ascontiguousarray(p, np.float32)
    dp = np.ascontiguousarray(dp, np.float32)
    ds = np.empty(int(ptr[-1]), np.float32)
    _lib.oracle_edge_softmax_backward_f32(_p(ptr), _p(p), _p(dp), _p(ds), len(ptr) - 1, int(bool(ftz)), int(nthreads))
    return ds


def softmax_exp(x, ftz=True):
    """The engine's exp routine (defined for x <= 0), elementwise."""
    x = np.ascontiguousarray(x, np.float32)
    y = np.empty_like(x)
    _lib.oracle_softmax_exp_array(_p(x), _p(y), x.size, int(bool(ftz)))
    return y


def softmax_exp_check(ftz=True, nthreads=0):
    """-> (values checked, violations, worst ulp) of the exp contract over every float32 in [-87.5, 0]."""
    stats = np.zeros(3, np.float64)
    _lib.oracle_softmax_exp_check(int(bool(ftz)), int(nthreads), _p(stats))
    return int(stats[0]), int(stats[1]), float(stats[2])
