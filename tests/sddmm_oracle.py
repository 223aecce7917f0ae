"""ctypes access to tests/sddmm_oracle.c — TEST INFRASTRUCTURE ONLY (the CPU restatement of spmm_b200_sddmm).

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

_SRC = os.path.join(os.path.dirname(os.path.abspath(__file__)), "sddmm_oracle.c")


def _load():
    src = open(_SRC, "rb").read()
    tag = hashlib.sha1(src).hexdigest()[:16]
    so = os.path.join(tempfile.gettempdir(), f"hpc_b200_sddmm_oracle_{os.getuid()}_{tag}.so")
    if not os.path.exists(so):
        tmp = f"{so}.{os.getpid()}.tmp"
        subprocess.run(["gcc", "-O3", "-mavx2", "-mfma", "-ffp-contract=off", "-fopenmp", "-fPIC", "-shared", "-o", tmp,
                        _SRC, "-lm"], check=True, capture_output=True)
        os.replace(tmp, so)
    lib = C.CDLL(so)
    P, I = C.c_void_p, C.c_int
    lib.oracle_sddmm_f32.argtypes = [P, P, P, P, P, I, I, I, I]
    lib.oracle_sddmm_f32.restype = None
    lib.oracle_sddmm_f64.argtypes = [P, P, P, P, P, P, I, I, I]
    lib.oracle_sddmm_f64.restype = None
    return lib


_lib = _load()


def _p(a):
    return a.ctypes.data_as(C.c_void_p) if a is not None else None


def _args(ptr, idx, x_row, x_col):
    return (np.ascontiguousarray(ptr, np.int32), np.ascontiguousarray(idx, np.int32),
            np.ascontiguousarray(x_row, np.float32), np.ascontiguousarray(x_col, np.float32))


def sddmm_f32(ptr, idx, x_row, x_col, feat, ftz=True, nthreads=0):
    """out[e] = <x_row[row(e)], x_col[idx[e]]> in the engine's order (sddmm.cu); ftz models its -ftz=true build."""
    ptr, idx, x_row, x_col = _args(ptr, idx, x_row, x_col)
    m = len(ptr) - 1
    out = np.empty(int(ptr[-1]), np.float32)
    _lib.oracle_sddmm_f32(_p(ptr), _p(idx), _p(x_row), _p(x_col), _p(out), m, int(feat), int(bool(ftz)), int(nthreads))
    return out


def sddmm_f64(ptr, idx, x_row, x_col, feat, nthreads=0):
    """-> (fp64 dot, fp64 sum of |terms|) per nonzero."""
    ptr, idx, x_row, x_col = _args(ptr, idx, x_row, x_col)
    m = len(ptr) - 1
    n = int(ptr[-1])
    out, ab = np.empty(n, np.float64), np.empty(n, np.float64)
    _lib.oracle_sddmm_f64(_p(ptr), _p(idx), _p(x_row), _p(x_col), _p(out), _p(ab), m, int(feat), int(nthreads))
    return out, ab
