"""ctypes access to tests/reduce_oracle.c — TEST INFRASTRUCTURE ONLY (the CPU restatement of spmm_b200_reduce and
spmm_b200_reduce_backward).

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

_SRC = os.path.join(os.path.dirname(os.path.abspath(__file__)), "reduce_oracle.c")
OPS = {"amax": 1, "amin": 2}


def _load():
    src = open(_SRC, "rb").read()
    tag = hashlib.sha1(src).hexdigest()[:16]
    so = os.path.join(tempfile.gettempdir(), f"hpc_b200_reduce_oracle_{os.getuid()}_{tag}.so")
    if not os.path.exists(so):
        tmp = f"{so}.{os.getpid()}.tmp"
        subprocess.run(["gcc", "-O3", "-mavx2", "-mfma", "-ffp-contract=off", "-fopenmp", "-fPIC", "-shared", "-o", tmp,
                        _SRC, "-lm"], check=True, capture_output=True)
        os.replace(tmp, so)
    lib = C.CDLL(so)
    P, I = C.c_void_p, C.c_int
    lib.oracle_reduce_f32.argtypes = [P, P, P, P, P, P, I, I, I, I, I]
    lib.oracle_reduce_f32.restype = None
    lib.oracle_reduce_backward_f32.argtypes = [P, P, P, P, P, P, P, P, I, I, I, I, I]
    lib.oracle_reduce_backward_f32.restype = None
    lib.oracle_reduce_backward_f64.argtypes = [P, P, P, P, P, P, P, P, P, P, P, I, I, I]
    lib.oracle_reduce_backward_f64.restype = None
    lib.oracle_reduce_tile.restype = I
    return lib


_lib = _load()
TILE = _lib.oracle_reduce_tile()


def _p(a):
    return a.ctypes.data_as(C.c_void_p) if a is not None else None


def _i32(a):
    return np.ascontiguousarray(a, np.int32)


def _f32(a):
    return np.ascontiguousarray(a, np.float32)


def reduce_f32(ptr, idx, val, vin, feat, op, ftz=True, nthreads=0):
    """-> (vout[num_v, K], arg[num_v, K]) in the engine's contract (reduce.cu); op "amax" | "amin"."""
    ptr, idx, val, vin = _i32(ptr), _i32(idx), _f32(val), _f32(vin)
    m = len(ptr) - 1
    vout = np.empty((m, feat), np.float32)
    arg = np.empty((m, feat), np.int32)
    _lib.oracle_reduce_f32(_p(ptr), _p(idx), _p(val), _p(vin), _p(vout), _p(arg), m, int(feat), int(OPS[op] == 1),
                           int(bool(ftz)), int(nthreads))
    return vout, arg


def reduce_backward_f32(ptr, idx, val, dc, arg, vin, b_rows, feat, db=True, dval=True, ftz=True, nthreads=0):
    """-> (db[b_rows, K] or None, dval[num_e] or None) in the engine's orders (tiles of TILE entries; sddmm's order)."""
    ptr, idx, val, dc, arg = _i32(ptr), _i32(idx), _f32(val), _f32(dc), _i32(arg)
    vin = _f32(vin) if dval else None
    m = len(ptr) - 1
    o_db = np.empty((b_rows, feat), np.float32) if db else None
    o_dv = np.empty(int(ptr[-1]), np.float32) if dval else None
    _lib.oracle_reduce_backward_f32(_p(ptr), _p(idx), _p(val), _p(dc), _p(arg), _p(vin), _p(o_db), _p(o_dv), m,
                                    int(b_rows), int(feat), int(bool(ftz)), int(nthreads))
    return o_db, o_dv


def reduce_backward_f64(ptr, idx, val, dc, arg, vin, b_rows, feat):
    """-> dict of fp64 db, db_abs (sum |terms|), db_terms (matched terms per element), dval, dval_abs."""
    ptr, idx, val, dc, arg, vin = _i32(ptr), _i32(idx), _f32(val), _f32(dc), _i32(arg), _f32(vin)
    m = len(ptr) - 1
    n = int(ptr[-1])
    out = {"db": np.empty((b_rows, feat)), "db_abs": np.empty((b_rows, feat)),
           "db_terms": np.empty((b_rows, feat), np.int32), "dval": np.empty(n), "dval_abs": np.empty(n)}
    _lib.oracle_reduce_backward_f64(_p(ptr), _p(idx), _p(val), _p(dc), _p(arg), _p(vin), _p(out["db"]),
                                    _p(out["db_abs"]), _p(out["dval"]), _p(out["dval_abs"]), _p(out["db_terms"]), m,
                                    int(b_rows), int(feat))
    return out
