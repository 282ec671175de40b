"""ctypes binding of feature_knn_oracle.c, the CPU reference of tknn_feature_knn — TEST INFRASTRUCTURE ONLY.

The library is compiled on first use into a fresh temporary directory (never into the source tree), with the same
compiler and flags as oracle/Makefile: OpenMP, and -ffp-contract=off so that the fp32 distance rule is evaluated exactly
as written.
"""
from __future__ import annotations

import ctypes as C
import os
import subprocess
import tempfile

import numpy as np

_SRC = os.path.join(os.path.dirname(os.path.abspath(__file__)), "feature_knn_oracle.c")
_lib = None
FLT_MAX = np.float32(np.finfo(np.float32).max)


def lib() -> C.CDLL:
    global _lib
    if _lib is None:
        out = os.path.join(tempfile.mkdtemp(prefix="tknn_feature_knn_oracle_"), "libfeature_knn_oracle.so")
        cc = "/usr/bin/gcc" if os.path.exists("/usr/bin/gcc") else "gcc"  # the system gcc ships libgomp
        subprocess.run([cc, "-O2", "-std=gnu11", "-fPIC", "-fopenmp", "-ffp-contract=off", "-fvisibility=hidden",
                        "-shared", "-o", out, _SRC, "-lm"], check=True)
        L = C.CDLL(out)
        L.tkfk_knn.restype = C.c_int
        L.tkfk_knn.argtypes = [C.c_void_p, C.c_int64, C.c_int, C.c_int64, C.c_void_p, C.c_void_p, C.c_int64, C.c_int64,
                               C.c_void_p, C.c_int64, C.c_void_p, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p]
        _lib = L
    return _lib


def offsets_of(sizes):
    return np.concatenate([[0], np.cumsum(np.asarray(sizes, dtype=np.int64))]).astype(np.uint64)


def knn(x, y, k, x_off=None, y_off=None, self_ids=None, f=None, squared=True, rows=None):
    """(idx [nq, k] int32, dist [nq, k] float32) of tknn_feature_knn: x [n, >= f], y [nq, >= f] (f defaults to
    x.shape[1]; further columns are skipped through the row pitch), x_off / y_off the segment offsets (None: one
    segment), self_ids one global data index per query row (None: no exclusion).  dist is d2 (squared) or sqrtf(d2);
    FLT_MAX pads rows with fewer eligible points.  rows (optional bool [nq]): only those rows are computed, the others
    stay -1 / NaN."""
    x = np.ascontiguousarray(x, dtype=np.float32)
    y = np.ascontiguousarray(y, dtype=np.float32)
    n, nq = x.shape[0], y.shape[0]
    f = x.shape[1] if f is None else int(f)
    xo = np.array([0, n], np.uint64) if x_off is None else np.ascontiguousarray(x_off, dtype=np.uint64)
    yo = np.array([0, nq], np.uint64) if y_off is None else np.ascontiguousarray(y_off, dtype=np.uint64)
    assert xo.shape == yo.shape and int(xo[-1]) == n and int(yo[-1]) == nq
    sid = None if self_ids is None else np.ascontiguousarray(self_ids, dtype=np.int32)
    rm = None if rows is None else np.ascontiguousarray(rows, dtype=np.uint8)
    idx = np.full((max(nq, 1), k), -1, np.int32)
    d2 = np.full((max(nq, 1), k), np.nan, np.float32)
    rc = lib().tkfk_knn(x.ctypes.data, n, f, x.shape[1], xo.ctypes.data, y.ctypes.data, nq, y.shape[1], yo.ctypes.data,
                        xo.shape[0] - 1, None if sid is None else sid.ctypes.data, int(k),
                        None if rm is None else rm.ctypes.data, idx.ctypes.data, d2.ctypes.data)
    if rc != 0:
        raise ValueError(f"tkfk_knn failed ({rc})")
    idx, d2 = idx[:nq], d2[:nq]
    if squared:
        return idx, d2
    return idx, np.where(idx >= 0, np.sqrt(d2), d2).astype(np.float32)
