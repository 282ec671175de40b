"""ctypes binding of interpolate_oracle.c, the CPU reference of tknn_interpolate / tknn_interpolate_backward — TEST
INFRASTRUCTURE ONLY.

The library is compiled on first use into a fresh temporary directory (never into the source tree) with
-ffp-contract=off, so that every product and sum rounds on its own as the contract states.  knn_rows() takes the kNN
rows from the segmented-query reference (segment_query_oracle.knn with squared distances), so that the whole chain of
knn_interpolate is reference code.
"""
from __future__ import annotations

import ctypes as C
import os
import subprocess
import tempfile

import numpy as np

import segment_query_oracle as SQ

_SRC = os.path.join(os.path.dirname(os.path.abspath(__file__)), "interpolate_oracle.c")
_lib = None


def lib() -> C.CDLL:
    global _lib
    if _lib is None:
        out = os.path.join(tempfile.mkdtemp(prefix="tknn_interpolate_oracle_"), "libinterpolate_oracle.so")
        cc = "/usr/bin/gcc" if os.path.exists("/usr/bin/gcc") else "gcc"
        subprocess.run([cc, "-O2", "-std=gnu11", "-fPIC", "-ffp-contract=off", "-fvisibility=hidden", "-shared", "-o", out,
                        _SRC], check=True)
        L = C.CDLL(out)
        vp = C.c_void_p
        L.tki_forward.restype = None
        L.tki_forward.argtypes = [vp, vp, C.c_int64, C.c_int, vp, C.c_int, C.c_int, vp, vp, vp]
        L.tki_backward.restype = None
        L.tki_backward.argtypes = [vp, vp, vp, C.c_int64, C.c_int, vp, C.c_int, C.c_int64, C.c_int, vp]
        _lib = L
    return _lib


def forward(idx, d2, x, f=None):
    """(out [nq, f], weight [nq, k], den [nq]) of the contract.  x: [n, pitch] float32, the first f columns are read."""
    idx = np.ascontiguousarray(idx, np.int32)
    d2 = np.ascontiguousarray(d2, np.float32)
    x = np.ascontiguousarray(x, np.float32)
    nq, k = idx.shape
    f = x.shape[1] if f is None else f
    out = np.empty((nq, f), np.float32)
    w = np.empty((nq, k), np.float32)
    den = np.empty(nq, np.float32)
    lib().tki_forward(idx.ctypes.data, d2.ctypes.data, nq, k, x.ctypes.data, f, x.shape[1], out.ctypes.data,
                      w.ctypes.data, den.ctypes.data)
    return out, w, den


def backward(idx, weight, den, grad_out, n, f=None):
    """grad_x [n, f] of the contract.  grad_out: [nq, pitch] float32, the first f columns are read."""
    idx = np.ascontiguousarray(idx, np.int32)
    weight = np.ascontiguousarray(weight, np.float32)
    den = np.ascontiguousarray(den, np.float32)
    g = np.ascontiguousarray(grad_out, np.float32)
    nq, k = idx.shape
    f = g.shape[1] if f is None else f
    gx = np.empty((n, f), np.float32)
    lib().tki_backward(idx.ctypes.data, weight.ctypes.data, den.ctypes.data, nq, k, g.ctypes.data, g.shape[1], n, f,
                       gx.ctypes.data)
    return gx


def knn_rows(pos_x, pos_y, k, x_sizes=None, y_sizes=None):
    """(idx [nq, k] int32, d2 [nq, k] float32) of knn_interpolate's query: the k nearest points of pos_x in the query's
    cloud by (d2, index), -1 / FLT_MAX past the cloud's size.  Sizes: points per cloud (None: one cloud)."""
    nx, ny = len(pos_x), len(pos_y)
    xo = SQ.offsets_of([nx] if x_sizes is None else x_sizes)
    yo = SQ.offsets_of([ny] if y_sizes is None else y_sizes)
    return SQ.knn(pos_x, pos_y, xo, yo, k, squared=True)
