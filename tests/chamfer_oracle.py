"""ctypes binding of chamfer_oracle.c, the CPU reference of tknn_knn_backward / tknn_segment_reduce, and the whole
chamfer_distance chain on top of it — TEST INFRASTRUCTURE ONLY.

The library is compiled on first use into a fresh temporary directory (never into the source tree) with
-ffp-contract=off, so that every product and sum rounds on its own as the contract states.  The neighbours come from the
segmented-query reference (segment_query_oracle.knn with squared distances), and the reductions' backward (the gather
and the division by the count) and autograd's sum of the two directions' gradients are restated in numpy float32, so
the whole chain of chamfer_distance, forward and backward, is reference code.
"""
from __future__ import annotations

import ctypes as C
import os
import subprocess
import tempfile

import numpy as np

import segment_query_oracle as SQ

_SRC = os.path.join(os.path.dirname(os.path.abspath(__file__)), "chamfer_oracle.c")
_lib = None


def lib() -> C.CDLL:
    global _lib
    if _lib is None:
        out = os.path.join(tempfile.mkdtemp(prefix="tknn_chamfer_oracle_"), "libchamfer_oracle.so")
        cc = "/usr/bin/gcc" if os.path.exists("/usr/bin/gcc") else "gcc"
        subprocess.run([cc, "-O2", "-std=gnu11", "-fPIC", "-ffp-contract=off", "-fvisibility=hidden", "-shared", "-o", out,
                        _SRC], check=True)
        L = C.CDLL(out)
        vp = C.c_void_p
        L.tkc_knn_backward.restype = None
        L.tkc_knn_backward.argtypes = [vp, C.c_int64, C.c_int, vp, C.c_int64, C.c_int, C.c_int, vp, C.c_int, vp, vp, vp]
        L.tkc_segment_reduce.restype = None
        L.tkc_segment_reduce.argtypes = [vp, C.c_int, C.c_int, vp, C.c_int64, C.c_int, vp]
        _lib = L
    return _lib


def knn_backward(q, p, idx, g, dim=None):
    """(grad_q [nq, dim], grad_p [n, dim]) of the contract.  q / p: [rows, pitch] float32, the first dim columns read."""
    q = np.ascontiguousarray(q, np.float32)
    p = np.ascontiguousarray(p, np.float32)
    idx = np.ascontiguousarray(idx, np.int32)
    g = np.ascontiguousarray(g, np.float32)
    nq, k = idx.shape
    dim = min(q.shape[1], 3) if dim is None else dim
    gq = np.empty((nq, dim), np.float32)
    gp = np.empty((len(p), dim), np.float32)
    lib().tkc_knn_backward(q.ctypes.data, nq, q.shape[1], p.ctypes.data if len(p) else None, len(p), p.shape[1], dim,
                           idx.ctypes.data, k, g.ctypes.data, gq.ctypes.data, gp.ctypes.data)
    return gq, gp


def segment_reduce(x, offsets, reduce="sum"):
    """[n_seg, f] (or [n_seg] for a 1-D x) float32 of the contract; offsets: the n_seg + 1 segment offsets."""
    x = np.ascontiguousarray(x, np.float32)
    rows = x.reshape(-1, 1) if x.ndim == 1 else x
    off = np.ascontiguousarray(offsets, np.uint64)
    n_seg, f = len(off) - 1, rows.shape[1]
    out = np.empty((n_seg, f), np.float32)
    lib().tkc_segment_reduce(rows.ctypes.data if len(rows) else None, f, f, off.ctypes.data, n_seg,
                             2 if reduce == "sum" else 0, out.ctypes.data)
    return out.reshape(n_seg) if x.ndim == 1 else out


def offsets_of(sizes):
    return np.concatenate([[0], np.cumsum(np.asarray(sizes, np.int64))]).astype(np.uint64)


def nearest(x, y, x_sizes, y_sizes):
    """(idx [len(x), 1] int32, d2 [len(x), 1] float32): for every point of x its nearest point of y in the same cloud."""
    return SQ.knn(y, x, offsets_of(y_sizes), offsets_of(x_sizes), 1, squared=True)


def _reduce_backward(g, sizes, how):
    """The reductions' backward: the gather g[segment], divided by (float)count for the mean."""
    sizes = np.asarray(sizes, np.int64)
    seg = np.repeat(np.arange(len(sizes)), sizes)
    out = np.asarray(g, np.float32)[seg]
    if how == "mean":
        out = (out / sizes.astype(np.float32)[seg]).astype(np.float32)
    return out


def chamfer(x, y, x_sizes, y_sizes, point_reduction="mean", batch_reduction="mean", single_directional=False,
            grad=None):
    """(loss, grad_x, grad_y) of chamfer_distance over clouds of x_sizes / y_sizes points.  grad: the gradient of the
    loss (default 1 per entry of the loss); for point_reduction None it is the pair (g_a, g_b) of per-point gradients and
    the loss is (a, b)."""
    x, y = np.ascontiguousarray(x, np.float32), np.ascontiguousarray(y, np.float32)
    B = len(x_sizes)
    ia, a = nearest(x, y, x_sizes, y_sizes)
    ib, b = (None, None) if single_directional else nearest(y, x, y_sizes, x_sizes)
    a = a[:, 0]
    b = None if b is None else b[:, 0]
    if point_reduction is None:
        loss = (a, b)
        ga, gb = grad
    else:
        X = segment_reduce(a, offsets_of(x_sizes), point_reduction)
        Y = None if single_directional else segment_reduce(b, offsets_of(y_sizes), point_reduction)
        if batch_reduction is not None:
            X = segment_reduce(X, [0, B], batch_reduction)[0]
            Y = None if Y is None else segment_reduce(Y, [0, B], batch_reduction)[0]
        loss = X if Y is None else np.float32(X + Y)
        g = np.ones_like(np.asarray(loss, np.float32)) if grad is None else np.asarray(grad, np.float32)
        gX = g
        if batch_reduction is not None:
            gX = _reduce_backward(np.reshape(g, 1), [B], batch_reduction)
        ga = _reduce_backward(gX, x_sizes, point_reduction)
        gb = None if single_directional else _reduce_backward(gX, y_sizes, point_reduction)
    gq_a, gp_a = knn_backward(x, y, ia, ga.reshape(-1, 1))
    if single_directional:
        return loss, gq_a, gp_a
    gq_b, gp_b = knn_backward(y, x, ib, np.asarray(gb, np.float32).reshape(-1, 1))
    return loss, (gq_a + gp_b).astype(np.float32), (gp_a + gq_b).astype(np.float32)
