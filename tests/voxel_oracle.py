"""ctypes binding of voxel_oracle.c, the CPU reference of tknn_voxel_grid / _members / _pool — TEST INFRASTRUCTURE ONLY.

The library is compiled on first use into a fresh temporary directory (never into the source tree) with
-ffp-contract=off, so that the fp32 formula and the chunked sums are evaluated exactly as written.
"""
from __future__ import annotations

import ctypes as C
import os
import subprocess
import tempfile

import numpy as np

_SRC = os.path.join(os.path.dirname(os.path.abspath(__file__)), "voxel_oracle.c")
_lib = None


def lib() -> C.CDLL:
    global _lib
    if _lib is None:
        out = os.path.join(tempfile.mkdtemp(prefix="tknn_voxel_oracle_"), "libvoxel_oracle.so")
        cc = "/usr/bin/gcc" if os.path.exists("/usr/bin/gcc") else "gcc"
        subprocess.run([cc, "-O2", "-std=gnu11", "-fPIC", "-ffp-contract=off", "-fvisibility=hidden", "-shared", "-o", out,
                        _SRC], check=True)
        L = C.CDLL(out)
        vp = C.c_void_p
        L.tkv_grid.restype = C.c_int64
        L.tkv_grid.argtypes = [vp, C.c_int64, C.c_int, C.c_int, vp, C.c_int64, vp, vp, vp, vp, vp, vp, vp, vp, vp]
        L.tkv_pool.restype = None
        L.tkv_pool.argtypes = [vp, C.c_int, C.c_int, vp, vp, C.c_int64, C.c_int, vp]
        _lib = L
    return _lib


def _cols(a, dim):
    a = np.asarray(a, dtype=np.float32)
    return np.ascontiguousarray(np.broadcast_to(a, (dim,)))


def _p(a):
    return None if a is None else a.ctypes.data


def grid(points, size, start=None, end=None, off=None, dim=None):
    """dict(raw int64 [n], cluster int32 [n], offsets uint64 [nv + 1], members int32 [n], first int32 [nv], seg int32
    [nv], n_voxels) of the contract.  points: [n, stride] float32 (the first dim columns are the position); off: the
    n_clouds + 1 cloud offsets or None; size / start / end: scalars or per-axis values (start / end may be None)."""
    pts = np.ascontiguousarray(points, dtype=np.float32)
    n, stride = pts.shape
    dim = min(stride, 3) if dim is None else dim
    size, start, end = _cols(size, dim), None if start is None else _cols(start, dim), None if end is None else _cols(end, dim)
    off = None if off is None else np.ascontiguousarray(off, dtype=np.uint64)
    raw = np.empty(n, np.int64)
    cluster = np.empty(n, np.int32)
    vox_off = np.empty(n + 1, np.uint64)
    members = np.empty(n, np.int32)
    first = np.empty(n, np.int32)
    seg = np.empty(n, np.int32)
    nv = lib().tkv_grid(_p(pts), n, dim, stride, _p(off), 0 if off is None else off.shape[0] - 1, _p(size), _p(start),
                        _p(end), _p(raw), _p(cluster), _p(vox_off), _p(members), _p(first), _p(seg))
    return dict(raw=raw, cluster=cluster, offsets=vox_off[: nv + 1].copy(), members=members, first=first[:nv].copy(),
                seg=seg[:nv].copy(), n_voxels=int(nv))


def pool(x, g, reduce="mean"):
    """[nv, f] float32: the rows x ([n, stride] float32, all columns pooled) over the clustering g of grid()."""
    x = np.ascontiguousarray(x, dtype=np.float32)
    if x.ndim == 1:
        x = x.reshape(-1, 1)
    f = x.shape[1]
    out = np.empty((g["n_voxels"], f), np.float32)
    lib().tkv_pool(_p(x), f, f, _p(g["offsets"]), _p(g["members"]), g["n_voxels"], 1 if reduce == "max" else 0, _p(out))
    return out


def numpy_raw(points, size, start=None, end=None, batch=None):
    """The raw-id formula restated in numpy float32 / int64 (torch_cluster's grid rule on [pos | batch])."""
    pos = np.asarray(points, dtype=np.float32)
    dim = pos.shape[1]
    size = _cols(size, dim)
    if batch is not None:
        b = np.asarray(batch, dtype=np.float32).reshape(-1, 1)
        pos = np.concatenate([pos, b], 1)
        size = np.concatenate([size, [np.float32(1)]]).astype(np.float32)
        start = None if start is None else np.concatenate([_cols(start, dim), [np.float32(0)]]).astype(np.float32)
        end = None if end is None else np.concatenate([_cols(end, dim), [b.max()]]).astype(np.float32)
    s0 = pos.min(0) if start is None else _cols(start, pos.shape[1])
    e0 = pos.max(0) if end is None else _cols(end, pos.shape[1])
    cnt = ((e0 - s0) / size).astype(np.int64) + 1
    mult = np.concatenate([[1], np.cumprod(cnt)[:-1]]).astype(np.int64)
    return (((pos - s0) / size).astype(np.int64) * mult).sum(1)
