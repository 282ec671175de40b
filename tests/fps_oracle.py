"""ctypes binding of fps_oracle.c, the CPU reference of tknn_fps — TEST INFRASTRUCTURE ONLY.

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

_SRC = os.path.join(os.path.dirname(os.path.abspath(__file__)), "fps_oracle.c")
_lib = None
FLT_MAX = np.float32(np.finfo(np.float32).max)


def lib() -> C.CDLL:
    global _lib
    if _lib is None:
        out = os.path.join(tempfile.mkdtemp(prefix="tknn_fps_oracle_"), "libfps_oracle.so")
        cc = "/usr/bin/gcc" if os.path.exists("/usr/bin/gcc") else "gcc"  # the system gcc ships libgomp
        subprocess.run([cc, "-O2", "-std=gnu11", "-fPIC", "-fopenmp", "-ffp-contract=off", "-fvisibility=hidden",
                        "-shared", "-o", out, _SRC, "-lm"], check=True)
        L = C.CDLL(out)
        L.tkf_num_threads.restype = C.c_int
        L.tkf_fps.restype = C.c_int
        L.tkf_fps.argtypes = [C.c_void_p, C.c_int64, C.c_void_p, C.c_void_p, C.c_int64, C.c_void_p, C.c_int64, C.c_void_p,
                              C.c_void_p]
        _lib = L
    return _lib


def _xyz(a):
    x = np.ascontiguousarray(a, dtype=np.float32)
    if x.shape[1] == 2:
        x = np.concatenate([x, np.zeros((x.shape[0], 1), np.float32)], 1)
    return np.ascontiguousarray(x[:, :3])


def offsets_of(sizes):
    return np.concatenate([[0], np.cumsum(np.asarray(sizes, dtype=np.int64))]).astype(np.uint64)


def fps(xyz, off=None, counts=None, starts=None, limit=None, squared=True):
    """(idx int32 [M], dist float32 [M]) of the contract: off the cloud offsets (None: one cloud), counts the samples per
    cloud, starts one global index per cloud (None: each cloud's first point).  dist is d2 (squared) or sqrtf(d2), with
    FLT_MAX for sample 0.  limit: only the first `limit` samples of each cloud are computed; the rest of idx is -1 and of
    dist NaN."""
    x = _xyz(xyz)
    n = x.shape[0]
    off = np.array([0, n], np.uint64) if off is None else np.ascontiguousarray(off, dtype=np.uint64)
    S = off.shape[0] - 1
    counts = np.asarray(counts, dtype=np.int64).reshape(S)
    soff = offsets_of(counts)
    st = off[:-1].astype(np.int32) if starts is None else np.ascontiguousarray(starts, dtype=np.int32)
    total = int(soff[-1])
    idx = np.full(max(total, 1), -1, np.int32)
    d2 = np.full(max(total, 1), np.nan, np.float32)
    rc = lib().tkf_fps(x.ctypes.data, n, off.ctypes.data, soff.ctypes.data, S, st.ctypes.data,
                       -1 if limit is None else int(limit), idx.ctypes.data, d2.ctypes.data)
    if rc != 0:
        raise ValueError(f"tkf_fps failed ({rc})")
    idx, d2 = idx[:total], d2[:total]
    dist = d2 if squared else np.sqrt(d2)
    dist[soff[:-1][counts > 0].astype(np.int64)] = FLT_MAX
    return idx, dist


def prefix_mask(counts, limit):
    """Positions of the first `limit` samples of every cloud in the concatenated output."""
    counts = np.asarray(counts, dtype=np.int64)
    soff = offsets_of(counts).astype(np.int64)
    rank = np.arange(int(soff[-1])) - np.repeat(soff[:-1], counts)
    return rank < limit
