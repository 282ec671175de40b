"""ctypes binding of radius_oracle.c, the CPU reference of tknn_radius_search / tknn_radius_query — TEST INFRASTRUCTURE
ONLY.

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

_SRC = os.path.join(os.path.dirname(os.path.abspath(__file__)), "radius_oracle.c")
_lib = None


def lib() -> C.CDLL:
    global _lib
    if _lib is None:
        out = os.path.join(tempfile.mkdtemp(prefix="tknn_radius_oracle_"), "libradius_oracle.so")
        cc = "/usr/bin/gcc" if os.path.exists("/usr/bin/gcc") else "gcc"  # the system gcc ships libgomp
        subprocess.run([cc, "-O2", "-std=gnu11", "-fPIC", "-fopenmp", "-ffp-contract=off", "-fvisibility=hidden",
                        "-shared", "-o", out, _SRC, "-lm"], check=True)
        L = C.CDLL(out)
        L.tkr_num_threads.restype = C.c_int
        L.tkr_radius_lists.restype = C.c_int
        L.tkr_radius_lists.argtypes = [C.c_void_p, C.c_int64, C.c_void_p, C.c_int64, C.c_void_p, C.c_float, C.c_void_p,
                                       C.POINTER(C.POINTER(C.c_uint64))]
        L.tkr_free.argtypes = [C.c_void_p]
        _lib = L
    return _lib


def num_threads() -> int:
    """OpenMP threads the reference runs on."""
    return int(lib().tkr_num_threads())


def _xyz(a):
    x = np.ascontiguousarray(a, dtype=np.float32)
    if x.shape[1] == 2:
        x = np.concatenate([x, np.zeros((x.shape[0], 1), np.float32)], 1)
    return np.ascontiguousarray(x[:, :3])


def radius_lists(xyz, r: float, queries=None, self_ids=None):
    """(offsets [nq + 1] int64, idx int32, d2 float32) of the contract: all points (queries None, self = the point) or a
    separate query set with optional self ids; 2-D input gets z = 0.  Rows sorted by (d2, index)."""
    x = _xyz(xyz)
    n = x.shape[0]
    q = None if queries is None else _xyz(queries)
    nq = n if q is None else q.shape[0]
    sid = None if self_ids is None else np.ascontiguousarray(self_ids, dtype=np.int32)
    off = np.empty(nq + 1, np.int64)
    keys_p = C.POINTER(C.c_uint64)()
    rc = lib().tkr_radius_lists(x.ctypes.data, n, None if q is None else q.ctypes.data, nq,
                                None if sid is None else sid.ctypes.data, C.c_float(r), off.ctypes.data, C.byref(keys_p))
    if rc != 0:
        raise ValueError(f"tkr_radius_lists failed (n={n}, nq={nq}, r={r})")
    total = int(off[-1])
    try:
        keys = np.ctypeslib.as_array(keys_p, shape=(max(total, 1),))[:total].copy()
    finally:
        lib().tkr_free(keys_p)
    idx = (keys & np.uint64(0xFFFFFFFF)).astype(np.uint32).view(np.int32)
    d2 = (keys >> np.uint64(32)).astype(np.uint32).view(np.float32)
    return off, idx, d2
