"""ctypes binding of dbscan_oracle.c, the CPU reference of tknn_dbscan — TEST INFRASTRUCTURE ONLY.

The library is compiled on first use into a fresh temporary directory (never into the source tree), with the
same compiler and flags as oracle/Makefile: OpenMP, and -ffp-contract=off so that the fp32 distance rule is
evaluated exactly as written.
"""
from __future__ import annotations

import ctypes as C
import os
import subprocess
import tempfile

import numpy as np

_SRC = os.path.join(os.path.dirname(os.path.abspath(__file__)), "dbscan_oracle.c")
_lib = None


def lib() -> C.CDLL:
    global _lib
    if _lib is None:
        out = os.path.join(tempfile.mkdtemp(prefix="tknn_dbscan_oracle_"), "libdbscan_oracle.so")
        cc = "/usr/bin/gcc" if os.path.exists("/usr/bin/gcc") else "gcc"  # the system gcc ships libgomp
        subprocess.run([cc, "-O2", "-std=gnu11", "-fPIC", "-fopenmp", "-ffp-contract=off", "-fvisibility=hidden",
                        "-shared", "-o", out, _SRC, "-lm"], check=True)
        L = C.CDLL(out)
        L.tkd_num_threads.restype = C.c_int
        L.tkd_dbscan.restype = C.c_int
        L.tkd_dbscan.argtypes = [C.POINTER(C.c_float), C.c_int64, C.c_float, C.c_int, C.POINTER(C.c_int32),
                                 C.POINTER(C.c_uint8), C.POINTER(C.c_int64)]
        _lib = L
    return _lib


def num_threads() -> int:
    """OpenMP threads the reference runs on."""
    return int(lib().tkd_num_threads())


def dbscan(xyz, eps: float, min_pts: int):
    """(labels [n] int32, core [n] uint8, C) of the tknn_dbscan contract; 2-D input gets z = 0."""
    x = np.ascontiguousarray(xyz, dtype=np.float32)
    if x.shape[1] == 2:
        x = np.ascontiguousarray(np.concatenate([x, np.zeros((x.shape[0], 1), np.float32)], 1))
    x = np.ascontiguousarray(x[:, :3])
    n = x.shape[0]
    labels = np.empty(n, np.int32)
    core = np.empty(n, np.uint8)
    c = C.c_int64(0)
    rc = lib().tkd_dbscan(x.ctypes.data_as(C.POINTER(C.c_float)), n, C.c_float(eps), int(min_pts),
                          labels.ctypes.data_as(C.POINTER(C.c_int32)), core.ctypes.data_as(C.POINTER(C.c_uint8)), C.byref(c))
    if rc != 0:
        raise ValueError(f"tkd_dbscan failed (n={n}, eps={eps}, min_pts={min_pts})")
    return labels, core, int(c.value)
