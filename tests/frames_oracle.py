"""ctypes binding of frames_oracle.c, the CPU reference of tknn_local_frames — TEST INFRASTRUCTURE ONLY.

The library is compiled on first use into a fresh temporary directory (never into the source tree) with
-ffp-contract=off, so that every product and sum rounds on its own as the contract states.  `pytorch3d_frames64` is a
float64 numpy restatement of PyTorch3D's estimate_pointcloud_local_coord_frames body (gather, mean, covariance mean,
eigh, the sign rule anchored at the point, y = cross(n, z)), for checking agreement in meaning, not in bits.
"""
from __future__ import annotations

import ctypes as C
import os
import subprocess
import tempfile

import numpy as np

_SRC = os.path.join(os.path.dirname(os.path.abspath(__file__)), "frames_oracle.c")
_lib = None


def lib() -> C.CDLL:
    global _lib
    if _lib is None:
        out = os.path.join(tempfile.mkdtemp(prefix="tknn_frames_oracle_"), "libframes_oracle.so")
        cc = "/usr/bin/gcc" if os.path.exists("/usr/bin/gcc") else "gcc"
        subprocess.run([cc, "-O2", "-std=gnu11", "-fPIC", "-ffp-contract=off", "-fvisibility=hidden", "-shared", "-o", out,
                        _SRC, "-lm"], check=True)
        L = C.CDLL(out)
        vp = C.c_void_p
        L.tlf_local_frames.restype = None
        L.tlf_local_frames.argtypes = [vp, C.c_int, vp, C.c_int64, C.c_int, C.c_int, vp, vp, vp, vp]
        _lib = L
    return _lib


def local_frames(points, idx, disambiguate=False, with_cov=False):
    """(eigvals [m, 3], frames [m, 3, 3]) of the contract, plus (cov [m, 6], sweeps [m]) when with_cov.  points:
    [n, pitch] float32 (the first 3 columns read); idx: [m, k] int32, -1 for an empty slot."""
    p = np.ascontiguousarray(points, np.float32)
    idx = np.ascontiguousarray(idx, np.int32)
    m, k = idx.shape
    eig = np.empty((m, 3), np.float32)
    frames = np.empty((m, 3, 3), np.float32)
    cov = np.empty((m, 6), np.float32)
    sweeps = np.empty(m, np.int32)
    if m:
        lib().tlf_local_frames(p.ctypes.data if p.size else None, p.shape[1], idx.ctypes.data, m, k, int(disambiguate),
                               eig.ctypes.data, frames.ctypes.data, cov.ctypes.data, sweeps.ctypes.data)
    return (eig, frames, cov, sweeps) if with_cov else (eig, frames)


def own_rows(nbr_idx):
    """[n, k - 1] neighbour rows -> [n, k] rows with each point's own index prepended (PyTorch3D's neighbourhood)."""
    nbr_idx = np.asarray(nbr_idx, np.int32)
    return np.concatenate([np.arange(len(nbr_idx), dtype=np.int32)[:, None], nbr_idx], 1)


def pytorch3d_frames64(points, idx):
    """PyTorch3D's body in float64 on full rows (no -1 slots): (curvatures [m, 3], frames [m, 3, 3]) with the
    disambiguated n, z and y = cross(n, z); anchor = the point of slot 0."""
    p = np.asarray(points, np.float64)[:, :3]
    nb = p[np.asarray(idx)]  # [m, k, 3]
    K = nb.shape[1]
    diff = nb - nb.mean(1, keepdims=True)
    cov = np.einsum("mki,mkj->mij", diff, diff) / K
    w, v = np.linalg.eigh(cov)
    df = nb - nb[:, :1]

    def sign(vec):
        proj = (vec[:, None, :] * df).sum(2)
        flip = (proj > 0).sum(1) < 0.5 * K
        return np.where(flip[:, None], -vec, vec)

    n, z = sign(v[:, :, 0]), sign(v[:, :, 2])
    return w, np.stack([n, np.cross(n, z), z], 2)
