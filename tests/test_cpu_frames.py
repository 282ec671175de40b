"""The CPU reference of tknn_local_frames (tests/frames_oracle.py) checked without a GPU: its covariance against a numpy
float32 restatement of the chunked rule, its Jacobi against numpy.linalg.eigh in float64 on the same covariance, known
normals of sampled planes, spheres and cylinders, the frames' shape and signs against a float64 restatement of
PyTorch3D's body, the edge cases of the contract, and the argument checks and library calls of the Python layer (through
the recording fake of test_cpu_wrapper_calls.py, no GPU)."""
import numpy as np
import pytest
from scipy.spatial import cKDTree

import frames_oracle as F
from owlraytracing_b200 import _lib, estimate_pointcloud_local_coord_frames, estimate_pointcloud_normals
from owlraytracing_b200 import trueknn as T

torch = pytest.importorskip("torch")

from test_cpu_wrapper_calls import _fill_knn, fake, t, trace  # noqa: E402,F401  (fixtures and the call trace)

IU = [(0, 0), (0, 1), (0, 2), (1, 1), (1, 2), (2, 2)]


def bits(a):
    return np.ascontiguousarray(a, np.float32).view(np.uint32)


def random_neighbourhoods(rng, count, k_max=64):
    """Anisotropic neighbourhoods (flatness down to 1e-3) at scales 1e-3 .. 1e3 and offsets up to 1e3, each its own
    points; rows padded with -1 up to k_max."""
    pts, rows, off = [], np.full((count, k_max), -1, np.int32), 0
    for i in range(count):
        k = int(rng.integers(3, k_max + 1))
        p = rng.random((k, 3)) * [1, 1, rng.choice([1e-1, 1e-2, 1e-3])]
        r, _ = np.linalg.qr(rng.normal(size=(3, 3)))
        pts.append(p @ r.T * rng.choice([1e-3, 1, 1e3]) + rng.normal(size=3) * rng.choice([0, 10, 1000]))
        rows[i, :k] = np.arange(off, off + k)
        off += k
    return np.concatenate(pts).astype(np.float32), rows


def sym(cov):
    a = np.zeros((len(cov), 3, 3))
    for e, (i, j) in enumerate(IU):
        a[:, i, j] = a[:, j, i] = cov[:, e]
    return a


def chunked_sum(terms):
    """[m, k] float32 terms (NaN = skipped slot) -> the chunked sum of every row, in numpy float32."""
    m, k = terms.shape
    acc = np.zeros(m, np.float32)
    part = np.zeros(m, np.float32)
    cnt = np.zeros(m, np.int64)
    for s in range(k):
        live = ~np.isnan(terms[:, s])
        part = np.where(live, (part + np.where(live, terms[:, s], 0)).astype(np.float32), part)
        cnt += live
        full = live & (cnt % 32 == 0)
        acc = np.where(full, (acc + part).astype(np.float32), acc)
        part = np.where(full, np.float32(0), part)
    return np.where(cnt % 32 != 0, (acc + part).astype(np.float32), acc)


def test_covariance_is_the_chunked_rule():
    rng = np.random.default_rng(0)
    p = (rng.random((5000, 3)) * 10 + 100).astype(np.float32)
    idx = rng.integers(0, 5000, (300, 100)).astype(np.int32)
    idx[rng.random(idx.shape) < 0.2] = -1  # -1 slots anywhere: the chunks count valid slots only
    _, _, cov, _ = F.local_frames(p, idx, with_cov=True)
    g = np.where((idx >= 0)[:, :, None], p[np.maximum(idx, 0)], np.nan).astype(np.float32)
    c = (idx >= 0).sum(1).astype(np.float32)
    mean = np.stack([(chunked_sum(g[:, :, d]) / c).astype(np.float32) for d in range(3)], 1)
    e = (g - mean[:, None, :]).astype(np.float32)
    for col, (a, b) in enumerate(IU):
        ref = (chunked_sum((e[:, :, a] * e[:, :, b]).astype(np.float32)) / c).astype(np.float32)
        assert (bits(cov[:, col]) == bits(ref)).all(), (a, b)


def test_jacobi_against_float64_eigh():
    rng = np.random.default_rng(1)
    pts, rows = random_neighbourhoods(rng, 20_000)
    eig, frames, cov, sweeps = F.local_frames(pts, rows, with_cov=True)
    w64, v64 = np.linalg.eigh(sym(cov))  # float64, on the reference's own fp32 covariance
    lam2 = w64[:, 2]
    assert (np.abs(eig - w64).max(1) <= 1e-6 * lam2).all()
    n = frames[:, :, 0].astype(np.float64)
    n /= np.linalg.norm(n, axis=1, keepdims=True)
    angle = np.degrees(np.arccos(np.clip(np.abs((n * v64[:, :, 0]).sum(1)), 0, 1)))
    gapped = (w64[:, 1] - w64[:, 0]) / lam2 > 1e-3
    assert gapped.mean() > 0.95 and angle[gapped].max() < 0.05
    assert sweeps.max() <= 6 and sweeps.min() >= 1  # the 8-sweep cap is never reached here
    f64 = frames.astype(np.float64)
    assert np.abs(np.einsum("mij,mik->mjk", f64, f64) - np.eye(3)).max() < 1e-5
    assert (np.diff(eig, axis=1) >= 0).all()


def neighbour_rows(p, k):
    """Each point's own index, then its k - 1 nearest other points (the rows estimate_pointcloud_normals builds)."""
    _, nb = cKDTree(p.astype(np.float64)).query(p.astype(np.float64), k)
    return nb.astype(np.int32)


def angle_deg(a, b):
    a = a / np.linalg.norm(a, axis=1, keepdims=True)
    b = b / np.linalg.norm(b, axis=1, keepdims=True)
    return np.degrees(np.arccos(np.clip(np.abs((a * b).sum(1)), 0, 1)))


def test_analytic_normals():
    rng = np.random.default_rng(2)
    # a tilted plane through (3, -2, 5)
    u, v = rng.random((2, 4000)) * 4 - 2
    r, _ = np.linalg.qr(rng.normal(size=(3, 3)))
    plane = (np.stack([u, v, np.zeros_like(u)], 1) @ r.T + [3, -2, 5]).astype(np.float32)
    _, fr = F.local_frames(plane, neighbour_rows(plane, 16))
    assert angle_deg(fr[:, :, 0], np.broadcast_to(r[:, 2], (len(plane), 3))).max() < 0.05
    # Curved surfaces: a one-sided k-NN cap tilts the fitted plane by O(r / R) (0.6 deg and 1.0 deg at most here,
    # 1.7 deg and 2.7 deg with a tenth of the points), so the samples are dense.  The sign rule points a normal to the
    # side where most neighbours lie: inward on a convex surface, except where the tilt outweighs the curvature.
    d = rng.normal(size=(200_000, 3))
    d /= np.linalg.norm(d, axis=1, keepdims=True)
    sphere = (d * 2 + 1).astype(np.float32)  # radius 2 around (1, 1, 1)
    _, fr = F.local_frames(sphere, neighbour_rows(sphere, 20), disambiguate=True)
    assert angle_deg(fr[:, :, 0], d).max() < 1.0
    assert ((fr[:, :, 0] * d).sum(1) < 0).mean() > 0.99
    phi, z = rng.random(200_000) * 2 * np.pi, rng.random(200_000) * 6
    cyl = np.stack([np.cos(phi), np.sin(phi), z], 1).astype(np.float32)  # radius 1 along z
    _, fr = F.local_frames(cyl, neighbour_rows(cyl, 20), disambiguate=True)
    radial = np.stack([np.cos(phi), np.sin(phi), np.zeros_like(phi)], 1)
    assert angle_deg(fr[:, :, 0], radial).max() < 1.5
    assert ((fr[:, :, 0] * radial).sum(1) < 0).mean() > 0.99


def test_disambiguated_frames_against_pytorch3d_body():
    rng = np.random.default_rng(3)
    m, k = 5000, 24
    centres = rng.normal(size=(m, 3)) * 50
    axes = np.stack([np.linalg.qr(rng.normal(size=(3, 3)))[0] for _ in range(m)])
    local = rng.normal(size=(m, k, 3)) * [3.0, 1.5, 0.2] + rng.normal(size=(m, 1, 3)) * [0.5, 0.5, 0.05]
    local[:, 0] = rng.normal(size=(m, 3)) * [1.0, 0.5, 0.05]  # the anchor, somewhere inside its neighbourhood
    pts = (np.einsum("mij,mkj->mki", axes, local) + centres[:, None]).reshape(-1, 3).astype(np.float32)
    rows = np.arange(m * k, dtype=np.int32).reshape(m, k)
    eig, fr = F.local_frames(pts, rows, disambiguate=True)
    w64, f64 = F.pytorch3d_frames64(pts, rows)
    det = np.linalg.det(fr.astype(np.float64))
    assert np.abs(det + 1).max() < 1e-5  # [n, n x z, z]: columns (2, 1, 0) are right-handed, as in PyTorch3D
    assert np.abs(np.linalg.det(fr[:, :, ::-1].astype(np.float64)) - 1).max() < 1e-5
    # well-conditioned rows: distinct eigenvalues and sign counts away from the tie 2 n_pos = k
    gaps = np.diff(w64, axis=1).min(1) / w64[:, 2]
    df = pts[rows].astype(np.float64) - pts[rows[:, :1]]
    clear = gaps > 1e-2
    for col in (0, 2):
        proj = (f64[:, None, :, col] * df).sum(2)
        clear &= np.abs(2 * (proj > 0).sum(1) - k) >= 2
        clear &= (np.abs(proj[:, 1:]) > 1e-4 * np.abs(proj).max(1, keepdims=True)).all(1)
    assert clear.mean() > 0.5
    for col in range(3):
        dots = (fr[clear, :, col].astype(np.float64) * f64[clear, :, col]).sum(1)
        assert (dots > 0.999).all(), col
    np.testing.assert_allclose(eig[clear], w64[clear], rtol=1e-4, atol=1e-6 * w64[clear, 2:].max())


def test_edge_cases():
    rng = np.random.default_rng(4)
    p = rng.random((10, 4)).astype(np.float32)  # pitch 4: the fourth column is never read
    p[:, 3] = np.nan
    dup = np.float32([[0.1, 0.7, 0.3, 0]])
    p = np.concatenate([p, np.repeat(dup, 40, 0)])
    idx = np.full((6, 40), -1, np.int32)
    idx[1, 7] = 3  # c = 1
    idx[2, [5, 30]] = [2, 8]  # c = 2
    idx[3, :] = np.arange(10, 50)  # 40 coincident points
    idx[4, ::3] = 2  # one point 14 times
    idx[5, 0] = 1  # disambiguated below
    for disamb in (False, True):
        eig, fr, cov, sweeps = F.local_frames(p, idx, disamb, with_cov=True)
        assert np.isnan(eig[0]).all() and np.isnan(fr[0]).all()  # c = 0
        assert (bits(eig[1]) == 0).all() and not cov[1].any() and sweeps[1] == 0
        if not disamb:
            assert (fr[1] == np.eye(3, dtype=np.float32)).all()
        else:  # no slot projects positively: columns 0 and 2 flip, and y = n x z
            assert (fr[1] == np.diag(np.float32([-1, -1, -1]))).all()
        # c = 2: a rank-one covariance; the normal and column 1 are perpendicular to the segment
        seg = (p[8, :3] - p[2, :3]).astype(np.float64)
        assert eig[2, 0] == 0 or abs(eig[2, 0]) < 1e-7 * eig[2, 2]
        np.testing.assert_allclose(eig[2, 2], (seg @ seg) / 4, rtol=1e-5)
        assert abs(fr[2, :, 0] @ seg) < 1e-5 * np.linalg.norm(seg) and abs(fr[2, :, 2] @ seg) > 0.9999 * np.linalg.norm(seg)
        for r in (3, 4):  # duplicates: a (near) zero covariance and an orthonormal frame
            assert np.isfinite(eig[r]).all() and np.abs(eig[r]).max() < 1e-12
            f64 = fr[r].astype(np.float64)
            assert np.abs(f64.T @ f64 - np.eye(3)).max() < 1e-6


def test_argument_checks_need_no_device():
    x = np.zeros((4, 3), np.float32)
    with pytest.raises(ValueError, match="neighborhood_size"):
        estimate_pointcloud_normals(x, 0)
    with pytest.raises(ValueError, match=r"\[n, 3\]"):
        estimate_pointcloud_normals(x[:, :2])
    with pytest.raises(ValueError, match=r"\[n, 3\]"):
        estimate_pointcloud_local_coord_frames(np.zeros((4, 4), np.float32))
    with pytest.raises(ValueError, match="above 512"):
        estimate_pointcloud_normals(np.zeros((600, 3), np.float32), 513)
    with pytest.raises(ValueError, match="CUDA"):
        estimate_pointcloud_normals(torch.zeros((4, 3)))
    with pytest.raises(ValueError, match="non-decreasing"):
        estimate_pointcloud_normals(x, 1, batch=np.array([1, 0, 0, 0]))
    n = estimate_pointcloud_normals(x[:0])
    c, f = estimate_pointcloud_local_coord_frames(x[:0])
    assert n.shape == (0, 3) and c.shape == (0, 3) and f.shape == (0, 3, 3) and n.dtype == np.float32


@pytest.mark.parametrize("kind", ["numpy", "torch"])
def test_local_frames_calls(t, fake, kind):
    conv = (lambda a: torch.from_numpy(a)) if kind == "torch" else (lambda a: a)
    p = conv(np.zeros((7, 4), np.float32))
    idx = conv(np.zeros((5, 3), np.int32))
    eig, fr = t.local_frames(p, idx, disambiguate=True)
    assert trace(fake, p=p, idx=idx, eig=eig, fr=fr) == [
        ("tknn_local_frames", ("ctx", "p", 7, 4, "idx", 5, 3, 1, "eig", "fr"))]
    assert tuple(eig.shape) == (5, 3) and tuple(fr.shape) == (5, 3, 3) and T._is_tensor(eig) == (kind == "torch")
    eig, fr = t.local_frames(p[:0], idx)  # no points: every slot must be -1, checked by the library
    assert trace(fake, idx=idx, eig=eig, fr=fr) == [
        ("tknn_local_frames", ("ctx", None, 0, 4, "idx", 5, 3, 0, "eig", "fr"))]
    eig, fr = t.local_frames(p, idx[:0])  # no rows: no call
    assert trace(fake) == [] and tuple(fr.shape) == (0, 3, 3)


def test_local_frames_inputs(t, fake):
    p, idx = np.zeros((7, 3), np.float32), np.zeros((5, 3), np.int32)
    with pytest.raises(ValueError, match="points"):
        t.local_frames(p[:, :2], idx)
    with pytest.raises(ValueError, match="idx"):
        t.local_frames(p, idx[0])
    with pytest.raises(TypeError, match="idx"):
        t.local_frames(torch.from_numpy(p), torch.from_numpy(idx).long())
    with pytest.raises(TypeError, match="points"):
        t.local_frames(torch.from_numpy(p).double(), torch.from_numpy(idx))
    assert trace(fake) == []
    t.local_frames(p.astype(np.float64), idx.tolist())  # numpy input is cast
    assert trace(fake) == [("tknn_local_frames", ("ctx", "ptr", 7, 3, "ptr", 5, 3, 0, "ptr", "ptr"))]


def test_estimate_functions_calls(fake):
    pos = np.random.default_rng(5).random((4, 3), dtype=np.float32)
    _fill_knn(fake, [[1, 2], [0, 2], [3, 0], [2, -1]])
    seen = []
    fake.hooks["tknn_local_frames"] = lambda *a: seen.append(np.ctypeslib.as_array(
        (T.C.c_int32 * (a[5] * a[6])).from_address(a[4].value)).reshape(a[5], a[6]).copy())
    n = estimate_pointcloud_normals(pos, 3, batch=np.array([0, 0, 0, 1]), device=1)
    assert trace(fake) == [("tknn_create", (1, "&")), ("tknn_build_segments", ("ctx", "ptr", 4, 3, 3, "ptr", 2)),
                           ("tknn_search", ("ctx", 2, 0.0, "ptr", None)),
                           ("tknn_local_frames", ("ctx", "ptr", 4, 3, "ptr", 4, 3, 1, "ptr", "ptr")),
                           ("tknn_destroy", ("ctx",))]
    assert seen[-1].tolist() == [[0, 1, 2], [1, 0, 2], [2, 3, 0], [3, 2, -1]]  # own index first
    assert n.shape == (4, 3) and n.flags["C_CONTIGUOUS"]
    c, f = estimate_pointcloud_local_coord_frames(pos, 50, disambiguate_directions=False)  # k clamps to n = 4
    assert [(name, a[5:8]) for name, a in trace(fake) if name in ("tknn_search", "tknn_local_frames")] == [
        ("tknn_search", ()), ("tknn_local_frames", (4, 4, 0))]
    estimate_pointcloud_normals(pos, 1)  # k = 1: no build, no search, each row the point alone
    assert [name for name, _ in trace(fake)] == ["tknn_create", "tknn_local_frames", "tknn_destroy"]
    assert seen[-1].tolist() == [[0], [1], [2], [3]]
    assert _lib.TKNN_MAX_K == 512
