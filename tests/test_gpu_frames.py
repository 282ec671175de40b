"""Surface normals and local frames on the GPU (tknn_local_frames, TrueKNN.local_frames, estimate_pointcloud_normals,
estimate_pointcloud_local_coord_frames): bit for bit against the CPU reference (tests/frames_oracle.py) for k = 1 to 512
with -1 slots anywhere in a row, with and without disambiguation, padded pitches, host and device arrays, NULL outputs
and a torch side stream; the whole normals pipeline on batches with empty clouds and clouds smaller than k, LiDAR-like
clouds, lattices (exact ties, degenerate planes), duplicate clusters and the 3-D extreme clouds, its neighbour rows
checked against the exact kNN reference; repeatability; every error code; and the independence of a built context from
the call."""
import numpy as np
import pytest

import extreme_clouds as X
import frames_oracle as F
import segment_oracle as S
from owlraytracing_b200 import (TrueKNN, _lib, datasets, estimate_pointcloud_local_coord_frames,
                                estimate_pointcloud_normals)
from owlraytracing_b200.trueknn import TrueKNNError

pytestmark = pytest.mark.gpu
torch = pytest.importorskip("torch")


def _np(a):
    return a.detach().cpu().numpy() if hasattr(a, "cpu") else np.asarray(a)


def bits_equal(a, b, what):
    a, b = np.asarray(_np(a), np.float32), np.asarray(b, np.float32)
    assert a.shape == b.shape, f"{what}: shape {a.shape} vs {b.shape}"
    a = np.where(np.isnan(a), np.float32(np.nan), a).view(np.uint32)  # NaN sign and payload are not part of the contract
    b = np.where(np.isnan(b), np.float32(np.nan), b).view(np.uint32)
    bad = np.argwhere(a != b)
    assert bad.size == 0, f"{what}: {len(bad)} entries differ, first at {tuple(bad[0])}"


def check(got, points, idx, disambiguate, what):
    eig, fr = F.local_frames(points, idx, disambiguate)
    bits_equal(got[0], eig, f"{what} eigvals")
    bits_equal(got[1], fr, f"{what} frames")


def random_rows(rng, n, m, k):
    """m rows of k indices into n points: -1 slots anywhere (20 %), plus rows with no, one and two valid slots."""
    idx = rng.integers(0, n, (m, k)).astype(np.int32)
    idx[rng.random(idx.shape) < 0.2] = -1
    idx[:4] = -1
    idx[1, k // 2] = 7
    idx[2, [0, k - 1]] = [3, 9]
    idx[3, :] = 5  # one point in every slot
    return idx


@pytest.mark.parametrize("k", [1, 3, 16, 50, 64, 512])
@pytest.mark.parametrize("disambiguate", [False, True])
def test_k_and_empty_slots(knn, k, disambiguate):
    rng = np.random.default_rng(k + 1000 * disambiguate)
    n, m = 30_000, 20_000 if k <= 64 else 4000
    p = (rng.random((n, 3)) * [4, 2, 0.1] + [100, -50, 7]).astype(np.float32)
    idx = random_rows(rng, n, m, k)
    got = knn.local_frames(p, idx, disambiguate)
    check(got, p, idx, disambiguate, f"k {k}")
    st = knn.stats()
    assert st["rounds"] == 1 and st["round_queries"] == [m] and st["k"] == k and st["n_queries"] == m


def _pitched(a, pad):
    buf = torch.full((a.shape[0], a.shape[1] + pad), float("nan"), device="cuda")
    buf[:, :a.shape[1]] = torch.from_numpy(a).cuda()
    return buf, a.shape[1] + pad


def test_pitches_host_device_null_outputs_and_streams(knn):
    rng = np.random.default_rng(1)
    n, m, k = 50_000, 30_000, 20
    p = rng.normal(size=(n, 3)).astype(np.float32)
    idx = random_rows(rng, n, m, k)
    reig, rfr = F.local_frames(p, idx, True)
    L, h = _lib.load(), knn._h
    pb, ps = _pitched(p, 5)
    di = torch.from_numpy(idx).cuda()
    eig, fr = torch.empty((m, 3), device="cuda"), torch.empty((m, 3, 3), device="cuda")
    torch.cuda.synchronize()
    assert L.tknn_local_frames(h, pb.data_ptr(), n, ps, di.data_ptr(), m, k, 1, eig.data_ptr(), fr.data_ptr()) == 0
    bits_equal(eig, reig, "pitched eigvals")
    bits_equal(fr, rfr, "pitched frames")
    # host in and out, each output alone, then neither (a no-op that leaves the outputs alone)
    p4 = np.concatenate([p, np.full((n, 1), np.nan, np.float32)], 1)
    he, hf = np.full((m, 3), 7, np.float32), np.full((m, 3, 3), 7, np.float32)
    assert L.tknn_local_frames(h, p4.ctypes.data, n, 4, idx.ctypes.data, m, k, 1, he.ctypes.data, None) == 0
    bits_equal(he, reig, "eigvals alone, host")
    assert L.tknn_local_frames(h, p.ctypes.data, n, 3, di.data_ptr(), m, k, 1, None, hf.ctypes.data) == 0
    bits_equal(hf, rfr, "frames alone, host points, device idx")
    he.fill(7)
    assert L.tknn_local_frames(h, p.ctypes.data, n, 3, idx.ctypes.data, m, k, 1, None, None) == 0
    assert L.tknn_local_frames(h, None, n, 3, None, 0, k, 1, he.ctypes.data, None) == 0  # m = 0
    assert (he == 7).all()
    # tensors on a torch side stream
    s = torch.cuda.Stream()
    with torch.cuda.stream(s):
        knn.set_stream(s.cuda_stream)
        te, tf = knn.local_frames(torch.from_numpy(p).cuda(), di, disambiguate=True)
        assert te.is_cuda and tf.is_cuda
    knn.set_stream(None)
    torch.cuda.synchronize()
    bits_equal(te, reig, "side stream eigvals")
    bits_equal(tf, rfr, "side stream frames")


def reference_frames(x, sizes, k, disambiguate=True):
    """The pipeline restated: exact kNN rows of every cloud (segment_oracle), own index first, the frames reference."""
    if k == 1:
        rows = np.arange(len(x), dtype=np.int32)[:, None]
    else:
        rows = F.own_rows(S.knn(x, S.offsets_of(sizes), k - 1)[0])
    return F.local_frames(x, rows, disambiguate)


def check_pipeline(x, sizes, neighborhood_size, what, disambiguate=True):
    k = min(neighborhood_size, len(x))
    reig, rfr = reference_frames(x, sizes, k, disambiguate)
    batch = np.repeat(np.arange(len(sizes)), sizes)
    xt, bt = torch.from_numpy(x).cuda(), torch.from_numpy(batch).cuda()
    curv, frames = estimate_pointcloud_local_coord_frames(xt, neighborhood_size, bt, disambiguate)
    bits_equal(curv, reig, f"{what} curvatures")
    bits_equal(frames, rfr, f"{what} frames")
    normals = estimate_pointcloud_normals(x, neighborhood_size, batch, disambiguate)  # numpy in, numpy out
    assert isinstance(normals, np.ndarray)
    bits_equal(normals, rfr[:, :, 0], f"{what} normals")
    return reig, rfr


@pytest.mark.parametrize("neighborhood_size", [1, 2, 16, 50])
def test_batches_with_empty_and_small_clouds(oracle, neighborhood_size):
    rng = np.random.default_rng(2)
    sizes = [0, 3000, 1, 0, 7, 49, 50, 51, 2000, 0]
    x = rng.random((sum(sizes), 3), dtype=np.float32)
    _, fr = check_pipeline(x, sizes, neighborhood_size, f"batch ns {neighborhood_size}")
    assert np.isfinite(fr).all()  # every row holds at least the point itself
    one = S.offsets_of(sizes)[2]  # the one-point cloud: frame -I (no slot projects positively), curvatures 0
    assert (fr[one] == -np.eye(3, dtype=np.float32)).all()


def test_lidar_lattice_and_duplicates(oracle):
    check_pipeline(datasets.lidar_like(200_000, seed=3), [200_000], 16, "lidar k 16")
    check_pipeline(datasets.lidar_like(60_000, seed=4), [60_000], 50, "lidar k 50", disambiguate=False)
    lat = datasets.lattice(24)
    _, fr = check_pipeline(lat, [len(lat)], 16, "lattice (ties)")
    plane = lat[lat[:, 2] == 0].copy()  # a degenerate plane: every covariance has a zero eigenvalue
    eig, fr = check_pipeline(plane, [len(plane)], 9, "lattice plane")
    assert (np.abs(fr[:, 2, 0]) == 1).all() and (eig[:, 0] == 0).all()
    rng = np.random.default_rng(5)
    dup = np.repeat(rng.random((3000, 3), dtype=np.float32), 40, 0)  # clusters of 40 coincident points
    check_pipeline(dup, [len(dup)], 50, "duplicate clusters")


@pytest.mark.parametrize("name", sorted(n for n in X.CLOUDS if not n.endswith("_2d")))
def test_extreme_clouds(oracle, name):
    x = X.cloud(name, 3000)
    check_pipeline(x, [len(x)], 16, name)


def test_repeatable(knn):
    rng = np.random.default_rng(6)
    x = torch.from_numpy(rng.random((1 << 20, 3), dtype=np.float32)).cuda()
    runs = [estimate_pointcloud_local_coord_frames(x, 32) for _ in range(2)]
    for a, b in zip(*runs):
        assert torch.equal(a.view(torch.int32), b.view(torch.int32))
    rows = torch.randint(0, 1 << 20, (4096, 32), device="cuda", dtype=torch.int32)
    bits_equal(knn.local_frames(x, rows, True)[1], F.local_frames(_np(x), _np(rows), True)[1], "random rows")


def test_error_codes(knn):
    L, h, E = _lib.load(), knn._h, _lib.EINVAL
    p = np.zeros((3, 3), np.float32)
    idx = np.int32([[0, 1], [2, -1]])
    eig, fr = np.empty((2, 3), np.float32), np.empty((2, 3, 3), np.float32)
    a = lambda v: None if v is None else v.ctypes.data

    def call(pp=p, n=3, s=3, i=idx, m=2, k=2, d=0, oe=eig, of=fr):
        return L.tknn_local_frames(h, a(pp), n, s, a(i), m, k, d, a(oe), a(of))

    assert call() == 0 and call(d=1) == 0 and call(oe=None) == 0 and call(of=None) == 0
    assert call(k=0) == E and call(k=513) == E and call(s=2) == E and call(n=1 << 31) == E and call(m=1 << 31) == E
    assert call(d=2) == E and call(d=-1) == E
    assert call(i=None) == E and call(pp=None) == E
    for bad in ([[0, 3], [2, -1]], [[0, 1], [-2, -1]]):  # outside {-1} and [0, n), found on the device
        assert call(i=np.int32(bad)) == E and call(i=np.int32(bad), d=1, oe=None) == E
    assert "outside" in L.tknn_last_error(h).decode()
    assert call(pp=None, n=0, i=np.int32([[-1, -1], [-1, -1]])) == 0 and np.isnan(fr).all()
    assert call(i=None, pp=None, m=0) == 0
    with pytest.raises(TrueKNNError):
        knn.local_frames(p, np.int32([[0, 9]]))


def test_build_and_search_unchanged(knn):
    rng = np.random.default_rng(7)
    pts = rng.random((30_000, 3), dtype=np.float32)
    idx0, d0 = knn.build(pts).search(8)
    rows = F.own_rows(idx0[:, :5])
    check(knn.local_frames(pts, rows, True), pts, rows, True, "after build")
    idx1, d1 = knn.search(8)
    assert (idx1 == idx0).all()
    bits_equal(d1, d0, "search dist after the call")


def test_keep_scratch_off():
    rng = np.random.default_rng(8)
    p = rng.random((5000, 3), dtype=np.float32)
    with TrueKNN(0, keep_scratch=0) as t:
        for k in (8, 40):
            idx = random_rows(rng, 5000, 3000, k)
            check(t.local_frames(p, idx, True), p, idx, True, f"keep_scratch 0 k {k}")
