"""Voxel-grid clustering and pooling on the GPU (tknn_voxel_grid / _members / _pool, TrueKNN.voxel_grid, grid_cluster,
voxel_grid, grid_sampling): every output bit for bit against the CPU reference (tests/voxel_oracle.py) — raw ids, dense
ids, offsets, members, representatives, voxel clouds, pooled mean and max bits — on 2-D / 3-D clouds, given and default
ranges, points outside them and on cell boundaries, long coincident voxels, big batches with empty clouds, padded
strides, f up to 1 024, device pointers and torch streams; every error code; and the independence of the clustering
from builds and searches."""
import ctypes as C

import numpy as np
import pytest

import voxel_oracle as V
from owlraytracing_b200 import TrueKNN, _lib, grid_cluster, grid_sampling, voxel_grid
from owlraytracing_b200.trueknn import TrueKNNError

pytestmark = pytest.mark.gpu


def _np(a):
    return a.cpu().numpy() if hasattr(a, "cpu") else np.asarray(a)


def bits_equal(a, b, what):
    a, b = _np(a), np.asarray(b)
    assert a.shape == b.shape, f"{what}: shape {a.shape} vs {b.shape}"
    if a.dtype == np.float32:
        a, b = a.view(np.uint32), b.view(np.uint32)
    bad = np.argwhere(a != b)
    assert bad.size == 0, f"{what}: {len(bad)} entries differ, first at {tuple(bad[0])}: {a[tuple(bad[0])]} vs {b[tuple(bad[0])]}"


def offsets_of(sizes):
    return np.concatenate([[0], np.cumsum(sizes)]).astype(np.uint64)


def check(t, pts, size, start=None, end=None, sizes=None, xs=(), dim=None):
    """Clusters pts with t (numpy or tensors) and compares everything with the reference; returns the reference."""
    off = None if sizes is None else offsets_of(sizes)
    batch = None if sizes is None else np.repeat(np.arange(len(sizes)), sizes)
    if batch is not None and hasattr(pts, "cuda"):
        import torch

        batch = torch.as_tensor(batch, device=pts.device)
    raw, cluster, nv = t.voxel_grid(pts, size, start, end, batch=batch, batch_size=None if sizes is None else len(sizes))
    g = V.grid(_np(pts), size, start, end, off=off, dim=dim)
    assert nv == g["n_voxels"]
    bits_equal(raw, g["raw"], "raw")
    bits_equal(cluster, g["cluster"], "cluster")
    o, m, first, seg = t.voxel_members()
    bits_equal(_np(o).astype(np.uint64), g["offsets"], "offsets")
    bits_equal(m, g["members"], "members")
    bits_equal(first, g["first"], "first")
    bits_equal(seg, g["seg"], "seg")
    for x in xs:
        for reduce in ("mean", "max"):
            bits_equal(t.voxel_pool(x, reduce), V.pool(_np(x), g, reduce), f"pool {reduce} f={_np(x).reshape(len(_np(x)), -1).shape[1]}")
    return g


def lidar_like(n, rng):
    r = rng.uniform(1.0, 40.0, n).astype(np.float32)
    a = rng.uniform(0, 2 * np.pi, n).astype(np.float32)
    z = rng.normal(0, 0.5, n).astype(np.float32)
    return np.stack([r * np.cos(a), r * np.sin(a), z], 1).astype(np.float32)


@pytest.mark.parametrize("dim", [2, 3])
@pytest.mark.parametrize("given", [False, True])
def test_clouds_against_reference(knn, dim, given):
    rng = np.random.default_rng(10 + dim)
    p = lidar_like(200_000, rng)[:, :dim].copy()
    start = np.float32([-25, -30, -1][:dim]) if given else None  # given ranges leave points outside on both sides
    end = np.float32([20, 25, 0.5][:dim]) if given else None
    x = rng.normal(size=(p.shape[0], 7)).astype(np.float32)
    check(knn, p, 0.25, start, end, xs=[p, x])
    check(knn, p, np.float32([0.5, 0.2, 0.1][:dim]), start, end, sizes=[50_000, 0, 100_000, 1, 49_999], xs=[x])


def test_coordinates_on_cell_boundaries(knn):
    rng = np.random.default_rng(2)
    size = np.float32(0.1)
    j = rng.integers(-20, 40, size=(50_000, 3)).astype(np.float32)
    p = (np.float32(-1.0) + j * size).astype(np.float32)  # exactly start + j * size in fp32
    check(knn, p, size, start=-1.0, end=2.0, xs=[p])
    check(knn, p, size, xs=[p])


@pytest.mark.parametrize("count", [33, 1025, 100_000])
def test_coincident_clusters(knn, count):
    rng = np.random.default_rng(count)
    bg = rng.random((20_000, 3), dtype=np.float32) * 10
    p = np.concatenate([bg[:7000], np.repeat(np.float32([[5.01, 5.01, 5.01]]), count, 0), bg[7000:]])
    x = (rng.normal(size=(p.shape[0], 3)) * 1e4).astype(np.float32)
    check(knn, p, 0.05, xs=[x, p])


def test_one_voxel_holds_the_whole_cloud(knn):
    rng = np.random.default_rng(4)
    p = rng.random((1_000_003, 3), dtype=np.float32)
    x = rng.normal(size=(p.shape[0], 2)).astype(np.float32)
    g = check(knn, p, 4.0, xs=[x])
    assert g["n_voxels"] == 1


def test_big_batch_and_empty_clouds(knn):
    rng = np.random.default_rng(6)
    sizes = np.full(65_536, 16)
    sizes[[0, 1, 7, 65_535]] = 0  # empty clouds, cloud 0 and the last one included
    p = rng.random((int(sizes.sum()), 3), dtype=np.float32)
    check(knn, p, 0.3, sizes=sizes, xs=[p])
    check(knn, p, 0.3, start=0.0, end=1.0, sizes=sizes)


def test_tiny_inputs(knn):
    raw, cluster, nv = knn.voxel_grid(np.zeros((0, 3), np.float32), 1.0)
    assert nv == 0 and raw.shape == (0,) and cluster.shape == (0,)
    o, m, first, seg = knn.voxel_members()
    assert list(o) == [0] and m.shape == (0,) and first.shape == (0,)
    assert knn.voxel_pool(np.zeros((0, 4), np.float32)).shape == (0, 4)
    check(knn, np.float32([[1.5, -2.0, 3.0]]), 0.5, xs=[np.float32([[7.0, -0.0]])])
    check(knn, np.float32([[1.5, -2.0, 3.0]]), 0.5, sizes=[0, 1, 0])


def test_padded_stride_and_wide_features(knn):
    rng = np.random.default_rng(8)
    n = 30_000
    p = rng.random((n, 3), dtype=np.float32) * 5
    p[rng.integers(0, n, 3000)] = p[0]  # one voxel above the long-voxel threshold
    L = _lib.load()
    padded = np.full((n, 5), np.nan, np.float32)  # garbage in the padding is never read
    padded[:, :3] = p
    nv = C.c_uint64()
    size = np.float32([0.2, 0.2, 0.2])
    raw = np.empty(n, np.int64)
    assert L.tknn_voxel_grid(knn._h, padded.ctypes.data, n, 3, 5, None, 1, size.ctypes.data, None, None, raw.ctypes.data,
                             None, C.byref(nv)) == 0
    g = V.grid(p, size)
    assert nv.value == g["n_voxels"]
    bits_equal(raw, g["raw"], "raw (padded)")
    for f in (1, 5, 33, 1024):
        pitch = f + 3
        x = np.full((n, pitch), np.inf, np.float32)
        x[:, :f] = rng.normal(size=(n, f)).astype(np.float32)
        for reduce, code in (("mean", 0), ("max", 1)):
            out = np.empty((nv.value, f), np.float32)
            assert L.tknn_voxel_pool(knn._h, x.ctypes.data, n, f, pitch, code, out.ctypes.data) == 0, knn._L.tknn_last_error(knn._h)
            bits_equal(out, V.pool(np.ascontiguousarray(x[:, :f]), g, reduce), f"pool {reduce} f={f} pitch={pitch}")


def test_wide_keys_take_the_pair_sort(knn):
    """Raw-id ranges above 2^33 do not fit beside the 31 index bits of a packed key: the (key, index) pair sort, the
    pair branch of the labels and the fold of long voxels must give the reference's outputs too."""
    rng = np.random.default_rng(13)
    p = (rng.random((150_000, 3), dtype=np.float32) * 100).astype(np.float32)
    p[rng.integers(0, len(p), 20_000)] = p[5]  # duplicates: multi-member voxels, one of them long
    p[rng.integers(0, len(p), 5_000)] = p[77]
    x = rng.normal(size=(len(p), 9)).astype(np.float32)
    g = check(knn, p, 0.01, xs=[p, x])
    assert int(g["raw"].max()) - int(g["raw"].min()) >= 2**33  # the key needs more than 33 bits
    sizes = [60_000, 0, 50_000, 40_000]  # the cloud id's multiplier is about 1e12
    g = check(knn, p, 0.01, sizes=sizes, xs=[x])
    assert int(g["raw"].max()) - int(g["raw"].min()) >= 2**33
    check(knn, p, 0.01, start=0.0, end=50.0, sizes=sizes, xs=[p])  # given range, points beyond it


def test_pool_in_column_passes(knn):
    """A long voxel whose chunk results exceed the per-pass bound (2^22 floats) at this width is pooled in several
    column passes; every column still equals the reference."""
    rng = np.random.default_rng(14)
    n_long, f = 300_000, 512
    bg = rng.random((20_000, 3), dtype=np.float32) * 10
    p = np.concatenate([bg[:9000], np.repeat(np.float32([[3.333, 3.333, 3.333]]), n_long, 0), bg[9000:]])
    assert (n_long + 31) // 32 * f > 2**22
    x = rng.normal(size=(len(p), f)).astype(np.float32)
    check(knn, p, 0.05, xs=[x])


def test_signed_zero_ties_under_max(knn):
    p = np.zeros((64, 3), np.float32)
    x = np.zeros((64, 2), np.float32)
    x[0::2, 0] = -0.0
    x[1::2, 1] = -0.0
    x[0, 1] = -0.0
    knn.voxel_grid(p, 1.0)
    got = knn.voxel_pool(x, "max")
    assert got.view(np.uint32)[0, 0] == np.float32(-0.0).view(np.uint32)  # the lowest index keeps the tie
    assert got.view(np.uint32)[0, 1] == np.float32(-0.0).view(np.uint32)
    x[0, 0] = 0.0
    assert knn.voxel_pool(x, "max").view(np.uint32)[0, 0] == 0


def test_device_pointers_and_torch_stream(knn):
    torch = pytest.importorskip("torch")
    rng = np.random.default_rng(9)
    sizes = [40_000, 0, 60_000]
    p = lidar_like(sum(sizes), rng)
    x = rng.normal(size=(p.shape[0], 64)).astype(np.float32)
    s = torch.cuda.Stream()
    with torch.cuda.stream(s):
        knn.set_stream(s.cuda_stream)
        pd, xd = torch.from_numpy(p).cuda(), torch.from_numpy(x).cuda()
        check(knn, pd, 0.3, sizes=sizes, xs=[xd])
        raw, cluster, nv = knn.voxel_grid(pd, 0.3)
        assert raw.is_cuda and raw.dtype == torch.int64 and cluster.dtype == torch.int32
    knn.set_stream(None)
    # host and device inputs, launch shapes and streams change nothing
    r2, c2, nv2 = knn.voxel_grid(p, 0.3)
    bits_equal(raw, r2, "raw host vs device")
    bits_equal(cluster, c2, "cluster host vs device")
    assert nv == nv2


def test_clustering_is_independent_of_builds_and_searches(knn):
    rng = np.random.default_rng(11)
    p = rng.random((50_000, 3), dtype=np.float32)
    idx0, d0 = knn.build(p).search(8)
    g = check(knn, p, 0.05)
    idx1, d1 = knn.search(8)
    bits_equal(idx1, idx0, "search idx after a voxel call")
    bits_equal(d1, d0, "search dist after a voxel call")
    knn.build(rng.random((1000, 3), dtype=np.float32))  # the clustering survives a build
    bits_equal(knn.voxel_pool(p), V.pool(p, g), "pool after a build")
    o, m, _, _ = knn.voxel_members()
    bits_equal(m, g["members"], "members after a build")


def test_error_codes(knn):
    L = _lib.load()
    h = knn._h
    p = np.random.default_rng(1).random((100, 3), dtype=np.float32)
    one = np.float32([1, 1, 1])
    nv = C.c_uint64()

    def grid(pts=p, n=100, dim=3, stride=3, off=None, nseg=1, size=one, start=None, end=None, nvp=C.byref(nv)):
        a = lambda v: None if v is None else v.ctypes.data
        return L.tknn_voxel_grid(h, a(pts), n, dim, stride, a(off), nseg, a(size), a(start), a(end), None, None, nvp)

    out = np.empty((100, 3), np.float32)
    assert L.tknn_voxel_pool(h, p.ctypes.data, 100, 3, 3, 0, out.ctypes.data) == _lib.ESTATE
    assert L.tknn_voxel_members(h, None, None, None, None) == _lib.ESTATE
    E = _lib.EINVAL
    assert grid(dim=4, stride=4) == E
    assert grid(dim=1) == E
    assert grid(stride=2) == E
    assert grid(size=np.float32([1, 0, 1])) == E
    assert grid(size=np.float32([1, -1, 1])) == E
    assert grid(size=np.float32([1, np.nan, 1])) == E
    assert grid(start=np.float32([0, np.inf, 0])) == E
    assert grid(end=np.float32([np.nan, 0, 0])) == E
    assert grid(nvp=None) == E
    assert grid(nseg=2) == E
    assert grid(off=np.uint64([0, 50, 99]), nseg=2) == E
    assert grid(off=np.uint64([0, 60, 50, 100]), nseg=3) == E
    assert grid(size=np.float32([1e-7, 1e-7, 1e-7])) == E  # the product of the cell counts overflows int64
    assert grid(size=np.float32([1e-20, 1, 1])) == E  # one axis' count overflows int64
    assert grid(start=np.float32([0, 0, 0]), end=np.float32([0, 0, 0]), size=np.float32([1e-20, 1, 1])) == E  # far outside
    bad = p.copy()
    bad[17, 1] = np.inf
    assert grid(pts=bad) == E
    assert grid() == 0
    assert L.tknn_voxel_pool(h, p.ctypes.data, 99, 3, 3, 0, out.ctypes.data) == E
    assert L.tknn_voxel_pool(h, p.ctypes.data, 100, 0, 3, 0, out.ctypes.data) == E
    assert L.tknn_voxel_pool(h, p.ctypes.data, 100, 1025, 1025, 0, out.ctypes.data) == E
    assert L.tknn_voxel_pool(h, p.ctypes.data, 100, 3, 2, 0, out.ctypes.data) == E
    assert L.tknn_voxel_pool(h, p.ctypes.data, 100, 3, 3, 2, out.ctypes.data) == E
    assert L.tknn_voxel_pool(h, None, 100, 3, 3, 0, out.ctypes.data) == E
    nan = p.copy()
    nan[3, 2] = np.nan
    assert L.tknn_voxel_pool(h, nan.ctypes.data, 100, 3, 3, 1, out.ctypes.data) == E
    with pytest.raises(TrueKNNError):
        knn.voxel_pool(np.zeros((7, 2), np.float32))


def torch_pipeline(pos, size, batch=None, x=None):
    """The plain-torch route: the formula, torch.unique, then float64 sums for the mean."""
    import torch

    p = pos
    sz = torch.full((pos.shape[1],), float(size), device=pos.device)
    if batch is not None:
        p = torch.cat([pos, batch.to(pos.dtype).view(-1, 1)], 1)
        sz = torch.cat([sz, torch.ones(1, device=pos.device)])
    s0, e0 = p.min(0).values, p.max(0).values
    cnt = ((e0 - s0) / sz).long() + 1
    mult = torch.cat([torch.ones(1, dtype=torch.long, device=pos.device), torch.cumprod(cnt, 0)[:-1]])
    raw = (((p - s0) / sz).long() * mult).sum(1)
    _, inv = torch.unique(raw, sorted=True, return_inverse=True)
    nv = int(inv.max()) + 1
    cnt = torch.bincount(inv, minlength=nv).double().view(-1, 1)
    mean = lambda a: (torch.zeros(nv, a.shape[1], dtype=torch.float64, device=a.device).index_add_(0, inv, a.double()) / cnt)
    return raw, inv, mean(pos), None if x is None else mean(x)


def test_module_functions_against_torch():
    torch = pytest.importorskip("torch")
    rng = np.random.default_rng(12)
    sizes = [30_000, 0, 50_000, 20_000]
    p = lidar_like(sum(sizes), rng)
    x = rng.normal(size=(p.shape[0], 16)).astype(np.float32)
    b = np.repeat(np.arange(len(sizes)), sizes)
    pd, xd, bd = torch.from_numpy(p).cuda(), torch.from_numpy(x).cuda(), torch.from_numpy(b).cuda()
    raw_t, inv_t, pm_t, xm_t = torch_pipeline(pd, 0.4, bd, xd)
    assert torch.equal(voxel_grid(pd, 0.4, bd), raw_t)
    raw0, inv0, _, _ = torch_pipeline(pd, 0.4)
    assert torch.equal(grid_cluster(pd, 0.4), raw0)
    assert (grid_cluster(p, 0.4) == raw0.cpu().numpy()).all()  # numpy in, numpy out
    pm, xm, bo, cl = grid_sampling(pd, 0.4, xd, bd)
    assert torch.equal(cl, inv_t)
    torch.testing.assert_close(pm.double(), pm_t, rtol=1e-5, atol=1e-5)
    torch.testing.assert_close(xm.double(), xm_t, rtol=1e-5, atol=1e-5)
    g = V.grid(p, 0.4, off=offsets_of(sizes))
    bits_equal(pm, V.pool(p, g), "grid_sampling pos")
    bits_equal(xm, V.pool(x, g), "grid_sampling x")
    bits_equal(bo, g["seg"].astype(np.int64), "grid_sampling batch")
    _, xmax, _, _ = grid_sampling(p, 0.4, x, b, reduce="max")
    bits_equal(xmax, V.pool(x, g, "max"), "grid_sampling max")
