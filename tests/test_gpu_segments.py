"""Segmented builds (tknn_build_segments / TrueKNN.build(batch=...)) on the GPU: bit for bit against the per-segment
CPU reference (tests/segment_oracle.py), plus the one-segment identity, the refused calls and the graph helpers."""
import ctypes

import numpy as np
import pytest

import segment_oracle as SO
from owlraytracing_b200 import TrueKNN, TrueKNNError, _lib, datasets, knn_graph, radius_graph

pytestmark = pytest.mark.gpu


def _np(a):
    return a.cpu().numpy() if hasattr(a, "cpu") else np.asarray(a)


def batch_of(sizes):
    return np.repeat(np.arange(len(sizes)), sizes).astype(np.int64)


def assert_rows(got, want, what):
    gi, gd = _np(got[0]), _np(got[1])
    wi, wd = want
    bad = np.flatnonzero((gi != wi).any(axis=1))
    assert bad.size == 0, f"{what}: {bad.size} rows differ in indices, first {bad[:5]}: {gi[bad[0]]} vs {wi[bad[0]]}"
    bad = np.flatnonzero((gd.view(np.uint32) != wd.view(np.uint32)).any(axis=1))
    assert bad.size == 0, f"{what}: {bad.size} rows differ in distances, first {bad[:5]}"


def check_knn(knn, x, sizes, k, squared=True, what="", **search):
    knn.set_option("squared_dist", 1 if squared else 0)
    got = knn.build(x, batch=batch_of(sizes)).search(k, **search)
    assert_rows(got, SO.knn(x, SO.offsets_of(sizes), k, squared=squared), what)
    return got


@pytest.fixture(scope="module")
def batch1024():
    return datasets.uniform(1024 * 4096, seed=11), [4096] * 1024


def uneven_sizes(k, seed=5):
    """half the segments smaller than k + 1 (0, 1, 2, k, and others), the rest 20 .. 3000 points"""
    rng = np.random.default_rng(seed)
    small = list(rng.choice([0, 1, 2, k], size=300)) + [k] * 10
    big = list(rng.integers(20, 3000, size=310)) + [k + 1] * 10
    sizes = np.array(small + big)
    rng.shuffle(sizes)
    return [int(s) for s in sizes]


@pytest.mark.parametrize("squared", [True, False])
def test_uniform_1024_clouds_k16(knn, batch1024, squared):
    x, sizes = batch1024
    check_knn(knn, x, sizes, 16, squared, "1024 x 4096")


@pytest.mark.parametrize("k", [16, 40])
def test_uneven_sizes_half_below_k_plus_1(knn, k):
    sizes = uneven_sizes(k)
    x = datasets.uniform(sum(sizes), seed=21)
    i, _ = check_knn(knn, x, sizes, k, what=f"uneven k={k}")
    assert (_np(i)[:, -1] == -1).any()


def test_lidar_sweeps_heap(knn):
    sizes = [100_000] * 16
    x = np.concatenate([datasets.lidar_like(100_000, seed=s) for s in range(16)])
    check_knn(knn, x, sizes, 64, what="16 lidar sweeps k=64")


def test_duplicate_heavy_segments_tie_variant(knn):
    rng = np.random.default_rng(3)
    parts = []
    for s in range(40):
        base = rng.random((50, 3), dtype=np.float32)
        parts.append(np.repeat(base, rng.integers(1, 40, size=50), axis=0))
    parts.append(np.repeat(parts[0][:5], 3, axis=0))  # a cloud coincident with points of cloud 0
    sizes = [len(p) for p in parts]
    x = np.concatenate(parts)
    for k in (8, 32):
        check_knn(knn, x, sizes, k, what=f"duplicates k={k}")
        assert knn.stats()["k"] == k


def test_two_dimensional_batch(knn):
    rng = np.random.default_rng(8)
    sizes = [int(s) for s in rng.integers(0, 2000, size=200)]
    x = rng.random((sum(sizes), 2), dtype=np.float32)
    check_knn(knn, x, sizes, 12, what="2-D")


@pytest.mark.parametrize("opt", ["approx_filter", "counters"])
def test_options(knn, batch1024, opt):
    x, sizes = batch1024
    knn.set_option(opt, 1)
    check_knn(knn, x[: 256 * 4096], sizes[:256], 16, what=opt)
    if opt == "counters":
        assert knn.stats()["filter_violations"] == 0


def test_device_outputs_and_input(knn, batch1024):
    torch = pytest.importorskip("torch")
    x, sizes = batch1024
    xt = torch.from_numpy(x[: 128 * 4096]).cuda()
    bt = torch.from_numpy(batch_of(sizes[:128])).cuda()
    knn.set_option("squared_dist", 1)
    i, d = knn.build(xt, batch=bt).search(16)
    assert i.is_cuda and d.is_cuda
    assert_rows((i, d), SO.knn(x[: 128 * 4096], SO.offsets_of(sizes[:128]), 16, squared=True), "device")


@pytest.mark.parametrize("chunks", [1, 5])
def test_file_order_chunks_host_outputs(knn, batch1024, chunks):
    x, sizes = batch1024
    knn.set_option("file_order_chunks", chunks)
    check_knn(knn, x, sizes, 16, squared=False, what=f"file-order chunks {chunks}")


def test_explicit_start_radius(knn):
    sizes = uneven_sizes(16, seed=9)
    x = datasets.uniform(sum(sizes), seed=4)
    check_knn(knn, x, sizes, 16, what="start radius", start_radius=0.001)
    assert knn.stats()["rounds"] >= 2


def test_estimate_with_tiny_segments_is_finite(knn):
    sizes = [3] * 5000 + [400] * 20
    x = datasets.uniform(sum(sizes), seed=6)
    knn.build(x, batch=batch_of(sizes))
    assert np.isfinite(knn.estimate_start_radius(16))
    sizes = [3] * 5000
    knn.build(datasets.uniform(sum(sizes), seed=6), batch=batch_of(sizes))
    assert knn.estimate_start_radius(2) > 0
    check_knn(knn, datasets.uniform(sum(sizes), seed=6), sizes, 4, what="all rows unfilled")


def test_radius_search_and_range_count(knn):
    sizes = uneven_sizes(16, seed=12)
    x = datasets.uniform(sum(sizes), seed=13)
    r = 0.05
    knn.set_option("squared_dist", 1)
    off, idx, d2 = knn.build(x, batch=batch_of(sizes)).radius_search(r)
    wo, wi, wd = SO.radius_lists(x, SO.offsets_of(sizes), r)
    np.testing.assert_array_equal(off, wo)
    np.testing.assert_array_equal(idx, wi)
    np.testing.assert_array_equal(d2.view(np.uint32), wd.view(np.uint32))
    np.testing.assert_array_equal(knn.range_count(r), np.diff(wo))


def test_radius_search_long_rows(knn):
    # dense clouds: rows longer than 1024 take the radix-sort tier
    rng = np.random.default_rng(14)
    sizes = [3000, 5, 2500, 0, 4000]
    x = (rng.random((sum(sizes), 3), dtype=np.float32) * 0.1).astype(np.float32)
    r = 0.06
    off, idx, d2 = knn.build(x, batch=batch_of(sizes)).radius_search(r)
    wo, wi, wd = SO.radius_lists(x, SO.offsets_of(sizes), r)
    assert np.diff(wo).max() > 1024
    np.testing.assert_array_equal(off, wo)
    np.testing.assert_array_equal(idx, wi)
    np.testing.assert_array_equal(np.asarray(d2), np.sqrt(wd))


def test_one_segment_is_a_plain_build(knn):
    x = datasets.uniform(300_000, seed=15)
    L = _lib.load()
    plain = TrueKNN(0)
    try:
        plain.build(x)
        knn.build(x, batch=np.zeros(len(x), np.int64))
        m = knn.stats()["n_leaves"]
        assert plain.stats()["n_leaves"] == m

        def bvh(t):
            nodes = np.empty((m - 1) * 16, np.float32)
            pts = np.empty(len(x) * 4, np.float32)
            ls = np.empty(m + 1, np.uint32)
            assert L.tknn_get_bvh(t._h, nodes.ctypes.data, pts.ctypes.data, ls.ctypes.data) == 0
            return nodes.view(np.uint32), pts.view(np.uint32), ls

        for a, b in zip(bvh(plain), bvh(knn)):
            np.testing.assert_array_equal(a, b)
        a, b = plain.search(16), knn.search(16)
        np.testing.assert_array_equal(a[0], b[0])
        np.testing.assert_array_equal(a[1].view(np.uint32), b[1].view(np.uint32))
    finally:
        plain.close()


def test_refused_calls_and_plain_rebuild(knn):
    sizes = [500, 700]
    x = datasets.uniform(1200, seed=16)
    knn.build(x, batch=batch_of(sizes))
    L = _lib.load()
    buf = np.zeros(1200 * 16, np.int32)
    fbuf = np.zeros(1200 * 16, np.float32)
    q = np.zeros((4, 3), np.float32)
    n_out = ctypes.c_uint64(0)
    off = np.zeros(8, np.uint64)
    calls = {
        "tknn_search_shard": lambda: L.tknn_search_shard(knn._h, 4, ctypes.c_float(0), 0, 2, buf.ctypes.data,
                                                         buf.ctypes.data, fbuf.ctypes.data, ctypes.byref(n_out)),
        "tknn_query": lambda: L.tknn_query(knn._h, q.ctypes.data, 4, 3, 3, None, None, 4, ctypes.c_float(0),
                                           buf.ctypes.data, fbuf.ctypes.data),
        "tknn_radius_query": lambda: L.tknn_radius_query(knn._h, q.ctypes.data, 4, 3, 3, None, ctypes.c_float(0.1),
                                                         off.ctypes.data, None, None, 0, ctypes.byref(n_out)),
        "tknn_dbscan": lambda: L.tknn_dbscan(knn._h, ctypes.c_float(0.1), 4, buf.ctypes.data, None, None),
        "tknn_brute_force": lambda: L.tknn_brute_force(knn._h, buf.ctypes.data, 4, 4, buf.ctypes.data, fbuf.ctypes.data),
        "tknn_partition_search": lambda: L.tknn_partition_search(knn._h, 4, ctypes.c_float(0), buf.ctypes.data,
                                                                 buf.ctypes.data, fbuf.ctypes.data, 1200,
                                                                 ctypes.byref(n_out)),
        "tknn_partition_verify": lambda: L.tknn_partition_verify(knn._h, 4, 4, buf.ctypes.data, buf.ctypes.data,
                                                                 fbuf.ctypes.data, 4, ctypes.byref(n_out),
                                                                 ctypes.byref(n_out)),
    }
    for name, call in calls.items():
        assert call() == _lib.ESTATE, name
        assert b"segmented" in L.tknn_last_error(knn._h), name
    # a plain build clears the segments: the whole cloud is one again
    i, d = knn.build(x).search(8)
    want = TrueKNN(0)
    try:
        wi, wd = want.build(x).search(8)
    finally:
        want.close()
    np.testing.assert_array_equal(i, wi)
    np.testing.assert_array_equal(d, wd)
    assert knn.query(q, 4)[0].shape == (4, 4)


@pytest.mark.parametrize("offsets", [[1, 600, 1200], [0, 700, 600, 1200], [0, 600, 1199], [0, 600, 1201]])
def test_invalid_offsets(knn, offsets):
    x = datasets.uniform(1200, seed=17)
    off = np.array(offsets, np.uint64)
    L = _lib.load()
    assert L.tknn_build_segments(knn._h, x.ctypes.data, 1200, 3, 3, off.ctypes.data, len(off) - 1) == _lib.EINVAL


def test_invalid_batch(knn):
    x = datasets.uniform(100, seed=18)
    with pytest.raises(ValueError):
        knn.build(x, batch=np.r_[np.zeros(50, np.int64), np.zeros(50, np.int64) - 1])
    with pytest.raises(ValueError):
        knn.build(x, batch=np.r_[np.ones(50, np.int64), np.zeros(50, np.int64)])


def test_knn_graph_and_radius_graph():
    torch = pytest.importorskip("torch")
    sizes = [40, 2, 0, 60]
    x = datasets.uniform(sum(sizes), seed=19)
    b = batch_of(sizes)
    off = SO.offsets_of(sizes)
    k = 6
    wi, _ = SO.knn(x, off, k)
    centre = np.repeat(np.arange(len(x)), k)
    keep = wi.reshape(-1) >= 0
    want = np.stack([wi.reshape(-1)[keep], centre[keep]]).astype(np.int64)
    e = knn_graph(x, k, b)
    assert e.dtype == np.int64 and e.shape == want.shape
    np.testing.assert_array_equal(e, want)
    et = knn_graph(torch.from_numpy(x).cuda(), k, torch.from_numpy(b).cuda())
    assert et.dtype == torch.int64 and et.is_cuda
    np.testing.assert_array_equal(et.cpu().numpy(), want)
    assert not (e[0] == e[1]).any()
    wo, wi, _ = SO.radius_lists(x, off, 0.3)
    want = np.stack([wi, np.repeat(np.arange(len(x)), np.diff(wo))]).astype(np.int64)
    np.testing.assert_array_equal(radius_graph(x, 0.3, b), want)
    rt = radius_graph(torch.from_numpy(x).cuda(), 0.3, torch.from_numpy(b).cuda())
    np.testing.assert_array_equal(rt.cpu().numpy(), want)
    # without a batch: one cloud
    wi, _ = SO.knn(x, SO.offsets_of([len(x)]), k)
    np.testing.assert_array_equal(knn_graph(x, k)[0], wi.reshape(-1))
