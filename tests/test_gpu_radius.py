"""tknn_radius_search / tknn_radius_query (TrueKNN.radius_search / radius_query) on the GPU: bit-exact against the CPU
reference (tests/radius_oracle.c), consistent with tknn_range_count and tknn_search."""
import ctypes

import numpy as np
import pytest

import radius_oracle as RO
from owlraytracing_b200 import MultiTrueKNN, TrueKNN, TrueKNNError, datasets
from owlraytracing_b200 import _lib
from test_gpu_dbscan import duplicate_cloud

pytestmark = pytest.mark.gpu

SHORT_MAX = 1024  # rows longer than this take the radix-sort tier (radius.cuh)


def _np(a):
    return a.cpu().numpy() if hasattr(a, "cpu") else np.asarray(a)


def assert_same(got, want, what="", squared=True):
    go, gi, gd = (_np(a) if a is not None else None for a in got)
    wo, wi, wd = want
    assert go.dtype == np.int64 and gi.dtype == np.int32
    bad = np.flatnonzero(go != wo)
    assert bad.size == 0, f"{what}: offsets differ at rows {bad[:10]}"
    bad = np.flatnonzero(gi != wi)
    assert bad.size == 0, f"{what}: {bad.size} indices differ, first at {bad[:10]}"
    if gd is not None:
        w = wd if squared else np.sqrt(wd)
        bad = np.flatnonzero(gd.view(np.uint32) != w.view(np.uint32))
        assert bad.size == 0, f"{what}: {bad.size} distances differ, first at {bad[:10]}"


def check(knn, x, r, what, squared=True):
    knn.set_option("squared_dist", 1 if squared else 0)
    got = knn.build(x).radius_search(r)
    want = RO.radius_lists(x, r)
    assert_same(got, want, what, squared)
    st = knn.stats()
    assert st["rounds"] == 3 and st["n_queries"] == len(x)
    lens = np.diff(want[0])
    # an empty result needs no second call: the wrapper's size call is the last one then
    filled = len(x) if want[0][-1] else 0
    assert st["round_queries"][:3] == [len(x), filled, int((lens > SHORT_MAX).sum())]
    return got


@pytest.fixture(scope="module")
def uniform200k():
    return datasets.uniform(200_000, seed=42)


@pytest.mark.parametrize("r", [0.0229, 0.0493])  # about 10 and 100 neighbours per point
@pytest.mark.parametrize("squared", [True, False])
def test_uniform_200k(knn, uniform200k, r, squared):
    off, _, _ = check(knn, uniform200k, r, f"uniform r={r}", squared)
    mean = off[-1] / len(uniform200k)
    assert (5 < mean < 15) if r < 0.03 else (60 < mean < 120)


@pytest.fixture(scope="module")
def lidar1m():
    return datasets.lidar_like(1_000_000, seed=7)


def test_lidar_1m(knn, lidar1m):
    check(knn, lidar1m, 0.05, "lidar r=0.05")


@pytest.mark.parametrize("r", [0.0, 0.03, 0.06])
def test_duplicates(knn, r):
    check(knn, duplicate_cloud(), r, f"duplicates r={r}")


def test_two_dimensional_input(knn):
    x = np.random.default_rng(21).random((50_000, 2)).astype(np.float32)
    check(knn, x, 0.01, "2-D")


def test_lattice_closed_ball(knn):
    x = datasets.lattice(20)
    off, idx, _ = check(knn, x, 1.0, "lattice r=1")
    g = x.astype(np.int64)
    interior = ((g > 0) & (g < 19)).all(1)
    assert (np.diff(off)[interior] == 6).all()
    off, _, _ = check(knn, x, float(np.nextafter(np.float32(1), np.float32(0))), "lattice r<1")
    assert off[-1] == 0


def test_special_radii_and_sizes(knn):
    x = np.repeat(np.random.default_rng(22).random((500, 3)).astype(np.float32), 3, axis=0)
    off, _, d = check(knn, x, 0.0, "r=0")
    assert (np.diff(off) == 2).all() and (d == 0).all()
    x = np.random.default_rng(23).random((300, 3)).astype(np.float32)
    off, _, _ = check(knn, x, np.inf, "r=inf")
    assert (np.diff(off) == 299).all()
    off, idx, _ = check(knn, x[:2], np.inf, "n=2")  # the smallest cloud a build accepts
    assert off.tolist() == [0, 1, 2] and idx.tolist() == [1, 0]
    off, idx, _ = check(knn, x[:2], 0.0, "n=2, r=0")
    assert off.tolist() == [0, 0, 0] and idx.size == 0
    off, idx, _ = check(knn, x[:3], np.inf, "n=3")
    assert off.tolist() == [0, 2, 4, 6]


def long_row_cloud():
    """A coincident cluster (rows ordered by index alone), a dense Gaussian blob (long rows of many distinct d2) and a
    uniform background (short rows)."""
    rng = np.random.default_rng(24)
    cluster = np.tile(np.array([[0.2, 0.2, 0.2]], np.float32), (12_000, 1))
    blob = rng.normal(0.7, 0.01, (30_000, 3))
    back = rng.random((50_000, 3))
    x = np.concatenate([back, cluster, blob]).astype(np.float32)
    return x[rng.permutation(len(x))]


def test_both_sort_tiers(knn):
    x = long_row_cloud()
    off, _, _ = check(knn, x, 0.01, "long rows")
    lens = np.diff(off)
    assert (lens == 11_999).sum() == 12_000, "the coincident cluster"
    blob_long = (lens > SHORT_MAX) & (lens != 11_999)
    assert blob_long.sum() > 1000 and np.unique(lens[blob_long]).size > 100
    assert ((lens > 1) & (lens <= SHORT_MAX)).sum() > 5_000


def test_cross_checks(knn, uniform200k):
    r = 0.0493
    knn.build(uniform200k)
    off, idx, dist = knn.radius_search(r)
    assert (np.diff(off) == knn.range_count(r).astype(np.int64)).all()
    lens = np.diff(off)
    for k in (10, 64):
        si, sd = knn.search(k)
        rows = np.flatnonzero(lens >= k)
        assert rows.size > len(uniform200k) // 2
        take = off[rows][:, None] + np.arange(k)[None, :]
        assert (idx[take] == si[rows]).all(), f"k={k}: indices"
        assert (dist[take].view(np.uint32) == sd[rows].view(np.uint32)).all(), f"k={k}: distances"


def test_query_form(knn):
    import torch

    x = datasets.uniform(100_000, seed=3)
    rng = np.random.default_rng(25)
    near = x[:3000] + rng.normal(0, 0.003, (3000, 3)).astype(np.float32)
    far = rng.random((1000, 3)).astype(np.float32) + np.float32(5.0)
    q = np.concatenate([near, far]).astype(np.float32)
    sid = np.full(len(q), -1, np.int32)
    sid[:1000] = np.arange(1000)                 # mostly inside the ball
    sid[1000:2000] = np.arange(50_000, 51_000)   # outside it
    r = 0.03
    knn.set_option("squared_dist", 1)
    knn.build(x)
    want = RO.radius_lists(x, r, q, sid)
    got = knn.radius_query(q, r, self_ids=sid)
    assert_same(got, want, "query form")
    lens = np.diff(want[0])
    assert (lens[3000:] == 0).all()
    inside = np.array([np.any(want[1][want[0][i]:want[0][i + 1]] == sid[i]) for i in range(1000)])
    assert not inside.any()
    assert_same(knn.radius_query(q, r), RO.radius_lists(x, r, q), "query form, no self ids")
    # device inputs and outputs
    got = knn.radius_query(torch.from_numpy(q).cuda(), r, self_ids=torch.from_numpy(sid).cuda())
    assert got[0].is_cuda and got[1].is_cuda and got[2].is_cuda
    assert_same(got, want, "query form, device")
    # 2-D queries against a 2-D build
    x2 = np.random.default_rng(26).random((20_000, 2)).astype(np.float32)
    q2 = np.random.default_rng(27).random((3000, 2)).astype(np.float32)
    knn.build(x2)
    assert_same(knn.radius_query(q2, 0.02), RO.radius_lists(x2, 0.02, q2), "2-D queries")
    # no queries
    off, idx, dist = knn.radius_query(np.empty((0, 3), np.float32), 0.02)
    assert off.tolist() == [0] and idx.size == 0


def test_sizing_protocol(knn):
    x = datasets.uniform(20_000, seed=8)
    r = 0.04
    knn.set_option("squared_dist", 1)
    knn.build(x)
    want = RO.radius_lists(x, r)
    total = int(want[0][-1])
    L, h = knn._L, knn._h
    off = np.zeros(len(x) + 1, np.uint64)
    t = ctypes.c_uint64(0)

    def call(idx, dist, cap):
        return L.tknn_radius_search(h, ctypes.c_float(r), ctypes.c_void_p(off.ctypes.data),
                                    None if idx is None else ctypes.c_void_p(idx.ctypes.data),
                                    None if dist is None else ctypes.c_void_p(dist.ctypes.data), cap, ctypes.byref(t))

    assert call(None, None, 0) == _lib.OK and t.value == total and (off.view(np.int64) == want[0]).all()
    idx, dist = np.empty(total, np.int32), np.empty(total, np.float32)
    off[:] = 0
    idx[:] = -7
    assert call(idx, dist, total - 1) == _lib.EINVAL
    assert t.value == total and (off.view(np.int64) == want[0]).all() and (idx == -7).all()
    assert call(idx, dist, total) == _lib.OK
    assert_same((off.view(np.int64), idx, dist), want, "exact capacity")
    idx[:] = -7
    assert call(idx, None, total) == _lib.OK and (idx == want[1]).all()
    o2, i2, d2 = knn.radius_search(r, indices_only=True)
    assert d2 is None and (i2 == want[1]).all()
    # out=: one call; too small raises naming the total
    o3, i3, d3 = knn.radius_search(r, out=(np.empty(len(x) + 1, np.int64), np.empty(total + 5, np.int32),
                                           np.empty(total + 5, np.float32)))
    assert_same((o3, i3, d3), want, "out=")
    with pytest.raises(TrueKNNError, match=str(total)):
        knn.radius_search(r, out=(np.empty(len(x) + 1, np.int64), np.empty(total - 1, np.int32), None))


def test_errors(knn):
    off = np.zeros(101, np.uint64)
    t = ctypes.c_uint64(0)

    def rc(ctx, r, o=off):
        return ctx._L.tknn_radius_search(ctx._h, ctypes.c_float(r), None if o is None else ctypes.c_void_p(o.ctypes.data),
                                         None, None, 0, ctypes.byref(t))

    assert rc(knn, 0.1) == _lib.ESTATE  # before a build
    knn.build(datasets.uniform(100, seed=3))
    assert rc(knn, float("nan")) == _lib.EINVAL
    assert rc(knn, -0.1) == _lib.EINVAL
    assert rc(knn, 0.1, None) == _lib.EINVAL
    assert rc(knn, 0.1) == _lib.OK
    assert rc(knn, float("inf")) == _lib.OK and t.value == 100 * 99
    with pytest.raises(TrueKNNError):
        knn.radius_query(np.zeros((4, 3), np.float32), -1.0)
    with pytest.raises(TrueKNNError):
        knn.radius_query(np.full((4, 3), np.nan, np.float32), 0.1)
    with MultiTrueKNN([0, 0], "partition") as m:
        m.build(datasets.uniform(4000, seed=4))
        view = m.rank(0)
        assert rc(view, 0.1, np.zeros(4001, np.uint64)) == _lib.ESTATE


def test_deterministic_stats_and_counters(lidar1m):
    r = 0.05
    outs = []
    for opts in ({}, {"blocks_per_sm": 1}, {"counters": 1}):
        with TrueKNN(0, **opts) as t:
            t.build(lidar1m)
            outs.append(t.radius_search(r))
            outs.append(t.radius_search(r))
            st = t.stats()
            assert st["rounds"] == 3 and st["round_queries"][:2] == [len(lidar1m), len(lidar1m)]
            assert st["search_ms"] > 0 and all(v >= 0 for v in st["round_ms"][:3])
            if opts.get("counters"):
                assert st["nodes_visited"] > 0 and st["points_tested"] > 0
                assert st["heap_inserts"] == int(outs[-1][0][-1])  # one per entry written by the fill pass
    for o in outs[1:]:
        for a, b in zip(o, outs[0]):
            assert (a.view(np.uint32 if a.dtype == np.float32 else a.dtype) ==
                    b.view(np.uint32 if b.dtype == np.float32 else b.dtype)).all()


def test_torch_sparse_csr(knn):
    import torch

    x = torch.from_numpy(datasets.uniform(50_000, seed=9)).cuda()
    off, idx, dist = knn.build(x).radius_search(0.03)
    assert off.is_cuda and off.dtype == torch.int64 and idx.dtype == torch.int32
    a = torch.sparse_csr_tensor(off, idx, dist, size=(50_000, 50_000))
    assert a.shape == (50_000, 50_000) and a._nnz() == int(off[-1])
    host = knn.build(x.cpu().numpy()).radius_search(0.03)
    assert (host[0] == off.cpu().numpy()).all() and (host[1] == idx.cpu().numpy()).all()
