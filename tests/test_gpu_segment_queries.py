"""Segmented query sets (tknn_query_segments / tknn_radius_query_segments, TrueKNN.query(batch=...),
TrueKNN.radius_query(batch=...), knn(), radius()) on the GPU: bit for bit against the per-segment CPU reference
(tests/segment_query_oracle.py), the two identities with the all-points and the unsegmented calls, and the errors."""
import ctypes

import numpy as np
import pytest

import segment_query_oracle as SQ
from owlraytracing_b200 import MultiTrueKNN, TrueKNN, TrueKNNError, _lib, datasets, knn, radius

pytestmark = pytest.mark.gpu


def _np(a):
    return a.cpu().numpy() if hasattr(a, "cpu") else np.asarray(a)


def batch_of(sizes):
    return np.repeat(np.arange(len(sizes)), sizes).astype(np.int64)


def rows_of(y_off, segments):
    return np.concatenate([np.arange(int(y_off[s]), int(y_off[s + 1])) for s in segments]).astype(np.int64)


def assert_rows(got, want, what, rows=None):
    gi, gd = _np(got[0]), _np(got[1])
    wi, wd = want
    if rows is not None:
        gi, gd, wi, wd = gi[rows], gd[rows], wi[rows], wd[rows]
    bad = np.flatnonzero((gi != wi).any(axis=1))
    assert bad.size == 0, f"{what}: {bad.size} rows differ in indices, first {bad[:5]}: {gi[bad[0]]} vs {wi[bad[0]]}"
    bad = np.flatnonzero((gd.view(np.uint32) != wd.view(np.uint32)).any(axis=1))
    assert bad.size == 0, f"{what}: {bad.size} rows differ in distances, first {bad[:5]}"


def assert_lists(got, want, what):
    off, idx, d = (_np(a) for a in got)
    wo, wi, wd = want
    np.testing.assert_array_equal(off.astype(np.int64), wo, err_msg=f"{what}: offsets")
    np.testing.assert_array_equal(idx, wi, err_msg=f"{what}: indices")
    np.testing.assert_array_equal(d.view(np.uint32), wd.view(np.uint32), err_msg=f"{what}: distance bits")


def check_query(t, x, y, x_sizes, y_sizes, k, squared=True, segments=None, self_ids=None, init_radius2=None,
                start_radius=0.0, what=""):
    t.set_option("squared_dist", 1 if squared else 0)
    t.build(x, batch=batch_of(x_sizes), batch_size=len(x_sizes))
    got = t.query(y, k, self_ids=self_ids, init_radius2=init_radius2, start_radius=start_radius, batch=batch_of(y_sizes))
    x_off, y_off = SQ.offsets_of(x_sizes), SQ.offsets_of(y_sizes)
    want = SQ.knn(x, y, x_off, y_off, k, self_ids=self_ids, caps2=init_radius2, squared=squared, segments=segments)
    assert_rows(got, want, what, None if segments is None else rows_of(y_off, segments))
    return got


@pytest.fixture(scope="module")
def set_abstraction():
    """1 024 uniform clouds x 4 096 points; every 4th point of each cloud is a query (PointNet++ set abstraction)."""
    x = datasets.uniform(1024 * 4096, seed=11)
    return x, [4096] * 1024, np.ascontiguousarray(x[::4]), [1024] * 1024


SAMPLE = range(0, 1024, 8)  # the sampled clouds of the large kNN checks


@pytest.mark.parametrize("squared", [True, False])
def test_set_abstraction_knn16(knn, set_abstraction, squared):
    x, xs, y, ys = set_abstraction
    check_query(knn, x, y, xs, ys, 16, squared, segments=SAMPLE, what="set abstraction k=16")


def test_set_abstraction_radius(knn, set_abstraction):
    x, xs, y, ys = set_abstraction
    knn.set_option("squared_dist", 1)
    got = knn.build(x, batch=batch_of(xs)).radius_query(y, 0.123, batch=batch_of(ys))
    assert_lists(got, SQ.radius_lists(x, y, SQ.offsets_of(xs), SQ.offsets_of(ys), 0.123), "set abstraction r=0.123")


def test_interpolation_knn3(knn, set_abstraction):
    x, xs, y, ys = set_abstraction
    check_query(knn, y, x, ys, xs, 3, segments=SAMPLE, what="interpolation k=3")


def uneven(k, seed):
    """data segments of 0, 1, k and k + 1 points among larger ones; half the query segments of 1 to 40 rows (32-query
    groups straddle many clouds), some empty, the rest larger"""
    rng = np.random.default_rng(seed)
    m = 400
    xs = [int(s) for s in rng.choice([0, 1, k, k + 1], size=m // 2)] + [int(s) for s in rng.integers(20, 2000, size=m // 2)]
    ys = [int(s) for s in rng.integers(1, 41, size=m // 2)] + [int(s) for s in rng.integers(0, 600, size=m // 2)]
    perm = rng.permutation(m)
    return [xs[i] for i in perm], [ys[i] for i in rng.permutation(m)]


@pytest.mark.parametrize("k", [16, 40])
def test_uneven_sizes(knn, k):
    xs, ys = uneven(k, 3)
    x = datasets.uniform(sum(xs), seed=31)
    y = datasets.uniform(sum(ys), seed=32)
    i, _ = check_query(knn, x, y, xs, ys, k, what=f"uneven k={k}")
    assert (_np(i)[:, 0] == -1).any() and (_np(i)[:, -1] == -1).any()
    knn.set_option("squared_dist", 1)
    got = knn.radius_query(y, 0.08, batch=batch_of(ys))
    assert_lists(got, SQ.radius_lists(x, y, SQ.offsets_of(xs), SQ.offsets_of(ys), 0.08), f"uneven radius k={k}")


def test_self_ids_inside_outside_and_none(knn):
    xs, ys = uneven(16, 4)
    x = datasets.uniform(sum(xs), seed=33)
    xo, yo = SQ.offsets_of(xs), SQ.offsets_of(ys)
    rng = np.random.default_rng(5)
    sid = rng.integers(-1, len(x), size=sum(ys)).astype(np.int32)  # mostly outside the query's data segment
    y = datasets.uniform(sum(ys), seed=34)
    for s in range(len(xs)):  # the first query of each segment sits on a point of its data segment and names it
        if ys[s] and xs[s]:
            p = int(xo[s]) + int(rng.integers(0, xs[s]))
            y[int(yo[s])] = x[p]
            sid[int(yo[s])] = p
    check_query(knn, x, y, xs, ys, 16, self_ids=sid, what="self ids")
    got = knn.radius_query(y, 0.1, self_ids=sid, batch=batch_of(ys))
    assert_lists(got, SQ.radius_lists(x, y, xo, yo, 0.1, self_ids=sid), "self ids radius")


def test_lidar_sweeps_heap(knn):
    xs = [100_000] * 16
    x = np.concatenate([datasets.lidar_like(100_000, seed=s) for s in range(16)])
    y = np.ascontiguousarray(x[::8] + np.float32(0.01))
    check_query(knn, x, y, xs, [12_500] * 16, 64, what="16 lidar sweeps k=64")


def test_duplicate_heavy_tie_variant(knn):
    rng = np.random.default_rng(3)
    parts = []
    for s in range(40):
        base = rng.random((50, 3), dtype=np.float32)
        parts.append(np.repeat(base, rng.integers(1, 40, size=50), axis=0))
    parts.append(np.repeat(parts[0][:5], 3, axis=0))  # a cloud coincident with points of cloud 0
    xs = [len(p) for p in parts]
    x = np.concatenate(parts)
    y = np.ascontiguousarray(np.concatenate([p[::3] for p in parts]))  # queries on the duplicates
    ys = [len(p[::3]) for p in parts]
    for k in (8, 32):
        check_query(knn, x, y, xs, ys, k, what=f"duplicates k={k}")


def test_two_dimensional(knn):
    rng = np.random.default_rng(8)
    xs = [int(s) for s in rng.integers(0, 2000, size=200)]
    ys = [int(s) for s in rng.integers(0, 300, size=200)]
    x = rng.random((sum(xs), 2), dtype=np.float32)
    y = rng.random((sum(ys), 2), dtype=np.float32)
    check_query(knn, x, y, xs, ys, 12, what="2-D")
    knn.set_option("squared_dist", 1)
    got = knn.radius_query(y, 0.05, batch=batch_of(ys))
    assert_lists(got, SQ.radius_lists(x, y, SQ.offsets_of(xs), SQ.offsets_of(ys), 0.05), "2-D radius")


def test_init_radius2_caps(knn):
    xs, ys = uneven(16, 6)
    x = datasets.uniform(sum(xs), seed=35)
    y = datasets.uniform(sum(ys), seed=36)
    caps = np.random.default_rng(7).choice([-1.0, 0.0004, 0.003, 0.02], size=sum(ys)).astype(np.float32)
    check_query(knn, x, y, xs, ys, 16, init_radius2=caps, what="caps")


@pytest.mark.parametrize("start_radius", [0.002, float("inf")])
def test_explicit_start_radius(knn, start_radius):
    xs, ys = uneven(16, 7)
    x = datasets.uniform(sum(xs), seed=37)
    y = datasets.uniform(sum(ys), seed=38)
    check_query(knn, x, y, xs, ys, 16, start_radius=start_radius, what=f"start radius {start_radius}")
    if start_radius < 1:
        assert knn.stats()["rounds"] >= 3


@pytest.mark.parametrize("opts", [{"warp_round_max": 0}, {"warp_round_max": 0, "sparse_divisor": 4},
                                  {"warp_round_max": 0, "sparse_divisor": 4, "sparse_team": 8}, {"approx_filter": 1},
                                  {"counters": 1}], ids=["dense", "sparse", "team8", "approx", "counters"])
def test_kernel_families(knn, set_abstraction, opts):
    x, xs, y, ys = set_abstraction
    x, xs, y, ys = x[: 128 * 4096], xs[:128], y[: 128 * 1024], ys[:128]
    for name, v in opts.items():
        knn.set_option(name, v)
    check_query(knn, x, y, xs, ys, 16, start_radius=0.01, segments=range(0, 128, 4), what=str(opts))
    if "counters" in opts:
        assert knn.stats()["filter_violations"] == 0
    got = knn.radius_query(y, 0.05, batch=batch_of(ys))
    assert_lists(got, SQ.radius_lists(x, y, SQ.offsets_of(xs), SQ.offsets_of(ys), 0.05), f"radius {opts}")


def test_device_inputs_and_outputs(knn, set_abstraction):
    torch = pytest.importorskip("torch")
    x, xs, y, ys = set_abstraction
    x, xs, y, ys = x[: 64 * 4096], xs[:64], y[: 64 * 1024], ys[:64]
    sid = np.arange(len(y), dtype=np.int32) * 4  # y = x[::4]: each query names its own data point
    knn.set_option("squared_dist", 1)
    knn.build(torch.from_numpy(x).cuda(), batch=torch.from_numpy(batch_of(xs)).cuda())
    i, d = knn.query(torch.from_numpy(y).cuda(), 16, self_ids=torch.from_numpy(sid).cuda(),
                     batch=torch.from_numpy(batch_of(ys)).cuda())
    assert i.is_cuda and d.is_cuda
    want = SQ.knn(x, y, SQ.offsets_of(xs), SQ.offsets_of(ys), 16, self_ids=sid, squared=True)
    assert_rows((i, d), want, "device")
    off, idx, d2 = knn.radius_query(torch.from_numpy(y).cuda(), 0.1, self_ids=torch.from_numpy(sid).cuda(),
                                    batch=torch.from_numpy(batch_of(ys)).cuda())
    assert off.is_cuda and idx.is_cuda
    assert_lists((off, idx, d2), SQ.radius_lists(x, y, SQ.offsets_of(xs), SQ.offsets_of(ys), 0.1, self_ids=sid),
                 "device radius")
    # device queries, self ids and offsets with host outputs, straight through the C ABI
    L = _lib.load()
    qd, sd = torch.from_numpy(y).cuda(), torch.from_numpy(sid).cuda()
    od = torch.from_numpy(SQ.offsets_of(ys).astype(np.int64)).cuda()
    hi = np.empty((len(y), 16), np.int32)
    hd = np.empty((len(y), 16), np.float32)
    assert L.tknn_query_segments(knn._h, qd.data_ptr(), len(y), 3, 3, od.data_ptr(), 64, sd.data_ptr(), None, 16,
                                 ctypes.c_float(0), hi.ctypes.data, hd.ctypes.data) == _lib.OK
    assert_rows((hi, hd), want, "device inputs, host outputs")


def test_run_to_run(knn):
    xs, ys = uneven(16, 9)
    x = datasets.uniform(sum(xs), seed=39)
    y = datasets.uniform(sum(ys), seed=40)
    knn.build(x, batch=batch_of(xs))
    a = knn.query(y, 16, batch=batch_of(ys))
    b = knn.query(y, 16, batch=batch_of(ys))
    np.testing.assert_array_equal(a[0], b[0])
    np.testing.assert_array_equal(a[1].view(np.uint32), b[1].view(np.uint32))
    ra = knn.radius_query(y, 0.07, batch=batch_of(ys))
    rb = knn.radius_query(y, 0.07, batch=batch_of(ys))
    for u, v in zip(ra, rb):
        np.testing.assert_array_equal(u.view(np.uint32) if u.dtype == np.float32 else u, v.view(np.uint32) if v.dtype == np.float32 else v)


@pytest.mark.parametrize("squared", [True, False])
def test_identity_with_the_all_points_calls(knn, set_abstraction, squared):
    x, xs, _, _ = set_abstraction
    b = batch_of(xs)
    knn.set_option("squared_dist", 1 if squared else 0)
    knn.build(x, batch=b)
    sid = np.arange(len(x), dtype=np.int32)
    want = knn.search(16)
    got = knn.query(x, 16, self_ids=sid, batch=b)
    np.testing.assert_array_equal(got[0], want[0])
    np.testing.assert_array_equal(got[1].view(np.uint32), want[1].view(np.uint32))
    want = knn.radius_search(0.06)
    got = knn.radius_query(x, 0.06, self_ids=sid, batch=b)
    for g, w in zip(got, want):
        np.testing.assert_array_equal(g.view(np.uint32) if g.dtype == np.float32 else g,
                                      w.view(np.uint32) if w.dtype == np.float32 else w)


def test_identity_with_the_unsegmented_calls(knn):
    x = datasets.uniform(300_000, seed=15)
    y = datasets.uniform(100_000, seed=16)
    sid = np.random.default_rng(1).integers(-1, len(x), size=len(y)).astype(np.int32)
    one = np.zeros(len(y), np.int64)
    knn.build(x)
    for k in (8, 64):
        a = knn.query(y, k, self_ids=sid)
        b = knn.query(y, k, self_ids=sid, batch=one)
        np.testing.assert_array_equal(a[0], b[0])
        np.testing.assert_array_equal(a[1].view(np.uint32), b[1].view(np.uint32))
    a = knn.radius_query(y, 0.02, self_ids=sid)
    b = knn.radius_query(y, 0.02, self_ids=sid, batch=one)
    for u, v in zip(a, b):
        np.testing.assert_array_equal(u.view(np.uint32) if u.dtype == np.float32 else u,
                                      v.view(np.uint32) if v.dtype == np.float32 else v)


def test_errors(knn):
    L = _lib.load()
    q = datasets.uniform(30, seed=41)
    qi = np.zeros(30 * 4, np.int32)
    qd = np.zeros(30 * 4, np.float32)
    t = ctypes.c_uint64(0)
    roff = np.zeros(31, np.uint64)

    def kq(ctx, off, n_seg, k=4, r=0.0):
        p = None if off is None else np.asarray(off, np.uint64).ctypes.data
        return L.tknn_query_segments(ctx._h, q.ctypes.data, 30, 3, 3, p, n_seg, None, None, k, ctypes.c_float(r),
                                     qi.ctypes.data, qd.ctypes.data)

    def rq(ctx, off, n_seg, r=0.1, idx=None, cap=0):
        p = None if off is None else np.asarray(off, np.uint64).ctypes.data
        return L.tknn_radius_query_segments(ctx._h, q.ctypes.data, 30, 3, 3, p, n_seg, None, ctypes.c_float(r),
                                            roff.ctypes.data, None if idx is None else idx.ctypes.data, None, cap,
                                            ctypes.byref(t))

    good = [0, 10, 10, 30]
    assert kq(knn, good, 3) == _lib.ESTATE  # before a build
    assert rq(knn, good, 3) == _lib.ESTATE
    knn.build(datasets.uniform(1200, seed=42), batch=batch_of([500, 0, 700]))
    assert kq(knn, good, 3) == _lib.OK and rq(knn, good, 3) == _lib.OK
    for bad_off, n_seg in [(good, 2), ([0, 30], 1), ([1, 10, 10, 30], 3), ([0, 12, 10, 30], 3), ([0, 10, 10, 29], 3),
                           ([0, 10, 10, 31], 3), (None, 3)]:
        assert kq(knn, bad_off, n_seg) == _lib.EINVAL, bad_off
        assert rq(knn, bad_off, n_seg) == _lib.EINVAL, bad_off
    torch = pytest.importorskip("torch")
    dev_bad = torch.tensor([0, 12, 10, 30], dtype=torch.int64, device="cuda")
    assert L.tknn_query_segments(knn._h, q.ctypes.data, 30, 3, 3, dev_bad.data_ptr(), 3, None, None, 4, ctypes.c_float(0),
                                 qi.ctypes.data, qd.ctypes.data) == _lib.EINVAL
    assert rq(knn, good, 3, r=float("nan")) == _lib.EINVAL
    assert kq(knn, good, 3, r=float("nan")) == _lib.EINVAL
    assert kq(knn, good, 3, k=0) == _lib.EINVAL
    # capacity below the total: the total is reported
    assert rq(knn, good, 3, r=0.5) == _lib.OK
    total = t.value
    assert total > 1
    small = np.zeros(total - 1, np.int32)
    t.value = 0
    assert rq(knn, good, 3, r=0.5, idx=small, cap=total - 1) == _lib.EINVAL and t.value == total
    with pytest.raises(TrueKNNError):
        knn.query(q, 4)  # the unsegmented form still refuses a segmented build
    with pytest.raises(ValueError):
        knn.query(q, 4, batch=np.full(30, 3))  # cloud id >= the build's batch size
    # a plain build: one segment only
    knn.build(datasets.uniform(1200, seed=42))
    assert kq(knn, [0, 30], 1) == _lib.OK and kq(knn, good, 3) == _lib.EINVAL
    with MultiTrueKNN([0, 0], "partition") as m:
        m.build(datasets.uniform(4000, seed=4))
        assert kq(m.rank(0), [0, 30], 1) == _lib.ESTATE
        assert rq(m.rank(0), [0, 30], 1) == _lib.ESTATE


def bipartite_want(x, y, bx, by, k=None, r=None, max_nn=None):
    size = max(int(bx.max()), int(by.max())) + 1
    xo = SQ.offsets_of(np.bincount(bx, minlength=size))
    yo = SQ.offsets_of(np.bincount(by, minlength=size))
    if k is not None:
        wi, _ = SQ.knn(x, y, xo, yo, min(k, len(x)))
        kk = wi.shape[1]
        q = np.repeat(np.arange(len(y)), kk)
        keep = wi.reshape(-1) >= 0
        return np.stack([q[keep], wi.reshape(-1)[keep]]).astype(np.int64)
    wo, wi, _ = SQ.radius_lists(x, y, xo, yo, r)
    q = np.repeat(np.arange(len(y)), np.diff(wo))
    if max_nn is not None:
        keep = np.arange(len(wi)) - wo[q] < max_nn
        q, wi = q[keep], wi[keep]
    return np.stack([q, wi]).astype(np.int64)


def test_knn_and_radius_helpers():
    torch = pytest.importorskip("torch")
    rng = np.random.default_rng(12)
    bx = np.repeat(np.arange(6), [40, 0, 7, 60, 3, 25]).astype(np.int64)  # clouds 0 .. 5
    by = np.repeat(np.arange(8), [10, 4, 0, 30, 5, 0, 0, 9]).astype(np.int64)  # clouds 0 .. 7: 6 and 7 have no data
    x = rng.random((len(bx), 3), dtype=np.float32)
    y = rng.random((len(by), 3), dtype=np.float32)
    for k in (5, 1000):  # 1000: clamped to len(x)
        want = bipartite_want(x, y, bx, by, k=k)
        e = knn(x, y, k, bx, by)
        assert e.dtype == np.int64
        np.testing.assert_array_equal(e, want)
        et = knn(torch.from_numpy(x).cuda(), torch.from_numpy(y).cuda(), k, torch.from_numpy(bx).cuda(),
                 torch.from_numpy(by).cuda())
        assert et.is_cuda and et.dtype == torch.int64
        np.testing.assert_array_equal(et.cpu().numpy(), want)
    for max_nn in (None, 3):
        want = bipartite_want(x, y, bx, by, r=0.35, max_nn=max_nn)
        np.testing.assert_array_equal(radius(x, y, 0.35, bx, by, max_num_neighbors=max_nn), want)
        rt = radius(torch.from_numpy(x).cuda(), torch.from_numpy(y).cuda(), 0.35, torch.from_numpy(bx).cuda(),
                    torch.from_numpy(by).cuda(), max_num_neighbors=max_nn)
        assert rt.is_cuda
        np.testing.assert_array_equal(rt.cpu().numpy(), want)
    # no batches: one cloud, and no self exclusion (a query on a data point finds it at distance 0)
    e = knn(x, x[:5], 2)
    np.testing.assert_array_equal(e[1][::2], np.arange(5))
    # empty inputs
    assert knn(x[:0], y, 3).shape == (2, 0) and radius(x, y[:0], 0.1).shape == (2, 0)
    assert knn(torch.from_numpy(x[:0]).cuda(), torch.from_numpy(y).cuda(), 3).shape == (2, 0)
    with pytest.raises(TrueKNNError):
        knn(np.random.default_rng(1).random((5000, 3), dtype=np.float32), y, 2000)  # above TKNN_MAX_K


def test_trailing_empty_clouds_via_batch_size(knn):
    x = datasets.uniform(300, seed=43)
    knn.build(x, batch=np.zeros(300, np.int64), batch_size=3)
    assert knn.n_segments == 3
    y = datasets.uniform(9, seed=44)
    by = np.array([0, 0, 0, 1, 1, 2, 2, 2, 2])
    i, d = knn.query(y, 4, batch=by)
    want = SQ.knn(x, y, [0, 300, 300, 300], [0, 3, 5, 9], 4)
    assert_rows((i, d), want, "trailing empty clouds")
    assert (i[3:] == -1).all()
