"""k nearest neighbours in feature space on the GPU (tknn_feature_knn, TrueKNN.feature_knn, feature_knn_graph,
feature_knn): every case bit for bit against the CPU reference (tests/feature_knn_oracle.py), indices and distance bits,
in the sqrtf and the squared form; the identities with the LBVH path at f = 3 and f = 2; the split + merge path; pointer
kinds, streams and every error code."""
import ctypes as C

import numpy as np
import pytest

import feature_knn_oracle as FK
from owlraytracing_b200 import TrueKNN, _lib, feature_knn, feature_knn_graph
from owlraytracing_b200.trueknn import TrueKNNError

pytestmark = pytest.mark.gpu


def _np(a):
    return a.cpu().numpy() if hasattr(a, "cpu") else np.asarray(a)


def assert_same(got, want, what, rows=None):
    gi, gd = _np(got[0]), got[1]
    wi, wd = want
    if rows is not None:
        gi, wi = gi[rows], wi[rows]
    bad = np.argwhere(gi != wi)
    assert bad.size == 0, f"{what}: {len(bad)} indices differ, first at {tuple(bad[0])}: {gi[tuple(bad[0])]} vs {wi[tuple(bad[0])]}"
    if gd is None:
        return
    gd = _np(gd)
    if rows is not None:
        gd, wd = gd[rows], wd[rows]
    bad = np.argwhere(gd.view(np.uint32) != wd.view(np.uint32))
    assert bad.size == 0, f"{what}: {len(bad)} distances differ, first at {tuple(bad[0])}: {gd[tuple(bad[0])]} vs {wd[tuple(bad[0])]}"


def batch_of(sizes):
    return np.repeat(np.arange(len(sizes)), sizes).astype(np.int64)


def call(t, x, y, k, xo=None, yo=None, sid=None, f=None, out_idx=None, out_dist=None):
    """tknn_feature_knn straight through ctypes (host or device arrays, strides from the arrays)."""
    L = _lib.load()
    f = int(x.shape[1]) if f is None else f
    nq = int(y.shape[0])
    idx = np.empty((nq, k), np.int32) if out_idx is None else out_idx
    dist = np.empty((nq, k), np.float32) if out_dist is None and out_idx is None else out_dist

    def p(a):
        if a is None:
            return None
        return C.c_void_p(a.data_ptr()) if hasattr(a, "data_ptr") else C.c_void_p(a.ctypes.data)

    n_seg = 1 if xo is None else int(xo.shape[0]) - 1
    rc = L.tknn_feature_knn(t._h, p(x), int(x.shape[0]), f, int(x.shape[1]), p(xo), p(y), nq, int(y.shape[1]), p(yo),
                            n_seg, p(sid), int(k), p(idx), p(dist))
    return rc, idx, dist


def run(t, x, y, k, xo=None, yo=None, sid=None, f=None, squared=True):
    t.set_option("squared_dist", 1 if squared else 0)
    rc, idx, dist = call(t, x, y, k, xo, yo, sid, f)
    assert rc == 0, t._L.tknn_last_error(t._h).decode()
    return idx, dist


def check(t, x, y, k, xo=None, yo=None, sid=None, f=None, what="", both=True, rows=None):
    for squared in ((True, False) if both else (True,)):
        got = run(t, x, y, k, xo, yo, sid, f, squared)
        want = FK.knn(x, y, k, xo, yo, sid, f, squared, rows=rows)
        assert_same(got, want, f"{what} squared={squared}", rows)
    return t.stats()


X_SIZES = [300, 0, 1, 20, 700, 129, 64]
Y_SIZES = [100, 4, 3, 0, 256, 65, 1]


@pytest.mark.parametrize("f", [1, 2, 3, 4, 5, 31, 32, 33, 64, 100, 128, 1024])
def test_columns(knn, f):
    rng = np.random.default_rng(f)
    x = rng.standard_normal((sum(X_SIZES), f)).astype(np.float32)
    y = rng.standard_normal((sum(Y_SIZES), f)).astype(np.float32)
    xo, yo = FK.offsets_of(X_SIZES), FK.offsets_of(Y_SIZES)
    st = check(knn, x, y, 20, xo, yo, what=f"f={f}")
    assert st["rounds"] in (1, 2) and st["n_queries"] == len(y) and st["k"] == 20
    assert st["points_tested"] == sum(a * b for a, b in zip(X_SIZES, Y_SIZES))


@pytest.mark.parametrize("k", [1, 16, 20, 32, 33, 64, 512])
def test_k(knn, k):
    rng = np.random.default_rng(100 + k)
    xs, ys = [1500, 600, 10, 0], [130, 70, 5, 9]
    x = rng.standard_normal((sum(xs), 40)).astype(np.float32)
    y = rng.standard_normal((sum(ys), 40)).astype(np.float32)
    check(knn, x, y, k, FK.offsets_of(xs), FK.offsets_of(ys), what=f"k={k}")


def test_stride_padding_is_ignored(knn):
    rng = np.random.default_rng(5)
    f, pitch = 37, 45
    x = rng.standard_normal((900, pitch)).astype(np.float32)
    y = rng.standard_normal((200, pitch)).astype(np.float32)
    x[:, f:] = np.nan
    y[:, f:] = np.inf
    x[::3, f + 1] = 3e38
    check(knn, x, y, 24, f=f, what="pitch 45, f 37")
    # the same rows without padding give the same answer
    want = run(knn, np.ascontiguousarray(x[:, :f]), np.ascontiguousarray(y[:, :f]), 24)
    assert_same(run(knn, x, y, 24, f=f), want, "pitch vs packed")


def test_small_and_empty_segments(knn):
    rng = np.random.default_rng(6)
    xs = [0, 5, 1, 40, 0, 33, 2, 100]
    ys = [7, 0, 3, 40, 0, 33, 2, 0]
    x = rng.integers(-3, 4, (sum(xs), 12)).astype(np.float32)  # many exact ties
    sid = np.full(sum(ys), -1, np.int32)
    sid[:sum(ys) // 2] = rng.integers(0, sum(xs), sum(ys) // 2)
    y = rng.integers(-3, 4, (sum(ys), 12)).astype(np.float32)
    check(knn, x, y, 33, FK.offsets_of(xs), FK.offsets_of(ys), sid, what="small segments")


def test_many_tiny_clouds(knn):
    rng = np.random.default_rng(7)
    sizes = [16] * 65536
    x = rng.random((16 * 65536, 8), dtype=np.float32)
    off = FK.offsets_of(sizes)
    sid = np.arange(len(x), dtype=np.int32)
    st = check(knn, x, x, 20, off, off, sid, what="65536 x 16", both=False)
    assert st["rounds"] == 1
    idx = run(knn, x, x, 20, off, off, sid)[0]
    assert (idx[:, 15:] == -1).all() and (idx[:, :15] >= 0).all()


@pytest.mark.parametrize("k", [20, 512])
def test_split_and_merge(knn, k):
    rng = np.random.default_rng(8)
    x = rng.standard_normal((131072, 16)).astype(np.float32)
    y = rng.standard_normal((512, 16)).astype(np.float32)
    st = check(knn, x, y, k, what=f"131072 x 512 k={k}")
    assert st["rounds"] == 2 and st["round_queries"][:2] == [512, 512]
    # indices only: the merge writes its distances to scratch
    knn.set_option("squared_dist", 1)
    rc, idx, _ = call(knn, x, y, k, out_idx=np.empty((512, k), np.int32))
    assert rc == 0
    assert (idx == FK.knn(x, y, k)[0]).all()


def test_many_clouds_one_round(knn):
    rng = np.random.default_rng(9)
    x = rng.standard_normal((1024 * 1024, 8)).astype(np.float32)
    off = FK.offsets_of([1024] * 1024)
    sid = np.arange(len(x), dtype=np.int32)
    st = check(knn, x, x, 20, off, off, sid, what="1024 x 1024", both=False)
    assert st["rounds"] == 1 and st["points_tested"] == 1024 ** 3


def test_self_ids(knn):
    rng = np.random.default_rng(10)
    xs, ys = [200, 150], [60, 40]
    x = rng.standard_normal((350, 20)).astype(np.float32)
    y = rng.standard_normal((100, 20)).astype(np.float32)
    y[:10] = x[:10]           # queries on data rows
    x[10:13] = x[0]           # duplicates of query 0's row: only the named one is excluded
    sid = np.full(100, -1, np.int32)
    sid[:10] = np.arange(10)  # self inside the segment
    sid[10:20] = 250          # outside segment 0: excludes nothing
    sid[60:70] = 5            # outside segment 1
    sid[70:80] = np.arange(200, 210)
    check(knn, x, y, 8, FK.offsets_of(xs), FK.offsets_of(ys), sid, what="self ids")
    idx = run(knn, x, y, 8, FK.offsets_of(xs), FK.offsets_of(ys), sid)[0]
    assert list(idx[0, :3]) == [10, 11, 12]


def test_device_pointers_streams_and_indices_only():
    import torch

    rng = np.random.default_rng(11)
    sizes = [700, 300, 0, 24]
    x = rng.standard_normal((sum(sizes), 64)).astype(np.float32)
    b = batch_of(sizes)
    want = FK.knn(x, x, 20, FK.offsets_of(sizes), FK.offsets_of(sizes), squared=False)
    xt, bt = torch.from_numpy(x).cuda(), torch.from_numpy(b).cuda()
    with TrueKNN(0) as t:
        idx, dist = t.feature_knn(xt, xt, 20, batch_x=bt, batch_y=bt)
        assert idx.is_cuda and dist.is_cuda
        assert_same((idx, dist), want, "device")
        s = torch.cuda.Stream()
        t.set_stream(s.cuda_stream)
        with torch.cuda.stream(s):
            idx, dist = t.feature_knn(xt, xt, 20, batch_x=bt, batch_y=bt)
        s.synchronize()
        assert_same((idx, dist), want, "torch stream")
        t.set_stream(None)
        idx, dist = t.feature_knn(x, x, 20, batch_x=b, batch_y=b, indices_only=True)
        assert dist is None and isinstance(idx, np.ndarray)
        assert (idx == want[0]).all()
        # device offsets and self ids through the C call
        sid = torch.arange(len(x), dtype=torch.int32, device="cuda")
        off = torch.from_numpy(FK.offsets_of(sizes).astype(np.int64)).cuda()
        t.set_option("squared_dist", 1)
        out_i = torch.empty((len(x), 20), dtype=torch.int32, device="cuda")
        out_d = torch.empty((len(x), 20), dtype=torch.float32, device="cuda")
        rc, _, _ = call(t, xt, xt, 20, off, off, sid, out_idx=out_i, out_dist=out_d)
        torch.cuda.synchronize()
        assert rc == 0
        assert_same((out_i, out_d), FK.knn(x, x, 20, FK.offsets_of(sizes), FK.offsets_of(sizes), np.arange(len(x))),
                    "device offsets")


@pytest.mark.parametrize("f", [2, 3])
def test_low_dims_equal_lbvh_queries(knn, f):
    rng = np.random.default_rng(12 + f)
    xs, ys = [4000, 0, 3, 2500], [500, 7, 2, 300]
    x = rng.random((sum(xs), f), dtype=np.float32)
    y = rng.random((sum(ys), f), dtype=np.float32)
    sid = rng.integers(-1, sum(xs), sum(ys)).astype(np.int32)
    k = 12
    knn.set_option("squared_dist", 1)
    knn.build(x, batch=batch_of(xs), batch_size=len(xs))
    lbvh = knn.query(y, k, self_ids=sid, batch=batch_of(ys))
    got = run(knn, x, y, k, FK.offsets_of(xs), FK.offsets_of(ys), sid)
    assert_same(got, (lbvh[0], lbvh[1]), f"f={f} vs tknn_query_segments")
    # all points, self excluded: tknn_search on a plain build
    knn.set_option("squared_dist", 0)
    knn.build(x)
    s_idx, s_dist = knn.search(k)
    got = run(knn, x, x, k, sid=np.arange(len(x), dtype=np.int32), squared=False)
    assert_same(got, (s_idx, s_dist), f"f={f} vs tknn_search")


def test_build_untouched(knn):
    rng = np.random.default_rng(13)
    pts = rng.random((50_000, 3), dtype=np.float32)
    f = rng.standard_normal((3000, 64)).astype(np.float32)
    x0 = run(knn, f, f, 20)  # before any build
    assert_same(x0, FK.knn(f, f, 20), "before a build")
    knn.build(pts)
    a = knn.search(10)
    run(knn, f, f, 20)
    b = knn.search(10)
    assert_same(b, (a[0], a[1]), "search after feature_knn")


def test_errors(knn):
    L = _lib.load()
    x = np.zeros((10, 8), np.float32)
    idx = np.empty((10, 4), np.int32)
    dist = np.empty((10, 4), np.float32)
    off = np.array([0, 5, 10], np.uint64)

    def rc(x=x, n=10, f=8, xs=8, xo=None, y=x, nq=10, ys=8, yo=None, S=1, k=4, idx=idx):
        p = (lambda a: None if a is None else C.c_void_p(a.ctypes.data))
        return L.tknn_feature_knn(knn._h, p(x), n, f, xs, p(xo), p(y), nq, ys, p(yo), S, None, k, p(idx), p(dist))

    E = _lib.EINVAL
    assert rc() == 0
    assert rc(f=0) == E and rc(f=1025) == E
    assert rc(xs=7) == E and rc(ys=7) == E
    assert rc(k=0) == E and rc(k=11) == E and rc(k=513) == E
    assert rc(n=1 << 31) == E and rc(nq=1 << 31) == E
    assert rc(x=None) == E and rc(y=None) == E and rc(idx=None) == E
    assert rc(xo=off, S=2) == E and rc(yo=off, S=2) == E  # one offset array only
    assert rc(S=2) == E                                   # no offsets, n_segments != 1
    assert rc(xo=off, yo=off, S=2) == 0
    for bad in (np.array([1, 5, 10], np.uint64), np.array([0, 6, 5], np.uint64), np.array([0, 5, 9], np.uint64)):
        assert rc(xo=bad, yo=off, S=2) == E and rc(xo=off, yo=bad, S=2) == E
    assert rc(nq=0) == 0
    for v in (np.nan, np.inf, -np.inf):
        bad = x.copy()
        bad[3, 7] = v
        assert rc(x=bad) == E and rc(y=bad) == E
    big = np.zeros((10, 1030), np.float32)
    assert rc(x=big, y=big, f=1025, xs=1030, ys=1030) == E
    with pytest.raises(TrueKNNError):
        knn.feature_knn(x, x, 11)


def test_module_functions_numpy_and_cuda():
    import torch

    rng = np.random.default_rng(14)
    sizes_x, sizes_y = [500, 0, 40, 300], [60, 10, 0, 80]
    x = rng.standard_normal((sum(sizes_x), 64)).astype(np.float32)
    y = rng.standard_normal((sum(sizes_y), 64)).astype(np.float32)
    bx, by = batch_of(sizes_x), batch_of(sizes_y)
    xo, yo = FK.offsets_of(sizes_x), FK.offsets_of(sizes_y)
    k = 20
    # feature_knn_graph: neighbour / centre rows, a point is never its own neighbour
    gi, _ = FK.knn(x, x, k, xo, xo, np.arange(len(x)))
    keep = gi.reshape(-1) >= 0
    centre = np.repeat(np.arange(len(x)), k)[keep]
    want_graph = np.stack([gi.reshape(-1)[keep], centre]).astype(np.int64)
    e = feature_knn_graph(x, k, bx)
    assert e.dtype == np.int64 and (e == want_graph).all()
    et = feature_knn_graph(torch.from_numpy(x).cuda(), k, torch.from_numpy(bx).cuda())
    assert et.is_cuda and (et.cpu().numpy() == want_graph).all()
    # feature_knn: query / data rows, no self exclusion, k clamped to len(x)
    qi, _ = FK.knn(x, y, k, xo, yo)
    keep = qi.reshape(-1) >= 0
    want = np.stack([np.repeat(np.arange(len(y)), k)[keep], qi.reshape(-1)[keep]]).astype(np.int64)
    assert (feature_knn(x, y, k, bx, by) == want).all()
    et = feature_knn(torch.from_numpy(x).cuda(), torch.from_numpy(y).cuda(), k, torch.from_numpy(bx).cuda(),
                     torch.from_numpy(by).cuda())
    assert et.is_cuda and (et.cpu().numpy() == want).all()
    small = x[:5]
    assert feature_knn(small, small, 50).shape == (2, 25)
    # DynamicEdgeConv's knn(x, x, k, b, b) keeps the point itself
    e = feature_knn(x, x, k, bx, bx)
    assert (e[1].reshape(-1, k)[:, 0] == np.arange(len(x))).all()
