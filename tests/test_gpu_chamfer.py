"""Gradients of kNN distances, segment reductions and the Chamfer distance on the GPU (tknn_knn_backward,
tknn_segment_reduce, TrueKNN.knn_backward / segment_reduce, knn_points, chamfer_distance): bit for bit against the CPU
reference (tests/chamfer_oracle.py) in 2-D and 3-D up to k = 64 with -1 slots, padded pitches, host and device arrays,
torch side streams and NULL outputs; one data point referenced by 2^20 edges (the long-run chunk path); segments empty,
long and up to 1 024 columns wide; every reduction of chamfer_distance on big batches with empty clouds, LiDAR-like
clouds, lattice ties, duplicates and the extreme clouds; repeatability; a plain-torch Chamfer on the GPU; every error
code; and the independence of a built context from the calls."""
import numpy as np
import pytest

import chamfer_oracle as R
import extreme_clouds as X
from owlraytracing_b200 import TrueKNN, _lib, chamfer_distance, datasets, knn_points
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


def batched(rng, sizes, dim=3):
    return rng.random((sum(sizes), dim), dtype=np.float32)


def rows(p, q, p_sizes, q_sizes, k):
    """The reference kNN rows of q against p (squared distances), and the library's, which must be the same."""
    ridx, rd2 = R.SQ.knn(p, q, R.offsets_of(p_sizes), R.offsets_of(q_sizes), k, squared=True)
    bp = np.repeat(np.arange(len(p_sizes)), p_sizes)
    bq = np.repeat(np.arange(len(q_sizes)), q_sizes)
    d2, idx = knn_points(p, q, k, bp, bq)
    assert (idx == ridx).all()
    bits_equal(np.where(ridx >= 0, d2, 0), np.where(ridx >= 0, rd2, 0), "knn_points d2")
    return ridx, rd2


@pytest.mark.parametrize("dim", [2, 3])
@pytest.mark.parametrize("k", [1, 3, 16, 64])
def test_knn_backward(knn, dim, k):
    rng = np.random.default_rng(10 * dim + k)
    ps, qs = [3000, 0, 5, k - 1 if k > 1 else 2, 900], [8000, 40, 300, 50, 2000]  # clouds smaller than k: -1 slots
    p, q = batched(rng, ps, dim), batched(rng, qs, dim)
    idx, _ = rows(p, q, ps, qs, k)
    g = rng.normal(size=idx.shape).astype(np.float32)
    gq, gp = knn.knn_backward(q, p, idx, g)
    rq, rp = R.knn_backward(q, p, idx, g)
    bits_equal(gq, rq, f"grad_q dim {dim} k {k}")
    bits_equal(gp, rp, f"grad_p dim {dim} k {k}")
    st = knn.stats()
    assert st["rounds"] == 3 and st["round_queries"] == [len(q), len(q) * k, len(p)] and st["k"] == k


def _pitched(a, pad):
    buf = torch.full((a.shape[0], a.shape[1] + pad), float("nan"), device="cuda")
    buf[:, :a.shape[1]] = torch.from_numpy(a).cuda()
    return buf, a.shape[1] + pad


def test_pitches_null_outputs_and_streams(knn):
    rng = np.random.default_rng(1)
    p, q = rng.random((5000, 3), dtype=np.float32), rng.random((20_000, 3), dtype=np.float32)
    idx, _ = rows(p, q, [5000], [20_000], 8)
    g = rng.normal(size=idx.shape).astype(np.float32)
    rq, rp = R.knn_backward(q, p, idx, g)
    L, h = _lib.load(), knn._h
    pb, ps = _pitched(p, 5)
    qb, qs = _pitched(q, 1)
    di, dg = torch.from_numpy(idx).cuda(), torch.from_numpy(g).cuda()
    gq = torch.empty((20_000, 3), device="cuda")
    gp = torch.empty((5000, 3), device="cuda")
    torch.cuda.synchronize()
    assert L.tknn_knn_backward(h, qb.data_ptr(), 20_000, qs, pb.data_ptr(), 5000, ps, 3, di.data_ptr(), 8, dg.data_ptr(),
                               gq.data_ptr(), gp.data_ptr()) == 0
    bits_equal(gq, rq, "pitched grad_q")
    bits_equal(gp, rp, "pitched grad_p")
    # NULL outputs: each side alone, then neither (a no-op)
    hq, hp = np.full((20_000, 3), 7, np.float32), np.full((5000, 3), 7, np.float32)
    assert L.tknn_knn_backward(h, qb.data_ptr(), 20_000, qs, pb.data_ptr(), 5000, ps, 3, di.data_ptr(), 8, dg.data_ptr(),
                               hq.ctypes.data, None) == 0
    bits_equal(hq, rq, "grad_q alone, host out")
    assert knn.stats()["round_queries"] == [20_000, 0, 0]
    assert L.tknn_knn_backward(h, q.ctypes.data, 20_000, 3, p.ctypes.data, 5000, 3, 3, idx.ctypes.data, 8, g.ctypes.data,
                               None, hp.ctypes.data) == 0
    bits_equal(hp, rp, "grad_p alone, host in and out")
    assert L.tknn_knn_backward(h, None, 20_000, 3, None, 5000, 3, 3, None, 8, None, None, None) == 0
    # nq = 0: grad_p is +0
    hp.fill(7)
    assert L.tknn_knn_backward(h, None, 0, 3, p.ctypes.data, 5000, 3, 3, None, 8, None, None, hp.ctypes.data) == 0
    assert not hp.any() and not np.signbit(hp).any()
    # tensors on a torch side stream
    s = torch.cuda.Stream()
    with torch.cuda.stream(s):
        knn.set_stream(s.cuda_stream)
        tq, tp = knn.knn_backward(torch.from_numpy(q).cuda(), torch.from_numpy(p).cuda(), di, dg)
        assert tq.is_cuda and tp.is_cuda
    knn.set_stream(None)
    torch.cuda.synchronize()
    bits_equal(tq, rq, "side stream grad_q")
    bits_equal(tp, rp, "side stream grad_p")


def test_one_point_referenced_by_2pow20_edges():
    rng = np.random.default_rng(2)
    nq = 1 << 20
    x = torch.tensor([[0.5, 0.5, 0.5]], device="cuda", requires_grad=True)
    yn = rng.random((nq, 3), dtype=np.float32)
    y = torch.from_numpy(yn).cuda().requires_grad_(True)
    d2, idx = knn_points(x, y, 4)  # k clamps to 1; one data point takes the feature-space search
    assert d2.shape == (nq, 1) and (idx == 0).all()
    g = torch.from_numpy(rng.normal(size=(nq, 1)).astype(np.float32)).cuda()
    (d2 * g).sum().backward()
    ridx, rd2 = R.SQ.knn(x.detach().cpu().numpy(), yn, R.offsets_of([1]), R.offsets_of([nq]), 1, squared=True)
    bits_equal(d2, rd2, "d2")
    rq, rp = R.knn_backward(yn, x.detach().cpu().numpy(), ridx, g.cpu().numpy())
    bits_equal(y.grad, rq, "queries' grad")
    bits_equal(x.grad, rp, "grad of the one point (a run of 2^20 edges)")


@pytest.mark.parametrize("reduce", ["sum", "mean"])
def test_segment_reduce(knn, reduce):
    rng = np.random.default_rng(3)
    sizes = [0, 1, 31, 32, 33, 256, 257, 0, 5000, 100_000, 3, 0]  # empty, short and long (> 256 rows) segments
    off = R.offsets_of(sizes)
    batch = np.repeat(np.arange(len(sizes)), sizes)
    x = rng.normal(size=(sum(sizes), 6)).astype(np.float32)
    out = knn.segment_reduce(x, batch, len(sizes), reduce)
    bits_equal(out, R.segment_reduce(x, off, reduce), f"{reduce} 6 columns")
    assert not _np(out)[[0, 7, 11]].any()
    v = torch.from_numpy(x[:, 2].copy()).cuda()
    bits_equal(knn.segment_reduce(v, torch.from_numpy(batch).cuda(), len(sizes), reduce),
               R.segment_reduce(x[:, 2], off, reduce), f"{reduce} 1-D")
    bits_equal(knn.segment_reduce(x, reduce=reduce), R.segment_reduce(x, [0, len(x)], reduce), f"{reduce} one segment")
    L = _lib.load()
    code = _lib.REDUCE_SUM if reduce == "sum" else _lib.REDUCE_MEAN
    for f in (1, 3, 32, 33, 256, 1024):
        sz = [0, 700, 20, 300]
        xf = rng.normal(size=(sum(sz), f)).astype(np.float32)
        xb, xs = _pitched(xf, 3)
        o = torch.from_numpy(R.offsets_of(sz).astype(np.int64)).cuda()
        out = torch.empty((4, f), device="cuda")
        torch.cuda.synchronize()
        assert L.tknn_segment_reduce(knn._h, xb.data_ptr(), sum(sz), f, xs, o.data_ptr(), 4, code, out.data_ptr()) == 0
        bits_equal(out, R.segment_reduce(xf, R.offsets_of(sz), reduce), f"{reduce} f {f} pitched")


def _batch(sizes):
    return torch.repeat_interleave(torch.arange(len(sizes), device="cuda"), torch.tensor(sizes, device="cuda"))


def check_chamfer(xn, yn, xs, ys, what, **kw):
    """chamfer_distance on CUDA tensors: the loss, x.grad and y.grad against the reference; returns them.  The batch
    has B = the last cloud with a point + 1 clouds (PyG's batch_size), so trailing empty clouds are not counted."""
    nz = np.nonzero(np.asarray(xs) + np.asarray(ys))[0]
    xs, ys = list(xs)[:nz[-1] + 1], list(ys)[:nz[-1] + 1]
    x = torch.from_numpy(xn).cuda().requires_grad_(True)
    y = torch.from_numpy(yn).cuda().requires_grad_(True)
    loss = chamfer_distance(x, y, _batch(xs), _batch(ys), **kw)
    if kw.get("point_reduction", "mean") is None:
        a, b = loss
        rng = np.random.default_rng(len(xn))
        ga = rng.normal(size=len(xn)).astype(np.float32)
        gb = rng.normal(size=len(yn)).astype(np.float32)
        s = (a * torch.from_numpy(ga).cuda()).sum()
        if b is not None:
            s = s + (b * torch.from_numpy(gb).cuda()).sum()
        s.backward()
        (ra, rb), rgx, rgy = R.chamfer(xn, yn, xs, ys, grad=(ga, gb), **kw)
        bits_equal(a, ra, f"{what} a")
        assert (b is None) == (rb is None)
        if b is not None:
            bits_equal(b, rb, f"{what} b")
    else:
        loss.sum().backward()
        rloss, rgx, rgy = R.chamfer(xn, yn, xs, ys, **kw)
        bits_equal(loss, rloss, f"{what} loss")
    bits_equal(x.grad, rgx, f"{what} x.grad")
    bits_equal(y.grad, rgy, f"{what} y.grad")
    return loss, x.grad, y.grad


@pytest.mark.parametrize("point_reduction,batch_reduction",  # point_reduction=None needs batch_reduction=None
                         [(p, b) for p in ("mean", "sum") for b in ("mean", "sum", None)] + [(None, None)])
@pytest.mark.parametrize("single_directional", [False, True])
def test_chamfer_reductions(point_reduction, batch_reduction, single_directional):
    rng = np.random.default_rng(4)
    xs = rng.integers(1, 60, 1024)
    ys = rng.integers(1, 60, 1024)
    xs[[0, 17, 500, 1023]] = ys[[0, 17, 500, 1023]] = 0  # empty on both sides: +0
    if single_directional:
        xs[[3, 900]] = 0  # y without x is allowed one way
    check_chamfer(batched(rng, xs), batched(rng, ys), list(xs), list(ys), "1024 clouds",
                  point_reduction=point_reduction, batch_reduction=batch_reduction,
                  single_directional=single_directional)


def test_chamfer_lidar_ties_duplicates_and_self():
    rng = np.random.default_rng(5)
    fine = [datasets.lidar_like(60_000, seed=s).astype(np.float32) for s in range(2)]
    check_chamfer(np.concatenate([f[::2] for f in fine]), np.concatenate([f[1::2] for f in fine]), [30_000] * 2,
                  [30_000] * 2, "lidar")
    g = np.stack(np.meshgrid(*[np.arange(10, dtype=np.float32)] * 3, indexing="ij"), -1).reshape(-1, 3)
    xl = g * np.float32(0.5)
    yl = np.concatenate([xl + np.float32(0.25), xl[:100]])  # cell centres: 8 equidistant lattice points each
    check_chamfer(xl, yl, [len(xl)], [len(yl)], "lattice ties", point_reduction="sum")
    _, idx = knn_points(xl, yl[:1], 1)  # 8 equidistant lattice points: the lowest index is the nearest
    assert idx.tolist() == [[0]]
    dup = np.repeat(rng.random((500, 3), dtype=np.float32), 3, 0)
    _, gx, gy = check_chamfer(dup, dup[::-1].copy(), [1500], [1500], "duplicates")
    assert not _np(gx).any() and not _np(gy).any()  # every nearest point coincides: zero gradient
    xn = rng.random((4000, 3), dtype=np.float32)
    loss, gx, gy = check_chamfer(xn, xn, [4000], [4000], "self")
    assert float(loss.detach()) == 0 and not _np(gx).any() and not _np(gy).any()


@pytest.mark.parametrize("name", sorted(X.CLOUDS))
def test_chamfer_extreme_clouds(name):
    c = X.cloud(name, 3000)
    x, y = c[0::2].copy(), c[1::2].copy()
    check_chamfer(x, y, [len(x)], [len(y)], name, point_reduction="sum")


def test_one_sided_empty_raises_and_numpy_result():
    x = torch.rand((10, 3), device="cuda")
    with pytest.raises(ValueError, match="none in y"):
        chamfer_distance(x, x[:5], _batch([5, 5]), _batch([5, 0]))
    with pytest.raises(ValueError, match="none in x"):
        chamfer_distance(x[:5], x, _batch([5, 0]), _batch([5, 5]))
    rng = np.random.default_rng(6)
    xn, yn = rng.random((300, 3), dtype=np.float32), rng.random((200, 3), dtype=np.float32)
    out = chamfer_distance(xn, yn)
    assert isinstance(out, (np.ndarray, np.floating)) and np.asarray(out).dtype == np.float32
    bits_equal(np.asarray(out), R.chamfer(xn, yn, [300], [200])[0], "numpy loss")
    assert float(chamfer_distance(xn[:5], yn, np.zeros(5, np.int64), np.r_[np.zeros(100), np.ones(100)].astype(np.int64),
                                  single_directional=True, batch_reduction="sum")) >= 0


def test_repeatable_and_against_plain_torch():
    rng = np.random.default_rng(7)
    xs, ys = [20_000] * 8, [15_000] * 8
    x = torch.from_numpy(batched(rng, xs)).cuda().requires_grad_(True)
    y = torch.from_numpy(batched(rng, ys)).cuda().requires_grad_(True)
    runs = []
    for _ in range(2):
        x.grad = y.grad = None
        loss = chamfer_distance(x, y, _batch(xs), _batch(ys))
        loss.backward()
        runs.append((loss.detach().clone(), x.grad.clone(), y.grad.clone()))
    for a, b in zip(*runs):
        assert torch.equal(a.view(torch.int32), b.view(torch.int32))
    # plain torch: cdist per cloud, min, mean, autograd (its scatter of the gradients uses atomics)
    xr, yr = x.detach().clone().requires_grad_(True), y.detach().clone().requires_grad_(True)
    total = 0
    for c in range(8):
        d = torch.cdist(xr[c * 20_000:(c + 1) * 20_000], yr[c * 15_000:(c + 1) * 15_000],
                        compute_mode="donot_use_mm_for_euclid_dist") ** 2
        total = total + d.min(1).values.mean() + d.min(0).values.mean()
    (total / 8).backward()
    torch.testing.assert_close(runs[0][0], total.detach() / 8, rtol=1e-4, atol=1e-9)
    for ours, ref in ((runs[0][1], xr.grad), (runs[0][2], yr.grad)):
        # a near-tie that fp32 resolves the other way moves one point's gradient: allow a handful of such points
        off = ((ours - ref).abs() > 1e-3 * ref.abs() + 1e-9).any(1)
        assert int(off.sum()) <= 5, int(off.sum())


def test_error_codes(knn):
    L, h, E = _lib.load(), knn._h, _lib.EINVAL
    q = np.zeros((2, 3), np.float32)
    p = np.zeros((3, 3), np.float32)
    idx = np.int32([[0, 1], [2, -1]])
    g = np.ones((2, 2), np.float32)
    gq, gp = np.empty((2, 3), np.float32), np.empty((3, 3), np.float32)
    a = lambda v: None if v is None else v.ctypes.data

    def bwd(qq=q, nq=2, qs=3, pp=p, n=3, ps=3, dim=3, i=idx, k=2, gg=g, oq=gq, op=gp):
        return L.tknn_knn_backward(h, a(qq), nq, qs, a(pp), n, ps, dim, a(i), k, a(gg), a(oq), a(op))

    assert bwd() == 0 and bwd(dim=2) == 0
    assert bwd(dim=1) == E and bwd(dim=4) == E and bwd(qs=2) == E and bwd(ps=2) == E
    assert bwd(k=0) == E and bwd(k=513) == E and bwd(n=1 << 31) == E and bwd(nq=1 << 31) == E
    assert bwd(nq=(1 << 28) + 1, k=4) == E  # above the sort's 2^30 - 1 edges, checked before any access
    for kw in ({"qq": None}, {"pp": None}, {"i": None}, {"gg": None}):
        assert bwd(**kw) == E
    for bad in ([[0, 3], [2, -1]], [[0, 1], [-2, -1]]):  # outside {-1} and [0, n), found on the device
        assert bwd(i=np.int32(bad)) == E
        assert bwd(i=np.int32(bad), op=None) == E
        assert bwd(i=np.int32(bad), oq=None) == E
    assert "outside" in L.tknn_last_error(h).decode()
    assert bwd(n=0, pp=None, i=np.int32([[-1, -1], [-1, -1]])) == 0
    x = np.ones((5, 4), np.float32)
    out = np.empty((2, 4), np.float32)
    off = np.uint64([0, 2, 5])

    def red(xx=x, n=5, f=4, s=4, o=off, m=2, r=_lib.REDUCE_SUM, oo=out):
        return L.tknn_segment_reduce(h, a(xx), n, f, s, a(o), m, r, a(oo))

    assert red() == 0 and red(r=_lib.REDUCE_MEAN) == 0 and red(o=None, m=1) == 0
    assert red(f=0) == E and red(f=1025, s=1025) == E and red(s=3) == E and red(r=_lib.REDUCE_MAX) == E and red(r=7) == E
    assert red(o=None) == E and red(m=0) == E and red(xx=None) == E and red(oo=None) == E
    assert red(o=np.uint64([1, 2, 5])) == E and red(o=np.uint64([0, 3, 2])) == E and red(o=np.uint64([0, 2, 4])) == E
    with pytest.raises(TrueKNNError):
        knn.knn_backward(q, p, np.int32([[0, 9], [1, 1]]), g)


def test_build_and_search_unchanged(knn):
    rng = np.random.default_rng(8)
    pts = rng.random((30_000, 3), dtype=np.float32)
    idx0, d0 = knn.build(pts).search(8)
    q = rng.random((10_000, 3), dtype=np.float32)
    idx, _ = rows(pts, q, [30_000], [10_000], 3)
    g = rng.normal(size=idx.shape).astype(np.float32)
    gq, gp = knn.knn_backward(q, pts, idx, g)
    bits_equal(gp, R.knn_backward(q, pts, idx, g)[1], "grad_p after build")
    knn.segment_reduce(pts, reduce="mean")
    idx1, d1 = knn.search(8)
    assert (idx1 == idx0).all()
    bits_equal(d1, d0, "search dist after the calls")


def test_keep_scratch_off():
    rng = np.random.default_rng(9)
    p, q = rng.random((1000, 3), dtype=np.float32), rng.random((5000, 3), dtype=np.float32)
    idx, _ = rows(p, q, [1000], [5000], 3)
    with TrueKNN(0, keep_scratch=0) as t:
        for _ in range(2):
            g = rng.normal(size=idx.shape).astype(np.float32)
            gq, gp = t.knn_backward(q, p, idx, g)
            rq, rp = R.knn_backward(q, p, idx, g)
            bits_equal(gq, rq, "keep_scratch 0 grad_q")
            bits_equal(gp, rp, "keep_scratch 0 grad_p")
            x = rng.normal(size=(5000, 3)).astype(np.float32)
            bits_equal(t.segment_reduce(x, np.repeat(np.arange(5), 1000), reduce="mean"),
                       R.segment_reduce(x, R.offsets_of([1000] * 5), "mean"), "keep_scratch 0 mean")
