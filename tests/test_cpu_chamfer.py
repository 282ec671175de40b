"""The CPU reference of the Chamfer distance and its gradients (tests/chamfer_oracle.py) checked without a GPU: the
whole chain against an independent float64 autograd of the same loss over brute-force distances, knn_backward against
its terms restated in torch float32 (a plain slot sum for grad_q, index_add_ in edge order for grad_p), segment_reduce
against the voxel-mean reference, and the argument checks and library calls of the Python layer (through the recording
fake of test_cpu_wrapper_calls.py, no GPU)."""
import numpy as np
import pytest

import chamfer_oracle as R
import voxel_oracle as V
from owlraytracing_b200 import chamfer_distance, knn_points

torch = pytest.importorskip("torch")

from test_cpu_wrapper_calls import fake, t, trace  # noqa: E402,F401  (fixtures and the call trace)


def bits(a):
    return np.ascontiguousarray(a, np.float32).view(np.uint32)


def clouds(rng, x_sizes, y_sizes, dim=3):
    return (rng.random((sum(x_sizes), dim), dtype=np.float32), rng.random((sum(y_sizes), dim), dtype=np.float32))


def chamfer64(x, y, xs, ys, point_reduction, batch_reduction, single_directional):
    """The loss in float64 torch over brute-force distances, and its gradients by autograd."""
    xt = torch.from_numpy(x).double().requires_grad_(True)
    yt = torch.from_numpy(y).double().requires_grad_(True)
    bx = torch.repeat_interleave(torch.arange(len(xs)), torch.tensor(xs))
    by = torch.repeat_interleave(torch.arange(len(ys)), torch.tensor(ys))
    d = ((xt[:, None, :] - yt[None, :, :]) ** 2).sum(-1)
    d = torch.where(bx[:, None] == by[None, :], d, torch.full_like(d, float("inf")))
    parts = [(d.min(1).values, bx, xs)] + ([] if single_directional else [(d.min(0).values, by, ys)])
    loss = 0
    for v, b, sizes in parts:
        per = torch.zeros(len(sizes), dtype=torch.float64).index_add(0, b, v)
        if point_reduction == "mean":
            per = per / torch.tensor(sizes, dtype=torch.float64).clamp(min=1)
        if batch_reduction == "sum":
            per = per.sum()
        elif batch_reduction == "mean":
            per = per.mean()
        loss = loss + per
    loss.sum().backward()
    return loss.detach().numpy(), xt.grad.numpy(), yt.grad.numpy()


@pytest.mark.parametrize("point_reduction", ["mean", "sum"])
@pytest.mark.parametrize("batch_reduction", ["mean", "sum", None])
@pytest.mark.parametrize("single_directional", [False, True])
def test_reference_against_float64_autograd(oracle, point_reduction, batch_reduction, single_directional):
    rng = np.random.default_rng(len(str(point_reduction)) + 3 * len(str(batch_reduction)) + single_directional)
    xs, ys = [300, 0, 40, 1, 120], [200, 0, 60, 3, 500]
    x, y = clouds(rng, xs, ys)
    loss, gx, gy = R.chamfer(x, y, xs, ys, point_reduction, batch_reduction, single_directional)
    l64, gx64, gy64 = chamfer64(x, y, xs, ys, point_reduction, batch_reduction, single_directional)
    np.testing.assert_allclose(loss, l64, rtol=2e-5, atol=1e-9)
    for g, g64 in ((gx, gx64), (gy, gy64)):
        np.testing.assert_allclose(g, g64, rtol=1e-4, atol=1e-6 * np.abs(g64).max())
    assert gx.dtype == np.float32 and gy.dtype == np.float32


def test_reference_per_point_and_2d(oracle):
    rng = np.random.default_rng(2)
    xs, ys = [100, 7], [50, 90]
    x, y = clouds(rng, xs, ys, dim=2)
    ga, gb = rng.normal(size=sum(xs)).astype(np.float32), rng.normal(size=sum(ys)).astype(np.float32)
    (a, b), gx, gy = R.chamfer(x, y, xs, ys, None, None, grad=(ga, gb))
    xt, yt = torch.from_numpy(x).double().requires_grad_(True), torch.from_numpy(y).double().requires_grad_(True)
    bx = torch.repeat_interleave(torch.arange(2), torch.tensor(xs))
    by = torch.repeat_interleave(torch.arange(2), torch.tensor(ys))
    d = ((xt[:, None] - yt[None]) ** 2).sum(-1)
    d = torch.where(bx[:, None] == by[None, :], d, torch.full_like(d, float("inf")))
    a64, b64 = d.min(1).values, d.min(0).values
    ((a64 * torch.from_numpy(ga).double()).sum() + (b64 * torch.from_numpy(gb).double()).sum()).backward()
    np.testing.assert_allclose(a, a64.detach().numpy(), rtol=1e-5, atol=1e-12)
    np.testing.assert_allclose(b, b64.detach().numpy(), rtol=1e-5, atol=1e-12)
    np.testing.assert_allclose(gx, xt.grad.numpy(), rtol=1e-4, atol=1e-6)
    np.testing.assert_allclose(gy, yt.grad.numpy(), rtol=1e-4, atol=1e-6)


def torch_knn_backward(q, p, idx, g):
    """grad_q as a plain sum over the slots in slot order, grad_p as index_add_ of term_p in edge order, torch float32."""
    qt, pt, gt = torch.from_numpy(q), torch.from_numpy(p), torch.from_numpy(g)
    it = torch.from_numpy(idx).long()
    nq, k = idx.shape
    gq = torch.zeros((nq, q.shape[1]))
    terms_p, js = [], []
    for s in range(k):
        ok = it[:, s] >= 0
        j = it[:, s].clamp(min=0)
        t = 2 * gt[:, s:s + 1]
        gq = torch.where(ok[:, None], gq + t * (qt - pt[j]), gq)
    flat = it.reshape(-1)
    e = torch.nonzero(flat >= 0)[:, 0]
    i, j = e // k, flat[e]
    term_p = (2 * gt.reshape(-1)[e])[:, None] * (pt[j] - qt[i])
    gp = torch.zeros((len(p), q.shape[1])).index_add_(0, j, term_p)
    return gq.numpy(), gp.numpy()


@pytest.mark.parametrize("dim", [2, 3])
@pytest.mark.parametrize("k", [1, 3, 16])
def test_knn_backward_reference_against_torch(oracle, dim, k):
    rng = np.random.default_rng(40 + 10 * dim + k)
    xs, ys = [2000, 5, 0, 700], [1500, 300, 20, 900]
    p, q = clouds(rng, xs, ys, dim)
    idx, _ = R.SQ.knn(p, q, R.offsets_of(xs), R.offsets_of(ys), k, squared=True)
    g = rng.normal(size=idx.shape).astype(np.float32)
    gq, gp = R.knn_backward(q, p, idx, g)
    tq, tp = torch_knn_backward(q, p, idx, g)
    assert (bits(gq) == bits(tq)).all()  # k <= 32 slots: the chunked sum is the plain one
    runs = np.bincount(idx[idx >= 0], minlength=len(p))
    short = runs <= 32
    assert short.sum() > 0.9 * len(p)
    assert (bits(gp[short]) == bits(tp[short])).all()
    np.testing.assert_allclose(gp, tp, rtol=1e-5, atol=1e-5 * np.abs(tp).max())
    assert not gp[runs == 0].any() and not np.signbit(gp[runs == 0]).any()  # unreferenced rows: +0
    assert np.isnan(np.where(idx < 0, np.nan, 0)).any()  # the 20 queries of the empty data cloud end in -1


def test_knn_backward_reference_long_runs_and_rows(oracle):
    rng = np.random.default_rng(50)
    p = rng.random((3, 3), dtype=np.float32)
    q = rng.random((5000, 3), dtype=np.float32)
    idx, _ = R.SQ.knn(p, q, R.offsets_of([3]), R.offsets_of([5000]), 3, squared=True)
    g = rng.normal(size=idx.shape).astype(np.float32)
    gq, gp = R.knn_backward(q, p, idx, g)
    tq, tp = torch_knn_backward(q, p, idx, g)
    assert (bits(gq) == bits(tq)).all()
    np.testing.assert_allclose(gp, tp, rtol=1e-4, atol=1e-6 * np.abs(tp).max())  # 5 000 edges per run: chunked
    # a row of 64 slots: two chunks
    idx = rng.integers(0, 3, (7, 64)).astype(np.int32)
    idx[2, 10] = idx[5, 40:] = -1
    g = rng.normal(size=idx.shape).astype(np.float32)
    gq, _ = R.knn_backward(q[:7], p, idx, g)
    tq, _ = torch_knn_backward(q[:7], p, idx, g)
    np.testing.assert_allclose(gq, tq, rtol=1e-5, atol=1e-6 * np.abs(tq).max())
    terms = [2 * g[0, s] * (q[0] - p[idx[0, s]]) for s in range(64)]
    c0 = np.float32(0)
    for v in terms[:32]:
        c0 = np.float32(c0 + v[0])
    c1 = np.float32(0)
    for v in terms[32:]:
        c1 = np.float32(c1 + v[0])
    assert bits(gq[0, 0]) == bits(np.float32(np.float32(0 + c0) + c1))


def test_segment_reduce_reference(oracle):
    rng = np.random.default_rng(60)
    sizes = [1, 31, 32, 33, 300, 2, 1000]
    x = rng.normal(size=(sum(sizes), 5)).astype(np.float32)
    off = R.offsets_of(sizes)
    g = dict(offsets=off, members=np.arange(sum(sizes), dtype=np.int32), n_voxels=len(sizes))
    mean = R.segment_reduce(x, off, "mean")
    assert (bits(mean) == bits(V.pool(x, g, "mean"))).all()
    total = R.segment_reduce(x, off, "sum")
    assert (bits(mean) == bits(total / np.float32(1) / np.asarray(sizes, np.float32)[:, None])).all()
    empty = R.segment_reduce(x, R.offsets_of([0, 5, 0]), "mean")
    assert not empty[[0, 2]].any() and not np.signbit(empty[[0, 2]]).any()


def test_argument_checks_need_no_device():
    x = np.zeros((4, 3), np.float32)
    with pytest.raises(ValueError, match="point_reduction"):
        chamfer_distance(x, x, point_reduction="max")
    with pytest.raises(ValueError, match="batch_reduction"):
        chamfer_distance(x, x, batch_reduction="min")
    with pytest.raises(ValueError, match="needs batch_reduction=None"):
        chamfer_distance(x, x, point_reduction=None)
    with pytest.raises(ValueError, match="columns"):
        chamfer_distance(x, x[:, :2])
    with pytest.raises(ValueError, match="x must be"):
        chamfer_distance(np.zeros((4, 4), np.float32), x)
    with pytest.raises(ValueError, match="none in y"):
        chamfer_distance(x, x, np.array([0, 0, 1, 1]), np.array([0, 0, 0, 0]))
    with pytest.raises(ValueError, match="none in x"):
        chamfer_distance(x, x, np.array([0, 0, 0, 0]), np.array([0, 0, 1, 1]))
    with pytest.raises(ValueError, match="none in y"):
        chamfer_distance(x, x[:0])
    with pytest.raises(ValueError, match="k = 0"):
        knn_points(x, x, 0)
    with pytest.raises(ValueError, match="columns"):
        knn_points(x, x[:, :2], 1)


def test_knn_backward_calls(t, fake):
    q = np.zeros((5, 3), np.float32)
    p = np.zeros((7, 3), np.float32)
    idx = np.zeros((5, 2), np.int32)
    g = np.ones((5, 2), np.float32)
    gq, gp = t.knn_backward(q, p, idx, g)
    assert trace(fake, q=q, p=p, idx=idx, g=g, gq=gq, gp=gp) == [
        ("tknn_knn_backward", ("ctx", "q", 5, 3, "p", 7, 3, 3, "idx", 2, "g", "gq", "gp"))]
    assert gq.shape == (5, 3) and gp.shape == (7, 3) and gq.dtype == np.float32
    gq, gp = t.knn_backward(q, p, idx, g, need_points=False)
    assert trace(fake, q=q, p=p, idx=idx, g=g, gq=gq) == [
        ("tknn_knn_backward", ("ctx", "q", 5, 3, "p", 7, 3, 3, "idx", 2, "g", "gq", None))] and gp is None
    qt, pt, it, gt = (torch.from_numpy(a) for a in (q[:, :2], p[:, :2], idx, g))
    gq, gp = t.knn_backward(qt.contiguous(), pt.contiguous(), it, gt, need_queries=False)
    assert trace(fake, it=it, gt=gt, gp=gp)[0][1][3:] == (2, "ptr", 7, 2, 2, "it", 2, "gt", None, "gp")
    assert gq is None and isinstance(gp, torch.Tensor) and gp.shape == (7, 2)
    gq, gp = t.knn_backward(q[:0], p, idx[:0], g[:0])  # no edge: no call, grad_p is +0
    assert trace(fake) == [] and gq.shape == (0, 3) and not gp.any()
    with pytest.raises(ValueError, match="shapes"):
        t.knn_backward(q, p, idx, g[:, :1])
    with pytest.raises(ValueError, match="columns"):
        t.knn_backward(q, p[:, :2], idx, g)
    with pytest.raises(TypeError, match="grad_d2"):
        t.knn_backward(q, p, idx, g.astype(np.float64))


def test_segment_reduce_calls(t, fake):
    x = np.zeros((10, 4), np.float32)
    out = t.segment_reduce(x, batch=np.array([0] * 6 + [2] * 4), reduce="mean")
    assert trace(fake, x=x, out=out) == [("tknn_segment_reduce", ("ctx", "x", 10, 4, 4, "ptr", 3, 0, "out"))]
    assert out.shape == (3, 4)
    v = torch.zeros(10)
    out = t.segment_reduce(v)
    assert trace(fake, v=v, out=out) == [("tknn_segment_reduce", ("ctx", "v", 10, 1, 1, None, 1, 2, "out"))]
    assert isinstance(out, torch.Tensor) and out.shape == (1,)
    with pytest.raises(ValueError, match="reduce"):
        t.segment_reduce(x, reduce="max")
    with pytest.raises(ValueError, match="batch_size"):
        t.segment_reduce(x, batch_size=3)
    with pytest.raises(TypeError, match="x"):
        t.segment_reduce(x.astype(np.float64))
    assert trace(fake) == []
