"""k-NN interpolation on the GPU (tknn_interpolate / tknn_interpolate_backward, TrueKNN.interpolate /
interpolate_backward, knn_interpolate): out, weight, den and grad_x bit for bit against the CPU reference
(tests/interpolate_oracle.py) on single clouds in 2-D and 3-D up to k = 64, big batches with empty and small clouds,
queries on data points and lattice ties, f from 1 to 1 500 with padded pitches, a point that 2^20 queries reference,
host and device arrays and torch side streams; repeatability; autograd through knn_interpolate; PyG's body in torch on
the GPU; every error code; and the independence of a built context from the calls."""
import ctypes as C

import numpy as np
import pytest

import interpolate_oracle as I
from owlraytracing_b200 import TrueKNN, _lib, knn_interpolate
from owlraytracing_b200.trueknn import TrueKNNError

pytestmark = pytest.mark.gpu


def _np(a):
    return a.cpu().numpy() if hasattr(a, "cpu") else np.asarray(a)


def bits_equal(a, b, what):
    a, b = _np(a), np.asarray(b)
    assert a.shape == b.shape, f"{what}: shape {a.shape} vs {b.shape}"
    if a.dtype == np.float32:  # every NaN is one value: its sign and payload are not part of the contract
        a = np.where(np.isnan(a), np.float32(np.nan), a).view(np.uint32)
        b = np.where(np.isnan(b), np.float32(np.nan), b).view(np.uint32)
    bad = np.argwhere(a != b)
    assert bad.size == 0, f"{what}: {len(bad)} entries differ, first at {tuple(bad[0])}: {a[tuple(bad[0])]} vs {b[tuple(bad[0])]}"


def check(t, idx, d2, x, rng=None, what=""):
    """interpolate + interpolate_backward on t against the reference; returns (out, weight, den, grad_x)."""
    out, w, den = t.interpolate(idx, d2, x)
    r_out, r_w, r_den = I.forward(_np(idx), _np(d2), _np(x))
    bits_equal(w, r_w, f"weight {what}")
    bits_equal(den, r_den, f"den {what}")
    bits_equal(out, r_out, f"out {what}")
    rng = rng or np.random.default_rng(0)
    g = rng.normal(size=r_out.shape).astype(np.float32)
    if hasattr(x, "cuda"):
        import torch

        g = torch.from_numpy(g).to(x.device)
    gx = t.interpolate_backward(idx, w, den, g, int(x.shape[0]))
    bits_equal(gx, I.backward(_np(idx), r_w, r_den, _np(g), int(x.shape[0])), f"grad_x {what}")
    return out, w, den, gx


def query_rows(pos_x, pos_y, k, x_sizes=None, y_sizes=None):
    """The library's kNN rows with squared distances, checked against the reference's."""
    batch = (lambda s: np.repeat(np.arange(len(s)), s)) if x_sizes is not None else (lambda s: None)
    with TrueKNN(0, squared_dist=1) as t:
        t.build(pos_x, batch=batch(x_sizes), batch_size=None if x_sizes is None else len(x_sizes))
        idx, d2 = t.query(pos_y, k, batch=batch(y_sizes))
    r_idx, r_d2 = I.knn_rows(pos_x, pos_y, k, x_sizes, y_sizes)
    bits_equal(idx, r_idx, "kNN idx")
    bits_equal(np.where(r_idx >= 0, _np(d2), 0), np.where(r_idx >= 0, r_d2, 0), "kNN d2")
    return idx, d2


@pytest.mark.parametrize("dim", [2, 3])
@pytest.mark.parametrize("k", [1, 3, 16, 64])
def test_single_cloud(knn, dim, k):
    rng = np.random.default_rng(10 * dim + k)
    pos_x = rng.random((4000, dim), dtype=np.float32)
    pos_y = rng.random((16_000, dim), dtype=np.float32)
    x = rng.normal(size=(4000, 24)).astype(np.float32)
    idx, d2 = query_rows(pos_x, pos_y, k)
    check(knn, idx, d2, x, rng, f"dim {dim} k {k}")
    bits_equal(knn_interpolate(x, pos_x, pos_y, k=k), I.forward(idx, d2, x)[0], "knn_interpolate")


@pytest.mark.parametrize("k", [3, 16])
def test_batches_with_empty_and_small_clouds(knn, k):
    rng = np.random.default_rng(100 + k)
    xs = rng.integers(0, 40, 1024)
    ys = rng.integers(0, 160, 1024)
    xs[[0, 5, 77, 1023]] = 0  # empty data clouds: NaN rows
    ys[[1, 6, 500]] = 0       # empty query clouds
    xs[[2, 3, 4]] = [1, 2, k - 1]  # data clouds smaller than k
    pos_x = rng.random((int(xs.sum()), 3), dtype=np.float32)
    pos_y = rng.random((int(ys.sum()), 3), dtype=np.float32)
    x = rng.normal(size=(len(pos_x), 7)).astype(np.float32)
    idx, d2 = query_rows(pos_x, pos_y, k, xs, ys)
    out, _, _, _ = check(knn, idx, d2, x, rng, "batch")
    yo = np.concatenate([[0], np.cumsum(ys)])
    for c in (0, 5, 77, 1023):
        assert np.isnan(out[yo[c]:yo[c + 1]]).all()
    bx, by = np.repeat(np.arange(1024), xs), np.repeat(np.arange(1024), ys)
    bits_equal(knn_interpolate(x, pos_x, pos_y, bx, by, k=k), I.forward(idx, d2, x)[0], "knn_interpolate batch")


def test_queries_on_data_points_and_lattice_ties(knn):
    rng = np.random.default_rng(7)
    g = np.stack(np.meshgrid(*[np.arange(12, dtype=np.float32)] * 3, indexing="ij"), -1).reshape(-1, 3)
    pos_x = g * np.float32(0.25)
    pos_y = np.concatenate([pos_x[::3], pos_x[::5] + np.float32(0.125), pos_x[:50]])  # on points, on cell centres
    x = rng.normal(size=(len(pos_x), 5)).astype(np.float32)
    for k in (1, 6, 27):
        idx, d2 = query_rows(pos_x, pos_y, k)
        assert (_np(d2)[: len(pos_x[::3]), 0] == 0).all()  # d2 = 0: the clamped weight 1e16
        _, w, _, _ = check(knn, idx, d2, x, rng, f"lattice k {k}")
        assert (_np(w)[: len(pos_x[::3]), 0] == np.float32(1e16)).all()


def _pitched(torch, a, pad):
    """a [rows, f] on the device inside rows of f + pad floats; returns (storage, row pitch)."""
    rows, f = a.shape
    buf = torch.full((rows, f + pad), float("nan"), device="cuda")
    buf[:, :f] = torch.from_numpy(a).cuda()
    return buf, f + pad


@pytest.mark.parametrize("f", [1, 3, 31, 32, 33, 256, 1024, 1500])
def test_widths_and_padded_pitches(knn, f):
    torch = pytest.importorskip("torch")
    rng = np.random.default_rng(f)
    nx, ny, k = 3000, 6000 if f <= 256 else 1500, 4
    pos_x = rng.random((nx, 3), dtype=np.float32)
    pos_y = rng.random((ny, 3), dtype=np.float32)
    idx, d2 = query_rows(pos_x, pos_y, k)
    x = rng.normal(size=(nx, f)).astype(np.float32)
    g = rng.normal(size=(ny, f)).astype(np.float32)
    check(knn, idx, d2, x, rng, f"f {f}")  # dense rows through the Python layer
    L, h = _lib.load(), knn._h
    xb, xs = _pitched(torch, x, 5)
    gb, gs = _pitched(torch, g, 3)
    di, dd = torch.from_numpy(idx).cuda(), torch.from_numpy(d2).cuda()
    out = torch.empty((ny, f), device="cuda")
    w = torch.empty((ny, k), device="cuda")
    den = torch.empty((ny,), device="cuda")
    torch.cuda.synchronize()
    assert L.tknn_interpolate(h, di.data_ptr(), dd.data_ptr(), ny, k, xb.data_ptr(), nx, f, xs, out.data_ptr(),
                              w.data_ptr(), den.data_ptr()) == 0
    r_out, r_w, r_den = I.forward(idx, d2, x)
    bits_equal(out, r_out, f"pitched out f {f}")
    gx = torch.empty((nx, f), device="cuda")
    assert L.tknn_interpolate_backward(h, di.data_ptr(), w.data_ptr(), den.data_ptr(), ny, k, gb.data_ptr(), gs, nx, f,
                                       gx.data_ptr()) == 0
    bits_equal(gx, I.backward(idx, r_w, r_den, g, nx), f"pitched grad_x f {f}")


def test_hot_point():
    torch = pytest.importorskip("torch")
    rng = np.random.default_rng(3)
    nq = 1 << 20
    pos_x = np.float32([[0.5, 0.5, 0.5]])
    pos_y = rng.random((nq, 3), dtype=np.float32)
    x = rng.normal(size=(1, 128)).astype(np.float32)
    xd = torch.from_numpy(x).cuda().requires_grad_(True)
    out = knn_interpolate(xd, torch.from_numpy(pos_x).cuda(), torch.from_numpy(pos_y).cuda(), k=3)  # k clamps to 1
    g = torch.from_numpy(rng.normal(size=(nq, 128)).astype(np.float32)).cuda()
    (out * g).sum().backward()
    idx, d2 = I.knn_rows(pos_x, pos_y, 1)
    r_out, r_w, r_den = I.forward(idx, d2, x)
    bits_equal(out.detach(), r_out, "hot out")
    bits_equal(xd.grad, I.backward(idx, r_w, r_den, g.cpu().numpy(), 1), "hot grad_x")


def test_host_device_and_side_stream(knn):
    torch = pytest.importorskip("torch")
    rng = np.random.default_rng(4)
    pos_x = rng.random((5000, 3), dtype=np.float32)
    pos_y = rng.random((20_000, 3), dtype=np.float32)
    x = rng.normal(size=(5000, 40)).astype(np.float32)
    idx, d2 = query_rows(pos_x, pos_y, 5)
    ref = check(knn, idx, d2, x, np.random.default_rng(40), "host")  # numpy in, numpy out
    assert isinstance(ref[0], np.ndarray)
    s = torch.cuda.Stream()
    with torch.cuda.stream(s):
        knn.set_stream(s.cuda_stream)
        di, dd, dx = (torch.from_numpy(a).cuda() for a in (idx, d2, x))
        got = check(knn, di, dd, dx, np.random.default_rng(40), "side stream")  # the same grad_out
        assert got[0].is_cuda and got[3].is_cuda
    knn.set_stream(None)
    for a, b, what in zip(got, ref, ("out", "weight", "den", "grad_x")):
        bits_equal(a, b, f"{what} device vs host")
    # device inputs, host outputs through the C ABI
    L = _lib.load()
    out = np.empty((20_000, 40), np.float32)
    w = np.empty((20_000, 5), np.float32)
    den = np.empty(20_000, np.float32)
    torch.cuda.synchronize()
    assert L.tknn_interpolate(knn._h, di.data_ptr(), dd.data_ptr(), 20_000, 5, dx.data_ptr(), 5000, 40, 40,
                              out.ctypes.data, w.ctypes.data, den.ctypes.data) == 0
    bits_equal(out, ref[0], "device in, host out")


def test_repeated_calls_are_identical(knn):
    torch = pytest.importorskip("torch")
    rng = np.random.default_rng(5)
    pos_x = rng.random((2000, 3), dtype=np.float32)
    pos_y = rng.random((200_000, 3), dtype=np.float32)  # about 300 edges per data row
    idx, d2 = query_rows(pos_x, pos_y, 3)
    di, dd = torch.from_numpy(idx).cuda(), torch.from_numpy(d2).cuda()
    x = torch.randn((2000, 64), device="cuda")
    g = torch.randn((200_000, 64), device="cuda")
    first = None
    for _ in range(3):
        out, w, den = knn.interpolate(di, dd, x)
        gx = knn.interpolate_backward(di, w, den, g, 2000)
        if first is None:
            first = (out.clone(), gx.clone())
        else:
            assert torch.equal(out.view(torch.int32), first[0].view(torch.int32))
            assert torch.equal(gx.view(torch.int32), first[1].view(torch.int32))
    st = knn.stats()
    assert st["rounds"] == 3 and st["round_queries"] == [200_000, 600_000, 2000] and st["k"] == 3
    knn.interpolate(di, dd, x)
    st = knn.stats()
    assert st["rounds"] == 1 and st["round_queries"] == [200_000] and st["search_ms"] > 0


def test_knn_interpolate_autograd():
    torch = pytest.importorskip("torch")
    rng = np.random.default_rng(6)
    xs, ys = [500, 0, 300, 2], [2000, 100, 1200, 50]
    pos_x = torch.from_numpy(rng.random((sum(xs), 3), dtype=np.float32)).cuda().requires_grad_(True)
    pos_y = torch.from_numpy(rng.random((sum(ys), 3), dtype=np.float32)).cuda().requires_grad_(True)
    bx = torch.repeat_interleave(torch.arange(4, device="cuda"), torch.tensor(xs, device="cuda"))
    by = torch.repeat_interleave(torch.arange(4, device="cuda"), torch.tensor(ys, device="cuda"))
    x = torch.randn((sum(xs), 32), device="cuda", requires_grad=True)
    out = knn_interpolate(x, pos_x, pos_y, bx, by, k=3)
    g = torch.randn_like(out)
    (out * g).nan_to_num().sum().backward()
    idx, d2 = I.knn_rows(pos_x.detach().cpu().numpy(), pos_y.detach().cpu().numpy(), 3, xs, ys)
    r_out, r_w, r_den = I.forward(idx, d2, x.detach().cpu().numpy())
    bits_equal(out.detach(), r_out, "autograd out")
    gn = torch.where(torch.isnan(out), torch.zeros_like(g), g)  # nan_to_num's gradient is 0 on the NaN rows
    bits_equal(x.grad, I.backward(idx, r_w, r_den, gn.cpu().numpy(), sum(xs)), "autograd x.grad")
    assert pos_x.grad is None and pos_y.grad is None
    # an empty query set and an empty data set keep the graph
    e = knn_interpolate(x, pos_x, pos_y[:0], bx, by[:0])
    assert e.shape == (0, 32) and e.requires_grad
    nanrows = knn_interpolate(x[:0], pos_x[:0], pos_y, None, None)
    assert nanrows.shape == (sum(ys), 32) and torch.isnan(nanrows).all()


def test_against_pyg_body_on_gpu():
    torch = pytest.importorskip("torch")
    rng = np.random.default_rng(8)
    xs, ys = [4096] * 16, [16384] * 16
    pos_x = torch.from_numpy(rng.random((sum(xs), 3), dtype=np.float32)).cuda()
    pos_y = torch.from_numpy(rng.random((sum(ys), 3), dtype=np.float32)).cuda()
    bx = torch.arange(16, device="cuda").repeat_interleave(4096)
    by = torch.arange(16, device="cuda").repeat_interleave(16384)
    x = torch.randn((sum(xs), 64), device="cuda", requires_grad=True)
    out = knn_interpolate(x, pos_x, pos_y, bx, by, k=3)
    g = torch.randn_like(out)
    (out * g).sum().backward()
    ours = x.grad.clone()
    x.grad = None
    with TrueKNN(0, squared_dist=1) as t:
        t.build(pos_x, batch=bx)
        idx, d2 = t.query(pos_y, 3, batch=by)
    keep = idx.reshape(-1) >= 0
    y_idx = torch.arange(len(pos_y), device="cuda").repeat_interleave(3)[keep]
    x_idx = idx.reshape(-1).long()[keep]
    with torch.no_grad():
        wts = (1.0 / torch.clamp(d2.reshape(-1)[keep], min=1e-16)).view(-1, 1)
    num = torch.zeros((len(pos_y), 64), device="cuda").index_add_(0, y_idx, x[x_idx] * wts)
    ref = num / torch.zeros((len(pos_y), 1), device="cuda").index_add_(0, y_idx, wts)
    (ref * g).sum().backward()
    torch.testing.assert_close(out, ref, rtol=1e-5, atol=1e-6)
    torch.testing.assert_close(ours, x.grad, rtol=1e-4, atol=1e-5)


def test_error_codes(knn):
    L = _lib.load()
    h = knn._h
    E = _lib.EINVAL
    idx = np.int32([[0, 1], [2, -1]])
    d2 = np.float32([[1, 2], [3, 4]])
    x = np.ones((3, 4), np.float32)
    out = np.empty((2, 4), np.float32)
    w = np.empty((2, 2), np.float32)
    den = np.empty(2, np.float32)
    gx = np.empty((3, 4), np.float32)
    p = lambda a: None if a is None else a.ctypes.data

    def fwd(i=idx, d=d2, nq=2, k=2, xx=x, n=3, f=4, xs=4, o=out):
        return L.tknn_interpolate(h, p(i), p(d), nq, k, p(xx), n, f, xs, p(o), p(w), p(den))

    def bwd(i=idx, ww=w, dn=den, nq=2, k=2, g=out, gs=4, n=3, f=4, o=gx):
        return L.tknn_interpolate_backward(h, p(i), p(ww), p(dn), nq, k, p(g), gs, n, f, p(o))

    assert fwd() == 0 and bwd() == 0
    assert fwd(k=0) == E and fwd(k=513) == E and bwd(k=0) == E and bwd(k=513) == E
    assert fwd(f=0) == E and fwd(xs=3) == E and bwd(f=0) == E and bwd(gs=3) == E
    assert fwd(n=1 << 31) == E and fwd(nq=1 << 31) == E and bwd(n=1 << 31) == E and bwd(nq=1 << 31) == E
    assert bwd(nq=(1 << 28) + 1, k=4) == E  # above the sort's 2^30 - 1 edges, checked before any access
    for kw in ({"i": None}, {"d": None}, {"xx": None}, {"o": None}):
        assert fwd(**kw) == E
    for kw in ({"i": None}, {"ww": None}, {"dn": None}, {"g": None}, {"o": None}):
        assert bwd(**kw) == E
    assert fwd(nq=0, i=None, d=None, xx=None, o=None) == 0  # nq = 0 is a no-op
    assert fwd(n=0, xx=None, i=np.int32([[-1, -1], [-1, -1]])) == 0
    for bad in ([[0, 3], [2, -1]], [[0, 1], [-2, -1]]):  # outside {-1} and [0, n)
        assert fwd(i=np.int32(bad)) == E
        assert bwd(i=np.int32(bad)) == E
    assert "outside" in L.tknn_last_error(h).decode()
    gx.fill(7)
    assert bwd(nq=0, i=None, ww=None, dn=None, g=None) == 0 and not gx.any()  # no edge: +0
    with pytest.raises(TrueKNNError):
        knn.interpolate(np.int32([[5]]), np.float32([[1]]), x)
    with pytest.raises(ValueError):
        knn.interpolate(idx, d2[:, :1], x)


def test_build_and_search_unchanged(knn):
    rng = np.random.default_rng(9)
    p = rng.random((30_000, 3), dtype=np.float32)
    idx0, d0 = knn.build(p).search(8)
    q_idx, q_d2 = query_rows(p, rng.random((10_000, 3), dtype=np.float32), 3)
    check(knn, q_idx, q_d2, rng.normal(size=(30_000, 16)).astype(np.float32), rng, "after build")
    idx1, d1 = knn.search(8)
    bits_equal(idx1, idx0, "search idx after interpolate")
    bits_equal(d1, d0, "search dist after interpolate")


def test_keep_scratch_off():
    rng = np.random.default_rng(11)
    pos_x = rng.random((1000, 3), dtype=np.float32)
    pos_y = rng.random((5000, 3), dtype=np.float32)
    idx, d2 = query_rows(pos_x, pos_y, 3)
    with TrueKNN(0, keep_scratch=0) as t:
        for _ in range(2):
            check(t, idx, d2, rng.normal(size=(1000, 9)).astype(np.float32), rng, "keep_scratch 0")
