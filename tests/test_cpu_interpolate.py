"""The CPU reference of k-NN interpolation (tests/interpolate_oracle.py) checked without a GPU: against a numpy float32
restatement of the contract, against PyG's knn_interpolate body restated in plain torch on the CPU (forward, and x.grad
through autograd), against a float64 evaluation within a rounding bound, and the argument checks of knn_interpolate()
that run before any device is touched."""
import numpy as np
import pytest

import interpolate_oracle as I
from owlraytracing_b200 import knn_interpolate

EPS = np.float32(np.finfo(np.float32).eps)


def clouds(rng, x_sizes, y_sizes, dim=3, f=5):
    pos_x = rng.random((sum(x_sizes), dim), dtype=np.float32)
    pos_y = rng.random((sum(y_sizes), dim), dtype=np.float32)
    x = rng.normal(size=(sum(x_sizes), f)).astype(np.float32)
    return pos_x, pos_y, x


def numpy_forward(idx, d2, x):
    """The contract in numpy float32, slot by slot (vectorised over rows)."""
    nq, k = idx.shape
    f = x.shape[1]
    den = np.zeros(nq, np.float32)
    num = np.zeros((nq, f), np.float32)
    w = np.zeros((nq, k), np.float32)
    for s in range(k):
        ok = idx[:, s] >= 0
        d = d2[:, s]
        ws = np.where(ok, np.float32(1) / np.where(d < np.float32(1e-16), np.float32(1e-16), d), np.float32(0))
        w[:, s] = ws
        den = np.where(ok, den + ws, den).astype(np.float32)
        num = np.where(ok[:, None], num + x[np.maximum(idx[:, s], 0)] * ws[:, None], num).astype(np.float32)
    with np.errstate(invalid="ignore", divide="ignore"):
        return num / den[:, None], w, den


def numpy_backward(idx, w, den, g, n):
    """The backward contract in numpy float32: the edges grouped by data row (stable, so ascending edge number), then
    the r-th edge of every run added in round r."""
    flat = idx.reshape(-1)
    e = np.nonzero(flat >= 0)[0]
    j = flat[e]
    order = np.argsort(j, kind="stable")
    e, j = e[order], j[order]
    start = np.searchsorted(j, j, side="left")
    rank = np.arange(len(j)) - start
    gx = np.zeros((n, g.shape[1]), np.float32)
    k = idx.shape[1]
    for r in range(int(rank.max()) + 1 if len(rank) else 0):
        sel = rank == r
        ee, jj = e[sel], j[sel]
        i = ee // k
        term = (g[i] / den[i][:, None]) * w.reshape(-1)[ee][:, None]
        gx[jj] = gx[jj] + term.astype(np.float32)
    return gx


def bits(a):
    return np.ascontiguousarray(a, np.float32).view(np.uint32)


@pytest.mark.parametrize("k", [1, 3, 16])
def test_reference_equals_numpy_contract(oracle, k):
    rng = np.random.default_rng(k)
    x_sizes, y_sizes = [300, 0, 5, 200], [800, 40, 100, 0]
    pos_x, pos_y, x = clouds(rng, x_sizes, y_sizes)
    idx, d2 = I.knn_rows(pos_x, pos_y, k, x_sizes, y_sizes)
    out, w, den = I.forward(idx, d2, x)
    ref_out, ref_w, ref_den = numpy_forward(idx, d2, x)
    assert (bits(w) == bits(ref_w)).all()
    assert (bits(den) == bits(ref_den)).all()
    assert (bits(out) == bits(ref_out)).all()
    assert np.isnan(out[800:840]).all()  # the empty data cloud: 0 / 0
    g = rng.normal(size=out.shape).astype(np.float32)
    gx = I.backward(idx, w, den, g, len(x))
    assert (bits(gx) == bits(numpy_backward(idx, w, den, g, len(x)))).all()
    assert not gx[np.setdiff1d(np.arange(len(x)), idx[idx >= 0])].any()  # unreferenced rows: +0


def test_reference_edge_cases():
    idx = np.int32([[0, -1, 1], [-1, -1, -1], [2, 2, -1], [1, 0, 2]])
    d2 = np.float32([[0.0, 9.0, np.inf], [1, 1, 1], [1e-30, 4.0, 1], [np.nan, 1.0, -0.0]])
    x = np.float32([[1, -2], [3, 4], [-5, 6]])
    out, w, den = I.forward(idx, d2, x)
    assert bits(w[0]).tolist() == bits([1e16, 0, 0]).tolist()  # d2 = 0 clamps, -1 gives +0, +inf gives 0
    assert np.isnan(out[1]).all() and den[1] == 0  # no filled slot
    assert w[2, 0] == np.float32(1e16) and w[2, 1] == np.float32(0.25)
    assert np.isnan(w[3, 0]) and np.isnan(out[3]).all()  # NaN propagates
    ref = numpy_forward(idx, d2, x)
    for a, b in zip((out, w, den), ref):
        assert (bits(a) == bits(b)).all()
    g = np.ones((4, 2), np.float32)
    assert (bits(I.backward(idx, w, den, g, 3)) == bits(numpy_backward(idx, w, den, g, 3))).all()


def pyg_body(torch, x, idx, d2, nq):
    """PyG's knn_interpolate body in plain torch (torch_geometric is not needed), fed the same edges and d2."""
    k = idx.shape[1]
    flat = torch.as_tensor(idx).reshape(-1).long()
    keep = flat >= 0
    y_idx = torch.arange(nq).repeat_interleave(k)[keep]
    x_idx = flat[keep]
    with torch.no_grad():
        weights = 1.0 / torch.clamp(torch.as_tensor(d2).reshape(-1)[keep], min=1e-16)
        weights = weights.view(-1, 1)
    f = x.shape[1]
    num = torch.zeros((nq, f), dtype=x.dtype).index_add_(0, y_idx, x[x_idx] * weights)
    den = torch.zeros((nq, 1), dtype=x.dtype).index_add_(0, y_idx, weights)
    return num / den


@pytest.mark.parametrize("k", [3, 8])
def test_reference_against_pyg_body_in_torch(oracle, k):
    torch = pytest.importorskip("torch")
    rng = np.random.default_rng(20 + k)
    x_sizes, y_sizes = [256, 64, 3], [1024, 256, 50]
    pos_x, pos_y, x = clouds(rng, x_sizes, y_sizes, f=16)
    idx, d2 = I.knn_rows(pos_x, pos_y, k, x_sizes, y_sizes)
    xt = torch.from_numpy(x.copy()).requires_grad_(True)
    out_t = pyg_body(torch, xt, idx, d2, len(pos_y))
    g = rng.normal(size=out_t.shape).astype(np.float32)
    (out_t * torch.from_numpy(g)).sum().backward()
    out, w, den = I.forward(idx, d2, x)
    gx = I.backward(idx, w, den, g, len(x))
    np.testing.assert_allclose(out, out_t.detach().numpy(), rtol=1e-6, atol=0)
    # torch's CPU index_add_ sums in edge order, so the forward agrees bit for bit
    assert (bits(out) == bits(out_t.detach().numpy())).all()
    # the backward's index_put_(accumulate=True) sums each row in its own order: the per-edge terms are the same, but a
    # sum that cancels differs in its last bits, so the bound is relative to the sum of the absolute terms
    flat = idx.reshape(-1)
    e = np.nonzero(flat >= 0)[0]
    ab = np.zeros(gx.shape)
    np.add.at(ab, flat[e], np.abs(g[e // k].astype(np.float64) / den[e // k][:, None] * w.reshape(-1)[e][:, None]))
    assert (np.abs(gx - xt.grad.numpy()) <= 1e-6 * ab).all()
    # the same terms summed by index_add_ (edge order) give the reference's bits
    term = torch.from_numpy((g[e // k] / den[e // k][:, None]) * w.reshape(-1)[e][:, None])
    seq = torch.zeros(gx.shape).index_add_(0, torch.from_numpy(flat[e]).long(), term)
    assert (bits(gx) == bits(seq.numpy())).all()


@pytest.mark.parametrize("k", [3, 16])
def test_reference_against_float64(oracle, k):
    rng = np.random.default_rng(30 + k)
    x_sizes, y_sizes = [500, 40], [2000, 300]
    pos_x, pos_y, x = clouds(rng, x_sizes, y_sizes, dim=2, f=8)
    idx, d2 = I.knn_rows(pos_x, pos_y, k, x_sizes, y_sizes)
    out, w, den = I.forward(idx, d2, x)
    ok = idx >= 0
    w64 = np.where(ok, 1.0 / np.maximum(d2.astype(np.float64), 1e-16), 0.0)
    xs = x.astype(np.float64)[np.maximum(idx, 0)]  # [nq, k, f]
    num64 = (xs * w64[:, :, None]).sum(1)
    den64 = w64.sum(1)
    # each of the k products, k additions, the division and the weights round once: a bound of (2k + 3) eps relative to
    # the sum of the absolute terms
    scale = (np.abs(xs) * w64[:, :, None]).sum(1) / den64[:, None]
    assert (np.abs(out - num64 / den64[:, None]) <= (2 * k + 3) * EPS * scale + 1e-30).all()
    g = rng.normal(size=out.shape).astype(np.float32)
    gx = I.backward(idx, w, den, g, len(x))
    gx64 = np.zeros(gx.shape)
    ab = np.zeros(gx.shape)
    flat = idx.reshape(-1)
    e = np.nonzero(flat >= 0)[0]
    term = g.astype(np.float64)[e // k] / den64[e // k][:, None] * w64.reshape(-1)[e][:, None]
    np.add.at(gx64, flat[e], term)
    np.add.at(ab, flat[e], np.abs(term))
    runs = np.bincount(flat[e], minlength=len(x))[:, None]
    assert (np.abs(gx - gx64) <= (runs + 2 * k + 5) * EPS * ab + 1e-30).all()


def test_host_argument_checks():
    rng = np.random.default_rng(1)
    p3 = rng.random((10, 3), dtype=np.float32)
    x = rng.normal(size=(10, 4)).astype(np.float32)
    with pytest.raises(ValueError):
        knn_interpolate(x, rng.random((10, 4), dtype=np.float32), p3)  # 4-D positions
    with pytest.raises(ValueError):
        knn_interpolate(x, p3, rng.random((5, 1), dtype=np.float32))  # 1-D positions
    with pytest.raises(ValueError):
        knn_interpolate(x, p3, p3[:, :2])  # mismatched widths
    with pytest.raises(ValueError):
        knn_interpolate(x[:9], p3, p3)  # x rows != pos_x rows
    with pytest.raises(ValueError):
        knn_interpolate(x[:, 0], p3, p3)  # x must be [n, f]
    with pytest.raises(TypeError):
        knn_interpolate(x.astype(np.float64), p3, p3)
    with pytest.raises(ValueError):
        knn_interpolate(x, p3, p3, k=0)


def test_empty_inputs_need_no_device():
    x = np.ones((4, 6), np.float32)
    p = np.zeros((4, 3), np.float32)
    out = knn_interpolate(x, p, np.zeros((0, 3), np.float32))
    assert out.shape == (0, 6) and out.dtype == np.float32
    out = knn_interpolate(np.zeros((0, 6), np.float32), np.zeros((0, 2), np.float32), np.zeros((3, 2), np.float32))
    assert out.shape == (3, 6) and np.isnan(out).all()
