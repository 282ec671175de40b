"""The CPU reference of the voxel grid (tests/voxel_oracle.py) checked without a GPU: raw ids against a numpy float32
restatement of torch_cluster's formula and against a torch CPU pipeline (formula, torch.unique, float64 mean); the
chunk rule of the mean; negative truncation and aliasing outside [start, end]; and the argument checks of the Python
layer that run before any device is touched."""
import numpy as np
import pytest

import voxel_oracle as V
from owlraytracing_b200 import grid_cluster, grid_sampling, voxel_grid


def lidar_like(n, rng):
    r = rng.uniform(1.0, 40.0, n).astype(np.float32)
    a = rng.uniform(0, 2 * np.pi, n).astype(np.float32)
    z = rng.normal(0, 0.5, n).astype(np.float32)
    return np.stack([r * np.cos(a), r * np.sin(a), z], 1).astype(np.float32)


@pytest.mark.parametrize("dim", [2, 3])
@pytest.mark.parametrize("given", [False, True])
def test_raw_ids_equal_numpy_formula(dim, given):
    rng = np.random.default_rng(dim)
    p = lidar_like(5000, rng)[:, :dim]
    size = np.float32([0.7, 0.5, 0.3][:dim])
    start = np.float32([-30, -35, -1][:dim]) if given else None
    end = np.float32([30, 35, 1][:dim]) if given else None
    g = V.grid(p, size, start, end)
    assert (g["raw"] == V.numpy_raw(p, size, start, end)).all()
    sizes = [0, 1200, 0, 3000, 800]
    b = np.repeat(np.arange(len(sizes)), sizes)
    off = np.concatenate([[0], np.cumsum(sizes)]).astype(np.uint64)
    g = V.grid(p, size, start, end, off=off)
    assert (g["raw"] == V.numpy_raw(p, size, start, end, batch=b)).all()


def test_reference_equals_torch_pipeline():
    torch = pytest.importorskip("torch")
    rng = np.random.default_rng(3)
    sizes = [2000, 0, 1500, 10, 2500]
    p = lidar_like(sum(sizes), rng)
    x = rng.normal(size=(p.shape[0], 5)).astype(np.float32)
    b = np.repeat(np.arange(len(sizes)), sizes)
    off = np.concatenate([[0], np.cumsum(sizes)]).astype(np.uint64)
    g = V.grid(p, 0.8, off=off)
    pos = torch.cat([torch.from_numpy(p), torch.from_numpy(b).float().view(-1, 1)], 1)
    size = torch.tensor([0.8, 0.8, 0.8, 1.0])
    s0, e0 = pos.min(0).values, pos.max(0).values
    cnt = ((e0 - s0) / size).long() + 1
    mult = torch.cat([torch.ones(1, dtype=torch.long), torch.cumprod(cnt, 0)[:-1]])
    raw = (((pos - s0) / size).long() * mult).sum(1)
    uniq, inv = torch.unique(raw, sorted=True, return_inverse=True)
    assert (raw.numpy() == g["raw"]).all()
    assert (inv.numpy() == g["cluster"]).all()
    assert g["n_voxels"] == uniq.numel()
    xd = torch.from_numpy(x).double()
    mean = torch.zeros(uniq.numel(), 5, dtype=torch.float64).index_add_(0, inv, xd)
    mean /= torch.bincount(inv).double().view(-1, 1)
    np.testing.assert_allclose(V.pool(x, g), mean.numpy(), rtol=1e-5, atol=1e-6)
    mx = torch.full((uniq.numel(), 5), -np.inf, dtype=torch.float32).scatter_reduce(
        0, inv.view(-1, 1).expand(-1, 5), torch.from_numpy(x), "amax")
    assert (V.pool(x, g, "max") == mx.numpy()).all()
    # the voxel cloud is every member's cloud, and the representative the lowest member
    assert (g["seg"][g["cluster"]] == b).all()
    assert (g["first"] == np.array([np.flatnonzero(g["cluster"] == v).min() for v in range(g["n_voxels"])])).all()


def test_chunk_rule_is_plain_sum_up_to_32():
    rng = np.random.default_rng(5)
    p = np.repeat(np.float32([[0, 0], [10, 10], [20, 20]]), [1, 32, 33], 0)
    x = rng.normal(size=(p.shape[0], 2)).astype(np.float32) * np.float32(1e3)
    g = V.grid(p, 1.0)
    got = V.pool(x, g)
    for v, (a, b) in enumerate(zip(g["offsets"][:-1].astype(int), g["offsets"][1:].astype(int))):
        rows = x[g["members"][a:b]]
        s = np.float32(0)
        for r in rows:  # plain sequential sum
            s = np.float32(s + r)
        plain = s / np.float32(b - a)
        if b - a <= 32:
            assert (got[v] == plain).all()
        else:  # 33 members: the 32-member chunk, then the last member
            c0 = np.float32(0)
            for r in rows[:32]:
                c0 = np.float32(c0 + r)
            want = np.float32(np.float32(np.float32(0) + c0) + np.float32(np.float32(0) + rows[32])) / np.float32(33)
            assert (got[v] == want).all()


def test_negative_truncation_and_aliasing():
    p = np.float32([[0.0, 0.0], [-0.5, 0.0], [-1.5, 0.0], [2.5, 0.0], [0.0, 1.0], [3.2, 0.0]])
    g = V.grid(p, 1.0, start=0.0, end=[2.0, 1.0])
    # counts: 3 along x; a point up to a voxel below start is cell 0, further below gives -1, beyond end aliases
    assert list(g["raw"]) == [0, 0, -1, 2, 3, 3]
    assert (g["raw"] == V.numpy_raw(p, 1.0, 0.0, [2.0, 1.0])).all()
    assert g["n_voxels"] == 4
    assert list(g["cluster"]) == [1, 1, 0, 2, 3, 3]


@pytest.mark.parametrize("call", [
    lambda: grid_cluster(np.zeros((4, 1), np.float32), 1.0),
    lambda: grid_cluster(np.zeros((4, 3), np.float32), 0.0),
    lambda: grid_cluster(np.zeros((4, 3), np.float32), [1.0, -1.0, 1.0]),
    lambda: grid_cluster(np.zeros((4, 3), np.float32), [1.0, 1.0]),
    lambda: grid_cluster(np.zeros((4, 3), np.float32), np.nan),
    lambda: grid_cluster(np.zeros((4, 3), np.float32), 1.0, start=[0, np.inf, 0]),
    lambda: voxel_grid(np.zeros((4, 2), np.float32), 1.0, end=[1.0, 2.0, 3.0]),
    lambda: grid_sampling(np.zeros((4, 3), np.float32), 1.0, reduce="sum"),
    lambda: grid_cluster(np.zeros((4, 4), np.float32), 1.0),  # xyz + time: torch_cluster clusters all four columns
    lambda: voxel_grid(np.zeros((4, 4), np.float32), 1.0, np.zeros(4, np.int64)),
    lambda: grid_sampling(np.zeros((4, 5), np.float32), 1.0),
])
def test_host_argument_checks(call):
    with pytest.raises(ValueError):
        call()
