"""The cell-grid round-1 kernel (grid.cuh) against the LBVH path: every row bit-identical (indices and distance bits)."""
import numpy as np
import pytest

from owlraytracing_b200 import TrueKNN, datasets

pytestmark = pytest.mark.gpu

torch = pytest.importorskip("torch")


def _ctx(**opts):
    # warp_round_max = 0: small clouds run a dense round 1 too (else one warp per query, which never takes the grid)
    return TrueKNN(0, warp_round_max=0, **opts)


def _same(a, b):
    """Equal outputs of two searches: every array bit for bit (distances compared as int32 bits)."""
    assert len(a) == len(b)
    for x, y in zip(a, b):
        if x is None or y is None:
            assert x is None and y is None
            continue
        if isinstance(x, np.ndarray):
            assert x.dtype == y.dtype and x.shape == y.shape
            assert np.array_equal(x.view(np.int32), y.view(np.int32))
        else:
            assert x.dtype == y.dtype and x.shape == y.shape
            assert torch.equal(x.view(torch.int32), y.view(torch.int32))


def _pair(points, run, grid_opts=None, **opts):
    """run(ctx) on the grid path (auto unless grid_opts) and on the LBVH path; returns (grid result, its build stats, lbvh result)."""
    with _ctx(**(grid_opts or {}), **opts) as g, _ctx(grid=1, **opts) as t:
        g.build(points)
        gs = g.stats()
        rg = run(g)
        t.build(points)
        assert t.stats()["grid_level"] == 0  # off: no table is made
        rt = run(t)
    return rg, gs, rt


def _dev_uniform(n, seed=42):
    x = torch.empty((n, 3), dtype=torch.float32, device="cuda")
    with TrueKNN(0) as t:
        t.generate_uniform(seed, 0, n, out=x)
    torch.cuda.synchronize()
    return x


@pytest.mark.parametrize("n", [1_000, 30_000, 1_000_000, 10_000_000])
@pytest.mark.parametrize("k", [1, 5, 10, 16, 24])
def test_uniform_matches_lbvh(n, k):
    x = _dev_uniform(n)
    rg, gs, rt = _pair(x, lambda c: c.search(k))
    assert gs["grid_selected"] == 1 and gs["grid_split_cells"] == 0
    _same(rg, rt)


def test_grid_kernel_runs_and_counts():
    """The counting build walks cells: cells tested and points tested are reported, few groups are deferred."""
    x = _dev_uniform(1_000_000, seed=5)
    with _ctx(counters=1) as g:
        g.build(x)
        g.search(10)
        s = g.stats()
    assert s["grid_selected"] == 1
    assert s["warp_node_visits"] > 0 and s["warp_leaf_visits"] > 0 and s["points_tested"] > 0 and s["heap_inserts"] > 0
    assert s["grid_deferred"] * 32 < 1_000_000 // 100


@pytest.mark.parametrize("host", [False, True])
def test_search_shard_matches_lbvh(host):
    n, k, shards = 1_000_000, 10, 3
    x = _dev_uniform(n, seed=9)
    if host:
        x = x.cpu().numpy()  # host input: host outputs, searched in Morton slices whose copies overlap
    rg, gs, rt = _pair(x, lambda c: [a.copy() if host else a.clone() for s in range(shards) for a in c.search_shard(k, s, shards)])
    assert gs["grid_selected"] == 1
    _same(rg, rt)


def test_file_order_host_search_matches_lbvh():
    """tknn_search with host outputs: round 1 runs on slices by original index (a queue of every 5th point)."""
    x = datasets.uniform(1_000_000, seed=11)
    rg, gs, rt = _pair(x, lambda c: c.search(10))
    assert gs["grid_selected"] == 1
    _same(rg, rt)


@pytest.mark.parametrize("radius", [1e-3, 0.05, 0.3, 1.5])
def test_explicit_start_radius(radius):
    """Small radii leave most rows to later rounds; large ones exceed the cell cap, and the LBVH rounds finish the groups."""
    x = _dev_uniform(1_000_000, seed=3)
    rg, gs, rt = _pair(x, lambda c: c.search(10, start_radius=radius))
    _same(rg, rt)
    if radius == 0.3:  # 0.3 spans ~40 cells of 1/64 per axis: every group is deferred
        with _ctx(counters=1) as g:
            g.build(x)
            g.search(10, start_radius=radius)
            assert g.stats()["grid_deferred"] > 0


@pytest.mark.parametrize("offset,scale", [(1.0e4, 100.0), (-3.0e3, 50.0), (0.25, 1e-3)])
def test_offset_scaled_cloud(offset, scale):
    x = datasets.uniform(500_000, seed=21) * np.float32(scale) + np.float32(offset)
    rg, gs, rt = _pair(x, lambda c: c.search(10))
    assert gs["grid_split_cells"] == 0
    _same(rg, rt)


@pytest.mark.parametrize("grid", [0, 2])
def test_flat_cloud(grid):
    x = np.ascontiguousarray(datasets.uniform(300_000, seed=13)[:, :2])
    rg, gs, rt = _pair(x, lambda c: c.search(8), grid_opts={"grid": grid})
    assert gs["grid_split_cells"] == 0
    _same(rg, rt)


def test_lidar_rejected_and_forced():
    """A LiDAR-like scan fails the occupancy test (LBVH path); forced onto the grid it still matches bit for bit."""
    x = datasets.lidar_like(1_000_000, seed=7)
    rg, gs, rt = _pair(x, lambda c: c.search(10))
    assert gs["grid_selected"] == 0
    _same(rg, rt)
    rg, gs, rt = _pair(x, lambda c: c.search(10), grid_opts={"grid": 2})
    if gs["grid_level"]:
        assert gs["grid_selected"] == 1 and gs["grid_max_cell"] > 64  # runs longer than the staging area are split
    _same(rg, rt)


def test_coincident_cluster_rejected():
    x = datasets.uniform(200_000, seed=17)
    x[1000:6000] = x[1000]
    rg, gs, rt = _pair(x, lambda c: c.search(10))
    assert gs["grid_level"] == 0 and gs["grid_selected"] == 0  # coincident-point leaves: no table at all
    _same(rg, rt)


@pytest.mark.parametrize("opts", [{}, {"curve": 1}, {"sort_mode": 1}, {"grid_level": 2}, {"grid_level": 5}, {"grid_level": 8}])
def test_table_contiguity(opts):
    """Each cell's points are one contiguous run of the sorted order (the key's quantisation, bit for bit), for either curve,
    either key layout and any level; the results match the LBVH at every level."""
    x = _dev_uniform(300_000, seed=23)
    rg, gs, rt = _pair(x, lambda c: c.search(10), grid_opts={"grid": 2, **opts})
    assert gs["grid_level"] >= 1 and gs["grid_split_cells"] == 0
    assert gs["grid_selected"] == 1
    if "grid_level" in opts:
        assert gs["grid_level"] == opts["grid_level"]
    _same(rg, rt)
