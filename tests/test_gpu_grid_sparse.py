"""The sparse rounds on the cell grid (grid.cuh: grid_sparse_kernel, one thread per leftover query) against the LBVH path
(grid = 1) and against the CPU oracle: every row bit-identical (indices and distance bits), and the same queries active in
every round.

A sparse round takes the grid on a grid build when it is not final; warp_round_max = 0 keeps small rounds off the
warp-per-query kernel, sparse_divisor = 1 makes every round after the first a sparse one, and speculative_max = 0 keeps a
search of at most 2^20 queries from launching its second round as the final one.
"""
import numpy as np
import pytest

from helpers import assert_knn_equal
from owlraytracing_b200 import TrueKNN, datasets
from test_cpu_grid_model import quantised

pytestmark = pytest.mark.gpu

torch = pytest.importorskip("torch")

f32 = np.float32
SPARSE = dict(warp_round_max=0, sparse_divisor=1, speculative_max=0)


def _dev_uniform(n, seed=42):
    x = torch.empty((n, 3), dtype=torch.float32, device="cuda")
    with TrueKNN(0) as t:
        t.generate_uniform(seed, 0, n, out=x)
    torch.cuda.synchronize()
    return x


def _bits(a):
    if isinstance(a, np.ndarray):
        return a.view(np.int32)
    return a.view(torch.int32).cpu().numpy()


def _run(points, search, **opts):
    """search(ctx) on a fresh context; returns (its outputs as int32 bit patterns, the search's stats)."""
    with TrueKNN(0, **opts) as t:
        t.build(points)
        out = search(t)
        st = t.stats()
        return [None if a is None else _bits(a).copy() for a in out], st


def _pair(points, search, same_rounds=True, **opts):
    """The grid path and the LBVH path (grid = 1): equal outputs bit for bit and, unless a query is capped, equal round sizes.
    Returns the grid run's stats."""
    rg, sg = _run(points, search, **opts)
    rt, st = _run(points, search, grid=1, **opts)
    assert sg["grid_level"] > 0 and st["grid_level"] == 0
    if same_rounds:
        assert sg["round_queries"] == st["round_queries"]
    assert len(rg) == len(rt)
    for a, b in zip(rg, rt):
        assert (a is None) == (b is None)
        if a is not None:
            assert a.shape == b.shape and np.array_equal(a, b)
    return sg


def _sparse_rounds(st):
    """Rounds after the first one: with SPARSE, each of them runs on the grid unless it is the final one (radius beyond
    twice the scene's diagonal)."""
    return max(0, st["rounds"] - 1)


@pytest.fixture(scope="module")
def uniform10m():
    return _dev_uniform(10_000_000)


@pytest.fixture(scope="module")
def uniform1m():
    return _dev_uniform(1_000_000, seed=8)


@pytest.mark.parametrize("k", [1, 5, 10, 16, 24])
def test_uniform_10m_default(uniform10m, k):
    """The default routing at 10 M points: round 2 (about 1 % of the queries) is a sparse round on the grid."""
    st = _pair(uniform10m, lambda c: c.search(k))
    assert st["rounds"] >= 2 and st["round_queries"][1] > 0


@pytest.mark.parametrize("k", [1, 5, 10, 16, 24])
def test_uniform_1m_sparse(uniform1m, k):
    _pair(uniform1m, lambda c: c.search(k), **SPARSE)


@pytest.mark.parametrize("k", [5, 24])
def test_many_sparse_rounds(uniform1m, k):
    """A start radius far below the k-th distance: round 1 resolves almost nothing and three or more sparse rounds follow."""
    st = _pair(uniform1m, lambda c: c.search(k, start_radius=1.5e-3), **SPARSE)
    assert _sparse_rounds(st) >= 3


@pytest.mark.parametrize("host", [False, True])
def test_search_shard(uniform1m, host):
    """tknn_search_shard with device outputs, and with host outputs (Morton slices, each with its own rounds)."""
    k, shards = 10, 3
    x = uniform1m.cpu().numpy() if host else uniform1m
    _pair(x, lambda c: [a for s in range(shards) for a in c.search_shard(k, s, shards, start_radius=4e-3)], **SPARSE)


def test_search_file_order_host(uniform1m):
    """tknn_search with host outputs: the queries are searched in slices by original index."""
    _pair(uniform1m.cpu().numpy(), lambda c: c.search(10, start_radius=4e-3), **SPARSE)


def _hollow(n=1_000_000, seed=12):
    """Uniform on [0, 1]^3 with the box [0, 0.3]^3 thinned to every 400th point: its queries are left over after the dense
    rounds and need radii of several cells, where the grid kernel's cell cap is reached."""
    x = datasets.uniform(n, seed=seed)
    inside = (x < f32(0.3)).all(axis=1)
    keep = ~inside | (np.cumsum(inside) % 400 == 0)
    return np.ascontiguousarray(x[keep])


def test_capped_queries_finish_on_lbvh():
    """Queries whose cell range exceeds the cap stay unresolved until the final round on the LBVH finishes them (so the round
    sizes differ from the LBVH path's); the counting build shows the grid kernel ran after round 1 (cells staged, queries
    deferred) against the same search whose later rounds run one warp per query."""
    x = torch.from_numpy(_hollow()).cuda()
    n = x.shape[0]
    _pair(x, lambda c: c.search(10), same_rounds=False, **SPARSE)
    _, a = _run(x, lambda c: c.search(10), counters=1, **SPARSE)
    _, b = _run(x, lambda c: c.search(10), counters=1, warp_round_max=n - 1, sparse_divisor=1, speculative_max=0)
    assert a["round_queries"][1] == b["round_queries"][1] and _sparse_rounds(a) >= 3
    assert a["warp_leaf_visits"] > b["warp_leaf_visits"]  # cells staged by grid_sparse_kernel (the LBVH kernels add none)
    assert a["grid_deferred"] > b["grid_deferred"]


def test_sparse_kernel_counts(uniform1m):
    """Counting build: the grid kernel stages cells in the rounds after the first, and defers none of their queries.  The
    reference search runs those rounds one warp per query: at radius 0.02 a few hundred queries are left after round 1, far
    below the three waves of the warp kernel from which a small round takes the grid."""
    _, a = _run(uniform1m, lambda c: c.search(10, start_radius=0.02), counters=1, **SPARSE)
    _, b = _run(uniform1m, lambda c: c.search(10, start_radius=0.02), counters=1, warp_round_max=999_999, sparse_divisor=1,
                speculative_max=0)
    assert a["round_queries"] == b["round_queries"] and a["round_queries"][1] > 0
    assert a["warp_leaf_visits"] > b["warp_leaf_visits"]
    assert a["grid_deferred"] == b["grid_deferred"]


# ---- against the CPU oracle: tie-heavy, boundary-aligned and tiny-scale clouds, most rows finished by the sparse rounds ----

def _oracle_check(oracle, x, k, start_radius):
    x3 = x if x.shape[1] == 3 else np.concatenate([x, np.zeros((x.shape[0], 1), f32)], 1)
    ref_i, ref_d = oracle.knn_kdtree(x3, k)
    (idx, dist), st = _run(torch.from_numpy(x).cuda(), lambda c: c.search(k, start_radius=start_radius), **SPARSE)
    assert st["round_queries"][1] > x.shape[0] // 10 and _sparse_rounds(st) >= 1
    assert_knn_equal(idx, dist.view(f32), ref_i, ref_d, f"k={k} r={start_radius}")
    assert np.array_equal(dist, ref_d.view(np.int32))


@pytest.mark.parametrize("k", [6, 18, 24])
def test_oracle_lattice(oracle, k):
    """The 100^3 unit lattice from radius 0.3: the rounds at 1.2 and 2.4 meet whole shells of exact ties at 1, sqrt 2, sqrt 3."""
    _oracle_check(oracle, datasets.lattice(100), k, 0.3)


@pytest.mark.parametrize("k", [7, 19])
def test_oracle_shifted_quantised(oracle, k):
    """1 M points of the 2^-7 lattice on [-0.5, 0.5]^3 (cell boundaries on lattice planes, across zero) from radius 2^-9:
    the round at 2^-7 has its bound exactly at the nearest shell."""
    x = (quantised(1_000_000) - f32(0.5)).astype(f32)
    _oracle_check(oracle, x, k, 2.0 ** -9)


@pytest.mark.parametrize("k", [10, 24])
def test_oracle_tiny_scale(oracle, k):
    """1 M uniform points scaled to 1e-20 from radius 1e-23: the bounds of the first rounds are 0 or subnormal, and most
    neighbour distances are a few subnormal steps, full of ties."""
    x = (datasets.uniform(1_000_000, seed=3) * f32(1e-20)).astype(f32)
    _oracle_check(oracle, x, k, 1e-23)
