"""The cell-grid round-1 kernel (grid.cuh) against the CPU oracle, bit for bit, on the clouds its exactness argument is about:
exact distance ties, points on cell boundaries and on the top cell's clamp, clouds across zero, coincident points, and
distances whose square is subnormal or underflows to 0.

Every case asserts that the build selected the grid (grid_selected == 1), compares indices and distance bits with
oracle.knn_kdtree (itself pinned on a sample of rows by knn_brute_queries), and runs the same case on the LBVH path
(grid = 1) against the oracle, so that a mismatch of the grid alone points at the grid and not at the shared k-list code.
"""
import numpy as np
import pytest

from helpers import assert_knn_equal
from owlraytracing_b200 import TrueKNN, datasets
from test_cpu_grid_model import quantised

pytestmark = pytest.mark.gpu

torch = pytest.importorskip("torch")

f32 = np.float32
N = 1_000_000
_refs = {}


def _pad3(x):
    return x if x.shape[1] == 3 else np.concatenate([x, np.zeros((x.shape[0], 1), f32)], 1)


def _ref(oracle, name, x, k, squared=False):
    """oracle.knn_kdtree(x, k), kept per (cloud, k, squared); ~1000 of its rows checked against knn_brute_queries."""
    key = (name, k, squared)
    if key not in _refs:
        x3 = _pad3(x)
        oracle.set_squared_output(squared)
        try:
            idx, dist = oracle.knn_kdtree(x3, k)
            sub = np.arange(0, x3.shape[0], max(1, x3.shape[0] // 1000), dtype=np.int32)
            bi, bd = oracle.knn_brute_queries(x3, x3[sub], k, self_ids=sub)
        finally:
            oracle.set_squared_output(False)
        assert np.array_equal(bi, idx[sub]) and np.array_equal(bd.view(np.int32), dist[sub].view(np.int32)), name
        _refs[key] = (idx, dist)
    return _refs[key]


def _search(x, k, device=True, start_radius=0.0, **opts):
    """search(k) on a fresh context; returns (idx, dist) as numpy and the build's stats."""
    with TrueKNN(0, **opts) as t:
        t.build(torch.from_numpy(x).cuda() if device else x)
        st = t.stats()
        idx, dist = t.search(k, start_radius=start_radius)
        if device:
            idx, dist = idx.cpu().numpy(), dist.cpu().numpy()
    return idx, dist, st


def _exact(idx, dist, ref, what):
    assert_knn_equal(idx, dist, *ref, what)
    bad = np.nonzero((dist.view(np.int32) != ref[1].view(np.int32)).any(axis=1))[0]
    assert bad.size == 0, f"{what}: {bad.size} rows differ in distance bits; first row {bad[0]}: {dist[bad[0]]} vs {ref[1][bad[0]]}"


def _check(oracle, name, x, k, grid_opts=None, **kw):
    """The grid run (auto unless grid_opts) and the LBVH run, both against the oracle.  Returns the grid run's results."""
    ref = _ref(oracle, name, x, k, squared=bool(kw.get("squared_dist")))
    idx, dist, st = _search(x, k, **(grid_opts or {}), **kw)
    assert st["grid_selected"] == 1 and st["grid_split_cells"] == 0, (name, st["grid_level"], st["grid_max_cell"])
    _exact(idx, dist, ref, f"{name} k={k} grid {grid_opts or ''}")
    li, ld, lst = _search(x, k, grid=1, **kw)
    assert lst["grid_level"] == 0
    _exact(li, ld, ref, f"{name} k={k} lbvh")
    return idx, dist, st


@pytest.fixture(scope="module")
def quant():
    """1 M distinct points of the 2^-7 lattice on [0, 1]^3, corners included: lo = 0, hi = 1, scale = 2^21, so at the auto
    level 6 every cell boundary is a lattice plane and the points at 1.0 sit in the clamped top cell.  Checked once with the
    counting build: round 1 walks the grid (cell tests are counted) and resolves most groups there."""
    x = quantised(N)
    with TrueKNN(0, counters=1) as t:
        t.build(torch.from_numpy(x).cuda())
        t.search(24)
        st = t.stats()
    assert st["grid_selected"] == 1 and st["grid_level"] == 6
    assert st["warp_node_visits"] > 0 and st["points_tested"] > 0
    assert st["grid_deferred"] < N // 32
    return x


@pytest.mark.parametrize("k", [1, 6, 7, 18, 19, 24])
def test_quantised(oracle, quant, k):
    _check(oracle, "quantised", quant, k)


@pytest.mark.parametrize("level", [1, 3, 8])
def test_quantised_forced_level(oracle, quant, level):
    """Level 1: a cell's run far exceeds the 64-point staging area and continues after each flush.  Level 8: cells of half
    a lattice step, every other one empty."""
    _, _, st = _check(oracle, "quantised", quant, 19, grid_opts={"grid": 2, "grid_level": level})
    assert st["grid_level"] == level


def test_quantised_k24_k25(oracle, quant):
    """k = 24 (the largest grid k) and k = 25 (the heap kernel, no grid round): both exact, and one the other's prefix."""
    i24, d24, _ = _check(oracle, "quantised", quant, 24)
    i25, d25, _ = _check(oracle, "quantised", quant, 25)
    assert np.array_equal(i25[:, :24], i24) and np.array_equal(d25[:, :24], d24)


def test_quantised_squared_dist(oracle, quant):
    _check(oracle, "quantised", quant, 10, squared_dist=1)


def test_quantised_host_file_order(oracle, quant):
    """Host input and outputs: round 1 runs on slices of the original order."""
    _check(oracle, "quantised", quant, 10, device=False)


@pytest.mark.parametrize("cloud,k", [("shifted", 7), ("shifted", 24), ("centred", 10), ("centred", 24)])
def test_across_zero(oracle, quant, cloud, k):
    """Clouds across 0: the bisection of the cell boundaries over ordered float bits crosses the sign."""
    if cloud == "shifted":  # the quantised cloud on [-0.5, 0.5]^3 (exact)
        x = (quant - f32(0.5)).astype(f32)
    else:  # uniform, centred on 0, extent 2e-3
        x = ((datasets.uniform(N, seed=31) - f32(0.5)) * f32(2e-3)).astype(f32)
    _check(oracle, cloud, x, k)


@pytest.mark.parametrize("k", [6, 18, 24])
def test_lattice(oracle, k):
    """The 100^3 unit lattice (cells not aligned with it): shells at 1 (6 points), sqrt 2 (12) and sqrt 3 (8), each shell
    in ascending index order; at k = 24 the six lowest indices of the sqrt 3 shell."""
    m = 100
    x = datasets.lattice(m)
    idx, dist, _ = _check(oracle, "lattice", x, k)
    g = x.astype(np.int64)
    inner = np.nonzero(((g >= 1) & (g <= m - 2)).all(axis=1))[0]
    shells = [(0, 6, f32(1.0)), (6, 18, np.sqrt(f32(2.0))), (18, 24, np.sqrt(f32(3.0)))]
    for a, b, d in shells:
        if a >= k:
            break
        b = min(b, k)
        assert (dist[inner, a:b] == d).all()
        assert (np.diff(idx[inner, a:b], axis=1) > 0).all()
    if k == 24:  # the corners of the unit cube around q with the lowest indices: all with x - 1, then two with x + 1
        i = inner[len(inner) // 2]
        want = sorted(i + dx * m * m + dy * m + dz for dx in (-1, 1) for dy in (-1, 1) for dz in (-1, 1))[:6]
        assert list(idx[i, 18:24]) == want


@pytest.mark.parametrize("k", [1, 10])
def test_coincident_groups(oracle, k):
    """2 % of 1 M uniform points get 1 to 6 extra copies: groups below the coincident-leaf size keep the grid selected.  At
    k = 1 every member of a group has its lowest-index twin at distance 0."""
    rng = np.random.default_rng(7)
    base = datasets.uniform(N, seed=41)
    src = rng.choice(N, N // 50, replace=False)
    reps = rng.integers(1, 7, src.size)
    x = np.concatenate([base, base[np.repeat(src, reps)]])
    perm = rng.permutation(x.shape[0])
    x = np.ascontiguousarray(x[perm])
    idx, dist, _ = _check(oracle, "coincident", x, k)
    orig = perm.copy()  # orig[i] = the base point of output row i
    orig[perm >= N] = np.repeat(src, reps)[perm[perm >= N] - N]
    members = np.isin(orig, src)
    assert (dist[members, 0] == 0).all()
    if k == 1:
        groups = {}
        for i in np.nonzero(members)[0]:  # ascending: each group's rows in index order
            groups.setdefault(orig[i], []).append(i)
        for rows in groups.values():
            assert idx[rows[0], 0] == rows[1] and (idx[rows[1:], 0] == rows[0]).all()


# sizes keep the oracle's tie-heavy kd-tree walk to seconds: at 1e-22 every pair's d2 is a few subnormal steps
TINY = {1e-20: N, 1e-21: 300_000, 1e-22: 60_000}


@pytest.mark.parametrize("start_radius", [0.0, 1e-23])
@pytest.mark.parametrize("k", [10, 24])
@pytest.mark.parametrize("scale", list(TINY))
def test_tiny_scale(oracle, scale, k, start_radius):
    """Uniform clouds scaled to 1e-20 .. 1e-22: neighbour d2 is subnormal or underflows to 0, so most rows hold far more
    than k points at d2 <= the round-1 bound, and the answer is the lowest indices among all of them, across cells.  The
    round-1 bound is the estimator's (start_radius 0) or 1e-23^2, which is 0 in fp32."""
    x = (datasets.uniform(TINY[scale], seed=3) * f32(scale)).astype(f32)
    _check(oracle, f"tiny{scale}", x, k, start_radius=start_radius)


def test_two_dimensional(oracle):
    """dim = 2 (z = 0): 200 K distinct points of the 2^-9 lattice on [0, 1]^2.  Auto selection rejects a flat cloud at
    level 5 (about 200 points per cell), so the grid is forced at level 8: cell boundaries on every other lattice line."""
    x = quantised(200_000, seed=2, b=9, dim=2)
    _, _, st = _check(oracle, "flat", x, 10, grid_opts={"grid": 2, "grid_level": 8})
    assert st["grid_level"] == 8
