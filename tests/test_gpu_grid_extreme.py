"""Both cell-grid kNN kernels (grid.cuh: grid_knn_kernel for the dense round 1, grid_sparse_kernel for the later rounds) on
the extreme clouds of tests/extreme_clouds.py, bit for bit against the CPU oracle (indices and distance bits, in the d2 and
the sqrt form) and against the same search on the LBVH alone (grid = 1).

Every case routes its rounds onto the grid and checks that they ran there (tknn_stats::grid_rounds, bit r = round r ran a
grid kernel): grid = 2 uses the table whatever its occupancy, warp_round_max = 0 keeps small rounds off the warp-per-query
kernel, and for the sparse rounds sparse_divisor = 1 makes every round after the first a sparse one and speculative_max = 0
keeps round 2 from being launched as the final one.  The clouds put the grid where it gets awkward: a frame of scale 0
(every point in cell 0), a normal cloud inside one cell beside an outlier, round radii whose square is +inf in a round
that is not final, coarse-ulp ties on cell faces, signed zeros, zero and subnormal bounds, a z axis one cell wide.
"""
import numpy as np
import pytest

import extreme_clouds as E
import segment_oracle as SO
from oracle import oracle as O
from owlraytracing_b200 import TrueKNN

pytestmark = [pytest.mark.gpu, pytest.mark.filterwarnings("ignore:overflow encountered")]

U32 = np.uint32
FLT_MAX = np.float32(np.finfo(np.float32).max)
DENSE = dict(grid=2, warp_round_max=0)
SPARSE = dict(grid=2, warp_round_max=0, sparse_divisor=1, speculative_max=0)
NAMES = sorted(E.CLOUDS)
K_REF = 25


def size_of(name):
    return 6000 if name == "near_max" else 20_000


_REF = {}


def ref(name, n):
    """(x, idx, d2) of the all-points kNN at k = 25 (rows of smaller k are prefixes), cached per (cloud, n)."""
    key = (name, n)
    if key not in _REF:
        x = E.cloud(name, n)
        O.set_squared_output(True)
        try:
            i, d = O.knn_kdtree(E.xyz3(x), K_REF)
        finally:
            O.set_squared_output(False)
        _REF[key] = (x, i, d)
    return _REF[key]


def sqrt_form(d2):
    return np.where(d2 == FLT_MAX, d2, np.sqrt(d2)).astype(np.float32)


def same(got, want, what):
    g, w = np.asarray(got), np.asarray(want)
    assert g.shape == w.shape, f"{what}: shape {g.shape} != {w.shape}"
    if w.dtype == np.float32:
        g, w = g.view(U32), w.view(U32)
    bad = np.flatnonzero((g != w).any(axis=-1) if g.ndim > 1 else g != w)
    assert bad.size == 0, f"{what}: {bad.size} / {len(w)} rows differ, first {bad[:6]}: {np.asarray(got)[bad[0]]} vs " \
                          f"{np.asarray(want)[bad[0]]}"


def run(x, k, start_radius=0.0, **opts):
    """search(k) in the d2 and the sqrt form on one build; returns (idx, d2, sqrt dist, stats of the second search)."""
    with TrueKNN(0, **opts) as t:
        t.build(x)
        t.set_option("squared_dist", 1)
        i, d = t.search(k, start_radius=start_radius)
        s1 = t.stats()
        t.set_option("squared_dist", 0)
        i2, ds = t.search(k, start_radius=start_radius)
        st = t.stats()
    same(i2, i, "the sqrt-form search returns the d2-form rows")
    assert s1["grid_rounds"] == st["grid_rounds"] and s1["round_queries"] == st["round_queries"]
    return i, d, ds, st


def check(name, n, k, start_radius=0.0, x=None, **opts):
    """The grid run against the oracle (both forms) and against the LBVH run (grid = 1) bit for bit; equal round sizes
    unless a counting run shows the grid deferred a group or query.  Returns the grid run's stats."""
    xr, ri, rd = ref(name, n)
    x = xr if x is None else x
    ri, rd = ri[:, :k], rd[:, :k]
    what = f"{name} n={n} k={k} r0={start_radius!r} {opts}"
    i, d, ds, st = run(x, k, start_radius, **opts)
    assert st["grid_level"] > 0, what + ": no cell table"
    same(i, ri, what + " idx vs oracle")
    same(d, rd, what + " d2 vs oracle")
    same(ds, sqrt_form(rd), what + " sqrt dist vs oracle")
    li, ld, _, lst = run(x, k, start_radius, **dict(opts, grid=1))
    assert lst["grid_rounds"] == 0 and lst["grid_level"] == 0
    same(i, li, what + " idx vs grid=1")
    same(d, ld, what + " d2 vs grid=1")
    if st["round_queries"] != lst["round_queries"]:
        with TrueKNN(0, counters=1, **opts) as t:
            t.build(x)
            t.search(k, start_radius=start_radius)
            assert t.stats()["grid_deferred"] > 0, f"{what}: round sizes differ from grid=1 without a deferred query " \
                                                   f"({st['round_queries']} vs {lst['round_queries']})"
    return st


def grid_sparse_rounds(st):
    """Sparse rounds that ran on the grid, after checking that round 1 did and that every round but the last did (each
    round before the last is not final, so with SPARSE it is a sparse round on the grid)."""
    bits, rounds = st["grid_rounds"], st["rounds"]
    want = (1 << min(rounds - 1, 32)) - 1
    assert bits & want == want, f"grid_rounds {bits:#x}, {rounds} rounds"
    return bin(bits).count("1") - 1


def start_radius_for(name, k, n):
    """A start radius below the k-th neighbour distance of 90 % of the queries (a quarter of its 10 % quantile), so that
    round 1 leaves most queries to the sparse rounds."""
    _, _, rd = ref(name, n)
    kth = rd[:, k - 1].astype(np.float64)
    if not np.isfinite(kth).any():
        return 1e19  # near_max: every d2 is +inf
    q = np.quantile(kth[np.isfinite(kth)], 0.1)
    return float(max(0.25 * np.sqrt(q), 1e-30))


# ---------------------------------------------------------------- dense round 1 (grid_knn_kernel)

@pytest.mark.parametrize("k", [1, 4, 10, 23, 24])
@pytest.mark.parametrize("name", NAMES)
def test_dense_round(name, k):
    st = check(name, size_of(name), k, **DENSE)
    assert st["grid_rounds"] & 1, f"round 1 did not run on the grid: {st['grid_rounds']:#x}"


# ---------------------------------------------------------------- sparse rounds (grid_sparse_kernel)

@pytest.mark.parametrize("k", [4, 24])
@pytest.mark.parametrize("name", NAMES)
def test_sparse_rounds(name, k):
    n = size_of(name)
    r0 = start_radius_for(name, k, n)
    st = check(name, n, k, start_radius=r0, **SPARSE)
    assert st["round_queries"][1] > n // 10, st["round_queries"][:4]
    assert grid_sparse_rounds(st) >= 2, (st["rounds"], hex(st["grid_rounds"]))


INF_RUNS = {"near_max": 1e19, "overflow_1e20": 2e19, "far_clusters": 2e19}


@pytest.mark.parametrize("name", sorted(INF_RUNS))
def test_rounds_with_infinite_r2(name):
    """Rounds that are not final but whose r^2 is +inf: the sparse kernel defers every query there (it tests nothing), so
    no round on the grid resolves a query; the final LBVH round finishes them all.  near_max from r = 1e19 (round 1 finds
    no finite d2, then r^2 overflows until the round cap makes a round final); overflow_1e20 and far_clusters from r = 2e19
    (r^2 = +inf from round 1 on, below twice the scene's diagonal)."""
    n, k, r0 = size_of(name), 10, INF_RUNS[name]
    st = check(name, n, k, start_radius=r0, **SPARSE)
    rounds, rq = st["rounds"], st["round_queries"]
    assert grid_sparse_rounds(st) >= 2
    r = np.float32(r0) * np.float32(2.0) ** np.arange(rounds, dtype=np.float32)
    inf_rounds = [j for j in range(1, rounds - 1) if np.isposinf(r[j] * r[j])]
    assert inf_rounds, "no non-final round with r^2 = +inf"
    for j in inf_rounds:
        assert rq[j + 1] == rq[j], f"round {j + 1} (r^2 = +inf) resolved queries: {rq}"
    with TrueKNN(0, counters=1, **SPARSE) as t:
        t.build(ref(name, n)[0])
        t.search(k, start_radius=r0)
        assert t.stats()["grid_deferred"] >= rq[inf_rounds[0]]


# ---------------------------------------------------------------- forced levels

@pytest.mark.parametrize("level", [1, 3, 8])
@pytest.mark.parametrize("name", ["offset_1e6", "across_zero", "mixed_scales", "offset_1e6_2d"])
def test_forced_levels(name, level):
    """Level 1: cells of thousands of points, runs far longer than the 64-point staging area; level 8: ranges wider than
    MAX_SPAN cells and more than TKNN_GRID_CAP cells (deferred groups and queries)."""
    n, k = size_of(name), 10
    st = check(name, n, k, grid_level=level, **DENSE)
    assert st["grid_level"] == level and st["grid_rounds"] & 1
    st = check(name, n, k, start_radius=start_radius_for(name, k, n), grid_level=level, **SPARSE)
    assert grid_sparse_rounds(st) >= 2


# ---------------------------------------------------------------- larger clouds: the auto level and many rings

@pytest.mark.parametrize("name", ["offset_1e4", "across_zero", "outlier_1e30"])
def test_larger_clouds(name):
    n, k = 200_000, 16
    st = check(name, n, k, **DENSE)
    assert st["grid_level"] >= 5 and st["grid_rounds"] & 1
    st = check(name, n, k, start_radius=start_radius_for(name, k, n), **SPARSE)
    assert grid_sparse_rounds(st) >= 2


# ---------------------------------------------------------------- search_shard and host outputs

@pytest.mark.parametrize("name", ["offset_1e4", "across_zero"])
def test_shards_and_host_outputs(name):
    """Host outputs of search at 300 K points (file-order slices, each with its own rounds: grid_rounds ORs them) and
    search_shard with 3 shards, host outputs too."""
    n, k, shards = 300_000, 10, 3
    x, ri, rd = ref(name, n)
    ri, rd = ri[:, :k], rd[:, :k]
    r0 = start_radius_for(name, k, n)
    with TrueKNN(0, squared_dist=1, **SPARSE) as t:
        t.build(x)
        i, d = t.search(k, start_radius=r0)
        st = t.stats()
        same(i, ri, f"{name} host search idx")
        same(d, rd, f"{name} host search d2")
        assert grid_sparse_rounds(st) >= 2
        for s in range(shards):
            qid, i, d = t.search_shard(k, s, shards, start_radius=r0)
            st = t.stats()
            same(i, ri[qid], f"{name} shard {s} idx")
            same(d, rd[qid], f"{name} shard {s} d2")
            assert st["grid_rounds"] & 3 == 3, hex(st["grid_rounds"])
        t.set_option("squared_dist", 0)
        i, d = t.search(k)
        same(i, ri, f"{name} host search (estimated radius) idx")
        same(d, sqrt_form(rd), f"{name} host search (estimated radius) dist")
        assert t.stats()["grid_rounds"] & 1


# ---------------------------------------------------------------- controls: routes that must stay off the grid

@pytest.mark.parametrize("name", ["offset_1e6", "mixed_scales"])
def test_k25_stays_on_lbvh(name):
    n, k = size_of(name), 25
    x, ri, rd = ref(name, n)
    for opts, r0 in ((DENSE, 0.0), (SPARSE, start_radius_for(name, 24, n))):
        i, d, ds, st = run(x, k, r0, **opts)
        assert st["grid_level"] > 0 and st["grid_rounds"] == 0
        same(i, ri, f"{name} k=25 idx")
        same(d, rd, f"{name} k=25 d2")
        same(ds, sqrt_form(rd), f"{name} k=25 dist")


def test_segmented_build_stays_on_lbvh():
    parts = [E.cloud("offset_1e6", 7000), E.cloud("across_zero", 5000), E.cloud("outlier_1e30", 6000)]
    x = np.concatenate(parts).astype(np.float32)
    sizes = [len(p) for p in parts]
    off = SO.offsets_of(sizes)
    batch = np.repeat(np.arange(len(sizes)), sizes)
    with TrueKNN(0, **SPARSE) as t:
        t.build(x, batch=batch, batch_size=len(sizes))
        for squared in (1, 0):
            t.set_option("squared_dist", squared)
            for k in (10, 24):
                wi, wd = SO.knn(x, off, k, squared=bool(squared))
                i, d = t.search(k)
                st = t.stats()
                same(i, wi, f"segmented k={k} idx")
                same(d, wd, f"segmented k={k} dist squared={squared}")
                assert st["grid_rounds"] == 0 and st["grid_level"] == 0
