"""The start-radius quantile of gridded searches (TKNN_OPT_GRID_RADIUS_QUANTILE) and the phase accounting of the counting
grid_knn_kernel.

A lower quantile only moves queries from round 1 to later rounds, and every round is exact, so at every quantile the rows
must equal the CPU oracle's and the LBVH path's (grid = 1) bit for bit: on a tie-heavy integer lattice and on the extreme
clouds of tests/extreme_clouds.py.  The rounds are routed onto the grid as in test_gpu_grid_extreme.py (grid = 2 uses the
table whatever its occupancy, warp_round_max = 0 keeps small rounds off the warp-per-query kernel, sparse_divisor = 1 and
speculative_max = 0 send every non-final round after the first to grid_sparse_kernel) and tknn_stats::grid_rounds shows
that they ran there.
"""
import numpy as np
import pytest

import extreme_clouds as E
from oracle import oracle as O
from owlraytracing_b200 import TrueKNN, TrueKNNError

pytestmark = [pytest.mark.gpu, pytest.mark.filterwarnings("ignore:overflow encountered")]

U32 = np.uint32
ROUTE = dict(grid=2, warp_round_max=0, sparse_divisor=1, speculative_max=0)
K_REF = 16


def lattice(n_side=26, seed=3):
    """An integer lattice in shuffled order: every query has many neighbours at exactly the k-th distance, so the rows
    depend on the lowest-index tie rule in every round."""
    g = np.arange(n_side, dtype=np.float32)
    x = np.stack(np.meshgrid(g, g, g, indexing="ij"), axis=-1).reshape(-1, 3)
    return np.ascontiguousarray(x[np.random.default_rng(seed).permutation(len(x))])


_REF = {}


def ref(name):
    """(cloud, idx, d2) of the all-points kNN at k = K_REF (rows of smaller k are prefixes), cached per cloud."""
    if name not in _REF:
        x = lattice() if name == "lattice" else E.cloud(name, 6000 if name == "near_max" else 20_000)
        O.set_squared_output(True)
        try:
            i, d = O.knn_kdtree(E.xyz3(x), K_REF)
        finally:
            O.set_squared_output(False)
        _REF[name] = (x, i, d)
    return _REF[name]


def same(got, want, what):
    g, w = np.asarray(got), np.asarray(want)
    assert g.shape == w.shape, f"{what}: shape {g.shape} != {w.shape}"
    if w.dtype == np.float32:
        g, w = g.view(U32), w.view(U32)
    bad = np.flatnonzero((g != w).any(axis=-1))
    assert bad.size == 0, f"{what}: {bad.size} / {len(w)} rows differ, first {bad[:6]}"


def search(x, k, **opts):
    with TrueKNN(0, squared_dist=1, **opts) as t:
        t.build(x)
        i, d = t.search(k)
        return i, d, t.stats()


def check(name, k, q):
    x, ri, rd = ref(name)
    what = f"{name} k={k} grid_radius_quantile={q}"
    i, d, st = search(x, k, grid_radius_quantile=q, **ROUTE)
    assert st["grid_level"] > 0, what + ": no cell table"
    same(i, ri[:, :k], what + " idx vs oracle")
    same(d, rd[:, :k], what + " d2 vs oracle")
    li, ld, lst = search(x, k, grid_radius_quantile=q, **dict(ROUTE, grid=1))
    assert lst["grid_rounds"] == 0
    same(i, li, what + " idx vs grid=1")
    same(d, ld, what + " d2 vs grid=1")
    # round 1 ran on the grid, and so did every later round but the last (none of them is final; rounds from 32 on have no
    # bit)
    want = (1 << min(st["rounds"] - 1, 32)) - 1
    assert st["grid_rounds"] & want == want, f"{what}: grid_rounds {st['grid_rounds']:#x}, {st['rounds']} rounds"
    return st, lst


@pytest.mark.parametrize("q", [0, 100, 500, 900, 990, 1000])
@pytest.mark.parametrize("k", [1, 10, 16])
def test_lattice(k, q):
    check("lattice", k, q)


@pytest.mark.parametrize("q", [100, 500])
def test_most_queries_left_to_later_rounds(q):
    """A start radius under most queries' k-th distance: round 2 on grid_sparse_kernel gets most of the cloud."""
    st, _ = check("offset_1e4", 10, q)
    assert st["round_queries"][1] > st["n_queries"] * (1000 - q) // 2000, st["round_queries"]
    assert st["grid_rounds"] & 2, f"round 2 did not run on the grid: {st['grid_rounds']:#x}, {st['rounds']} rounds"


@pytest.mark.parametrize("q", [100, 500])
@pytest.mark.parametrize("name", sorted(E.CLOUDS))
def test_extreme(name, q):
    check(name, 10, q)


def test_only_gridded_searches_use_it():
    """The option moves the start radius of a search whose round 1 walks the grid, and of no other."""
    x = ref("offset_1e4")[0]
    r = {}
    for grid in (2, 1):
        for q in (500, 990):
            _, _, st = search(x, 10, grid_radius_quantile=q, **dict(ROUTE, grid=grid))
            r[grid, q] = st["start_radius"]
    assert r[2, 500] < r[2, 990]
    assert r[1, 500] == r[1, 990]          # the LBVH path keeps TKNN_OPT_RADIUS_QUANTILE
    assert r[2, 990] == r[1, 990]          # both at 99 %: the same sample and the same quantile
    with TrueKNN(0) as t:
        for bad in (-1, 1001):
            with pytest.raises(TrueKNNError):
                t.set_option("grid_radius_quantile", bad)


def test_phase_counters():
    """The counting grid_knn_kernel charges its cycles to the six phases and counts its insert-loop trips: the loop runs at
    least as many lane-trips as round 1 inserts, and round 1 inserts at least k keys per query it resolves."""
    x = ref("offset_1e4")[0]
    k = 10
    with TrueKNN(0, counters=1, **ROUTE) as t:
        t.build(x)
        t.search(k)
        st = t.stats()
    assert st["grid_rounds"] & 1
    assert len(st["grid_phase_cycles"]) == 6 and all(c > 0 for c in st["grid_phase_cycles"]), st["grid_phase_cycles"]
    resolved = st["round_queries"][0] - (st["round_queries"][1] if st["rounds"] > 1 else 0)
    assert k * resolved <= st["grid_inserts"] <= st["heap_inserts"]
    assert st["grid_inserts"] <= 32 * st["grid_insert_iters"]
    with TrueKNN(0, **ROUTE) as t:  # the plain build reports none of them
        t.build(x)
        t.search(k)
        st = t.stats()
    assert sum(st["grid_phase_cycles"]) == 0 and st["grid_insert_iters"] == 0 and st["grid_inserts"] == 0
