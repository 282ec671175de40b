"""Round 1 on the cell grid (grid.cuh: grid_knn_kernel) with its 128-point staging area, bit for bit against the CPU oracle.

A warp stages up to 128 points (four warp-wide loads of a row gather) before it filters them into four survivor masks and
inserts the survivors, and writes one unresolved ballot word per 32-query group.  The cases put queries where that gets
awkward: nearly empty and partly valid last groups, queues of file-order slices instead of consecutive positions, k on
both ends of the ascending lists, groups whose cell range is capped so that all their queries go to the LBVH rounds,
round-1 bounds that leave a known set of queries underfilled, and coincident twins staged in the same flush as the query's
own point.  Every case checks that round 1 ran on the grid (tknn_stats::grid_rounds bit 0).
"""
import numpy as np
import pytest

from owlraytracing_b200 import TrueKNN, datasets

pytestmark = pytest.mark.gpu

torch = pytest.importorskip("torch")

U32 = np.uint32
DENSE = dict(grid=2, warp_round_max=0)  # the table whatever its occupancy; small rounds stay off the warp-per-query kernel
K_REF = 24
_REF = {}


def ref(oracle, name, x):
    """(idx, d2) of the all-points kNN at k = 24 (rows of smaller k are prefixes), cached per cloud."""
    if name not in _REF:
        oracle.set_squared_output(True)
        try:
            _REF[name] = oracle.knn_kdtree(np.ascontiguousarray(x, dtype=np.float32), K_REF)
        finally:
            oracle.set_squared_output(False)
    return _REF[name]


def same(got, want, what):
    g, w = np.asarray(got), np.asarray(want)
    assert g.shape == w.shape, f"{what}: shape {g.shape} != {w.shape}"
    if w.dtype == np.float32:
        g, w = g.view(U32), w.view(U32)
    bad = np.flatnonzero((g != w).any(axis=-1))
    assert bad.size == 0, f"{what}: {bad.size} / {len(w)} rows differ, first {bad[:6]}: {np.asarray(got)[bad[0]]} vs " \
                          f"{np.asarray(want)[bad[0]]}"


def search(x, k, start_radius=0.0, device=True, **opts):
    """search(k) with squared distances on a fresh context, from a device copy of x (one round sequence over all points) or
    from x on the host (host outputs: file-order slices, each with its own rounds).  Returns (idx, d2, stats)."""
    with TrueKNN(0, squared_dist=1, **DENSE, **opts) as t:
        t.build(torch.from_numpy(x).cuda() if device else x)
        i, d = t.search(k, start_radius=start_radius)
        st = t.stats()
    if device:
        i, d = i.cpu().numpy(), d.cpu().numpy()
    assert st["grid_level"] > 0 and st["grid_rounds"] & 1, f"round 1 did not run on the grid: {st['grid_rounds']:#x}"
    return i, d, st


def check(oracle, name, x, k, start_radius=0.0, device=True, **opts):
    ri, rd = ref(oracle, name, x)
    i, d, st = search(x, k, start_radius, device, **opts)
    what = f"{name} n={len(x)} k={k} r0={start_radius!r} {opts}"
    same(i, ri[:, :k], what + " idx")
    same(d, rd[:, :k], what + " d2")
    return st


def uniform(n, seed=5):
    return datasets.uniform(n, seed=seed)


@pytest.mark.parametrize("tail", [1, 31, 32, 33, 63])
def test_last_group(oracle, tail):
    """n mod 64 = tail: the last 32-query group holds 1, 31, 32 (full), 1 or 31 valid queries."""
    n = 64 * 300 + tail
    check(oracle, f"tail{tail}", uniform(n), 10)


@pytest.mark.parametrize("k", [1, 5, 10, 16, 24])
def test_k(oracle, k):
    check(oracle, "uniform50k", uniform(50_000, seed=9), k)


@pytest.mark.parametrize("k", [5, 24])
def test_file_order_slices(oracle, k):
    """Host input and outputs with three file-order slices: round 1 of each slice walks a queue of that slice's queries in
    curve order, so a group's queries are queue entries, not consecutive positions."""
    x = uniform(60_000 + 17, seed=13)
    check(oracle, "slices", x, k, device=False, file_order_chunks=3)


def test_capped_groups(oracle):
    """A start radius above the cloud's diagonal: every group's range is the whole 16^3-cell grid, more than TKNN_GRID_CAP
    cells, so round 1 tests nothing and the ballot words send all queries to the LBVH rounds.  (At half the extent the
    groups in a corner clip to 9^3 cells and resolve on the grid.)"""
    n = 64 * 200 + 40
    x = uniform(n, seed=17)
    st = check(oracle, "capped", x, 10, start_radius=2.0)
    assert st["round_queries"][:2] == [n, n], st["round_queries"]


@pytest.mark.parametrize("k", [4, 16])
def test_underfilled_queries(oracle, k):
    """A start radius between two k-th neighbour distances near their median: round 1 resolves exactly the queries with k
    points within it, so round 2 receives exactly the others."""
    n = 64 * 250 + 33
    x = uniform(n, seed=19)
    _, rd = ref(oracle, "underfilled", x)
    kth = np.sort(np.unique(rd[:, k - 1]))
    m = len(kth) // 2
    r0 = np.float32(np.sqrt((np.float64(kth[m]) + np.float64(kth[m + 1])) / 2))
    r2 = np.float32(r0 * r0)
    assert kth[m] < r2 < kth[m + 1]
    st = check(oracle, "underfilled", x, k, start_radius=float(r0))
    assert st["round_queries"][1] == int((rd[:, k - 1] > r2).sum()), st["round_queries"]


@pytest.mark.parametrize("k", [1, 5])
def test_coincident_twins(oracle, k):
    """Every point has a twin at distance 0 whose index is n / 2 away.  The twins sit in the same cell, so a query's own
    point and its twin are staged in the same flush, and the query must skip the one and take the other."""
    half = 64 * 150 + 31
    base = uniform(half, seed=23)
    x = np.concatenate([base, base])
    i, d, _ = search(x, k)
    ri, rd = ref(oracle, "twins", x)
    same(i, ri[:, :k], f"twins k={k} idx")
    same(d, rd[:, :k], f"twins k={k} d2")
    rows = np.arange(2 * half)
    assert (i[:, 0] == (rows + half) % (2 * half)).all() and (d[:, 0] == 0).all()
