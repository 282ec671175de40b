"""The CPU references on the extreme clouds of tests/extreme_clouds.py, against brute force on the full d2 matrix.

The GPU tests of test_gpu_extreme.py compare the library with these references bit for bit, so the references must
first be right where the fp32 rule gets awkward: +inf distances ordered by index, fl(r * r) = +inf admitting every
pair, subnormal and zero d2 between distinct points, signed zeros.  The facts the GPU tests rely on are pinned here.
"""
import numpy as np
import pytest

import dbscan_oracle as DO
import extreme_clouds as E
import fps_oracle as F
import radius_oracle as RO
from oracle import oracle as O
from test_cpu_dbscan import assert_same as assert_same_dbscan
from test_cpu_dbscan import d2_matrix, dbscan_brute

N = 2000
U32, U64 = np.uint32, np.uint64


def knn_squared(x, k, tree=True):
    O.set_squared_output(True)
    try:
        return O.knn_kdtree(x, k) if tree else O.knn_brute(x, k)
    finally:
        O.set_squared_output(False)


def brute_keys(D):
    """Per row, the sorted (d2 bits << 32 | index) keys of every other point."""
    keys = (D.view(U32).astype(U64) << U64(32)) | np.arange(len(D), dtype=U64)[None, :]
    np.fill_diagonal(keys, np.iinfo(U64).max)
    return np.sort(keys, axis=1)[:, :-1]


def radii_of(d2_5th):
    """0, the median 5th-neighbour distance, the same one ulp down, the last radius with a finite square, the first
    with an infinite one, and +inf."""
    med = np.float32(np.median(np.sqrt(d2_5th.astype(np.float64))))
    return [np.float32(0), med, E.next_down(med), E.R_LAST_FINITE, E.R_FIRST_INF, np.float32(np.inf)]


def assert_lists_equal_brute(got, D, r, what):
    off, idx, d2 = got
    n = len(D)
    ball = D <= np.float32(np.float32(r) * np.float32(r))
    np.fill_diagonal(ball, False)
    assert (np.diff(off) == ball.sum(1)).all(), f"{what}: row lengths"
    rows = np.repeat(np.arange(n), np.diff(off))
    assert ball[rows, idx].all(), f"{what}: a listed point is outside the ball"
    assert (d2.view(U32) == D[rows, idx].view(U32)).all(), f"{what}: d2 bits"
    keys = (d2.view(U32).astype(U64) << U64(32)) | idx.astype(U64)
    same = rows[1:] == rows[:-1]
    assert (keys[1:][same] > keys[:-1][same]).all(), f"{what}: rows not strictly ascending by (d2, index)"


def fps_brute(D, m):
    """The selection rule of tknn_fps on the d2 matrix: start 0, then the largest (bits(D) << 32 | ~index) key."""
    n = len(D)
    low = U64(0xFFFFFFFF) - np.arange(n, dtype=U64)
    dmin = np.full(n, np.inf, np.float32)
    idx, dist = [0], [np.float32(np.finfo(np.float32).max)]
    for _ in range(m - 1):
        dmin = np.minimum(dmin, D[idx[-1]])
        c = int(np.argmax((dmin.view(U32).astype(U64) << U64(32)) | low))
        idx.append(c)
        dist.append(dmin[c])
    return np.array(idx, np.int32), np.array(dist, np.float32)


@pytest.mark.filterwarnings("ignore:overflow encountered")  # fl(r * r) = +inf and d2 = +inf are the point here
@pytest.mark.parametrize("name", sorted(E.CLOUDS))
def test_references_equal_brute_force(name):
    x = E.xyz3(E.cloud(name, N))
    D = d2_matrix(x)
    keys = brute_keys(D)
    for k in (1, 10):
        ti, td = knn_squared(x, k)
        bi, bd = knn_squared(x, k, tree=False)
        assert (ti == bi).all() and (td.view(U32) == bd.view(U32)).all(), f"{name} k={k}: kd-tree != brute"
        want = keys[:, :k]
        assert (bi == (want & U64(0xFFFFFFFF)).astype(np.int32)).all(), f"{name} k={k}: indices"
        assert (bd.view(U32) == (want >> U64(32)).astype(U32)).all(), f"{name} k={k}: d2 bits"
    _, d5 = knn_squared(x, 5)
    for r in radii_of(d5[:, 4]):
        what = f"{name} r={r!r}"
        assert_lists_equal_brute(RO.radius_lists(x, r), D, r, what)
        ball = D <= np.float32(r) * np.float32(r)
        assert (O.range_count(x, r).astype(np.int64) == ball.sum(1) - 1).all(), f"{what}: range count"
        for m in (2, 5, 20):
            assert_same_dbscan(DO.dbscan(x, r, m), dbscan_brute(x, r, m, d2=D), f"{what} min_pts={m}")
    for squared in (True, False):
        gi, gd = F.fps(x, counts=[N // 3], squared=squared)
        bi, bd = fps_brute(D, N // 3)
        assert (gi == bi).all(), f"{name}: fps indices"
        if not squared:
            bd[1:] = np.sqrt(bd[1:])
        assert (gd.view(U32) == bd.view(U32)).all(), f"{name}: fps distances"


def test_near_max_every_distance_is_inf():
    x = E.cloud("near_max", N)
    for k in (1, 10):
        idx, d2 = knn_squared(x, k)
        lowest = np.array([[j for j in range(k + 1) if j != q][:k] for q in range(N)], np.int32)
        assert (idx == lowest).all() and np.isposinf(d2).all()
    for squared in (True, False):
        idx, dist = F.fps(x, counts=[N], squared=squared)
        assert (idx == np.arange(N)).all() and np.isposinf(dist[1:]).all()


def test_radius_total_flips_where_r_squared_overflows():
    with np.errstate(over="ignore"):
        assert np.isfinite(E.R_LAST_FINITE * E.R_LAST_FINITE) and np.isposinf(E.R_FIRST_INF * E.R_FIRST_INF)
    assert np.nextafter(E.R_LAST_FINITE, np.float32(np.inf)) == E.R_FIRST_INF
    x = E.cloud("near_max", N)
    assert RO.radius_lists(x, E.R_LAST_FINITE)[0][-1] == 0
    assert RO.radius_lists(x, E.R_FIRST_INF)[0][-1] == N * (N - 1)
    x = E.cloud("overflow_1e20", N)
    below = RO.radius_lists(x, E.R_LAST_FINITE)[0][-1]
    assert 0 < below < N * (N - 1) and RO.radius_lists(x, E.R_FIRST_INF)[0][-1] == N * (N - 1)


def test_tiny_cloud_has_zero_distances_between_distinct_points():
    x = E.cloud("tiny_1e-21", N)
    assert len(np.unique(x, axis=0)) == N
    _, d2 = knn_squared(x, 1)
    assert (d2[:, 0] == 0).mean() > 0.25
    assert ((d2[:, 0] > 0) & (d2[:, 0] < np.finfo(np.float32).tiny)).any(), "some d2 are subnormal"


def test_catalogue_is_finite_and_deterministic():
    for name in E.CLOUDS:
        a, b = E.cloud(name, 500), E.cloud(name, 500)
        assert a.dtype == np.float32 and np.isfinite(a).all() and (a.view(U32) == b.view(U32)).all(), name
    z = E.cloud("across_zero", N)
    assert (np.signbit(z) & (z == 0)).any() and (~np.signbit(z) & (z == 0)).any()
    with np.errstate(over="ignore"):
        x = E.cloud("near_max", N)
        assert np.isposinf(x.max(0) - x.min(0)).all(), "the extent overflows on every axis"
