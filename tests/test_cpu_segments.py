"""The per-segment CPU reference of segmented builds (tests/segment_oracle.py) against a direct brute force with a
same-segment mask, and the batch -> offsets conversion of TrueKNN.build(batch=...).  No GPU needed."""
import numpy as np
import pytest

import segment_oracle as SO
from oracle import oracle as O
from owlraytracing_b200 import batch_to_offsets

K = 5


def brute(x, offsets, k):
    """The contract read literally: same segment, index != q, smallest (d2, index) by the project's d2 rule."""
    x = SO._xyz3(x)
    n = x.shape[0]
    seg = np.searchsorted(np.asarray(offsets, np.int64), np.arange(n), side="right") - 1
    idx = np.full((n, k), -1, np.int32)
    d2 = np.full((n, k), SO.FLT_MAX, np.float32)
    for q in range(n):
        cand = [(float(O.dist2(x[q], x[p])), p) for p in range(n) if p != q and seg[p] == seg[q]]
        cand.sort()
        for j, (d, p) in enumerate(cand[:k]):
            idx[q, j] = p
            d2[q, j] = d
    return idx, d2


def brute_radius(x, offsets, r):
    x = SO._xyz3(x)
    n = x.shape[0]
    seg = np.searchsorted(np.asarray(offsets, np.int64), np.arange(n), side="right") - 1
    r2 = np.float32(r) * np.float32(r)
    rows, idx, d2 = [0], [], []
    for q in range(n):
        cand = sorted((float(O.dist2(x[q], x[p])), p) for p in range(n) if p != q and seg[p] == seg[q])
        cand = [(d, p) for d, p in cand if np.float32(d) <= r2]
        idx += [p for _, p in cand]
        d2 += [d for d, _ in cand]
        rows.append(len(idx))
    return np.array(rows, np.int64), np.array(idx, np.int32), np.array(d2, np.float32)


def rng_cloud(n, seed, dim=3):
    return np.random.default_rng(seed).random((n, dim), dtype=np.float32)


def check(x, offsets, k=K, r=0.3):
    want_i, want_d = brute(x, offsets, k)
    got_i, got_d = SO.knn(x, offsets, k, squared=True)
    np.testing.assert_array_equal(got_i, want_i)
    np.testing.assert_array_equal(got_d.view(np.uint32), want_d.view(np.uint32))
    got_i2, got_s = SO.knn(x, offsets, k, squared=False)
    np.testing.assert_array_equal(got_i2, want_i)
    filled = want_i >= 0
    np.testing.assert_array_equal(got_s[filled], np.sqrt(want_d[filled]))
    wo, wi, wd = brute_radius(x, offsets, r)
    go, gi, gd = SO.radius_lists(x, offsets, r)
    np.testing.assert_array_equal(go, wo)
    np.testing.assert_array_equal(gi, wi)
    np.testing.assert_array_equal(gd.view(np.uint32), wd.view(np.uint32))
    np.testing.assert_array_equal(SO.range_count(x, offsets, r), np.diff(wo))


def test_uneven_sizes_with_empty_and_tiny_segments():
    sizes = [0, 1, 2, K, K + 1, 0, 9, 30, 0]
    check(rng_cloud(sum(sizes), 1), SO.offsets_of(sizes))


def test_identical_copies():
    c = rng_cloud(40, 2)
    x = np.concatenate([c] * 4)
    off = SO.offsets_of([40] * 4)
    check(x, off)
    idx, _ = SO.knn(x, off, K)
    for s in range(1, 4):  # every copy has the neighbours of the first, shifted
        np.testing.assert_array_equal(idx[40 * s:40 * (s + 1)], idx[:40] + 40 * s)


def test_coincident_points_across_a_boundary_are_not_neighbours():
    x = rng_cloud(24, 3)
    x[11] = x[12]  # last point of segment 0 == first point of segment 1
    x[13] = x[12]
    off = SO.offsets_of([12, 12])
    check(x, off)
    idx, d = SO.knn(x, off, K, squared=True)
    assert 12 not in idx[11] and 11 not in idx[12] and 11 not in idx[13]
    assert idx[12, 0] == 13 and d[12, 0] == 0


def test_two_dimensional():
    sizes = [3, 17, 1, 25]
    check(rng_cloud(sum(sizes), 4, dim=2), SO.offsets_of(sizes))


def test_batch_to_offsets_numpy():
    off = batch_to_offsets(np.array([0, 0, 2, 2, 2, 3], np.int64), 6)
    assert off.dtype == np.uint64
    np.testing.assert_array_equal(off, [0, 2, 2, 5, 6])
    np.testing.assert_array_equal(batch_to_offsets(np.array([1, 1, 1], np.int32), 3), [0, 0, 3])
    np.testing.assert_array_equal(batch_to_offsets(np.zeros(4, np.uint8), 4), [0, 4])


def test_batch_to_offsets_torch():
    torch = pytest.importorskip("torch")
    off = batch_to_offsets(torch.tensor([0, 1, 1, 3, 3, 3]), 6)
    assert off.dtype == torch.int64
    assert off.tolist() == [0, 1, 3, 3, 6]


@pytest.mark.parametrize("bad", [[0, 1, 0], [-1, 0, 0], [0.0, 1.0, 1.0], [[0, 0, 1]], [0, 0]])
def test_batch_to_offsets_errors(bad):
    with pytest.raises(ValueError):
        batch_to_offsets(np.array(bad), 3)


def test_batch_to_offsets_errors_torch():
    torch = pytest.importorskip("torch")
    with pytest.raises(ValueError):
        batch_to_offsets(torch.tensor([0, 2, 1]), 3)
    with pytest.raises(ValueError):
        batch_to_offsets(torch.tensor([-1, 0, 0]), 3)
