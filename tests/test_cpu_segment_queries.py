"""The per-segment CPU reference of segmented query sets (tests/segment_query_oracle.py) against a direct brute force
with a same-segment mask, and batch_to_offsets with batch_size.  No GPU needed."""
import numpy as np
import pytest

import segment_query_oracle as SQ
from oracle import oracle as O
from owlraytracing_b200 import batch_to_offsets


def segment_ids(off, m):
    return np.searchsorted(np.asarray(off, np.int64), np.arange(m), side="right") - 1


def brute_rows(x, y, x_off, y_off, self_ids, caps2=None):
    """The contract read literally: per query, the (d2, index)-sorted list of data points of the same segment with index
    != self and d2 <= cap, by the project's d2 rule (oracle.dist2)."""
    x, y = SQ._xyz3(x), SQ._xyz3(y)
    sx, sy = segment_ids(x_off, len(x)), segment_ids(y_off, len(y))
    rows = []
    for j in range(len(y)):
        cand = [(np.float32(O.dist2(y[j], x[p])), p) for p in range(len(x)) if sx[p] == sy[j] and p != self_ids[j]]
        if caps2 is not None and caps2[j] >= 0:
            cand = [(d, p) for d, p in cand if d <= caps2[j]]
        rows.append(sorted(cand, key=lambda t: (float(t[0]), t[1])))
    return rows


@pytest.fixture(scope="module")
def case():
    """Empty data and query segments, a tiny data segment, duplicates across a boundary, self ids inside, outside and -1."""
    rng = np.random.default_rng(1)
    x_sizes = [30, 0, 1, 25, 4, 0, 40]
    y_sizes = [12, 5, 3, 0, 9, 6, 15]
    x = rng.random((sum(x_sizes), 3), dtype=np.float32)
    x[30 + 1] = x[3]  # a point of segment 2 coincident with one of segment 0
    y = rng.random((sum(y_sizes), 3), dtype=np.float32)
    y[:4] = x[:4]  # queries on data points: self exclusion matters
    x_off, y_off = SQ.offsets_of(x_sizes), SQ.offsets_of(y_sizes)
    self_ids = rng.integers(-1, len(x), size=len(y)).astype(np.int32)
    self_ids[:4] = np.arange(4)  # inside their data segment
    self_ids[4] = 31  # outside it (segment 2's point)
    self_ids[5] = -1
    return x, y, x_off, y_off, self_ids


@pytest.mark.parametrize("k", [1, 4, 30])
def test_knn_oracle_against_brute(case, k):
    x, y, x_off, y_off, sid = case
    caps = np.where(np.arange(len(y)) % 3 == 0, np.float32(0.1), np.float32(-1)).astype(np.float32)
    for cap in (None, caps):
        idx, d2 = SQ.knn(x, y, x_off, y_off, k, self_ids=sid, caps2=cap, squared=True)
        rows = brute_rows(x, y, x_off, y_off, sid, cap)
        for j, row in enumerate(rows):
            row = row[:k]
            np.testing.assert_array_equal(idx[j, : len(row)], [p for _, p in row])
            np.testing.assert_array_equal(d2[j, : len(row)].view(np.uint32), np.array([d for d, _ in row], np.float32).view(np.uint32))
            assert (idx[j, len(row):] == -1).all() and (d2[j, len(row):] == SQ.FLT_MAX).all()
    i2, d = SQ.knn(x, y, x_off, y_off, k, self_ids=sid)  # sqrtf(d2) form: the same rows
    wi, wd2 = SQ.knn(x, y, x_off, y_off, k, self_ids=sid, squared=True)
    np.testing.assert_array_equal(i2, wi)
    ok = wi >= 0
    np.testing.assert_array_equal(d[ok], np.sqrt(wd2[ok]))


def test_knn_oracle_segments_subset(case):
    x, y, x_off, y_off, sid = case
    full = SQ.knn(x, y, x_off, y_off, 4, self_ids=sid)
    part = SQ.knn(x, y, x_off, y_off, 4, self_ids=sid, segments=[0, 4])
    rows = np.r_[np.arange(y_off[0], y_off[1]), np.arange(y_off[4], y_off[5])].astype(np.int64)
    np.testing.assert_array_equal(part[0][rows], full[0][rows])
    rest = np.setdiff1d(np.arange(len(y)), rows)
    assert (part[0][rest] == -1).all()


@pytest.mark.parametrize("r", [0.0, 0.2, 0.5, np.inf])
def test_radius_oracle_against_brute(case, r):
    x, y, x_off, y_off, sid = case
    off, idx, d2 = SQ.radius_lists(x, y, x_off, y_off, r, self_ids=sid)
    r2 = np.float32(r) * np.float32(r)
    rows = [[(d, p) for d, p in row if d <= r2] for row in brute_rows(x, y, x_off, y_off, sid)]
    np.testing.assert_array_equal(np.diff(off), [len(row) for row in rows])
    np.testing.assert_array_equal(idx, [p for row in rows for _, p in row])
    np.testing.assert_array_equal(d2.view(np.uint32), np.array([d for row in rows for d, _ in row], np.float32).view(np.uint32))


def test_radius_oracle_without_self_ids(case):
    x, y, x_off, y_off, _ = case
    off, idx, _ = SQ.radius_lists(x, y, x_off, y_off, 0.3)
    rows = [[(d, p) for d, p in row if d <= np.float32(0.3) * np.float32(0.3)]
            for row in brute_rows(x, y, x_off, y_off, np.full(len(y), -1))]
    np.testing.assert_array_equal(idx, [p for row in rows for _, p in row])


def test_batch_to_offsets_batch_size():
    b = np.array([0, 0, 2, 2, 2])
    np.testing.assert_array_equal(batch_to_offsets(b, 5), [0, 2, 2, 5])
    np.testing.assert_array_equal(batch_to_offsets(b, 5, batch_size=5), [0, 2, 2, 5, 5, 5])
    np.testing.assert_array_equal(batch_to_offsets(b, 5, batch_size=3), [0, 2, 2, 5])
    assert batch_to_offsets(b, 5, batch_size=5).dtype == np.uint64
    np.testing.assert_array_equal(batch_to_offsets(np.zeros(0, np.int64), 0, batch_size=3), [0, 0, 0, 0])
    with pytest.raises(ValueError):
        batch_to_offsets(b, 5, batch_size=2)  # id 2 >= batch_size
    with pytest.raises(ValueError):
        batch_to_offsets(b, 5, batch_size=0)
    with pytest.raises(ValueError):
        batch_to_offsets(np.array([1, 0]), 2, batch_size=4)  # decreasing


def test_batch_to_offsets_batch_size_torch_cpu():
    torch = pytest.importorskip("torch")
    b = torch.tensor([0, 1, 1, 3])
    np.testing.assert_array_equal(batch_to_offsets(b, 4, batch_size=6).numpy(), [0, 1, 3, 3, 4, 4, 4])
    with pytest.raises(ValueError):
        batch_to_offsets(b, 4, batch_size=3)
