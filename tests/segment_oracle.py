"""CPU reference of segmented builds (tknn_build_segments, TrueKNN.build(batch=...)): the contract restated per segment
on the existing references.  Row q of a segmented search equals the unsegmented search of q's segment alone, with k'
= min(k, size - 1), the row padded with -1 / FLT_MAX, and the indices shifted by the segment's first offset (a shift
keeps the index order, so the (d2, index) tie-break is unchanged).  The radius lists restate the same way."""
import numpy as np

import radius_oracle as RO
from oracle import oracle as O

FLT_MAX = np.float32(np.finfo(np.float32).max)


def offsets_of(sizes):
    """Segment sizes -> the n_segments + 1 offsets (uint64)."""
    return np.concatenate([[0], np.cumsum(np.asarray(sizes, np.int64))]).astype(np.uint64)


def _xyz3(x):
    x = np.ascontiguousarray(x, dtype=np.float32)
    if x.shape[1] == 2:
        x = np.concatenate([x, np.zeros((x.shape[0], 1), np.float32)], axis=1)
    return np.ascontiguousarray(x[:, :3])


def knn(x, offsets, k, squared=False):
    """(idx [n, k] int32, dist [n, k] float32): sqrtf(d2), or d2 when squared."""
    x = _xyz3(x)
    n = x.shape[0]
    idx = np.full((n, k), -1, np.int32)
    dist = np.full((n, k), FLT_MAX, np.float32)
    off = np.asarray(offsets, np.int64)
    O.set_squared_output(squared)
    try:
        for s in range(len(off) - 1):
            a, b = int(off[s]), int(off[s + 1])
            kk = min(k, b - a - 1)
            if kk < 1:
                continue
            si, sd = O.knn_kdtree(x[a:b], kk)
            idx[a:b, :kk] = si + a
            dist[a:b, :kk] = sd
    finally:
        O.set_squared_output(False)
    return idx, dist


def radius_lists(x, offsets, r):
    """(offsets [n + 1] int64, idx int32, d2 float32) of tknn_radius_search after a segmented build."""
    x = _xyz3(x)
    off = np.asarray(offsets, np.int64)
    counts, idxs, d2s = [], [], []
    for s in range(len(off) - 1):
        a, b = int(off[s]), int(off[s + 1])
        if b == a:
            continue
        if b - a == 1:
            counts.append(np.zeros(1, np.int64))
            continue
        o, i, d = RO.radius_lists(x[a:b], r)
        counts.append(np.diff(o))
        idxs.append(i + np.int32(a))
        d2s.append(d)
    c = np.concatenate(counts) if counts else np.zeros(0, np.int64)
    rows = np.concatenate([[0], np.cumsum(c)]).astype(np.int64)
    idx = np.concatenate(idxs).astype(np.int32) if idxs else np.zeros(0, np.int32)
    d2 = np.concatenate(d2s).astype(np.float32) if d2s else np.zeros(0, np.float32)
    return rows, idx, d2


def range_count(x, offsets, r):
    o, _, _ = radius_lists(x, offsets, r)
    return np.diff(o).astype(np.uint32)
