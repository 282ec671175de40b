"""CPU reference of segmented query sets (tknn_query_segments, tknn_radius_query_segments, TrueKNN.query(batch=...),
TrueKNN.radius_query(batch=...)): the contract restated per segment on the existing references.  Query segment s
searches data segment s alone; a self id inside the data segment is mapped to its local index, one outside (or -1)
excludes nothing, and the indices are shifted back by the data segment's first offset (a shift keeps the index order,
so the (d2, index) tie-break is unchanged).  Rows with fewer eligible points end in -1 / FLT_MAX."""
import numpy as np

import radius_oracle as RO
from oracle import oracle as O
from segment_oracle import FLT_MAX, _xyz3, offsets_of  # noqa: F401  (offsets_of: re-exported for the tests)


def _local_self(self_ids, c, d, a, b):
    if self_ids is None:
        return None
    sid = np.asarray(self_ids, np.int64)[c:d]
    return np.where((sid >= a) & (sid < b), sid - a, -1).astype(np.int32)


def knn(x, y, x_off, y_off, k, self_ids=None, caps2=None, squared=False, segments=None):
    """(idx [nq, k] int32, dist [nq, k] float32: sqrtf(d2), or d2 when squared) of tknn_query_segments.  segments: the
    query segments to compute (default all); the rows of the others stay -1 / FLT_MAX."""
    x, y = _xyz3(x), _xyz3(y)
    xo, yo = np.asarray(x_off, np.int64), np.asarray(y_off, np.int64)
    idx = np.full((y.shape[0], k), -1, np.int32)
    dist = np.full((y.shape[0], k), FLT_MAX, np.float32)
    O.set_squared_output(squared)
    try:
        for s in (range(len(xo) - 1) if segments is None else segments):
            a, b, c, d = int(xo[s]), int(xo[s + 1]), int(yo[s]), int(yo[s + 1])
            if d == c or b == a:
                continue
            kk = min(k, b - a)
            local = _local_self(self_ids, c, d, a, b)
            if caps2 is None:  # the exact kd-tree (bit-identical to the brute force) keeps large batches fast
                tree = O.KdTree(x[a:b])
                try:
                    si, sd = tree.query(y[c:d], kk, self_ids=local)
                finally:
                    tree.close()
            else:
                si, sd = O.knn_brute_queries(x[a:b], y[c:d], kk, local, caps2=np.asarray(caps2, np.float32)[c:d])
            idx[c:d, :kk] = np.where(si >= 0, si + a, -1)
            dist[c:d, :kk] = sd
    finally:
        O.set_squared_output(False)
    return idx, dist


def radius_lists(x, y, x_off, y_off, r, self_ids=None):
    """(offsets [nq + 1] int64, idx int32, d2 float32) of tknn_radius_query_segments."""
    x, y = _xyz3(x), _xyz3(y)
    xo, yo = np.asarray(x_off, np.int64), np.asarray(y_off, np.int64)
    counts, idxs, d2s = [], [], []
    for s in range(len(xo) - 1):
        a, b, c, d = int(xo[s]), int(xo[s + 1]), int(yo[s]), int(yo[s + 1])
        if d == c:
            continue
        if b == a:
            counts.append(np.zeros(d - c, np.int64))
            continue
        o, i, dd = RO.radius_lists(x[a:b], r, queries=y[c:d], self_ids=_local_self(self_ids, c, d, a, b))
        counts.append(np.diff(o))
        idxs.append(i + np.int32(a))
        d2s.append(dd)
    cnt = np.concatenate(counts) if counts else np.zeros(0, np.int64)
    rows = np.concatenate([[0], np.cumsum(cnt)]).astype(np.int64)
    idx = np.concatenate(idxs).astype(np.int32) if idxs else np.zeros(0, np.int32)
    d2 = np.concatenate(d2s).astype(np.float32) if d2s else np.zeros(0, np.float32)
    return rows, idx, d2
