"""Caller arrays on the host and on the device, and TKNN_OPT_KEEP_SCRATCH = 0.

Every entry point takes arrays that may be host or device memory: host inputs are staged on the device and host
outputs are written to a staging buffer and copied back.  Here every combination of host and device arrays of
tknn_brute_force, tknn_sort_pairs (pairs and keys only), tknn_morton_codes, tknn_generate_uniform, tknn_range_count and
tknn_query gives the same bits, the calls that count device->host bytes count exactly the staged ones, and the calls
that leave tknn_stats alone still do.  A context that releases its build, query, radius-list and interpolation scratch
after every call (keep_scratch = 0) computes the same bits and statistics as one that keeps it, twice in a row, so
released buffers grow back."""
import ctypes as C
import itertools

import numpy as np
import pytest
import torch

from owlraytracing_b200 import TrueKNN

pytestmark = pytest.mark.gpu


def _np(a):
    return a.cpu().numpy() if torch.is_tensor(a) else np.asarray(a)


def bits_equal(a, b, what):
    a, b = _np(a), _np(b)
    assert a.shape == b.shape and a.dtype == b.dtype, f"{what}: {a.shape} {a.dtype} vs {b.shape} {b.dtype}"
    if a.dtype == np.float32:
        a, b = a.view(np.uint32), b.view(np.uint32)
    bad = np.argwhere(a != b)
    assert bad.size == 0, f"{what}: {len(bad)} entries differ, first at {tuple(bad[0])}"


def untimed(stats):
    return {k: v for k, v in stats.items() if not k.endswith("_ms")}


def on(a, device):
    """a (numpy) as a host array or as a CUDA tensor, complete before the context's own stream reads it"""
    a = np.ascontiguousarray(a)
    if not device:
        return a.copy()
    t = torch.from_numpy(a.view({np.dtype(np.uint64): np.int64, np.dtype(np.uint32): np.int32}.get(a.dtype, a.dtype))).cuda()
    torch.cuda.synchronize()
    return t


def ptr(a):
    return None if a is None else C.c_void_p(a.data_ptr() if torch.is_tensor(a) else a.ctypes.data)


def sides(n):
    """every host (False) / device (True) assignment of n arrays"""
    return list(itertools.product((False, True), repeat=n))


def cloud(n, seed):
    return np.random.default_rng(seed).random((n, 3), dtype=np.float32)


def test_brute_force_host_and_device(knn):
    pts = cloud(50_000, 1)
    knn.build(pts)
    ids = np.random.default_rng(2).permutation(50_000)[:3_000].astype(np.int32)
    nq, k = ids.shape[0], 12
    want = None
    for ids_dev, idx_dev, dist_dev in sides(3):
        idx, dist = on(np.empty((nq, k), np.int32), idx_dev), on(np.empty((nq, k), np.float32), dist_dev)
        before = knn.stats()
        ids_in = on(ids, ids_dev)  # held while the library reads it
        knn._check(knn._L.tknn_brute_force(knn._h, ptr(ids_in), nq, k, ptr(idx), ptr(dist)))
        assert knn.stats() == before, "tknn_brute_force changed tknn_stats"
        if want is None:
            want = (_np(idx), _np(dist))
        bits_equal(idx, want[0], f"brute idx {ids_dev, idx_dev, dist_dev}")
        bits_equal(dist, want[1], f"brute dist {ids_dev, idx_dev, dist_dev}")


def test_sort_pairs_host_and_device(knn):
    rng = np.random.default_rng(3)
    n = 300_001
    keys = rng.integers(0, 1 << 40, n, dtype=np.uint64)  # many ties: a stable sort keeps value order
    keys[::3] = keys[0]
    vals = np.arange(n, dtype=np.uint32)
    order = np.argsort(keys, kind="stable")
    for keys_dev, vals_dev in sides(2):
        k_, v_ = on(keys, keys_dev), on(vals, vals_dev)
        before = knn.stats()
        knn._check(knn._L.tknn_sort_pairs(knn._h, ptr(k_), ptr(v_), n))
        assert knn.stats() == before, "tknn_sort_pairs changed tknn_stats"
        bits_equal(_np(k_).view(np.uint64), keys[order], f"sorted keys {keys_dev, vals_dev}")
        bits_equal(_np(v_).view(np.uint32), order.astype(np.uint32), f"sorted values {keys_dev, vals_dev}")
    for keys_dev in (False, True):
        k_ = on(keys, keys_dev)
        knn._check(knn._L.tknn_sort_pairs(knn._h, ptr(k_), None, n))
        bits_equal(_np(k_).view(np.uint64), keys[order], f"keys only {keys_dev}")


def test_morton_codes_host_and_device(knn):
    pts = np.random.default_rng(4).normal(size=(100_000, 4)).astype(np.float32)  # stride 4, dim 3
    box = np.float32([-5, -5, -5, 5, 5, 5])
    n = pts.shape[0]
    want = None
    for pts_dev, box_dev, out_dev in sides(3):
        out = on(np.empty(n, np.uint64), out_dev)
        before = knn.stats()
        pts_in, box_in = on(pts, pts_dev), on(box, box_dev)
        knn._check(knn._L.tknn_morton_codes(knn._h, ptr(pts_in), n, 3, 4, ptr(box_in), ptr(out)))
        assert knn.stats() == before, "tknn_morton_codes changed tknn_stats"
        got = _np(out).view(np.uint64)
        if want is None:
            want = got
        bits_equal(got, want, f"morton {pts_dev, box_dev, out_dev}")


def test_generate_uniform_host_and_device(knn):
    n = 123_457
    outs = []
    for dev in (False, True):
        out = on(np.empty((n, 3), np.float32), dev)
        before = knn.stats()
        knn._check(knn._L.tknn_generate_uniform(knn._h, 7, 1000, n, ptr(out)))
        assert knn.stats() == before, "tknn_generate_uniform changed tknn_stats"
        outs.append(_np(out))
    bits_equal(outs[1], outs[0], "generate_uniform")


def test_range_count_and_query_host_and_device(knn):
    pts = cloud(200_000, 5)
    knn.build(pts)
    n = pts.shape[0]
    counts = []
    for dev in (False, True):
        out = on(np.empty(n, np.uint32), dev)
        knn._check(knn._L.tknn_range_count(knn._h, C.c_float(0.01), ptr(out)))
        assert knn.stats()["d2h_bytes"] == (0 if dev else 4 * n)
        counts.append(_np(out).view(np.uint32))
    bits_equal(counts[1], counts[0], "range_count")

    rng = np.random.default_rng(6)
    nq, k = 20_000, 10
    q = rng.random((nq, 3), dtype=np.float32)
    sid = rng.integers(-1, n, nq).astype(np.int32)
    r2 = rng.uniform(-1e-4, 4e-4, nq).astype(np.float32)  # negative: no cap
    want = None
    for q_dev, sid_dev, r2_dev, idx_dev, dist_dev in sides(5):
        idx, dist = on(np.empty((nq, k), np.int32), idx_dev), on(np.empty((nq, k), np.float32), dist_dev)
        q_in, sid_in, r2_in = on(q, q_dev), on(sid, sid_dev), on(r2, r2_dev)
        knn._check(knn._L.tknn_query(knn._h, ptr(q_in), nq, 3, 3, ptr(sid_in), ptr(r2_in), k,
                                     C.c_float(0), ptr(idx), ptr(dist)))
        st = untimed(knn.stats())
        assert st["d2h_bytes"] == 4 * nq * k * ((not idx_dev) + (not dist_dev))
        st.pop("d2h_bytes")
        if want is None:
            want = (_np(idx), _np(dist), st)
        case = (q_dev, sid_dev, r2_dev, idx_dev, dist_dev)
        bits_equal(idx, want[0], f"query idx {case}")
        bits_equal(dist, want[1], f"query dist {case}")
        assert st == want[2], f"query stats {case}"


def sequence(t, rng_seed):
    """Builds, searches, queries, counts, radius lists, a segmented batch and interpolation on t; returns every output
    and the untimed statistics of every call."""
    rng = np.random.default_rng(rng_seed)
    pts = cloud(200_000, 8)
    dev_pts = torch.from_numpy(pts).cuda()
    got = []

    def keep(name, *arrays):
        got.append((name, [None if a is None else _np(a).copy() for a in arrays], untimed(t.stats())))

    t.build(pts)
    keep("build")
    keep("search host", *t.search(8))
    n = pts.shape[0]
    keep("search device", *t.search(8, out=(torch.empty((n, 8), dtype=torch.int32, device="cuda"),
                                            torch.empty((n, 8), dtype=torch.float32, device="cuda"))))
    q = pts[:30_000] + rng.normal(0, 1e-3, (30_000, 3)).astype(np.float32)
    sid = np.arange(30_000, dtype=np.int32)
    r2 = rng.uniform(-1e-4, 4e-4, 30_000).astype(np.float32)
    keep("query", *t.query(q, 6, self_ids=sid, init_radius2=r2))
    q_idx, q_d = t.query(q, 6)
    keep("query plain", q_idx, q_d)
    keep("range_count", t.range_count(0.01))
    keep("radius_search", *t.radius_search(0.008))
    keep("radius_query", *t.radius_query(q, 0.008, self_ids=sid))
    t.build(dev_pts)
    keep("build device")
    keep("radius_search device", *t.radius_search(0.008))

    sizes = [3_000, 0, 5_000, 1, 2_000]
    small = cloud(sum(sizes), 9)
    batch = np.repeat(np.arange(len(sizes)), sizes)
    t.build(small, batch=batch)
    keep("segmented build")
    keep("segmented search", *t.search(5))
    qs = cloud(4_000, 10)
    q_batch = np.sort(rng.integers(0, len(sizes), 4_000))
    keep("segmented query", *t.query(qs, 5, batch=q_batch))
    keep("segmented radius query", *t.radius_query(qs, 0.05, batch=q_batch))

    x = rng.normal(size=(n, 9)).astype(np.float32)
    keep("interpolate", *t.interpolate(q_idx, q_d * q_d, x))
    return got


def test_keep_scratch_off_matches_default():
    with TrueKNN(0, keep_scratch=0) as off, TrueKNN(0) as kept:
        for rep in range(2):  # the second pass runs on released (keep_scratch 0) and on grown buffers
            a, b = sequence(off, 12), sequence(kept, 12)
            assert [s[0] for s in a] == [s[0] for s in b]
            for (name, xs, st_a), (_, ys, st_b) in zip(a, b):
                for i, (x, y) in enumerate(zip(xs, ys)):
                    bits_equal(x, y, f"pass {rep}: {name} output {i}")
                assert st_a == st_b, f"pass {rep}: {name} statistics differ"
