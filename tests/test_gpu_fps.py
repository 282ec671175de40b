"""Farthest point sampling on the GPU (tknn_fps, TrueKNN.fps, fps()): every case bit for bit against the CPU reference
(tests/fps_oracle.py), indices and distance bits, on both tiers (clouds of at most 14 336 points: one CTA each; larger:
the leaf-culled cooperative kernel), with the identities the contract states and every error code."""
import ctypes

import numpy as np
import pytest

import fps_oracle as F
from owlraytracing_b200 import MultiTrueKNN, TrueKNN, _lib, datasets, fps, radius
from owlraytracing_b200.trueknn import fps_counts

pytestmark = pytest.mark.gpu

CAP = 14336


def _np(a):
    return a.cpu().numpy() if hasattr(a, "cpu") else np.asarray(a)


def batch_of(sizes):
    return np.repeat(np.arange(len(sizes)), sizes).astype(np.int64)


def run(t, x, sizes, counts, starts=None, squared=True, plain=False):
    t.set_option("squared_dist", 1 if squared else 0)
    if plain:
        t.build(x)
    else:
        t.build(x, batch=batch_of(sizes), batch_size=len(sizes))
    return t.fps(num_samples=counts, start=starts, with_dist=True)


def assert_same(got, want, what, mask=None):
    gi, gd = _np(got[0]), _np(got[1])
    wi, wd = want
    if mask is not None:
        gi, gd, wi, wd = gi[mask], gd[mask], wi[mask], wd[mask]
    bad = np.flatnonzero(gi != wi)
    assert bad.size == 0, f"{what}: {bad.size} / {gi.size} samples differ, first at {bad[0]}: {gi[bad[0]]} vs {wi[bad[0]]}"
    bad = np.flatnonzero(gd.view(np.uint32) != wd.view(np.uint32))
    assert bad.size == 0, f"{what}: {bad.size} distances differ, first at {bad[0]}: {gd[bad[0]]} vs {wd[bad[0]]}"


def check(t, x, sizes, counts, starts=None, squared=True, limit=None, plain=False, what=""):
    got = run(t, x, sizes, counts, starts, squared, plain)
    want = F.fps(x, F.offsets_of(sizes), counts, starts, limit=limit, squared=squared)
    assert_same(got, want, what, None if limit is None else F.prefix_mask(counts, limit))
    return got


def non_increasing(dist, counts):
    d = _np(dist)
    off = F.offsets_of(counts).astype(np.int64)
    for s in range(len(counts)):
        seg = d[off[s] + 1: off[s + 1]]
        assert (np.diff(seg) <= 0).all(), f"cloud {s}: coverage radius increases"


@pytest.fixture(scope="module")
def clouds_4096():
    return datasets.uniform(1024 * 4096, seed=21), [4096] * 1024


@pytest.mark.parametrize("squared", [True, False])
def test_block_tier_1024_clouds(knn, clouds_4096, squared):
    x, sizes = clouds_4096
    counts = fps_counts(sizes, 0.25)
    got = check(knn, x, sizes, counts, squared=squared, what="1024 x 4096")
    st = knn.stats()
    assert st["rounds"] == 2 and st["round_queries"][0] == 1024 * 1024 and st["round_queries"][1] == 0
    non_increasing(got[1], counts)


def test_grid_tier_uniform(knn):
    x = datasets.uniform(300_000, seed=22)
    got = check(knn, x, [300_000], [6000], limit=1500, plain=True, what="uniform 300k")
    non_increasing(got[1], [6000])
    st = knn.stats()
    assert st["round_queries"][1] == 6000 and st["n_queries"] == 6000


def test_grid_tier_lidar(knn):
    x = datasets.lidar_like(200_000, seed=23)
    got = check(knn, x, [x.shape[0]], [3000], squared=False, limit=1200, plain=True, what="lidar 200k")
    non_increasing(got[1], [3000])


def test_grid_tier_lattice_ties(knn):
    x = datasets.lattice(40)  # 64 000 points, ties everywhere
    check(knn, x, [x.shape[0]], [2500], plain=True, what="lattice 40^3")
    x = datasets.lattice(25)
    check(knn, x, [x.shape[0]], [x.shape[0]], plain=True, what="lattice 25^3, every point")


def mixed():
    sizes = [CAP, CAP + 1, 0, 1, 5000, 20000, 3, 0, 40000, 64]
    counts = [CAP, 700, 0, 1, 0, 20000, 3, 0, 900, 1]
    x = datasets.uniform(sum(sizes), seed=24)
    return x, sizes, counts


@pytest.mark.parametrize("squared", [True, False])
def test_mixed_batch(knn, squared):
    x, sizes, counts = mixed()
    got = check(knn, x, sizes, counts, squared=squared, what="mixed")
    st = knn.stats()
    assert st["round_queries"][0] == CAP + 1 + 3 + 1 and st["round_queries"][1] == 700 + 20000 + 900
    non_increasing(got[1], counts)
    gi = _np(got[0])
    off = F.offsets_of(sizes).astype(np.int64)
    so = F.offsets_of(counts).astype(np.int64)
    assert sorted(gi[so[0]:so[1]].tolist()) == list(range(0, CAP))  # m = n: a permutation
    assert sorted(gi[so[5]:so[6]].tolist()) == list(range(off[5], off[6]))


def test_explicit_starts(knn):
    x, sizes, counts = mixed()
    rng = np.random.default_rng(9)
    off = F.offsets_of(sizes).astype(np.int64)
    starts = np.array([off[s] + rng.integers(0, max(n, 1)) for s, n in enumerate(sizes)], np.int32)
    got = check(knn, x, sizes, counts, starts=starts, what="mixed, explicit starts")
    so = F.offsets_of(counts).astype(np.int64)
    for s, m in enumerate(counts):
        if m:
            assert _np(got[0])[so[s]] == starts[s]


def test_device_and_host_arrays_and_stream(knn):
    torch = pytest.importorskip("torch")
    x, sizes, counts = mixed()
    want = F.fps(x, F.offsets_of(sizes), counts, squared=False)
    knn.set_option("squared_dist", 0)
    knn.build(torch.from_numpy(x).cuda(), batch=torch.from_numpy(batch_of(sizes)).cuda(), batch_size=len(sizes))
    got = knn.fps(num_samples=counts, with_dist=True)
    assert got[0].is_cuda and got[1].is_cuda
    assert_same(got, want, "device arrays")
    s = torch.cuda.Stream()
    with torch.cuda.stream(s):
        knn.set_stream(s.cuda_stream)
        idx = torch.empty(int(sum(counts)), dtype=torch.int32, device="cuda")
        dist = torch.empty(int(sum(counts)), dtype=torch.float32, device="cuda")
        knn.fps(num_samples=counts, out=(idx, dist))
        s.synchronize()
    knn.set_stream(None)
    assert_same((idx, dist), want, "torch stream")
    # host outputs from a device build, device offsets and starts through the C call
    L = _lib.load()
    soff = torch.from_numpy(F.offsets_of(counts).astype(np.int64)).cuda()
    starts = torch.from_numpy(F.offsets_of(sizes)[:-1].astype(np.int32)).cuda()
    hi = np.empty(int(sum(counts)), np.int32)
    hd = np.empty(int(sum(counts)), np.float32)
    torch.cuda.synchronize()
    assert L.tknn_fps(knn._h, ctypes.c_void_p(soff.data_ptr()), len(sizes), ctypes.c_void_p(starts.data_ptr()),
                      hi.ctypes.data, hd.ctypes.data) == _lib.OK
    assert_same((hi, hd), want, "host outputs, device offsets")
    assert L.tknn_fps(knn._h, ctypes.c_void_p(soff.data_ptr()), len(sizes), None, hi.ctypes.data, None) == _lib.OK
    np.testing.assert_array_equal(hi, want[0])


@pytest.mark.parametrize("leaf_size,curve", [(4, 0), (32, 1), (4, 1), (16, 0)])
def test_independent_of_build_options(leaf_size, curve):
    x, sizes, counts = mixed()
    want = F.fps(x, F.offsets_of(sizes), counts)
    with TrueKNN(0, leaf_size=leaf_size, curve=curve, sort_mode=1 if leaf_size == 16 else 0) as t:
        assert_same(run(t, x, sizes, counts), want, f"leaf {leaf_size} curve {curve}")
    y = datasets.uniform(100_000, seed=25)
    want = F.fps(y, None, [800])
    with TrueKNN(0, leaf_size=leaf_size, curve=curve, grid=2 if curve else 1) as t:
        assert_same(run(t, y, [100_000], [800], plain=True), want, f"plain, leaf {leaf_size} curve {curve}")


def test_repeated_calls_identical(knn):
    x, sizes, counts = mixed()
    a = run(knn, x, sizes, counts)
    b = knn.fps(num_samples=counts, with_dist=True)
    c = knn.fps(num_samples=counts, with_dist=True)
    for other in (b, c):
        np.testing.assert_array_equal(a[0], other[0])
        np.testing.assert_array_equal(a[1].view(np.uint32), other[1].view(np.uint32))


def test_batch_equals_alone(knn):
    x, sizes, counts = mixed()
    batch = run(knn, x, sizes, counts)
    off = F.offsets_of(sizes).astype(np.int64)
    so = F.offsets_of(counts).astype(np.int64)
    for s in (0, 1, 5, 8, 9):
        alone = run(knn, np.ascontiguousarray(x[off[s]:off[s + 1]]), [sizes[s]], [counts[s]], plain=True)
        np.testing.assert_array_equal(batch[0][so[s]:so[s + 1]], alone[0] + off[s])
        np.testing.assert_array_equal(batch[1][so[s]:so[s + 1]].view(np.uint32), alone[1].view(np.uint32))


def test_counters_same_samples(knn):
    x = datasets.uniform(200_000, seed=26)
    plain = run(knn, x, [200_000], [2000], plain=True)
    knn.set_option("counters", 1)
    counted = knn.fps(num_samples=[2000], with_dist=True)
    st = knn.stats()
    knn.set_option("counters", 0)
    np.testing.assert_array_equal(plain[0], counted[0])
    np.testing.assert_array_equal(plain[1].view(np.uint32), counted[1].view(np.uint32))
    leaves = knn.stats()["n_leaves"]
    assert 0 < st["warp_leaf_visits"] <= st["nodes_visited"] <= 1999 * leaves
    assert st["warp_leaf_visits"] < st["nodes_visited"]  # the cull skipped leaves
    assert st["points_tested"] >= st["warp_leaf_visits"]


def test_errors(knn):
    L = _lib.load()
    out_i = np.zeros(64, np.int32)
    out_d = np.zeros(64, np.float32)

    def call(ctx, soff, n_seg, starts=None, idx=out_i):
        s = None if starts is None else np.asarray(starts, np.int32).ctypes.data
        return L.tknn_fps(ctx._h, None if soff is None else np.asarray(soff, np.uint64).ctypes.data, n_seg, s,
                          None if idx is None else idx.ctypes.data, out_d.ctypes.data)

    assert call(knn, [0, 4], 1) == _lib.ESTATE  # before a build
    knn.build(datasets.uniform(30, seed=3), batch=batch_of([10, 0, 20]))
    assert call(knn, [0, 4, 4, 9], 3) == _lib.OK
    for bad in ([1, 4, 4, 9], [0, 4, 3, 9], [0, 11, 11, 12], [0, 4, 5, 9], [0, 4, 4, 25]):
        assert call(knn, bad, 3) == _lib.EINVAL, bad
    assert call(knn, None, 3) == _lib.EINVAL
    assert call(knn, [0, 4, 4, 9], 3, idx=None) == _lib.EINVAL
    assert call(knn, [0, 4, 9], 2) == _lib.EINVAL  # segment count mismatch
    assert call(knn, [0, 4, 4, 9], 3, starts=[0, 0, 10]) == _lib.OK
    assert call(knn, [0, 4, 4, 9], 3, starts=[0, 0, 9]) == _lib.EINVAL  # start outside its segment
    assert call(knn, [0, 4, 4, 9], 3, starts=[10, 0, 10]) == _lib.EINVAL
    assert call(knn, [0, 4, 4, 9], 3, starts=[-1, 0, 10]) == _lib.EINVAL
    assert call(knn, [0, 0, 0, 9], 3, starts=[-1, 77, 10]) == _lib.OK  # no samples: the start is not used
    with pytest.raises(ValueError):
        knn.fps(num_samples=[1, 2])
    with pytest.raises(ValueError):
        knn.fps(num_samples=[1, 0, 1], ratio=0.5)
    knn.build(datasets.uniform(30, seed=3))
    assert call(knn, [0, 30], 1) == _lib.OK and call(knn, [0, 4, 4, 9], 3) == _lib.EINVAL
    assert call(knn, [0, 31], 1) == _lib.EINVAL
    with MultiTrueKNN([0, 0], "partition") as m:
        m.build(datasets.uniform(4000, seed=4))
        assert call(m.rank(0), [0, 3], 1) == _lib.ESTATE


def test_fps_set_abstraction():
    torch = pytest.importorskip("torch")
    sizes = [4096] * 64 + [20000, 3, 0, 17]
    x = datasets.uniform(sum(sizes), seed=27)
    b = batch_of(sizes)
    idx = fps(x, b, 0.25, random_start=False, batch_size=len(sizes))
    counts = fps_counts(sizes, 0.25)
    want, _ = F.fps(x, F.offsets_of(sizes), counts)
    assert idx.dtype == np.int64
    np.testing.assert_array_equal(idx, want)
    xt, bt = torch.from_numpy(x).cuda(), torch.from_numpy(b).cuda()
    torch.manual_seed(5)
    it = fps(xt, bt, 0.25, random_start=True, batch_size=len(sizes))
    assert it.is_cuda and it.dtype == torch.int64 and it.shape[0] == int(counts.sum())
    torch.manual_seed(5)
    assert torch.equal(it, fps(xt, bt, 0.25, random_start=True, batch_size=len(sizes)))
    so = F.offsets_of(counts).astype(np.int64)
    starts = it.cpu().numpy()[so[:-1][counts > 0]].astype(np.int32)
    full_starts = F.offsets_of(sizes)[:-1].astype(np.int32)
    full_starts[counts > 0] = starts
    want_r, _ = F.fps(x, F.offsets_of(sizes), counts, full_starts)
    np.testing.assert_array_equal(it.cpu().numpy(), want_r)
    # one set abstraction step: the sampled centroids query the full cloud of their batch
    edges = radius(xt, xt[it], 0.1, bt, bt[it])
    assert edges.shape[0] == 2 and edges.shape[1] >= it.shape[0]
    assert bool((bt[edges[1]] == bt[it][edges[0]]).all())
    assert bool((edges[1][torch.cat([torch.ones(1, dtype=torch.bool, device="cuda"), edges[0][1:] != edges[0][:-1]])]
                 == it[edges[0].unique_consecutive()]).all())  # each centroid's nearest neighbour is itself


def test_readme_example():
    idx = fps(datasets.uniform(1024 * 4096), np.repeat(np.arange(1024), 4096), 0.25, random_start=False)
    assert idx.shape == (1048576,)
