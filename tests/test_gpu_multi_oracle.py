"""The multi-GPU drivers (csrc/dist.cu) on one GPU, bit for bit against the CPU oracle at the edges of the fp32 rule.

A device list naming device 0 several times runs that many ranks on it over the in-process transport.  Indices and
distance bits are compared with the exact kd-tree reference (no tolerances) on the extreme catalogue of
tests/extreme_clouds.py, on ties that straddle rank borders (lattice shells split by k, coarse-ulp offsets), at k
beyond the small-k kernels (the heap kernel in the local search and in the remote capped query, many merges per row),
under every build option, with 2-column and padded inputs, and into host, device and unaligned outputs.  The routing
of boundary queries is checked against the point rule of test_cpu_reach_model.py, whose split of the cloud into
ranks must be the driver's.
"""
import threading

import numpy as np
import pytest

import extreme_clouds as E
import test_cpu_reach_model as RM
from oracle import oracle as O
from owlraytracing_b200 import MultiTrueKNN, TrueKNNError, _lib, datasets
from test_cpu_grid_model import dist2

pytestmark = [pytest.mark.gpu, pytest.mark.filterwarnings("ignore:overflow encountered"),
              pytest.mark.filterwarnings("ignore:invalid value encountered")]

U32 = np.uint32
FLT_MAX = np.float32(np.finfo(np.float32).max)
N = 20_000


def sqrt_form(d2):
    """dist_out without TKNN_OPT_SQUARED_DIST: sqrtf(d2), FLT_MAX padding kept."""
    return np.where(d2 == FLT_MAX, d2, np.sqrt(d2)).astype(np.float32)


def squared_oracle(fn, *a, **kw):
    O.set_squared_output(True)
    try:
        return fn(*a, **kw)
    finally:
        O.set_squared_output(False)


_REF = {}


def ref(key, make, k):
    """(x, idx, d2) of the all-points kNN of a cloud, cached per key; rows of smaller k are prefixes."""
    if key not in _REF or _REF[key][1].shape[1] < k:
        x = make()
        i, d = squared_oracle(O.knn_kdtree, E.xyz3(x), k)
        _REF[key] = (x, i, d)
    return _REF[key]


def rows_equal(idx, dist, ref_i, ref_d, what, squared=False):
    """Every row identical: indices, and the distance bits of sqrtf(d2) (or d2)."""
    idx, dist = np.asarray(idx), np.asarray(dist)
    want = ref_d if squared else sqrt_form(ref_d)
    assert idx.shape == ref_i.shape, (what, idx.shape, ref_i.shape)
    bad = (idx != ref_i).any(1) | (dist.view(U32) != want.view(U32)).any(1)
    if bad.any():
        r = np.flatnonzero(bad)[0]
        raise AssertionError(f"{what}: {bad.sum()} of {len(bad)} rows differ; row {r}: got {idx[r]} {dist[r]}, "
                             f"want {ref_i[r]} {want[r]}")


def _run_ranks(m, fn):
    """Drive the per-rank C ABI from one Python thread per rank (ctypes releases the GIL); a hang fails the test."""
    out, err = [None] * m.n_ranks, [None] * m.n_ranks

    def body(r):
        try:
            out[r] = fn(r, m.rank(r))
        except Exception as e:  # noqa: BLE001
            err[r] = e

    th = [threading.Thread(target=body, args=(r,)) for r in range(m.n_ranks)]
    for t in th:
        t.start()
    for t in th:
        t.join(timeout=300)
    assert all(not t.is_alive() for t in th), "a rank hangs"
    for e in err:
        if e is not None:
            raise e
    return out


def _owned_min(x, ranks):
    owner = RM.split(x, ranks)
    return 0 if owner is None else int(np.bincount(owner, minlength=ranks).min())


def _still_usable(m):
    x = datasets.uniform(6000, seed=2)
    i, d = m.build(x).search(4)
    ri, rd = squared_oracle(O.knn_kdtree, x, 4)
    rows_equal(i, d, ri, rd, "a normal cloud after a refusal")


# ---------------------------------------------------------------- the extreme catalogue

@pytest.mark.parametrize("name", sorted(E.CLOUDS))
def test_catalogue_partitioned(name):
    """Every catalogue cloud at 2, 3 and 5 ranks, k in {1, 4, 10, 25}: exact, or refused (TKNN_EINVAL) exactly when the
    cell-aligned split leaves a rank with fewer than 2 points (build) or no more than k (search)."""
    x, ri, rd = ref(name, lambda: E.cloud(name, N), 25)
    for ranks in (2, 3, 5):
        owned = _owned_min(x, ranks)
        with MultiTrueKNN([0] * ranks, "partition") as m:
            try:
                m.build(x)
            except TrueKNNError as e:
                assert e.code == _lib.EINVAL and owned < 2, (name, ranks, owned, str(e))
                _still_usable(m)
                continue
            assert owned >= 2, (name, ranks, "the split leaves a rank with < 2 points, yet the build succeeded")
            for k in (1, 4, 10, 25):
                if owned <= k:
                    with pytest.raises(TrueKNNError) as e:
                        m.search(k)
                    assert e.value.code == _lib.EINVAL
                    continue
                i, d = m.search(k)
                rows_equal(i, d, ri[:, :k], rd[:, :k], f"{name} partition x{ranks} k={k}")


@pytest.mark.parametrize("name", sorted(E.CLOUDS))
def test_catalogue_sharded(name):
    x, ri, rd = ref(name, lambda: E.cloud(name, N), 25)
    for ranks in (2, 3):
        with MultiTrueKNN([0] * ranks, "shard") as m:
            m.build(x)
            for k in (1, 10, 25):
                i, d = m.search(k)
                rows_equal(i, d, ri[:, :k], rd[:, :k], f"{name} shard x{ranks} k={k}")


def test_refusals_reach_every_rank():
    """A build the split cannot serve (near_max: one curve cell) and a search with k >= a rank's points are refused by
    every rank with TKNN_EINVAL, and the handle then builds and searches a normal cloud."""
    x = E.cloud("near_max", 6000)
    with MultiTrueKNN([0] * 3, "partition") as m:
        def build(r, eng):
            lo, hi = len(x) * r // 3, len(x) * (r + 1) // 3
            try:
                eng.partition_build(x[lo:hi], lo)
            except TrueKNNError as e:
                return e.code
            return 0

        assert _run_ranks(m, build) == [_lib.EINVAL] * 3
        _still_usable(m)
        small = datasets.uniform(64, seed=3)

        def search(r, eng):
            eng.partition_build(small[16 * r:16 * (r + 1)], 16 * r)
            try:
                eng.partition_search(40)
            except TrueKNNError as e:
                return e.code
            return 0

        assert _run_ranks(m, search) == [_lib.EINVAL] * 3
        _still_usable(m)


# ---------------------------------------------------------------- ties across rank borders, large k

TIE_CLOUDS = {"lattice28": lambda: datasets.lattice(28), "offset_1e6": lambda: E.cloud("offset_1e6", N)}


@pytest.mark.parametrize("ranks", [2, 4, 7])
@pytest.mark.parametrize("name", sorted(TIE_CLOUDS))
def test_ties_across_rank_borders(name, ranks):
    """k = 7, 19, 27 split the lattice's 2nd, 3rd and 4th shells (12, 8 and 6 tied points): the remote capped search must
    return the points tied exactly at the cap, in global-index order, and the merge must keep the lower indices."""
    x, ri, rd = ref(name, TIE_CLOUDS[name], 28)
    with MultiTrueKNN([0] * ranks, "partition") as m:
        m.build(x)
        for k in (7, 19, 27):
            i, d = m.search(k)
            sent = sum(m.rank(r).dist_stats()["boundary_sent"] for r in range(ranks))
            assert sent > 0
            rows_equal(i, d, ri[:, :k], rd[:, :k], f"{name} partition x{ranks} k={k}")
    if name == "lattice28":
        assert all((rd[:, k - 1] == rd[:, k]).any() for k in (7, 19, 27)), "k does not split a shell"


LARGE = {"uniform": lambda: datasets.uniform(40_000, seed=21), "lidar": lambda: datasets.lidar_like(40_000, seed=9)}


@pytest.mark.parametrize("mode", ["partition", "shard"])
@pytest.mark.parametrize("kind", sorted(LARGE))
def test_large_k(kind, mode):
    x, ri, rd = ref(kind, LARGE[kind], 200)
    with MultiTrueKNN([0] * 3, mode) as m:
        m.build(x)
        for k in (24, 25, 64, 200):
            i, d = m.search(k)
            rows_equal(i, d, ri[:, :k], rd[:, :k], f"{kind} {mode} x3 k={k}")


# ---------------------------------------------------------------- build options

# {"grid": 2} builds the cell table on every rank, but covers no grid kernel: each rank's local search of about 7 000
# queries runs one warp per query (below warp_round_max), and test_gpu_grid_extreme.py covers the kernels themselves
OPTIONS = [{"squared_dist": 1}, {"grid": 2}, {"tie_pruning": 0}, {"tie_pruning": 1}, {"tie_pruning": 2},
           {"leaf_size": 4}, {"leaf_policy": 1}, {"curve": 1}, {"sort_mode": 1}, {"blocks_per_sm": 1},
           {"approx_filter": 1, "counters": 1}]
OPTION_CLOUDS = {"lattice28": lambda: datasets.lattice(28), "tiny_1e-21": lambda: E.cloud("tiny_1e-21", N)}


@pytest.mark.parametrize("opts", OPTIONS, ids=lambda o: ",".join(f"{k}={v}" for k, v in o.items()))
@pytest.mark.parametrize("name", sorted(OPTION_CLOUDS))
def test_options_change_no_result(name, opts):
    x, ri, rd = ref(name, OPTION_CLOUDS[name], 19)
    with MultiTrueKNN([0] * 3, "partition") as m:
        for key, v in opts.items():
            m.set_option(key, v)
        m.build(x)
        for k in (1, 7, 19):
            i, d = m.search(k)
            rows_equal(i, d, ri[:, :k], rd[:, :k], f"{name} {opts} k={k}", squared="squared_dist" in opts)
        if "approx_filter" in opts:
            assert all(m.rank(r).stats()["filter_violations"] == 0 for r in range(3))


# ---------------------------------------------------------------- inputs and outputs

def test_two_columns_and_padded_stride():
    x3 = datasets.uniform(N, seed=4)
    x2 = np.ascontiguousarray(x3[:, :2])
    pad = np.concatenate([x3, np.full((N, 2), np.nan, np.float32)], 1)   # stride 5: the padding must never be read
    for what, x, dim, pts in (("2 columns", x2, 2, E.xyz3(x2)), ("stride 5", pad, 3, x3)):
        _, ri, rd = ref(what, lambda: pts, 10)
        for mode in ("partition", "shard"):
            with MultiTrueKNN([0] * 3, mode) as m:
                i, d = m.build(x, dim=dim).search(10)
                rows_equal(i, d, ri, rd, f"{what} {mode}")
        with MultiTrueKNN([0] * 3, "partition") as m:
            def work(r, eng):
                lo, hi = N * r // 3, N * (r + 1) // 3
                eng.partition_build(x[lo:hi], lo, dim=dim)
                return eng.partition_search(10)

            for gid, i, d in _run_ranks(m, work):
                rows_equal(i, d, ri[gid], rd[gid], f"{what} per rank")


def test_partition_search_outputs():
    """Host arrays, CUDA tensors, and distance arrays one float past a 16-byte boundary (host, and device: the scalar
    path of sqrt_rows_kernel); the owned rows are the model's split."""
    import torch

    name, k, ranks = "tiny_1e-21", 10, 3
    x, ri, rd = ref(name, lambda: E.cloud(name, N), 25)
    owner = RM.split(x, ranks)
    with MultiTrueKNN([0] * ranks, "partition") as m:
        def work(r, eng):
            lo, hi = N * r // ranks, N * (r + 1) // ranks
            eng.partition_build(x[lo:hi], lo)
            n = eng.partition_owned()
            res = {"default": eng.partition_search(k)}
            res["host"] = eng.partition_search(k, out=(np.empty(n, np.int32), np.empty((n, k), np.int32),
                                                       np.empty((n, k), np.float32)))
            buf = np.empty(n * k + 1, np.float32)
            res["host unaligned"] = eng.partition_search(k, out=(np.empty(n, np.int32), np.empty((n, k), np.int32),
                                                                 buf[1:].reshape(n, k)))
            dev = torch.empty(n * k + 1, dtype=torch.float32, device="cuda")
            res["device"] = eng.partition_search(k, out=(torch.empty(n, dtype=torch.int32, device="cuda"),
                                                         torch.empty((n, k), dtype=torch.int32, device="cuda"),
                                                         torch.empty((n, k), dtype=torch.float32, device="cuda")))
            res["device unaligned"] = eng.partition_search(k, out=(torch.empty(n, dtype=torch.int32, device="cuda"),
                                                                   torch.empty((n, k), dtype=torch.int32, device="cuda"),
                                                                   dev[1:].view(n, k)))
            assert dev[1:].data_ptr() % 16 == 4
            return {w: tuple(a.cpu().numpy() if hasattr(a, "cpu") else np.asarray(a) for a in v) for w, v in res.items()}

        out = _run_ranks(m, work)
    for r, res in enumerate(out):
        gid = res["default"][0]
        assert np.array_equal(np.sort(gid), np.flatnonzero(owner == r)), f"rank {r} owns other points than the split model"
        for what, (g, i, d) in res.items():
            assert np.array_equal(g, gid), what
            rows_equal(i, d, ri[g, :k], rd[g, :k], f"rank {r} {what}")


# ---------------------------------------------------------------- partition_verify

@pytest.mark.parametrize("name,k", [("tiny_1e-21", 10), ("lattice28", 7)])
def test_partition_verify(name, k):
    """0 bad with every row of the smallest rank sampled (samples must match across ranks); one flipped distance bit,
    and two tied entries swapped out of index order, are each flagged once."""
    x, ri, rd = ref(name, OPTION_CLOUDS[name], 19)
    ranks = 3
    samples = _owned_min(x, ranks)
    with MultiTrueKNN([0] * ranks, "partition") as m:
        def work(r, eng):
            lo, hi = len(x) * r // ranks, len(x) * (r + 1) // ranks
            eng.partition_build(x[lo:hi], lo)
            gid, idx, dist = eng.partition_search(k)
            ok = eng.partition_verify(k, samples, gid, idx, dist)
            rows = [len(gid) * t // samples for t in range(samples)]
            row = rows[1]
            if r == 1:
                dist.view(U32)[row, k - 1] ^= 1
            flipped = eng.partition_verify(k, samples, gid, idx, dist)
            if r == 1:
                dist.view(U32)[row, k - 1] ^= 1
            tie = next((t, j) for t in rows for j in range(k - 1) if dist[t, j] == dist[t, j + 1])
            if r == 1:
                idx[tie[0], [tie[1], tie[1] + 1]] = idx[tie[0], [tie[1] + 1, tie[1]]]
            swapped = eng.partition_verify(k, samples, gid, idx, dist)
            return ok, flipped, swapped

        res = _run_ranks(m, work)
    for ok, flipped, swapped in res:
        assert ok == (ranks * samples, 0)
        assert flipped == (ranks * samples, 1)
        assert swapped == (ranks * samples, 1)


# ---------------------------------------------------------------- the reach kernel under the point rule

@pytest.mark.parametrize("ranks,k", [(2, 1), (4, 1), (4, 4)])
def test_reach_mask_flags_every_rank_a_point_needs(knn, ranks, k):
    """tknn_reach_mask on summaries of real points of the 1e-21 cloud: every rank holding a point p with the fp32
    dist2(q, p) <= r2 (r2 = q's local k-th d2, often 0 or subnormal) is flagged."""
    import torch

    x = RM.MODEL_CLOUDS["tiny_1e-21"]()
    lo, hi, _ = RM.frame(x)
    box6 = np.concatenate([lo, hi]).astype(np.float32)
    owner = RM.split(x, ranks)
    summ, _ = RM.summaries(x, owner, ranks, RM.frame(x))
    summ_d = torch.from_numpy(summ.reshape(ranks, -1)).cuda()
    missed, needed = 0, 0
    for r in range(ranks):
        qi = np.flatnonzero(owner == r)
        need = np.zeros(len(qi), np.int64)
        r2 = np.empty(len(qi), np.float32)
        for b in range(0, len(qi), 512):
            q = qi[b:b + 512]
            d = dist2(x[q][:, None, :], x[None, :, :])
            local = np.where(owner[None, :] == r, d, np.float32(np.inf))
            local[np.arange(len(q)), q] = np.inf
            r2[b:b + 512] = np.partition(local, k - 1, axis=1)[:, k - 1]
            for s in range(ranks):
                if s != r:
                    hit = ((d <= r2[b:b + 512, None]) & (owner[None, :] == s)).any(1)
                    need[b:b + 512] |= hit.astype(np.int64) << s
        got = knn.reach_mask(torch.from_numpy(x[qi]).cuda(), torch.from_numpy(r2).cuda(), box6, summ_d, r, 3)
        got = got.cpu().numpy().astype(np.int64) & ((1 << ranks) - 1)
        missed += int(((need & ~got) != 0).sum())
        needed += int((need != 0).sum())
    assert needed > 0
    assert missed == 0, f"{missed} of {needed} rows that need a remote rank do not flag it"
