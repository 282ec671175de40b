"""Every search of the library on the extreme clouds of tests/extreme_clouds.py, bit for bit against the CPU references
(indices, offsets and distance bits, in the d2 and the sqrt form; no tolerances).

The clouds put the fp32 rule where it gets awkward: +inf distances (some pairs, every pair, across clusters, from a query
outside the scene), an extent that overflows fp32 (curve-code scale 0), a normal cloud inside one curve cell beside an
outlier, subnormal and zero d2, signed zeros, exact ties from coarse ulps.  The builder, the leaf cut, the cell grid's
dense round (the grid cases route round 1 onto it and check tknn_stats::grid_rounds; test_gpu_grid_extreme.py covers both
grid kernels on every cloud), the query staging, the radius-list tiers, DBSCAN, both FPS tiers, segmented builds, feature kNN and every build option
run on them.  test_cpu_extreme_oracles.py checks the references themselves on the same clouds.
"""
import os
import subprocess
import sys

import numpy as np
import pytest

import dbscan_oracle as DO
import extreme_clouds as E
import feature_knn_oracle as FK
import fps_oracle as F
import radius_oracle as RO
import segment_oracle as SO
import segment_query_oracle as SQ
from oracle import oracle as O
from owlraytracing_b200 import TrueKNN
from test_cpu_extreme_oracles import radii_of

pytestmark = [pytest.mark.gpu, pytest.mark.filterwarnings("ignore:overflow encountered")]

U32 = np.uint32
FLT_MAX = np.float32(np.finfo(np.float32).max)
INF = np.float32(np.inf)
CAP = 14336  # FPS: clouds of at most this many points take the one-CTA tier, larger ones the leaf-culled grid tier


def _np(a):
    return a.cpu().numpy() if hasattr(a, "cpu") else np.asarray(a)


def same(got, want, what):
    g, w = _np(got), np.asarray(want)
    assert g.shape == w.shape, f"{what}: shape {g.shape} != {w.shape}"
    if w.dtype == np.float32:
        g, w = g.view(U32), w.view(U32)
    bad = np.flatnonzero(g.reshape(-1) != w.reshape(-1))
    assert bad.size == 0, f"{what}: {bad.size} / {w.size} entries differ, first at {bad[:8]}: " \
                          f"{_np(got).reshape(-1)[bad[:4]]} vs {np.asarray(want).reshape(-1)[bad[:4]]}"


def sqrt_form(d2):
    """dist_out without TKNN_OPT_SQUARED_DIST: sqrtf(d2), FLT_MAX padding kept."""
    return np.where(d2 == FLT_MAX, d2, np.sqrt(d2)).astype(np.float32)


def squared_oracle(fn, *a, **kw):
    O.set_squared_output(True)
    try:
        return fn(*a, **kw)
    finally:
        O.set_squared_output(False)


_KNN_REF = {}


def knn_ref(name, n, k=64):
    """(x, idx, d2) of the all-points kNN of a catalogue cloud; rows of smaller k are prefixes."""
    key = (name, n, k)
    if key not in _KNN_REF:
        x = E.cloud(name, n)
        i, d = squared_oracle(O.knn_kdtree, E.xyz3(x), k)
        _KNN_REF.clear()
        _KNN_REF[key] = (x, i, d)
    return _KNN_REF[key]


# ---------------------------------------------------------------- kNN: search and query on the uncovered families

KNN_FAMILIES = ["near_max", "outlier", "outlier_1e30", "mixed_scales", "far_clusters", "tiny_1e-21", "outlier_2d"]
KNN_N = {"near_max": 6000}


@pytest.mark.parametrize("k", [1, 10, 24, 25, 64])
@pytest.mark.parametrize("name", KNN_FAMILIES)
def test_knn(name, k):
    n = KNN_N.get(name, 20_000)
    x, ri, rd = knn_ref(name, n)
    ri, rd = ri[:, :k], rd[:, :k]
    q = E.cloud(name, 3000, seed=1)
    tree = O.KdTree(E.xyz3(x))
    try:
        qi, qd = squared_oracle(tree.query, E.xyz3(q), k)
    finally:
        tree.close()
    # grid = 2: the cell grid whenever its table is valid; warp_round_max = 0 keeps round 1 of these small clouds off the
    # warp-per-query kernel, so that it runs on grid_knn_kernel (k <= 24)
    for opts in ({"grid": 0}, {"grid": 2, "warp_round_max": 0}):
        grid = opts["grid"]
        with TrueKNN(0, **opts) as t:
            t.build(x)
            for squared in (1, 0):
                t.set_option("squared_dist", squared)
                form = (lambda d: d) if squared else sqrt_form
                what = f"{name} k={k} grid={grid} squared={squared}"
                i, d = t.search(k)
                same(i, ri, what + " search idx")
                same(d, form(rd), what + " search dist")
                if grid == 2:
                    st = t.stats()
                    assert st["grid_level"] > 0, what
                    assert st["grid_rounds"] & 1 if k <= 24 else st["grid_rounds"] == 0, f"{what}: {st['grid_rounds']:#x}"
                i, d = t.query(q, k)
                same(i, qi, what + " query idx")
                same(d, form(qd), what + " query dist")
            i, d = t.query(x, k, self_ids=np.arange(n, dtype=np.int32))
            same(i, ri, f"{name} k={k} grid={grid}: query of the built points")
    if name == "near_max":
        assert np.isposinf(rd).all()
        same(ri[:20], [[j for j in range(k + 1) if j != p][:k] for p in range(20)], "near_max: the k lowest indices")


@pytest.mark.parametrize("name", ["offset_1e4", "overflow_1e20", "far_clusters", "tiny_1e-21", "mixed_scales",
                                  "offset_1e6_2d"])
@pytest.mark.parametrize("k", [10, 25])
def test_queries_outside_the_scene(knn, name, k):
    """Queries at +-3e38: every d2 is +inf, so a row holds the k lowest indices; init_radius2 = FLT_MAX excludes +inf
    pairs, +inf and -1 (no cap) admit them, 0 admits nothing."""
    x = E.cloud(name, 20_000)
    dim = x.shape[1]
    rng = np.random.default_rng(3)
    far = (np.where(rng.random((200, dim)) < 0.5, -1.0, 1.0) * E.BIG).astype(np.float32)
    near = E.cloud(name, 200, seed=2)
    qs = np.concatenate([far, near, far[:50]]).astype(np.float32)
    caps = np.resize(np.array([FLT_MAX, INF, 0.0, -1.0, 1.0], np.float32), len(qs))
    knn.build(x)
    for squared in (1, 0):
        knn.set_option("squared_dist", squared)
        O.set_squared_output(bool(squared))
        try:
            want = O.knn_brute_queries(E.xyz3(x), E.xyz3(qs), k)
            want_c = O.knn_brute_queries(E.xyz3(x), E.xyz3(qs), k, caps2=caps)
        finally:
            O.set_squared_output(False)
        what = f"{name} k={k} squared={squared}"
        i, d = knn.query(qs, k)
        same(i, want[0], what + " idx")
        same(d, want[1], what + " dist")
        i, d = knn.query(qs, k, init_radius2=caps)
        same(i, want_c[0], what + " capped idx")
        same(d, want_c[1], what + " capped dist")
    same(want[0][:200], np.tile(np.arange(k, dtype=np.int32), (200, 1)), "far rows: the k lowest indices")
    assert np.isposinf(want[1][:200]).all()
    fmax_rows = np.flatnonzero(caps[:200] == FLT_MAX)
    assert (want_c[0][fmax_rows] == -1).all(), "a FLT_MAX cap excludes +inf pairs"


# ---------------------------------------------------------------- radius lists, range counts, DBSCAN

RADIUS_N = 2500


@pytest.fixture(scope="module")
def radius_clouds():
    out = {}
    for name in E.CLOUDS:
        x, _, d = knn_ref(name, RADIUS_N, 5)
        out[name] = (x, radii_of(d[:, 4]))
    return out


@pytest.mark.parametrize("name", sorted(E.CLOUDS))
def test_radius_lists_and_counts(knn, radius_clouds, name):
    x, radii = radius_clouds[name]
    q = E.cloud(name, 700, seed=4)
    knn.build(x)
    knn.set_option("squared_dist", 1)
    ki, kd = knn.search(5)
    for r in radii:
        what = f"{name} r={r!r}"
        want = RO.radius_lists(x, r)
        wq = RO.radius_lists(x, r, q)
        for squared in (1, 0):
            knn.set_option("squared_dist", squared)
            form = (lambda d: d) if squared else np.sqrt
            off, idx, dist = knn.radius_search(r)
            same(off, want[0], what + " offsets")
            same(idx, want[1], what + " idx")
            same(dist, form(want[2]), what + f" dist squared={squared}")
            off, idx, dist = knn.radius_query(q, r)
            same(off, wq[0], what + " query offsets")
            same(idx, wq[1], what + " query idx")
            same(dist, form(wq[2]), what + f" query dist squared={squared}")
        lens = np.diff(want[0])
        same(knn.range_count(r), lens.astype(np.uint32), what + " range count")
        rows = np.flatnonzero(lens >= 5)
        take = want[0][rows][:, None] + np.arange(5)[None, :]
        same(want[1][take], ki[rows], what + ": long rows start with the kNN row")
        same(want[2][take], kd[rows], what + ": ... and its distances")
    if name in ("near_max", "overflow_1e20", "far_clusters", "outlier", "mixed_scales"):
        n = len(x)
        assert RO.radius_lists(x, E.R_FIRST_INF)[0][-1] == n * (n - 1)


@pytest.mark.parametrize("name", sorted(E.CLOUDS))
def test_dbscan(knn, radius_clouds, name):
    x, radii = radius_clouds[name]
    knn.build(x)
    for r in radii:
        for m in (2, 5, 20):
            what = f"{name} eps={r!r} min_pts={m}"
            labels, core, c = knn.dbscan(r, m)
            wl, wc, wn = DO.dbscan(E.xyz3(x), r, m)
            assert c == wn, f"{what}: {c} clusters, want {wn}"
            same(core, wc, what + " core flags")
            same(labels, wl, what + " labels")


# ---------------------------------------------------------------- FPS, both tiers

def check_fps(t, x, m, what):
    t.build(x)
    for squared in (1, 0):
        t.set_option("squared_dist", squared)
        i, d = t.fps(num_samples=m, with_dist=True)
        wi, wd = F.fps(x, counts=[m], squared=bool(squared))
        same(i, wi, f"{what} squared={squared} idx")
        same(d, wd, f"{what} squared={squared} dist")
        st = t.stats()
        tier = 0 if len(x) <= CAP else 1
        assert st["round_queries"][tier] == m and st["round_queries"][1 - tier] == 0
    return wi, wd


@pytest.mark.parametrize("name", sorted(E.CLOUDS))
def test_fps_block_tier_every_point(knn, name):
    x = E.cloud(name, 3000)
    wi, wd = check_fps(knn, x, len(x), f"{name} m=n")
    if name == "near_max":
        same(wi, np.arange(len(x), dtype=np.int32), "near_max: index order")
        assert np.isposinf(wd[1:]).all()


@pytest.mark.parametrize("name", sorted(E.CLOUDS))
def test_fps_grid_tier(knn, name):
    x = E.cloud(name, 30_000)
    assert len(x) > CAP
    wi, wd = check_fps(knn, x, 3000, f"{name} n={len(x)}")
    if name == "near_max":
        same(wi, np.arange(3000, dtype=np.int32), "near_max: index order")
        assert np.isposinf(wd[1:]).all()


# ---------------------------------------------------------------- a batch of different families

BATCH = [("near_max", 1200), ("outlier", 1500), ("tiny_1e-21", 1200), ("empty", 0), ("mixed_scales", 1200),
         ("far_clusters", 1200), ("single", 1), ("offset_1e6", 1500), ("across_zero", 1000), ("overflow_1e20", 1200),
         ("outlier_1e30", 1200), ("offset_1e4", 2)]


def _batch(seed):
    parts = []
    for name, n in BATCH:
        if name == "empty":
            parts.append(np.zeros((0, 3), np.float32))
        elif name == "single":
            parts.append(np.full((1, 3), 1e20 * (1 + seed), np.float32))
        else:
            parts.append(E.cloud(name, n, seed))
    sizes = [len(p) for p in parts]
    return np.concatenate(parts).astype(np.float32), sizes


def test_batch_of_families(knn):
    x, sizes = _batch(0)
    q, qsizes = _batch(5)
    off, qoff = SO.offsets_of(sizes), SO.offsets_of(qsizes)
    batch = np.repeat(np.arange(len(sizes)), sizes)
    qbatch = np.repeat(np.arange(len(qsizes)), qsizes)
    knn.build(x, batch=batch, batch_size=len(sizes))
    for squared in (1, 0):
        knn.set_option("squared_dist", squared)
        for k in (10, 25):
            what = f"batch k={k} squared={squared}"
            wi, wd = SO.knn(x, off, k, squared=bool(squared))
            i, d = knn.search(k)
            same(i, wi, what + " knn graph idx")
            same(d, wd, what + " knn graph dist")
            wi, wd = SQ.knn(x, q, off, qoff, k, squared=bool(squared))
            i, d = knn.query(q, k, batch=qbatch)
            same(i, wi, what + " query idx")
            same(d, wd, what + " query dist")
        form = (lambda d: d) if squared else np.sqrt
        for r in (np.float32(0), np.float32(1e-3), E.R_LAST_FINITE, E.R_FIRST_INF):
            what = f"batch r={r!r} squared={squared}"
            want = SO.radius_lists(x, off, r)
            o, i, d = knn.radius_search(r)
            same(o, want[0], what + " radius graph offsets")
            same(i, want[1], what + " radius graph idx")
            same(d, form(want[2]), what + " radius graph dist")
            want = SQ.radius_lists(x, q, off, qoff, r)
            o, i, d = knn.radius_query(q, r, batch=qbatch)
            same(o, want[0], what + " radius query offsets")
            same(i, want[1], what + " radius query idx")
            same(d, form(want[2]), what + " radius query dist")
        counts = [s if s < 100 else s // 2 for s in sizes]
        i, d = knn.fps(num_samples=counts, with_dist=True)
        wi, wd = F.fps(x, off, counts, squared=bool(squared))
        same(i, wi, f"batch fps squared={squared} idx")
        same(d, wd, f"batch fps squared={squared} dist")


# ---------------------------------------------------------------- feature kNN

def features(kind, n, f=64, seed=0):
    rng = np.random.default_rng(seed)
    if kind == "overflow":  # rows at three scales: d2 finite between small rows, +inf where a huge row is involved
        scale = rng.choice([1.0, 1e17, E.BIG], size=(n, 1))
        return ((rng.random((n, f)) - 0.5) * 2 * scale).astype(np.float32)
    return (rng.random((n, f)) * 1e-21).astype(np.float32)  # "tiny": a subnormal accumulation


@pytest.mark.parametrize("kind", ["overflow", "tiny"])
@pytest.mark.parametrize("k", [16, 64])
def test_feature_knn(knn, kind, k):
    x = features(kind, 3000)
    y = features(kind, 1000, seed=1)
    sid = np.arange(len(x), dtype=np.int32)
    for squared in (1, 0):
        knn.set_option("squared_dist", squared)
        what = f"{kind} k={k} squared={squared}"
        i, d = knn.feature_knn(x, x, k, self_ids=sid)
        wi, wd = FK.knn(x, x, k, self_ids=sid, squared=bool(squared))
        same(i, wi, what + " all-points idx")
        same(d, wd, what + " all-points dist")
        i, d = knn.feature_knn(x, y, k)
        wi, wd = FK.knn(x, y, k, squared=bool(squared))
        same(i, wi, what + " query idx")
        same(d, wd, what + " query dist")
    wi, wd = FK.knn(x, x, k, self_ids=sid)
    if kind == "overflow":
        assert np.isposinf(wd).any() and np.isfinite(wd).any()
    else:
        assert ((wd > 0) & (wd < np.finfo(np.float32).tiny)).any(), "some d2 are subnormal"


def test_feature_knn_f3_equals_query(knn):
    x = E.cloud("overflow_1e20", 20_000)
    far = np.array([[E.BIG, -E.BIG, E.BIG], [-E.BIG, -E.BIG, -E.BIG]], np.float32)  # every d2 from these is +inf
    q = np.concatenate([E.cloud("overflow_1e20", 3000, seed=1), np.tile(far, (50, 1))]).astype(np.float32)
    knn.set_option("squared_dist", 1)
    for k in (10, 25):
        fi, fd = knn.feature_knn(x, q, k)
        qi, qd = knn.build(x).query(q, k)
        same(fi, qi, f"k={k}: feature kNN f=3 idx vs query")
        same(fd, qd, f"k={k}: feature kNN f=3 dist vs query")
        assert np.isposinf(qd).any()


# ---------------------------------------------------------------- every build option, one at a time

OPTIONS = [{"leaf_size": 4}, {"leaf_policy": 1}, {"curve": 1}, {"sort_mode": 1}, {"morton_bits": 4},
           {"tie_pruning": 1}, {"tie_pruning": 2}, {"approx_filter": 1, "counters": 1}, {"blocks_per_sm": 1},
           {"grid": 2}]


def outlier_with_duplicates(n):
    x = E.cloud("outlier", n - 1800)
    return np.concatenate([x[:n // 3], np.tile(x[7:8], (1500, 1)), np.tile(x[9:10], (300, 1)), x[n // 3:]])


OPTION_CLOUDS = {"outlier_dups": lambda: outlier_with_duplicates(20_000), "offset_1e6": lambda: E.cloud("offset_1e6", 20_000)}


def run_all(t, x, r, knn_only=False):
    t.set_option("squared_dist", 1)
    t.build(x)
    out = {}
    for k in (10, 25):
        out[f"search k={k}"] = t.search(k)
        out[f"grid_rounds k={k}"] = t.stats()["grid_rounds"]
    out["grid_level"] = t.stats()["grid_level"]
    if not knn_only:
        out["radius_search"] = t.radius_search(r)
        out["range_count"] = (t.range_count(r),)
        out["dbscan"] = t.dbscan(r, 5)
        out["fps"] = t.fps(num_samples=2000, with_dist=True)
    return out


@pytest.fixture(scope="module")
def option_refs():
    refs = {}
    for name, make in OPTION_CLOUDS.items():
        x = make()
        i, d = squared_oracle(O.knn_kdtree, x, 25)
        r = np.float32(np.median(np.sqrt(d[:, 4])))
        want = {"search k=10": (i[:, :10], d[:, :10]), "search k=25": (i, d),
                "radius_search": RO.radius_lists(x, r), "dbscan": DO.dbscan(x, r, 5),
                "fps": F.fps(x, counts=[2000])}
        want["range_count"] = (np.diff(want["radius_search"][0]).astype(np.uint32),)
        with TrueKNN(0) as t:
            default = run_all(t, x, r)
        refs[name] = (x, r, want, default)
    return refs


@pytest.mark.parametrize("opts", OPTIONS, ids=lambda o: ",".join(f"{k}={v}" for k, v in o.items()))
@pytest.mark.parametrize("name", sorted(OPTION_CLOUDS))
def test_build_options_change_no_result(option_refs, name, opts):
    x, r, want, default = option_refs[name]
    knn_only = "grid" in opts
    # grid = 2 with warp_round_max = 0: round 1 of these small clouds runs on the grid instead of one warp per query
    extra = {"warp_round_max": 0} if "grid" in opts else {}
    with TrueKNN(0, **opts, **extra) as t:
        got = run_all(t, x, r, knn_only)
        st = t.stats()
    for op, res in got.items():
        if op == "grid_level" or op.startswith("grid_rounds"):
            continue
        for j, (g, d, w) in enumerate(zip(res, default[op], want[op])):
            if w is None or isinstance(w, int):
                assert g == d == w, f"{name} {opts} {op}[{j}]"
                continue
            same(g, d, f"{name} {opts} {op}[{j}] vs the default build")
            same(g, w, f"{name} {opts} {op}[{j}] vs the reference")
    if "approx_filter" in opts:
        assert st["filter_violations"] == 0
    if "grid" in opts and name == "offset_1e6":
        assert got["grid_level"] > 0, "the cell grid was built"
    if "grid" in opts:  # outlier_dups has coincident-point leaves: no table, and the LBVH alone
        assert got["grid_rounds k=10"] & 1 if got["grid_level"] > 0 else got["grid_rounds k=10"] == 0
        assert got["grid_rounds k=25"] == 0


# ---------------------------------------------------------------- two ranks on one device

_MULTI = r"""
import sys
import numpy as np
import extreme_clouds as E
from oracle import oracle as O
from owlraytracing_b200 import MultiTrueKNN, TrueKNNError
x = E.cloud("outlier", 30000)
ri, rd = O.knn_kdtree(x, 10)
try:
    with MultiTrueKNN([0, 0], "partition") as m:
        i, d = m.build(x).search(10)
except TrueKNNError as e:
    print("refused:", e)
    sys.exit(0)
assert (i == ri).all(), "indices differ"
assert (d.view(np.uint32) == rd.view(np.uint32)).all(), "distances differ"
print("exact")
"""


def test_partitioned_outlier_returns():
    """A point-partitioned build of a cloud whose extent overflows a rank's frame either answers exactly or refuses;
    it must return either way (run in a child process, so that a hang fails the test instead of the suite)."""
    here = os.path.dirname(os.path.abspath(__file__))
    env = dict(os.environ, PYTHONPATH=os.pathsep.join([here, os.path.dirname(here), os.environ.get("PYTHONPATH", "")]))
    r = subprocess.run([sys.executable, "-c", _MULTI], cwd=here, env=env, capture_output=True, text=True, timeout=300)
    assert r.returncode == 0, r.stdout[-2000:] + r.stderr[-4000:]
    assert r.stdout.startswith(("exact", "refused:")), r.stdout
