"""The Python wrapper's calls into libtrueknn, traced through a recording fake of the library (no GPU, no build).

Every case runs a public method or module function and compares the tknn_* calls it made: their names, their scalar
arguments and, for every pointer, NULL or which input or output array it addresses ("ptr" for a staged copy or a
wrapper-made array such as batch offsets).  The arrays that come back are compared by type, dtype and shape.  Methods
that take arrays run with numpy input and with CPU torch tensors (which the wrapper passes like CUDA tensors, zero-copy).
"""
import ctypes as C

import numpy as np
import pytest

from owlraytracing_b200 import _lib
from owlraytracing_b200 import trueknn as T

torch = pytest.importorskip("torch")

HANDLE = 0x5A00  # the fake's context handle
COUNT = 3  # what every uint64 out-parameter receives
CAPACITY = 4  # what tknn_shard_capacity and tknn_partition_owned return
_BYREF = type(C.byref(C.c_int()))


class FakeLib:
    """Records (name, args) of every tknn_* call, returns TKNN_OK and fills the out-parameters."""

    def __init__(self):
        self.calls = []
        self.hooks = {}

    def __getattr__(self, name):
        if not name.startswith("tknn_"):
            raise AttributeError(name)

        def call(*args):
            self.calls.append((name, args))
            if name in ("tknn_shard_capacity", "tknn_partition_owned"):
                return CAPACITY
            if name == "tknn_multi_ctx":
                return HANDLE
            for a in args:
                obj = getattr(a, "_obj", None)
                if isinstance(obj, C.c_uint64):
                    obj.value = COUNT
                elif isinstance(obj, C.c_void_p):
                    obj.value = HANDLE
            if name in self.hooks:
                self.hooks[name](*args)
            return 0

        return call


@pytest.fixture()
def fake(monkeypatch):
    f = FakeLib()
    monkeypatch.setattr(_lib, "load", lambda: f)
    return f


@pytest.fixture()
def t(fake):
    ctx = T.TrueKNN(0)
    fake.calls.clear()
    yield ctx
    ctx.close()


def _addr(a):
    return a.data_ptr() if T._is_tensor(a) else a.ctypes.data


def trace(fake, **arrays):
    """The recorded calls with pointers named after `arrays` (None = NULL, "ctx" = the context), then forgotten."""
    names = {}
    for name, a in arrays.items():
        if a is not None and _addr(a):
            names.setdefault(_addr(a), name)

    def arg(a):
        if a is None:
            return None
        if isinstance(a, C.c_void_p):
            if not a.value:
                return None
            if a.value < 0x1000:  # a stream handle such as cudaStreamLegacy
                return a.value
            return "ctx" if a.value == HANDLE else names.get(a.value, "ptr")
        if isinstance(a, C.c_float):
            return float(a.value)
        if isinstance(a, _BYREF):
            return "&"
        if isinstance(a, C.Array):
            return list(a)
        return int(a)

    out = [(name, tuple(arg(a) for a in args)) for name, args in fake.calls]
    fake.calls.clear()
    return out


def desc(a):
    if a is None:
        return None
    if T._is_tensor(a):
        return ("torch", str(a.dtype).replace("torch.", ""), tuple(a.shape))
    return ("numpy", str(a.dtype), tuple(a.shape))


def kinds(np_name, torch_name):
    return {"numpy": np_name, "torch": torch_name}


KINDS = ["numpy", "torch"]


def as_kind(a, kind):
    return torch.from_numpy(np.ascontiguousarray(a)) if kind == "torch" else a


rng = np.random.default_rng(5)
P = rng.random((10, 4), dtype=np.float32)  # 10 points, stride 4: dim 3
Q = rng.random((5, 3), dtype=np.float32)
BATCH = np.array([0] * 6 + [1] * 4)


# ---- builds ----
@pytest.mark.parametrize("kind", KINDS)
def test_build(t, fake, kind):
    pts = as_kind(P, kind)
    assert t.build(pts) is t
    assert trace(fake, points=pts) == [("tknn_build", ("ctx", "points", 10, 3, 4))]
    t.build(pts, dim=2)
    assert trace(fake, points=pts) == [("tknn_build", ("ctx", "points", 10, 2, 4))]
    assert (t.n, t.n_segments) == (10, 1)
    assert t.cloud_sizes().tolist() == [10]


def test_build_casts_numpy(t, fake):
    t.build(P.astype(np.float64))  # a cast copy, not the caller's array
    assert trace(fake) == [("tknn_build", ("ctx", "ptr", 10, 3, 4))]
    t.build(P[:, :3].tolist())
    assert trace(fake) == [("tknn_build", ("ctx", "ptr", 10, 3, 3))]


@pytest.mark.parametrize("kind", KINDS)
def test_build_segments(t, fake, kind):
    pts = as_kind(P, kind)
    t.build(pts, batch=as_kind(BATCH, kind))
    assert trace(fake, points=pts) == [("tknn_build_segments", ("ctx", "points", 10, 3, 4, "ptr", 2))]
    assert t.n_segments == 2 and t.cloud_sizes().tolist() == [6, 4]
    t.build(pts, batch=as_kind(BATCH, kind), batch_size=4)
    assert trace(fake, points=pts) == [("tknn_build_segments", ("ctx", "points", 10, 3, 4, "ptr", 4))]
    assert t.cloud_sizes().tolist() == [6, 4, 0, 0]


def test_build_errors(t, fake):
    with pytest.raises(ValueError, match="points"):
        t.build(np.zeros(6, np.float32))
    with pytest.raises(TypeError, match="points"):
        t.build(torch.zeros((4, 3), dtype=torch.float64))
    with pytest.raises(ValueError, match="contiguous"):
        t.build(torch.zeros((3, 8), dtype=torch.float32).t())
    with pytest.raises(ValueError, match="batch_size"):
        t.build(P, batch_size=2)
    assert trace(fake) == []


@pytest.mark.parametrize("kind", KINDS)
def test_build_replicated_and_partition(t, fake, kind):
    pts = as_kind(P, kind)
    t.build_replicated(pts, 20, 40)
    assert trace(fake, points=pts) == [("tknn_build_replicated", ("ctx", "points", 10, 20, 40, 3, 4))]
    assert t.n == 40
    t.partition_build(pts, 20, dim=2)
    assert trace(fake, points=pts) == [("tknn_partition_build", ("ctx", "points", 10, 20, 2, 4)),
                                       ("tknn_partition_owned", ("ctx",))]
    assert t.n == CAPACITY
    gid, idx, dist = t.partition_search(2, 0.25)
    assert trace(fake, gid=gid, idx=idx, dist=dist) == [
        ("tknn_partition_owned", ("ctx",)),
        ("tknn_partition_search", ("ctx", 2, 0.25, "gid", "idx", "dist", CAPACITY, "&"))]
    assert [desc(a) for a in (gid, idx, dist)] == [(kind, "int32", (COUNT,)), (kind, "int32", (COUNT, 2)),
                                                   (kind, "float32", (COUNT, 2))]


# ---- searches on the built cloud ----
@pytest.mark.parametrize("kind", KINDS)
def test_search(t, fake, kind):
    t.build(as_kind(P, kind))
    fake.calls.clear()
    idx, dist = t.search(2)
    assert trace(fake, idx=idx, dist=dist) == [("tknn_search", ("ctx", 2, 0.0, "idx", "dist"))]
    assert [desc(idx), desc(dist)] == [(kind, "int32", (10, 2)), (kind, "float32", (10, 2))]
    idx, dist = t.search(3, indices_only=True)
    assert trace(fake, idx=idx) == [("tknn_search", ("ctx", 3, 0.0, "idx", None))]
    assert desc(idx) == (kind, "int32", (10, 3)) and dist is None


def test_search_out(t, fake):
    t.build(P)
    fake.calls.clear()
    oi, od = np.empty((10, 2), np.int32), np.empty((10, 2), np.float32)
    idx, dist = t.search(2, 0.5, out=(oi, od))
    assert idx is oi and dist is od
    assert trace(fake, oi=oi, od=od) == [("tknn_search", ("ctx", 2, 0.5, "oi", "od"))]
    t.search(2, out=(oi, None))
    assert trace(fake, oi=oi) == [("tknn_search", ("ctx", 2, 0.0, "oi", None))]
    with pytest.raises(TypeError, match="idx_out"):
        t.search(2, out=(od, None))
    with pytest.raises(TypeError, match="dist_out"):
        t.search(2, out=(oi, oi))


@pytest.mark.parametrize("kind", KINDS)
def test_search_shard(t, fake, kind):
    t.build(as_kind(P, kind))
    fake.calls.clear()
    qid, idx, dist = t.search_shard(2, 1, 3)
    assert trace(fake, qid=qid, idx=idx, dist=dist) == [
        ("tknn_shard_capacity", (10, 3)),
        ("tknn_search_shard", ("ctx", 2, 0.0, 1, 3, "qid", "idx", "dist", "&"))]
    assert [desc(a) for a in (qid, idx, dist)] == [(kind, "int32", (COUNT,)), (kind, "int32", (COUNT, 2)),
                                                   (kind, "float32", (COUNT, 2))]


def test_search_shard_out(t, fake):
    t.build(P)
    fake.calls.clear()
    out = (np.empty(8, np.int32), np.empty((8, 2), np.int32), np.empty((8, 2), np.float32))
    qid, idx, dist = t.search_shard(2, 0, 2, 0.5, out=out)
    assert trace(fake, qid=out[0], idx=out[1], dist=out[2]) == [
        ("tknn_shard_capacity", (10, 2)),
        ("tknn_search_shard", ("ctx", 2, 0.5, 0, 2, "qid", "idx", "dist", "&"))]
    assert qid.base is out[0] and qid.shape == (COUNT,)


@pytest.mark.parametrize("kind", KINDS)
def test_query(t, fake, kind):
    t.build(as_kind(P, kind))
    fake.calls.clear()
    q = as_kind(Q, kind)
    sid = as_kind(np.arange(5, dtype=np.int32), kind)
    cap = as_kind(np.ones(5, np.float32), kind)
    idx, dist = t.query(q, 2, self_ids=sid, init_radius2=cap, start_radius=0.5)
    assert trace(fake, queries=q, sid=sid, cap=cap, idx=idx, dist=dist) == [
        ("tknn_query", ("ctx", "queries", 5, 3, 3, "sid", "cap", 2, 0.5, "idx", "dist"))]
    assert [desc(idx), desc(dist)] == [(kind, "int32", (5, 2)), (kind, "float32", (5, 2))]
    idx, dist = t.query(q, 1, dim=2)
    assert trace(fake, queries=q, idx=idx, dist=dist) == [
        ("tknn_query", ("ctx", "queries", 5, 2, 3, None, None, 1, 0.0, "idx", "dist"))]


def test_query_casts_numpy(t, fake):
    t.build(P)
    fake.calls.clear()
    idx, dist = t.query(Q.astype(np.float64), 2, self_ids=[0, 1, 2, 3, 4], init_radius2=[1.0] * 5)
    assert trace(fake, idx=idx, dist=dist) == [
        ("tknn_query", ("ctx", "ptr", 5, 3, 3, "ptr", "ptr", 2, 0.0, "idx", "dist"))]


@pytest.mark.parametrize("kind", KINDS)
def test_query_segments(t, fake, kind):
    t.build(as_kind(P, kind), batch=as_kind(BATCH, kind))
    fake.calls.clear()
    q = as_kind(Q, kind)
    idx, dist = t.query(q, 2, batch=as_kind(np.array([0, 0, 1, 1, 1]), kind))
    assert trace(fake, queries=q, idx=idx, dist=dist) == [
        ("tknn_query_segments", ("ctx", "queries", 5, 3, 3, "ptr", 2, None, None, 2, 0.0, "idx", "dist"))]


@pytest.mark.parametrize("kind", KINDS)
def test_range_count(t, fake, kind):
    t.build(as_kind(P, kind))
    fake.calls.clear()
    out = t.range_count(0.5)
    assert trace(fake, out=out) == [("tknn_range_count", ("ctx", 0.5, "out"))]
    assert desc(out) == (kind, kinds("uint32", "int32")[kind], (10,))


@pytest.mark.parametrize("kind", KINDS)
def test_dbscan(t, fake, kind):
    t.build(as_kind(P, kind))
    fake.calls.clear()
    labels, core, c = t.dbscan(0.5, 4)
    assert trace(fake, labels=labels, core=core) == [("tknn_dbscan", ("ctx", 0.5, 4, "labels", "core", "&"))]
    assert [desc(labels), desc(core), c] == [(kind, "int32", (10,)), (kind, "uint8", (10,)), COUNT]
    labels, core, _ = t.dbscan(0.5, 4, with_core=False)
    assert trace(fake, labels=labels) == [("tknn_dbscan", ("ctx", 0.5, 4, "labels", None, "&"))]
    assert core is None
    ol, oc = as_kind(np.empty(10, np.int32), kind), as_kind(np.empty(10, np.uint8), kind)
    assert t.dbscan(0.5, 2, out=(ol, oc))[:2] == (ol, oc)
    assert trace(fake, ol=ol, oc=oc) == [("tknn_dbscan", ("ctx", 0.5, 2, "ol", "oc", "&"))]
    with pytest.raises(TypeError, match="core"):
        t.dbscan(0.5, 2, out=(ol, ol))


@pytest.mark.parametrize("kind", KINDS)
def test_radius_search(t, fake, kind):
    t.build(as_kind(P, kind))
    fake.calls.clear()
    off, idx, dist = t.radius_search(0.5)
    assert trace(fake, off=off, idx=idx, dist=dist) == [
        ("tknn_radius_search", ("ctx", 0.5, "off", None, None, 0, "&")),
        ("tknn_radius_search", ("ctx", 0.5, "off", "idx", "dist", COUNT, "&"))]
    assert [desc(off), desc(idx), desc(dist)] == [(kind, "int64", (11,)), (kind, "int32", (COUNT,)),
                                                  (kind, "float32", (COUNT,))]
    off, idx, dist = t.radius_search(0.5, indices_only=True)
    assert trace(fake, off=off, idx=idx) == [
        ("tknn_radius_search", ("ctx", 0.5, "off", None, None, 0, "&")),
        ("tknn_radius_search", ("ctx", 0.5, "off", "idx", None, COUNT, "&"))]
    assert dist is None


def test_radius_search_out(t, fake):
    t.build(P)
    fake.calls.clear()
    oo, oi, od = np.empty(11, np.int64), np.empty(8, np.int32), np.empty(6, np.float32)
    off, idx, dist = t.radius_search(0.5, out=(oo, oi, od))
    assert trace(fake, oo=oo, oi=oi, od=od) == [("tknn_radius_search", ("ctx", 0.5, "oo", "oi", "od", 6, "&"))]
    assert off is oo and idx.shape == (COUNT,) and dist.shape == (COUNT,)
    with pytest.raises(ValueError, match="offsets"):
        t.radius_search(0.5, out=(oo[:5], oi, od))
    with pytest.raises(TypeError, match="offsets"):
        t.radius_search(0.5, out=(oo.astype(np.int32), oi, od))
    assert trace(fake) == []


@pytest.mark.parametrize("kind", KINDS)
def test_radius_query(t, fake, kind):
    t.build(as_kind(P, kind))
    fake.calls.clear()
    q, sid = as_kind(Q, kind), as_kind(np.arange(5, dtype=np.int32), kind)
    off, idx, dist = t.radius_query(q, 0.5, self_ids=sid)
    assert trace(fake, queries=q, sid=sid, off=off, idx=idx, dist=dist) == [
        ("tknn_radius_query", ("ctx", "queries", 5, 3, 3, "sid", 0.5, "off", None, None, 0, "&")),
        ("tknn_radius_query", ("ctx", "queries", 5, 3, 3, "sid", 0.5, "off", "idx", "dist", COUNT, "&"))]
    assert [desc(off), desc(idx), desc(dist)] == [(kind, "int64", (6,)), (kind, "int32", (COUNT,)),
                                                  (kind, "float32", (COUNT,))]
    with pytest.raises(TypeError, match="self_ids"):
        t.radius_query(q, 0.5, self_ids=as_kind(np.arange(5, dtype=np.int64), "torch"))


@pytest.mark.parametrize("kind", KINDS)
def test_radius_query_segments(t, fake, kind):
    t.build(as_kind(P, kind), batch=as_kind(BATCH, kind))
    fake.calls.clear()
    q = as_kind(Q, kind)
    off, idx, dist = t.radius_query(q, 0.5, dim=2, indices_only=True, batch=as_kind(np.array([0, 0, 1, 1, 1]), kind))
    assert trace(fake, queries=q, off=off, idx=idx) == [
        ("tknn_radius_query_segments", ("ctx", "queries", 5, 2, 3, "ptr", 2, None, 0.5, "off", None, None, 0, "&")),
        ("tknn_radius_query_segments", ("ctx", "queries", 5, 2, 3, "ptr", 2, None, 0.5, "off", "idx", None, COUNT,
                                        "&"))]


@pytest.mark.parametrize("kind", KINDS)
def test_brute_force_and_merge(t, fake, kind):
    t.build(as_kind(P, kind))
    fake.calls.clear()
    ids = as_kind(np.array([1, 4, 7], np.int32), kind)
    idx, dist = t.brute_force(ids, 2)
    assert trace(fake, ids=ids, idx=idx, dist=dist) == [("tknn_brute_force", ("ctx", "ids", 3, 2, "idx", "dist"))]
    assert [desc(idx), desc(dist)] == [(kind, "int32", (3, 2)), (kind, "float32", (3, 2))]
    ip, dp = as_kind(np.zeros((2, 3, 4), np.int32), kind), as_kind(np.zeros((2, 3, 4), np.float32), kind)
    idx, dist = t.merge_topk(ip, dp)
    assert trace(fake, ip=ip, dp=dp, idx=idx, dist=dist) == [
        ("tknn_merge_topk", ("ctx", "ip", "dp", 2, 3, 4, "idx", "dist"))]
    assert [desc(idx), desc(dist)] == [(kind, "int32", (3, 4)), (kind, "float32", (3, 4))]


# ---- farthest point sampling ----
@pytest.mark.parametrize("kind", KINDS)
def test_fps(t, fake, kind):
    t.build(as_kind(P, kind), batch=as_kind(BATCH, kind))
    fake.calls.clear()
    idx, dist = t.fps([2, 3])
    assert trace(fake, idx=idx) == [("tknn_fps", ("ctx", "ptr", 2, None, "idx", None))]
    assert desc(idx) == (kind, "int32", (5,)) and dist is None
    start = as_kind(np.array([1, 7], np.int32), kind)
    idx, dist = t.fps(ratio=0.5, start=start, with_dist=True)
    assert trace(fake, idx=idx, dist=dist, start=start) == [("tknn_fps", ("ctx", "ptr", 2, "start", "idx", "dist"))]
    assert [desc(idx), desc(dist)] == [(kind, "int32", (5,)), (kind, "float32", (5,))]
    idx, dist = t.fps([0, 0], with_dist=True)  # nothing to sample: no call
    assert trace(fake) == []
    assert [desc(idx), desc(dist)] == [(kind, "int32", (0,)), (kind, "float32", (0,))]


def test_fps_start_and_errors(t, fake):
    t.build(P)
    fake.calls.clear()
    idx, _ = t.fps(4, start=3)
    assert trace(fake, idx=idx) == [("tknn_fps", ("ctx", "ptr", 1, "ptr", "idx", None))]
    with pytest.raises(ValueError, match="start"):
        t.fps(4, start=[1, 2])
    with pytest.raises(TypeError, match="start"):
        t.fps(4, start=torch.tensor([1], dtype=torch.int64))
    with pytest.raises(ValueError, match="num_samples"):
        t.fps(4, ratio=0.5)
    with pytest.raises(TypeError, match="idx"):
        t.fps(4, out=(np.empty(4, np.int64), None))
    assert trace(fake) == []


# ---- feature space ----
@pytest.mark.parametrize("kind", KINDS)
def test_feature_knn(t, fake, kind):
    x, y = as_kind(P, kind), as_kind(rng.random((5, 4), dtype=np.float32), kind)
    sid = as_kind(np.arange(5, dtype=np.int32), kind)
    idx, dist = t.feature_knn(x, y, 2, self_ids=sid)
    assert trace(fake, x=x, y=y, sid=sid, idx=idx, dist=dist) == [
        ("tknn_feature_knn", ("ctx", "x", 10, 4, 4, None, "y", 5, 4, None, 1, "sid", 2, "idx", "dist"))]
    assert [desc(idx), desc(dist)] == [(kind, "int32", (5, 2)), (kind, "float32", (5, 2))]
    idx, dist = t.feature_knn(x, x, 3, batch_x=as_kind(BATCH, kind), indices_only=True)
    assert trace(fake, x=x, idx=idx) == [
        ("tknn_feature_knn", ("ctx", "x", 10, 4, 4, "ptr", "x", 10, 4, "ptr", 2, None, 3, "idx", None))]
    assert desc(idx) == (kind, "int32", (10, 3)) and dist is None


@pytest.mark.parametrize("kind", KINDS)
def test_feature_knn_zero_rows(t, fake, kind):
    x = as_kind(P, kind)
    idx, dist = t.feature_knn(x, x[:0], 2)
    assert trace(fake) == []
    assert [desc(idx), desc(dist)] == [(kind, "int32", (0, 2)), (kind, "float32", (0, 2))]
    y = as_kind(Q, kind)
    idx, _ = t.feature_knn(as_kind(np.zeros((0, 3), np.float32), kind), y, 2, batch_y=as_kind(np.zeros(5, np.int64), kind))
    assert trace(fake, y=y, idx=idx) == [
        ("tknn_feature_knn", ("ctx", kinds("ptr", None)[kind], 0, 3, 3, None, "y", 5, 3, None, 1, None, 2, "idx",
                              "ptr"))]


def test_feature_knn_errors(t, fake):
    with pytest.raises(ValueError, match="columns"):
        t.feature_knn(P, Q, 2)
    with pytest.raises(ValueError, match="x and y"):
        t.feature_knn(P[0], Q, 2)
    with pytest.raises(TypeError, match="y"):
        t.feature_knn(torch.from_numpy(P), torch.zeros((2, 4), dtype=torch.float64), 2)
    with pytest.raises(TypeError, match="self_ids"):
        t.feature_knn(P, P, 2, self_ids=torch.zeros(10, dtype=torch.int64))
    assert trace(fake) == []


# ---- voxel grid ----
@pytest.mark.parametrize("kind", KINDS)
def test_voxel_grid(t, fake, kind):
    pts = as_kind(P, kind)
    raw, cluster, nv = t.voxel_grid(pts, 0.25, batch=as_kind(BATCH, kind))
    assert trace(fake, points=pts, raw=raw, cluster=cluster) == [
        ("tknn_voxel_grid", ("ctx", "points", 10, 3, 4, "ptr", 2, "ptr", None, None, "raw", "cluster", "&"))]
    assert [desc(raw), desc(cluster), nv] == [(kind, "int64", (10,)), (kind, "int32", (10,)), COUNT]
    offsets, members, first, seg = t.voxel_members()
    assert trace(fake, offsets=offsets, members=members, first=first, seg=seg) == [
        ("tknn_voxel_members", ("ctx", "offsets", "members", "first", "seg"))]
    assert [desc(a) for a in (offsets, members, first, seg)] == [
        (kind, kinds("uint64", "int64")[kind], (COUNT + 1,)), (kind, "int32", (10,)), (kind, "int32", (COUNT,)),
        (kind, "int32", (COUNT,))]
    x = as_kind(rng.random((10, 2), dtype=np.float32), kind)
    out = t.voxel_pool(x, "max")
    assert trace(fake, x=x, out=out) == [("tknn_voxel_pool", ("ctx", "x", 10, 2, 2, _lib.REDUCE_MAX, "out"))]
    assert desc(out) == (kind, "float32", (COUNT, 2))
    x1 = as_kind(np.zeros(10, np.float32), kind)
    out = t.voxel_pool(x1)
    assert trace(fake, x=x1, out=out) == [("tknn_voxel_pool", ("ctx", "x", 10, 1, 1, _lib.REDUCE_MEAN, "out"))]
    assert desc(out) == (kind, "float32", (COUNT, 1))
    raw, cluster, _ = t.voxel_grid(as_kind(P[:, :2], kind), [0.5, 0.25], start=0.0, end=[1, 1])
    assert trace(fake, raw=raw, cluster=cluster) == [
        ("tknn_voxel_grid", ("ctx", "ptr", 10, 2, 2, None, 1, "ptr", "ptr", "ptr", "raw", "cluster", "&"))]


@pytest.mark.parametrize("kind", KINDS)
def test_voxel_zero_rows(t, fake, kind):
    pts = as_kind(np.zeros((0, 3), np.float32), kind)
    raw, cluster, nv = t.voxel_grid(pts, 1.0)
    assert trace(fake) == [("tknn_voxel_grid", ("ctx", None, 0, 3, 3, None, 1, "ptr", None, None, None, None, "&"))]
    assert [desc(raw), desc(cluster)] == [(kind, "int64", (0,)), (kind, "int32", (0,))]
    offsets, members, first, seg = t.voxel_members()
    assert trace(fake, offsets=offsets) == [("tknn_voxel_members", ("ctx", "offsets", None, "ptr", "ptr"))]
    assert desc(members) == (kind, "int32", (0,))
    out = t.voxel_pool(as_kind(np.zeros((0, 2), np.float32), kind))
    assert trace(fake, out=out) == [("tknn_voxel_pool", ("ctx", None, 0, 2, 2, _lib.REDUCE_MEAN, "out"))]
    assert desc(out) == (kind, "float32", (COUNT, 2))


def test_voxel_errors(t, fake):
    with pytest.raises(T.TrueKNNError):
        t.voxel_pool(P)
    with pytest.raises(ValueError, match="points"):
        t.voxel_grid(P[:, :1], 1.0)
    with pytest.raises(ValueError, match="size"):
        t.voxel_grid(P, [1.0, 2.0])
    with pytest.raises(TypeError, match="points"):
        t.voxel_grid(torch.zeros((3, 3), dtype=torch.float64), 1.0)
    t.voxel_grid(P, 1.0)
    with pytest.raises(ValueError, match="reduce"):
        t.voxel_pool(P, "sum")
    with pytest.raises(ValueError, match="x"):
        t.voxel_pool(np.zeros((10, 2, 2), np.float32))
    with pytest.raises(TypeError, match="x"):
        t.voxel_pool(torch.zeros((10, 2), dtype=torch.float64))


# ---- interpolation ----
@pytest.mark.parametrize("kind", KINDS)
def test_interpolate(t, fake, kind):
    x = as_kind(rng.random((10, 3), dtype=np.float32), kind)
    idx = as_kind(np.zeros((5, 2), np.int32), kind)
    d2 = as_kind(np.ones((5, 2), np.float32), kind)
    out, weight, den = t.interpolate(idx, d2, x)
    assert trace(fake, x=x, idx=idx, d2=d2, out=out, weight=weight, den=den) == [
        ("tknn_interpolate", ("ctx", "idx", "d2", 5, 2, "x", 10, 3, 3, "out", "weight", "den"))]
    assert [desc(a) for a in (out, weight, den)] == [(kind, "float32", (5, 3)), (kind, "float32", (5, 2)),
                                                     (kind, "float32", (5,))]
    g = as_kind(np.ones((5, 3), np.float32), kind)
    grad = t.interpolate_backward(idx, weight, den, g, 10)
    assert trace(fake, idx=idx, weight=weight, den=den, g=g, grad=grad) == [
        ("tknn_interpolate_backward", ("ctx", "idx", "weight", "den", 5, 2, "g", 3, 10, 3, "grad"))]
    assert desc(grad) == (kind, "float32", (10, 3))


@pytest.mark.parametrize("kind", KINDS)
def test_interpolate_zero_rows(t, fake, kind):
    x = as_kind(np.zeros((0, 3), np.float32), kind)
    idx = as_kind(np.full((5, 2), -1, np.int32), kind)
    d2 = as_kind(np.ones((5, 2), np.float32), kind)
    out, weight, den = t.interpolate(idx, d2, x)
    assert trace(fake, idx=idx, d2=d2, out=out, weight=weight, den=den) == [
        ("tknn_interpolate", ("ctx", "idx", "d2", 5, 2, None, 0, 3, 3, "out", "weight", "den"))]
    out, weight, den = t.interpolate(idx[:0], d2[:0], x)  # no query rows: no call
    assert trace(fake) == []
    assert [desc(a) for a in (out, weight, den)] == [(kind, "float32", (0, 3)), (kind, "float32", (0, 2)),
                                                     (kind, "float32", (0,))]
    grad = t.interpolate_backward(idx[:0], weight, den, out, 4)
    assert trace(fake) == []
    assert desc(grad) == (kind, "float32", (4, 3)) and float(grad.sum()) == 0.0
    g = as_kind(np.ones((5, 3), np.float32), kind)
    w = as_kind(np.ones((5, 2), np.float32), kind)
    dn = as_kind(np.ones(5, np.float32), kind)
    grad = t.interpolate_backward(idx, w, dn, g, 0)
    assert trace(fake, idx=idx, w=w, dn=dn, g=g) == [
        ("tknn_interpolate_backward", ("ctx", "idx", "w", "dn", 5, 2, "g", 3, 0, 3, None))]
    assert desc(grad) == (kind, "float32", (0, 3))


def test_interpolate_inputs(t, fake):
    x = np.zeros((10, 3), np.float32)
    idx, d2 = np.zeros((5, 2), np.int32), np.ones((5, 2), np.float32)
    with pytest.raises(TypeError, match="x"):
        t.interpolate(idx, d2, x.astype(np.float64))  # x is not cast
    with pytest.raises(ValueError, match="x"):
        t.interpolate(idx, d2, x[0])
    with pytest.raises(ValueError, match="idx"):
        t.interpolate(idx[0], d2, x)
    with pytest.raises(ValueError, match="d2"):
        t.interpolate(idx, d2[:3], x)
    with pytest.raises(TypeError, match="idx"):
        t.interpolate(torch.from_numpy(idx).long(), torch.from_numpy(d2), torch.from_numpy(x))
    with pytest.raises(ValueError, match="shapes"):
        t.interpolate_backward(idx, d2, np.ones(4, np.float32), np.ones((5, 3), np.float32), 10)
    assert trace(fake) == []
    t.interpolate(idx.tolist(), d2.astype(np.float64), x)  # idx and d2 are cast
    assert trace(fake, x=x) == [("tknn_interpolate", ("ctx", "ptr", "ptr", 5, 2, "x", 10, 3, 3, "ptr", "ptr", "ptr"))]
    xt = torch.zeros((3, 10), dtype=torch.float32).t()  # a non-contiguous x is copied, not refused
    it, dt = torch.from_numpy(idx), torch.from_numpy(d2)
    t.interpolate(it, dt, xt)
    assert trace(fake, it=it, dt=dt) == [
        ("tknn_interpolate", ("ctx", "it", "dt", 5, 2, "ptr", 10, 3, 3, "ptr", "ptr", "ptr"))]


# ---- introspection ----
@pytest.mark.parametrize("kind", KINDS)
def test_morton_codes(t, fake, kind):
    pts = as_kind(P, kind)
    out = t.morton_codes(pts, [0, 0, 0, 1, 1, 1])
    assert trace(fake, points=pts, out=out) == [("tknn_morton_codes", ("ctx", "points", 10, 3, 4, "ptr", "out"))]
    assert desc(out) == (kind, kinds("uint64", "int64")[kind], (10,))


def test_reach_mask(t, fake):
    pts, r2 = torch.from_numpy(P), torch.ones(10)
    summ = torch.zeros((3, 8, 6))
    out = t.reach_mask(pts, r2, [0, 0, 0, 1, 1, 1], summ, 1, cell_bits=2)
    assert trace(fake, pts=pts, r2=r2, summ=summ, out=out) == [
        ("tknn_reach_mask", ("ctx", "pts", 10, 4, "r2", "ptr", "summ", 3, 2, 1, "out"))]
    assert desc(out) == ("torch", "int32", (10,))


def test_small_calls(t, fake):
    keys = np.arange(6, dtype=np.uint32)
    t.sort_pairs(keys)
    out = t.generate_uniform(3, 10, 7)
    t.estimate_start_radius(4)
    t.set_option("leaf_size", 8)
    t.set_stream(0)
    t.set_stream(None)
    assert trace(fake, keys=keys, out=out) == [
        ("tknn_sort_pairs", ("ctx", "keys", None, 6)), ("tknn_generate_uniform", ("ctx", 3, 10, 7, "out")),
        ("tknn_estimate_start_radius", ("ctx", 4, "&")), ("tknn_set_option", ("ctx", _lib.OPT_LEAF_SIZE, 8)),
        ("tknn_set_stream", ("ctx", 1)), ("tknn_set_stream", ("ctx", None))]
    assert desc(out) == ("numpy", "float32", (7, 3))


def test_rank_view(fake):
    m = T.MultiTrueKNN([0, 0])
    r = m.rank(1)
    assert trace(fake) == [("tknn_create_multi", ([0, 0], 2, _lib.SHARD_QUERIES, "&")), ("tknn_multi_ctx", ("ctx", 1))]
    assert r.stats()["n_points"] == 0
    for name in ("device", "n", "n_segments", "_offsets", "_like", "_own_stream"):
        assert hasattr(r, name), name
    assert r.cloud_sizes().tolist() == [0]
    m.close()


# ---- module functions (numpy in; device 0 unless given) ----
def test_fps_function(fake):
    idx = T.fps(P, batch=BATCH, ratio=0.5, random_start=False, device=1)
    assert trace(fake) == [("tknn_create", (1, "&")), ("tknn_build_segments", ("ctx", "ptr", 10, 3, 4, "ptr", 2)),
                           ("tknn_fps", ("ctx", "ptr", 2, None, "ptr", None)), ("tknn_destroy", ("ctx",))]
    assert desc(idx) == ("numpy", "int64", (5,))
    T.fps(P, ratio=0.5)
    assert [c[0] for c in trace(fake)] == ["tknn_create", "tknn_build", "tknn_fps", "tknn_destroy"]
    assert desc(T.fps(P[:0])) == ("numpy", "int64", (0,)) and trace(fake) == []


def _fill_knn(fake, rows):
    """The fake's searches write rows of neighbours (-1 = none) into their idx output."""
    r = np.asarray(rows, np.int32)

    def fill(at):
        return lambda *args: C.memmove(args[at].value, r.ctypes.data, r.nbytes)

    fake.hooks.update(tknn_search=fill(3), tknn_query_segments=fill(-2), tknn_feature_knn=fill(-2))


def _fill_lists(fake, offsets, idx):
    """The fake's radius calls write the CSR rows: the offsets on the size call, the indices on the second."""
    off, ix = np.asarray(offsets, np.uint64), np.asarray(idx, np.int32)

    def fill(*args):
        ptrs = [a for a in args if isinstance(a, C.c_void_p) and a.value and a.value != HANDLE]
        C.memmove(ptrs[-1 if args[-2] == 0 else -2].value, off.ctypes.data, off.nbytes)
        if args[-2]:
            C.memmove(ptrs[-1].value, ix.ctypes.data, ix.nbytes)
        args[-1]._obj.value = ix.shape[0]

    for name in ("tknn_radius_search", "tknn_radius_query", "tknn_radius_query_segments"):
        fake.hooks[name] = fill


def test_knn_graph_function(fake):
    _fill_knn(fake, [[1, 2], [0, -1], [0, 1]])
    e = T.knn_graph(P[:3], 2)
    assert trace(fake) == [("tknn_create", (0, "&")), ("tknn_build", ("ctx", "ptr", 3, 3, 4)),
                           ("tknn_search", ("ctx", 2, 0.0, "ptr", None)), ("tknn_destroy", ("ctx",))]
    assert desc(e) == ("numpy", "int64", (2, 5))
    assert e.tolist() == [[1, 2, 0, 0, 1], [0, 0, 1, 2, 2]]


def test_knn_function(fake):
    _fill_knn(fake, [[1, 2, -1], [0, -1, -1]])
    e = T.knn(P[:3], Q[:2], 5, batch_y=np.array([0, 0]), device=2)
    assert trace(fake) == [("tknn_create", (2, "&")), ("tknn_build_segments", ("ctx", "ptr", 3, 3, 4, "ptr", 1)),
                           ("tknn_query_segments", ("ctx", "ptr", 2, 3, 3, "ptr", 1, None, None, 3, 0.0, "ptr", "ptr")),
                           ("tknn_destroy", ("ctx",))]
    assert e.tolist() == [[0, 0, 1], [1, 2, 0]] and e.dtype == np.int64
    assert desc(T.knn(P[:0], Q, 2)) == ("numpy", "int64", (2, 0)) and trace(fake) == []


def test_radius_graph_function(fake):
    _fill_lists(fake, [0, 2, 2, 3], [1, 2, 0])
    e = T.radius_graph(P[:3], 0.5)
    assert trace(fake) == [("tknn_create", (0, "&")), ("tknn_build", ("ctx", "ptr", 3, 3, 4)),
                           ("tknn_radius_search", ("ctx", 0.5, "ptr", None, None, 0, "&")),
                           ("tknn_radius_search", ("ctx", 0.5, "ptr", "ptr", None, 3, "&")),
                           ("tknn_destroy", ("ctx",))]
    assert e.tolist() == [[1, 2, 0], [0, 0, 2]] and e.dtype == np.int64


def test_radius_function(fake):
    _fill_lists(fake, [0, 3, 4], [2, 0, 1, 1])
    e = T.radius(P[:3], Q[:2], 0.5, max_num_neighbors=2)
    assert trace(fake) == [
        ("tknn_create", (0, "&")), ("tknn_build", ("ctx", "ptr", 3, 3, 4)),
        ("tknn_radius_query", ("ctx", "ptr", 2, 3, 3, None, 0.5, "ptr", None, None, 0, "&")),
        ("tknn_radius_query", ("ctx", "ptr", 2, 3, 3, None, 0.5, "ptr", "ptr", None, 4, "&")),
        ("tknn_destroy", ("ctx",))]
    assert e.tolist() == [[0, 0, 1], [2, 0, 1]] and e.dtype == np.int64
    _fill_lists(fake, [0, 3, 4], [2, 0, 1, 1])
    assert T.radius(P[:3], Q[:2], 0.5, batch_x=np.zeros(3, np.int64)).tolist() == [[0, 0, 0, 1], [2, 0, 1, 1]]
    assert [c[0] for c in trace(fake)] == ["tknn_create", "tknn_build_segments", "tknn_radius_query_segments",
                                           "tknn_radius_query_segments", "tknn_destroy"]
    assert desc(T.radius(P, Q[:0], 0.5)) == ("numpy", "int64", (2, 0))


def test_feature_knn_functions(fake):
    _fill_knn(fake, [[1], [0], [-1]])
    e = T.feature_knn_graph(P[:3], 1, device=1)
    assert trace(fake) == [("tknn_create", (1, "&")),
                           ("tknn_feature_knn", ("ctx", "ptr", 3, 4, 4, None, "ptr", 3, 4, None, 1, "ptr", 1, "ptr",
                                                 None)), ("tknn_destroy", ("ctx",))]
    assert e.tolist() == [[1, 0], [0, 1]] and e.dtype == np.int64
    _fill_knn(fake, [[2, 1, -1], [0, -1, -1]])
    e = T.feature_knn(P[:3], P[:2], 4, batch_x=np.array([0, 0, 1]))
    assert trace(fake)[1] == ("tknn_feature_knn", ("ctx", "ptr", 3, 4, 4, "ptr", "ptr", 2, 4, "ptr", 2, None, 3, "ptr",
                                                   None))
    assert e.tolist() == [[0, 0, 1], [2, 1, 0]]
    assert desc(T.feature_knn_graph(P[:0], 2)) == ("numpy", "int64", (2, 0))


def test_voxel_functions(fake):
    raw = T.grid_cluster(P[:, :3], 0.5, device=1)
    assert trace(fake) == [("tknn_create", (1, "&")),
                           ("tknn_voxel_grid", ("ctx", "ptr", 10, 3, 3, None, 1, "ptr", None, None, "ptr", "ptr", "&")),
                           ("tknn_destroy", ("ctx",))]
    assert desc(raw) == ("numpy", "int64", (10,))
    with pytest.raises(ValueError, match="columns"):
        T.voxel_grid(P, 0.5)
    pos_mean, xp, batch_out, cluster = T.grid_sampling(P[:, :3], 0.5, x=P, batch=BATCH, reduce="max")
    assert [c[0] for c in trace(fake)] == ["tknn_create", "tknn_voxel_grid", "tknn_voxel_pool", "tknn_voxel_pool",
                                           "tknn_voxel_members", "tknn_destroy"]
    assert [desc(a) for a in (pos_mean, xp, batch_out, cluster)] == [
        ("numpy", "float32", (COUNT, 3)), ("numpy", "float32", (COUNT, 4)), ("numpy", "int64", (COUNT,)),
        ("numpy", "int64", (10,))]


def test_knn_interpolate_function(fake):
    x = rng.random((3, 2), dtype=np.float32)
    _fill_knn(fake, [[0, 1], [2, -1]])
    out = T.knn_interpolate(x, P[:3, :3], Q[:2], k=2)
    assert trace(fake, x=x, out=out) == [
        ("tknn_create", (0, "&")), ("tknn_set_option", ("ctx", _lib.OPT_SQUARED_DIST, 1)),
        ("tknn_build", ("ctx", "ptr", 3, 3, 3)),
        ("tknn_query", ("ctx", "ptr", 2, 3, 3, None, None, 2, 0.0, "ptr", "ptr")),
        ("tknn_interpolate", ("ctx", "ptr", "ptr", 2, 2, "x", 3, 2, 2, "out", "ptr", "ptr")),
        ("tknn_destroy", ("ctx",))]
    assert desc(out) == ("numpy", "float32", (2, 2))
    with pytest.raises(TypeError, match="x"):
        T.knn_interpolate(x.astype(np.float64), P[:3, :3], Q[:2])
    with pytest.raises(ValueError, match="pos_x"):
        T.knn_interpolate(x, P[:3], Q[:2])
    with pytest.raises(ValueError, match="x has"):
        T.knn_interpolate(x, P[:4, :3], Q[:2])
    assert desc(T.knn_interpolate(x, P[:3, :3], Q[:0])) == ("numpy", "float32", (0, 2))
    assert np.isnan(T.knn_interpolate(x[:0], P[:0, :3], Q[:2])).all()
    assert trace(fake) == []
