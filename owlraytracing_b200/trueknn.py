"""Host-side mirror of the reference's TrueKNN sample interface over the libtrueknn C ABI.

The reference has no library API for kNN — its interface is the command line of
samples/s01-trueknn (hostCode.cpp:66-73: file, n, dim, start radius, k, out file) and the in-memory
`Neigh` buffer (GeomTypes.h:22-28, read at hostCode.cpp:294).  `run_sample()` below keeps those six
positional arguments; `TrueKNN` is the object behind it.  Every array argument may be a numpy array
(host memory, staged inside the C call) or a CUDA `torch.Tensor` (device memory, zero-copy).
"""
from __future__ import annotations

import ctypes as C
import re
import time

import numpy as np

from . import _lib
from ._lib import Stats


class TrueKNNError(RuntimeError):
    def __init__(self, code: int, message: str):
        super().__init__(f"{_lib.ERROR_NAMES.get(code, code)}: {message}")
        self.code = code


def _is_tensor(a) -> bool:
    return hasattr(a, "data_ptr") and hasattr(a, "is_cuda")


def _ptr(a, null_if_empty: bool = False):
    """Raw address of a numpy array or torch tensor (None -> NULL; with null_if_empty, an array without rows too)."""
    if a is None or (null_if_empty and a.shape[0] == 0):
        return None
    if _is_tensor(a):
        if not a.is_contiguous():
            raise ValueError("tensor must be contiguous")
        return C.c_void_p(a.data_ptr())
    if not a.flags["C_CONTIGUOUS"]:
        raise ValueError("array must be C-contiguous")
    return C.c_void_p(a.ctypes.data)


def _torch_dtype(np_dtype):
    """The tensor dtype of an array the library reads or writes as np_dtype: uint32 and uint64 arrays travel as int32 and
    int64 tensors."""
    import torch

    return {np.float32: torch.float32, np.int32: torch.int32, np.uint32: torch.int32, np.int64: torch.int64,
            np.uint64: torch.int64, np.uint8: torch.uint8}[np_dtype]


def _check_dtype(a, np_dtype, name):
    """TypeError naming `name` unless `a` (None passes) holds np_dtype, or its tensor dtype (torch.uint32 for uint32 too)."""
    if a is None:
        return
    if _is_tensor(a):
        import torch

        want = _torch_dtype(np_dtype)
        if a.dtype != want and not (np_dtype is np.uint32 and a.dtype == torch.uint32):
            raise TypeError(f"{name}: expected {want}, got {a.dtype}")
    elif a.dtype != np_dtype:
        raise TypeError(f"{name}: expected {np.dtype(np_dtype)}, got {a.dtype}")


def _arg(a, np_dtype, name, ndim: int | None = None, cast: bool = True, copy: bool = False):
    """An input array (None passes) ready for _ptr: anything numpy takes becomes a C-contiguous array, cast to np_dtype
    unless cast is False (then another dtype raises); a tensor is passed in place, or as a contiguous copy when copy is
    set (otherwise _ptr refuses a non-contiguous one).  TypeError for another dtype, ValueError for another rank."""
    if a is None:
        return None
    if _is_tensor(a):
        a = a.contiguous() if copy else a
    else:
        a = np.ascontiguousarray(a, dtype=np_dtype if cast else None)
    _check_dtype(a, np_dtype, name)
    if ndim is not None and a.ndim != ndim:
        raise ValueError(f"{name} must be {ndim}-D, got shape {tuple(a.shape)}")
    return a


def _points(a, name, dim: int | None = None):
    """Positions [n, stride] float32 as the LBVH calls take them: (array, n, dim, stride), dim = min(stride, 3) unless
    given, so columns beyond the third are skipped through the stride."""
    a = _arg(a, np.float32, name, ndim=2)
    stride = int(a.shape[1])
    return a, int(a.shape[0]), min(stride, 3) if dim is None else int(dim), stride


def _empty_like_rows(like, shape, np_dtype):
    """An uninitialised array of `shape` beside `like`: a tensor on its device, or numpy."""
    if _is_tensor(like):
        import torch

        return torch.empty(shape, dtype=_torch_dtype(np_dtype), device=like.device)
    return np.empty(shape, np_dtype)


def _zeros_like_rows(like, shape, np_dtype):
    """_empty_like_rows, filled with zeros."""
    if _is_tensor(like):
        import torch

        return torch.zeros(shape, dtype=_torch_dtype(np_dtype), device=like.device)
    return np.zeros(shape, np_dtype)


def _arange_like(like, n: int, np_dtype=np.int64):
    """0 .. n - 1 beside `like`: a tensor on its device, or numpy."""
    if _is_tensor(like):
        import torch

        return torch.arange(n, dtype=_torch_dtype(np_dtype), device=like.device)
    return np.arange(n, dtype=np_dtype)


class TrueKNN:
    """One LBVH + traversal context on one CUDA device (`tknn_ctx`)."""

    def __init__(self, device: int = 0, **options):
        self._L = _lib.load()
        h = C.c_void_p()
        rc = self._L.tknn_create(int(device), C.byref(h))
        if rc != _lib.OK:
            raise TrueKNNError(rc, f"tknn_create(device={device}) failed — a CUDA sm_100 device is required, "
                                   "there is no CPU fallback")
        self._h = h
        self._init_state(device)
        for k, v in options.items():
            self.set_option(k, v)

    def _init_state(self, device: int):
        self.device = int(device)
        self._own_stream = True  # until set_stream() hands over a caller stream
        self.n = 0
        self.n_segments = 1  # clouds of the last build (batch_size of query(batch=...) / radius_query(batch=...))
        self._offsets = None  # the cloud offsets of a segmented build (numpy or a tensor), None for a plain build
        self._like = None  # the last build's points: outputs of searches on it follow their kind and device
        self._vx_like = None  # the points of the last voxel_grid(), None before the first

    # ---- plumbing ----
    def _check(self, rc: int):
        if rc != _lib.OK:
            raise TrueKNNError(rc, self._L.tknn_last_error(self._h).decode())

    def close(self):
        if getattr(self, "_h", None):
            self._L.tknn_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def __enter__(self):
        return self

    def __exit__(self, *exc):
        self.close()

    _OPTS = {
        "leaf_size": _lib.OPT_LEAF_SIZE, "counters": _lib.OPT_COUNTERS, "leaf_policy": _lib.OPT_LEAF_POLICY,
        "sample_groups": _lib.OPT_SAMPLE_GROUPS, "blocks_per_sm": _lib.OPT_BLOCKS_PER_SM,
        "squared_dist": _lib.OPT_SQUARED_DIST, "radius_quantile": _lib.OPT_RADIUS_QUANTILE,
        "keep_scratch": _lib.OPT_KEEP_SCRATCH, "sparse_divisor": _lib.OPT_SPARSE_DIVISOR,
        "approx_filter": _lib.OPT_APPROX_FILTER, "output_chunks": _lib.OPT_OUTPUT_CHUNKS,
        "file_order_chunks": _lib.OPT_FILE_ORDER_CHUNKS, "morton_bits": _lib.OPT_MORTON_BITS,
        "tie_pruning": _lib.OPT_TIE_PRUNING, "warp_round_max": _lib.OPT_WARP_ROUND_MAX, "curve": _lib.OPT_CURVE,
        "speculative_max": _lib.OPT_SPECULATIVE_MAX, "sparse_team": _lib.OPT_SPARSE_TEAM, "sort_mode": _lib.OPT_SORT_MODE,
        "grid": _lib.OPT_GRID, "grid_level": _lib.OPT_GRID_LEVEL,
        "grid_radius_quantile": _lib.OPT_GRID_RADIUS_QUANTILE,
    }

    def set_option(self, name: str, value: int):
        if name not in self._OPTS:
            raise KeyError(name)
        self._check(self._L.tknn_set_option(self._h, self._OPTS[name], int(value)))

    def set_stream(self, cuda_stream: int | None):
        """Run on a caller-owned cudaStream_t (e.g. torch.cuda.current_stream().cuda_stream).

        None = the context's own non-blocking stream.  0 is the LEGACY DEFAULT stream (what torch's default
        current stream is): it is passed as cudaStreamLegacy (0x1) so that the library's work is ordered with the
        caller's kernels and collectives on that stream instead of racing them from a private stream."""
        self._own_stream = cuda_stream is None
        if cuda_stream is None:
            handle = 0
        elif cuda_stream == 0:
            handle = 1  # cudaStreamLegacy
        else:
            handle = cuda_stream
        self._check(self._L.tknn_set_stream(self._h, C.c_void_p(handle)))

    def _settle(self, a):
        """While the context runs on its OWN stream, nothing orders torch's current stream before the library's work:
        a CUDA tensor torch produced there must be complete before the library reads it, and the caching allocator may
        hand back, as an output, a block that a kernel still pending there uses.  Settle torch's stream (nothing to do
        when the context was given torch's stream with set_stream)."""
        if self._own_stream and _is_tensor(a) and a.is_cuda:
            import torch

            torch.cuda.current_stream(a.device).synchronize()

    def _in(self, a, null_if_empty: bool = False):
        """Pointer of an INPUT array (see _settle)."""
        self._settle(a)
        return _ptr(a, null_if_empty)

    def _empty(self, like, shape, np_dtype):
        """An OUTPUT array of `shape` beside `like` (a tensor on its device, or numpy), settled (see _settle)."""
        out = _empty_like_rows(like, shape, np_dtype)
        self._settle(out)
        return out

    def stats(self) -> dict:
        s = Stats()
        self._check(self._L.tknn_get_stats(self._h, C.byref(s)))
        return s.as_dict()

    # ---- the path ----
    def build(self, points, dim: int | None = None, batch=None, batch_size: int | None = None):
        """Build the LBVH over `points` ([n, 2|3] float32; extra columns are skipped through the stride, so columns
        beyond the third are ignored: feature_knn() searches over all columns).

        batch (optional, torch_cluster's convention): one non-decreasing, non-negative integer cloud id per point, numpy
        or a CUDA tensor.  Each cloud then is searched on its own: search(), estimate_start_radius(), range_count() and
        radius_search() only find neighbours in the point's own cloud (tknn_build_segments).  batch_size (optional, with
        batch): the number of clouds, for trailing clouds without points.  A separate query set of a batch takes
        query(..., batch=) / radius_query(..., batch=); without a batch they, search_shard(), dbscan() and brute_force()
        raise TrueKNNError (TKNN_ESTATE) on such a build."""
        points, n, dim, stride = _points(points, "points", dim)
        if batch is None:
            if batch_size is not None:
                raise ValueError("batch_size needs a batch")
            self._check(self._L.tknn_build(self._h, self._in(points), n, dim, stride))
            self.n_segments = 1
            self._offsets = None
        else:
            offsets = batch_to_offsets(batch, n, batch_size)
            self._check(self._L.tknn_build_segments(self._h, self._in(points), n, dim, stride, self._in(offsets),
                                                    int(offsets.shape[0]) - 1))
            self.n_segments = int(offsets.shape[0]) - 1
            self._offsets = offsets
        self.n = n
        self._like = points
        return self

    def search(self, k: int, start_radius: float = 0.0, out=None, indices_only: bool = False):
        """All-points kNN. Returns (idx [n,k] int32, dist [n,k] float32), rows in build order.
        indices_only (or out = (idx, None)): dist_out = NULL — no distances are returned or copied."""
        if out is None:
            idx = self._empty(self._like, (self.n, k), np.int32)
            dist = None if indices_only else self._empty(self._like, (self.n, k), np.float32)
        else:
            idx, dist = out
        _check_dtype(idx, np.int32, "idx_out")
        _check_dtype(dist, np.float32, "dist_out")
        self._check(self._L.tknn_search(self._h, int(k), C.c_float(start_radius), _ptr(idx), _ptr(dist)))
        return idx, dist

    def shard_capacity(self, n_shards: int) -> int:
        return int(self._L.tknn_shard_capacity(self.n, int(n_shards)))

    def search_shard(self, k: int, shard: int, n_shards: int, start_radius: float = 0.0, out=None):
        """Query-sharded search: returns (qid [m], idx [m,k], dist [m,k]) for this shard's Morton slice."""
        cap = self.shard_capacity(n_shards)
        if out is None:
            qid = self._empty(self._like, (cap,), np.int32)
            idx = self._empty(self._like, (cap, k), np.int32)
            dist = self._empty(self._like, (cap, k), np.float32)
        else:
            qid, idx, dist = out
        m = C.c_uint64(0)
        self._check(self._L.tknn_search_shard(self._h, int(k), C.c_float(start_radius), int(shard), int(n_shards), _ptr(qid),
                                              _ptr(idx), _ptr(dist), C.byref(m)))
        m = int(m.value)
        return qid[:m], idx[:m], dist[:m]

    def query(self, queries, k: int, self_ids=None, init_radius2=None, start_radius: float = 0.0, dim: int | None = None,
              batch=None):
        """kNN of a separate query set against the built BVH; rows follow the query order.
        init_radius2: optional per-query cap on the squared distance (closed; negative = none).
        batch (after build(batch=...)): the cloud id of every query, as build()'s; the queries of cloud c search the points
        of cloud c only (tknn_query_segments), and a query whose cloud has too few points ends in -1 / FLT_MAX."""
        queries, nq, dim, stride = _points(queries, "queries", dim)
        self_ids = _arg(self_ids, np.int32, "self_ids")
        init_radius2 = _arg(init_radius2, np.float32, "init_radius2")
        idx = self._empty(queries, (nq, k), np.int32)
        dist = self._empty(queries, (nq, k), np.float32)
        if batch is None:
            self._check(self._L.tknn_query(self._h, self._in(queries), nq, dim, stride, self._in(self_ids),
                                           self._in(init_radius2), int(k), C.c_float(start_radius), _ptr(idx), _ptr(dist)))
        else:
            offsets = batch_to_offsets(batch, nq, self.n_segments)
            self._check(self._L.tknn_query_segments(self._h, self._in(queries), nq, dim, stride, self._in(offsets),
                                                    int(offsets.shape[0]) - 1, self._in(self_ids), self._in(init_radius2),
                                                    int(k), C.c_float(start_radius), _ptr(idx), _ptr(dist)))
        return idx, dist

    def range_count(self, radius: float):
        """Neighbours within the closed ball of `radius` for every point (DBSCAN core-point test; see dbscan()): uint32
        numpy, or an int32 tensor for a build from a tensor."""
        out = self._empty(self._like, (self.n,), np.uint32)
        self._check(self._L.tknn_range_count(self._h, C.c_float(radius), _ptr(out)))
        return out

    def dbscan(self, eps: float, min_pts: int, with_core: bool = True, out=None):
        """Exact DBSCAN of the built cloud (closed eps-ball, min_pts counts the point itself: scikit-learn's min_samples).

        Returns (labels [n] int32: cluster id in 0 .. C-1 or -1 for noise, core [n] uint8: 1 = core point (None when
        with_core is False), C).  Clusters are numbered in ascending order of their smallest core index; a border point
        takes the lowest id among the clusters of the core points in its ball.  numpy outputs for numpy input, CUDA
        tensors for CUDA tensor input; out = (labels, core) supplies the arrays (core may be None)."""
        if out is not None:
            labels, core = out
        else:
            labels = self._empty(self._like, (self.n,), np.int32)
            core = self._empty(self._like, (self.n,), np.uint8) if with_core else None
        _check_dtype(labels, np.int32, "labels")
        _check_dtype(core, np.uint8, "core")
        c = C.c_uint64(0)
        self._check(self._L.tknn_dbscan(self._h, C.c_float(eps), int(min_pts), _ptr(labels), _ptr(core), C.byref(c)))
        return labels, core, int(c.value)

    def cloud_sizes(self) -> np.ndarray:
        """Points per cloud of the last build (int64 numpy; [n] for a plain build)."""
        if self._offsets is None:
            return np.array([self.n], np.int64)
        off = self._offsets.cpu().numpy() if _is_tensor(self._offsets) else self._offsets
        return np.diff(off.astype(np.int64))

    def fps(self, num_samples=None, ratio: float | None = None, start=None, with_dist: bool = False, out=None):
        """Exact farthest point sampling of every cloud of the last build (tknn_fps; torch_cluster's fps selection rule).

        Exactly one of num_samples (an int for a plain build, or one count per cloud) and ratio (in (0, 1]: cloud s gets
        ceil(float32(n_s) * float32(ratio)) samples, fps_counts) is given.  start: None (the first point of every cloud)
        or one global index per cloud.  Sample 0 of a cloud is its start; each next sample is the point farthest from the
        samples so far (squared fp32 distance, ties to the lowest index).  Returns (idx [M] int32: global indices, cloud
        by cloud; dist [M] float32 or None: the distance of each sample from the earlier ones when it was picked, FLT_MAX
        for sample 0, d2 while squared_dist is set).  numpy outputs for numpy input, CUDA tensors for CUDA tensor input;
        out = (idx, dist) supplies the arrays (dist may be None)."""
        sizes = self.cloud_sizes()
        if (num_samples is None) == (ratio is None):
            raise ValueError("give exactly one of num_samples and ratio")
        if ratio is not None:
            counts = fps_counts(sizes, ratio)
        else:
            counts = np.atleast_1d(np.asarray(num_samples, dtype=np.int64))
            if counts.shape != sizes.shape:
                raise ValueError(f"num_samples: one count per cloud ({sizes.shape[0]}), got {counts.shape[0]}")
        if (counts < 0).any():
            raise ValueError("num_samples must be >= 0")
        soff = np.concatenate([[0], np.cumsum(counts)]).astype(np.uint64)
        total = int(soff[-1])
        start = _arg(start, np.int32, "start")  # a scalar becomes [1]
        if start is not None and int(start.shape[0]) != sizes.shape[0]:
            raise ValueError(f"start: one index per cloud ({sizes.shape[0]}), got {int(start.shape[0])}")
        if out is not None:
            idx, dist = out
        else:
            idx = self._empty(self._like, (total,), np.int32)
            dist = self._empty(self._like, (total,), np.float32) if with_dist else None
        _check_dtype(idx, np.int32, "idx")
        _check_dtype(dist, np.float32, "dist")
        if total:  # an empty torch tensor has no address, and there is nothing to sample
            self._check(self._L.tknn_fps(self._h, _ptr(soff), sizes.shape[0], self._in(start), _ptr(idx), _ptr(dist)))
        return idx, dist

    def feature_knn(self, x, y, k: int, batch_x=None, batch_y=None, self_ids=None, indices_only: bool = False):
        """Exact k nearest rows of x for every row of y in feature space (tknn_feature_knn): all f = x.shape[1] columns
        count, d2 = fmaf chain over the columns in order (include/trueknn.h).  Needs no build and leaves the last build
        untouched.  batch_x / batch_y (optional, torch_cluster's convention): cloud ids of the rows; the rows of y in
        cloud c search the rows of x in cloud c only (batch_size = max over both + 1; a missing one is all zeros).
        self_ids (optional): per row of y, a global index into x to exclude (-1 or outside its cloud: none).  Returns
        (idx [nq, k] int32, dist [nq, k] float32 or None when indices_only); rows ascend by (d2, index) and end in -1 /
        FLT_MAX when the cloud has fewer eligible rows; dist is d2 while squared_dist is set.  numpy outputs for numpy
        input, CUDA tensors (on x's device) for CUDA tensor input.  float32 only."""
        x, y = _arg(x, np.float32, "x"), _arg(y, np.float32, "y")
        if x.ndim != 2 or y.ndim != 2:
            raise ValueError("x and y must be [rows, f]")
        n, f, nq = int(x.shape[0]), int(x.shape[1]), int(y.shape[0])
        if int(y.shape[1]) != f:
            raise ValueError(f"x has {f} columns, y has {int(y.shape[1])}")
        self_ids = _arg(self_ids, np.int32, "self_ids")
        x_off = y_off = None
        n_seg = 1
        if (batch_x is not None or batch_y is not None) and n and nq:
            bx, by, size = _bipartite_setup(x, y, batch_x, batch_y)
            x_off, y_off = batch_to_offsets(bx, n, size), batch_to_offsets(by, nq, size)
            n_seg = size
        idx = self._empty(y, (nq, k), np.int32)
        dist = None if indices_only else self._empty(y, (nq, k), np.float32)
        if nq == 0:  # an empty torch tensor has no address, and there is nothing to search
            return idx, dist
        self._check(self._L.tknn_feature_knn(self._h, self._in(x), n, f, f, self._in(x_off), self._in(y), nq, f,
                                             self._in(y_off), n_seg, self._in(self_ids), int(k), _ptr(idx), _ptr(dist)))
        return idx, dist

    def voxel_grid(self, points, size, start=None, end=None, batch=None, batch_size: int | None = None):
        """Exact voxel-grid clustering of `points` ([n, >= 2] float32, the first 2 or 3 columns are the position;
        tknn_voxel_grid).  size: a scalar or one value per axis; start / end (optional): the same, by default the column
        min / max.  Raw id: torch_cluster's grid rule, c = sum_d (int64) fl(fl(p_d - start_d) / size_d) * m_d with m_d
        the product of the cell counts (int64) fl(fl(end_e - start_e) / size_e) + 1 of the earlier axes, truncation
        toward zero, evaluated in fp32 as written.  batch (optional, torch_cluster's convention) adds the cloud id as a
        last column of size 1, as PyG's voxel_grid does; batch_size pads trailing empty clouds.  Returns (raw [n] int64,
        cluster [n] int32: the rank of the raw id among the distinct ones, n_voxels).  numpy outputs for numpy input,
        CUDA tensors for CUDA tensor input.  The clustering stays in the context for voxel_members() and voxel_pool()
        until the next voxel_grid(); builds and searches do not touch it.  Unlike torch_cluster, ids that leave int64
        are rejected (TrueKNNError, TKNN_EINVAL) instead of wrapping."""
        points, dim, size, start, end = _voxel_args(points, size, start, end)
        n = int(points.shape[0])
        raw = self._empty(points, (n,), np.int64)
        cluster = self._empty(points, (n,), np.int32)
        offsets, n_seg = None, 1
        if batch is not None:
            offsets = batch_to_offsets(batch, n, batch_size)
            n_seg = int(offsets.shape[0]) - 1
        nv = C.c_uint64()
        self._check(self._L.tknn_voxel_grid(self._h, self._in(points, null_if_empty=True), n, dim, int(points.shape[1]),
                                            self._in(offsets), n_seg, _ptr(size), _ptr(start), _ptr(end),
                                            _ptr(raw, null_if_empty=True), _ptr(cluster, null_if_empty=True),
                                            C.byref(nv)))
        self._vx_like = points
        self._vx_n = n
        self._vx_nv = int(nv.value)
        return raw, cluster, self._vx_nv

    def voxel_members(self):
        """Members of the last voxel_grid()'s voxels (tknn_voxel_members): (offsets [nv + 1] CSR offsets, uint64 numpy or
        int64 tensor; members [n] int32 point indices voxel by voxel, ascending inside a voxel; first [nv] int32 the
        lowest point index of each voxel (PyG's consecutive_cluster returns an arbitrary member); seg [nv] int32 the
        cloud of each voxel)."""
        like = self._vx_like
        if like is None:
            raise TrueKNNError(_lib.ESTATE, "voxel_members before voxel_grid")
        n, nv = self._vx_n, self._vx_nv
        offsets = self._empty(like, (nv + 1,), np.uint64)
        members = self._empty(like, (n,), np.int32)
        first = self._empty(like, (nv,), np.int32)
        seg = self._empty(like, (nv,), np.int32)
        self._check(self._L.tknn_voxel_members(self._h, _ptr(offsets), _ptr(members, null_if_empty=True),
                                               _ptr(first, null_if_empty=True), _ptr(seg, null_if_empty=True)))
        return offsets, members, first, seg

    def voxel_pool(self, x, reduce: str = "mean"):
        """Pools the rows of x ([n] or [n, f] float32, 1 <= f <= 1024, n the clustering's point count) over the last
        voxel_grid() (tknn_voxel_pool).  Returns [n_voxels, f] float32.  reduce="mean": members in ascending index in
        chunks of 32, each chunk summed from +0 in order, the chunk sums summed in order, divided by the count, all in
        fp32 (no atomics, so the result is the same on every run); reduce="max": the first maximum in index order, and
        a non-finite value in x is TKNN_EINVAL.  Call it any number of times per clustering."""
        if reduce not in ("mean", "max"):
            raise ValueError(f"reduce must be 'mean' or 'max', got {reduce!r}")
        if self._vx_like is None:
            raise TrueKNNError(_lib.ESTATE, "voxel_pool before voxel_grid")
        x = _arg(x, np.float32, "x")
        if x.ndim == 1:
            x = x.reshape(-1, 1)
        if x.ndim != 2:
            raise ValueError("x must be [n] or [n, f]")
        n, f = int(x.shape[0]), int(x.shape[1])
        out = self._empty(x, (self._vx_nv, f), np.float32)
        code = _lib.REDUCE_MAX if reduce == "max" else _lib.REDUCE_MEAN
        self._check(self._L.tknn_voxel_pool(self._h, self._in(x, null_if_empty=True), n, f, f, code,
                                            _ptr(out, null_if_empty=True)))
        return out

    def interpolate(self, idx, d2, x):
        """k-NN interpolation of the rows of x ([n, f] float32) at nq query rows (tknn_interpolate): idx [nq, k] int32 and
        d2 [nq, k] float32 are kNN rows with squared distances (query() with squared_dist=1), -1 slots skipped.  Per row,
        w = 1 / max(d2, 1e-16), out = sum_s fl(x[idx_s] * w_s) / sum_s w_s, both sums in slot order from +0 in fp32, so
        the result is PyG's knn_interpolate on the same neighbours, bit for bit on every run.  Returns (out [nq, f],
        weight [nq, k] (+0 for skipped slots), den [nq]), the inputs of interpolate_backward().  Needs no build and
        leaves the last build untouched.  numpy outputs for numpy x, CUDA tensors (on x's device) for a CUDA tensor."""
        x = _arg(x, np.float32, "x", ndim=2, cast=False, copy=True)
        idx = _arg(idx, np.int32, "idx", ndim=2, copy=True)
        d2 = _arg(d2, np.float32, "d2", ndim=2, copy=True)
        nq, k = int(idx.shape[0]), int(idx.shape[1])
        if tuple(d2.shape) != (nq, k):
            raise ValueError(f"d2 has shape {tuple(d2.shape)}, idx {(nq, k)}")
        n, f = int(x.shape[0]), int(x.shape[1])
        out = self._empty(x, (nq, f), np.float32)
        weight = self._empty(x, (nq, k), np.float32)
        den = self._empty(x, (nq,), np.float32)
        if nq == 0:  # an empty torch tensor has no address, and there is nothing to compute
            return out, weight, den
        self._check(self._L.tknn_interpolate(self._h, self._in(idx), self._in(d2), nq, k, self._in(x, null_if_empty=True),
                                             n, f, f, _ptr(out), _ptr(weight), _ptr(den)))
        return out, weight, den

    def interpolate_backward(self, idx, weight, den, grad_out, n: int):
        """Gradient of interpolate()'s out with respect to x (tknn_interpolate_backward): grad_x [n, f] with
        grad_x[j] = sum over the slots (i, s) with idx[i, s] = j, in ascending i * k + s, of fl(fl(grad_out[i] / den[i]) *
        weight[i, s]), from +0 in fp32; +0 for a row no slot references.  No float atomics: the same bits on every run.
        idx / weight / den: what interpolate() took and returned; grad_out: [nq, f] float32.  numpy outputs for numpy
        grad_out, CUDA tensors for a CUDA tensor."""
        g = _arg(grad_out, np.float32, "grad_out", ndim=2, cast=False, copy=True)
        idx = _arg(idx, np.int32, "idx", ndim=2, copy=True)
        weight = _arg(weight, np.float32, "weight", ndim=2, copy=True)
        den = _arg(den, np.float32, "den")
        nq, k, f, n = int(idx.shape[0]), int(idx.shape[1]), int(g.shape[1]), int(n)
        if tuple(weight.shape) != (nq, k) or tuple(den.shape) != (nq,) or int(g.shape[0]) != nq:
            raise ValueError(f"shapes idx {tuple(idx.shape)}, weight {tuple(weight.shape)}, den {tuple(den.shape)}, "
                             f"grad_out {tuple(g.shape)} do not match")
        grad_x = self._empty(g, (n, f), np.float32)
        if nq == 0:  # no slot references a row
            grad_x[:] = 0
            return grad_x
        self._check(self._L.tknn_interpolate_backward(self._h, self._in(idx), self._in(weight), self._in(den), nq, k,
                                                      self._in(g), f, n, f, _ptr(grad_x, null_if_empty=True)))
        return grad_x

    def radius_search(self, radius: float, indices_only: bool = False, out=None):
        """Exact fixed-radius neighbour lists of every built point (closed ball, the point itself excluded).

        Returns CSR (offsets [n + 1] int64, idx [total] int32, dist [total] float32 or None when indices_only): row q is
        idx[offsets[q]:offsets[q + 1]], sorted by (distance, index), rows in build order; dist is d2 while squared_dist
        is set.  numpy outputs for numpy input, CUDA tensors for CUDA tensor input, so that
        torch.sparse_csr_tensor(offsets, idx, dist) works directly.  Without `out` a size call comes first;
        out = (offsets, idx, dist) (dist may be None) makes one call and raises TrueKNNError naming the total needed
        when idx is too short."""
        def call(off, idx, dist, cap, total):
            return self._L.tknn_radius_search(self._h, C.c_float(radius), _ptr(off), _ptr(idx), _ptr(dist), cap,
                                              C.byref(total))

        return self._radius_lists(self._like, self.n, indices_only, out, call)

    def radius_query(self, queries, radius: float, self_ids=None, dim: int | None = None, indices_only: bool = False,
                     out=None, batch=None):
        """Exact fixed-radius neighbour lists of a separate query set (rows in query order); self_ids (optional, -1 =
        none) names the data index each query excludes.  Returns (offsets, idx, dist) as radius_search().
        batch (after build(batch=...)): the cloud id of every query; the ball of a query holds points of its own cloud
        only (tknn_radius_query_segments)."""
        queries, nq, dim, stride = _points(queries, "queries", dim)
        self_ids = _arg(self_ids, np.int32, "self_ids")
        q_ptr, sid_ptr = self._in(queries), self._in(self_ids)
        if batch is not None:
            q_off = batch_to_offsets(batch, nq, self.n_segments)
            off_ptr, n_seg = self._in(q_off), int(q_off.shape[0]) - 1

        def call(off, idx, dist, cap, total):
            if batch is not None:
                return self._L.tknn_radius_query_segments(self._h, q_ptr, nq, dim, stride, off_ptr, n_seg, sid_ptr,
                                                          C.c_float(radius), _ptr(off), _ptr(idx), _ptr(dist), cap,
                                                          C.byref(total))
            return self._L.tknn_radius_query(self._h, q_ptr, nq, dim, stride, sid_ptr, C.c_float(radius), _ptr(off),
                                             _ptr(idx), _ptr(dist), cap, C.byref(total))

        return self._radius_lists(queries, nq, indices_only, out, call)

    def _radius_lists(self, like, nq: int, indices_only: bool, out, call):
        total = C.c_uint64(0)
        if out is not None:
            offsets, idx, dist = out
            _check_dtype(idx, np.int32, "idx")
            _check_dtype(dist, np.float32, "dist")
            if _is_tensor(offsets):
                _check_dtype(offsets, np.uint64, "offsets")
            elif offsets.dtype not in (np.int64, np.uint64):
                raise TypeError(f"offsets: expected int64, got {offsets.dtype}")
            if int(offsets.shape[0]) < nq + 1:
                raise ValueError(f"offsets holds {int(offsets.shape[0])} entries, {nq + 1} needed")
            cap = int(idx.shape[0]) if dist is None else min(int(idx.shape[0]), int(dist.shape[0]))
            rc = call(offsets, idx, dist, cap, total)
            if rc == _lib.EINVAL and total.value > cap:
                raise TrueKNNError(rc, f"the neighbour lists hold {total.value} entries, out has room for {cap}")
            self._check(rc)
            t = int(total.value)
            return offsets, idx[:t], dist[:t] if dist is not None else None
        offsets = self._empty(like, (nq + 1,), np.int64)
        self._check(call(offsets, None, None, 0, total))
        t = int(total.value)
        idx = self._empty(like, (t,), np.int32)
        dist = None if indices_only else self._empty(like, (t,), np.float32)
        if t:
            self._check(call(offsets, idx, dist, t, total))
        return offsets, idx, dist

    def estimate_start_radius(self, k: int) -> float:
        r = C.c_float(0)
        self._check(self._L.tknn_estimate_start_radius(self._h, int(k), C.byref(r)))
        return float(r.value)

    def brute_force(self, query_ids, k: int):
        """Exact tiled brute force on the GPU for selected data indices (second oracle)."""
        query_ids = _arg(query_ids, np.int32, "query_ids")
        nq = int(query_ids.shape[0])
        idx = self._empty(query_ids, (nq, k), np.int32)
        dist = self._empty(query_ids, (nq, k), np.float32)
        self._check(self._L.tknn_brute_force(self._h, self._in(query_ids), nq, int(k), _ptr(idx), _ptr(dist)))
        return idx, dist

    def merge_topk(self, idx_parts, d2_parts):
        """Merge [parts, nq, k] (idx, d2) device lists on (d2, index); returns (idx, dist=sqrt(d2))."""
        parts, nq, k = (int(x) for x in idx_parts.shape)
        idx = self._empty(idx_parts, (nq, k), np.int32)
        dist = self._empty(idx_parts, (nq, k), np.float32)
        self._check(self._L.tknn_merge_topk(self._h, self._in(idx_parts), self._in(d2_parts), parts, nq, k, _ptr(idx), _ptr(dist)))
        return idx, dist

    # ---- multi-GPU, one rank per process (include/trueknn.h "multi-GPU" (b)) ----
    @staticmethod
    def unique_id() -> bytes:
        """128 bytes from ncclGetUniqueId: rank 0 creates them, every rank passes them to comm_init."""
        L = _lib.load()
        buf = C.create_string_buffer(_lib.UNIQUE_ID_BYTES)
        rc = L.tknn_comm_unique_id(buf)
        if rc != _lib.OK:
            raise TrueKNNError(rc, "tknn_comm_unique_id failed (libnccl.so.2 not loadable?)")
        return buf.raw

    def comm_init(self, n_ranks: int, rank: int, unique_id: bytes):
        if len(unique_id) != _lib.UNIQUE_ID_BYTES:
            raise ValueError("unique_id must be 128 bytes")
        self._check(self._L.tknn_comm_init(self._h, int(n_ranks), int(rank), C.c_char_p(unique_id)))
        self.rank, self.n_ranks = int(rank), int(n_ranks)
        return self

    def comm_init_torch(self, group=None):
        """Communicator over the ranks of a torch.distributed group: the unique id travels through the group."""
        import torch.distributed as dist

        rank, world = dist.get_rank(group), dist.get_world_size(group)
        box = [self.unique_id() if rank == 0 else None]
        dist.broadcast_object_list(box, src=dist.get_global_rank(group, 0) if group is not None else 0, group=group)
        return self.comm_init(world, rank, box[0])

    def dist_stats(self) -> dict:
        s = _lib.DistStats()
        self._check(self._L.tknn_get_dist_stats(self._h, C.byref(s)))
        return s.as_dict()

    def build_replicated(self, local_points, first: int, n_total: int, dim: int | None = None):
        """TKNN_SHARD_QUERIES build: this rank's contiguous slice in, the replicated LBVH out (one ncclAllGather)."""
        local_points, n, dim, stride = _points(local_points, "local_points", dim)
        self._check(self._L.tknn_build_replicated(self._h, self._in(local_points), n, int(first), int(n_total), dim,
                                                  stride))
        self.n = int(n_total)
        self.n_segments = 1
        self._like = local_points
        return self

    def partition_build(self, local_points, first_index: int, dim: int | None = None):
        """TKNN_PARTITION_POINTS build: rows of global indices first_index.. in, one Morton range of the cloud owned."""
        local_points, n, dim, stride = _points(local_points, "local_points", dim)
        self._check(self._L.tknn_partition_build(self._h, self._in(local_points), n, int(first_index), dim, stride))
        self.n = int(self._L.tknn_partition_owned(self._h))
        self.n_segments = 1
        self._like = local_points
        return self

    def partition_owned(self) -> int:
        return int(self._L.tknn_partition_owned(self._h))

    def partition_search(self, k: int, start_radius: float = 0.0, out=None):
        """Exact kNN of the owned points against the global cloud: (gid [m], idx [m,k] global ids, dist [m,k])."""
        m = self.partition_owned()
        if out is None:
            gid = self._empty(self._like, (m,), np.int32)
            idx = self._empty(self._like, (m, k), np.int32)
            dist = self._empty(self._like, (m, k), np.float32)
        else:
            gid, idx, dist = out
        got = C.c_uint64(0)
        self._check(self._L.tknn_partition_search(self._h, int(k), C.c_float(start_radius), _ptr(gid), _ptr(idx), _ptr(dist),
                                                  int(gid.shape[0]), C.byref(got)))
        g = int(got.value)
        return gid[:g], idx[:g], dist[:g]

    def partition_verify(self, k: int, samples: int, gid, idx, dist):
        """Distributed brute-force check of `samples` sampled rows per rank; returns GLOBAL (checked, bad)."""
        a, b = C.c_uint64(0), C.c_uint64(0)
        self._check(self._L.tknn_partition_verify(self._h, int(k), int(samples), self._in(gid), self._in(idx), self._in(dist),
                                                  int(gid.shape[0]), C.byref(a), C.byref(b)))
        return int(a.value), int(b.value)

    # ---- introspection (tests / bench) ----
    def sort_pairs(self, keys, values=None):
        n = int(keys.shape[0])
        self._check(self._L.tknn_sort_pairs(self._h, self._in(keys), self._in(values), n))
        return keys, values

    def get_bvh(self):
        """Host copies: nodes [n_nodes,16] float32 (bit views for refs), points [n,4] float32, leaf_start [n_leaves+1]."""
        st = self.stats()
        nodes = np.empty((st["n_nodes"], 16), np.float32)
        pts = np.empty((self.n, 4), np.float32)
        leaf_start = np.empty((st["n_leaves"] + 1,), np.uint32)
        self._check(self._L.tknn_get_bvh(self._h, _ptr(nodes), _ptr(pts), _ptr(leaf_start)))
        return nodes, pts, leaf_start

    def morton_codes(self, points, box6, dim: int | None = None):
        """63-bit Morton codes on the cubic grid over `box6` = (lo.xyz, hi.xyz); int64/uint64 [n]."""
        points, n, dim, stride = _points(points, "points", dim)
        out = self._empty(points, (n,), np.uint64)
        if _is_tensor(points):
            import torch

            box = torch.as_tensor(box6, dtype=torch.float32).cpu().contiguous().numpy()
        else:
            box = np.ascontiguousarray(box6, dtype=np.float32)
        self._check(self._L.tknn_morton_codes(self._h, self._in(points), n, dim, stride, _ptr(box), _ptr(out)))
        return out

    def reach_mask(self, points, reach2, box6, summaries, self_rank: int, cell_bits: int = 3):
        """Bit mask of the remote ranks whose per-cell summary boxes the ball (p, sqrt(reach2)) touches (CUDA tensors)."""
        import torch

        n, stride = int(points.shape[0]), int(points.shape[1])
        n_ranks = int(summaries.shape[0])
        box = torch.as_tensor(box6, dtype=torch.float32, device=points.device).contiguous()
        summ = summaries.contiguous()
        out = self._empty(points, (n,), np.int32)
        self._check(self._L.tknn_reach_mask(self._h, self._in(points), n, stride, self._in(reach2.contiguous()), self._in(box),
                                            self._in(summ), n_ranks, int(cell_bits), int(self_rank), _ptr(out)))
        return out

    def generate_uniform(self, seed: int, first: int, n: int, out=None):
        if out is None:
            out = np.empty((n, 3), np.float32)
        self._check(self._L.tknn_generate_uniform(self._h, int(seed), int(first), int(n), _ptr(out)))
        return out

    def measure_bandwidth(self) -> dict:
        l2, hbm, sms, l2b = C.c_double(0), C.c_double(0), C.c_int(0), C.c_uint64(0)
        self._check(self._L.tknn_measure_bandwidth(self._h, C.byref(l2), C.byref(hbm), C.byref(sms), C.byref(l2b)))
        return {"l2_gbs": l2.value, "hbm_read_gbs": hbm.value, "sm_count": sms.value, "l2_bytes": int(l2b.value)}

    def measure_smem_bandwidth(self) -> dict:
        a, b = C.c_double(0), C.c_double(0)
        self._check(self._L.tknn_measure_smem_bandwidth(self._h, C.byref(a), C.byref(b)))
        return {"smem_conflict_free_gbs": a.value, "smem_broadcast_gbs": b.value}


class _RankView(TrueKNN):
    """A rank's context inside a MultiTrueKNN (owned by it): statistics and options only."""

    def __init__(self, L, handle, device: int):  # noqa: D401 — no tknn_create here
        self._L, self._h = L, handle
        self._init_state(device)

    def close(self):
        self._h = None


class MultiTrueKNN:
    """All devices from ONE process (`tknn_create_multi`): the device-list form of the reference's context
    (owlContextCreate(ids, n), owl/include/owl/owl_host.h:360).  Host arrays in, host arrays in file order out.

    mode: "shard" (BVH replicated, queries sharded) or "partition" (points partitioned by Morton range).
    Naming one device several times runs that many ranks on it (how the single-GPU tests exercise the paths)."""

    MODES = {"shard": _lib.SHARD_QUERIES, "partition": _lib.PARTITION_POINTS}

    def __init__(self, device_ids, mode: str = "shard", **options):
        self._L = _lib.load()
        self._device_ids = [int(d) for d in device_ids]  # rank r runs on device_ids[r]
        ids = (C.c_int * len(device_ids))(*self._device_ids)
        h = C.c_void_p()
        rc = self._L.tknn_create_multi(ids, len(device_ids), self.MODES[mode], C.byref(h))
        if rc != _lib.OK:
            raise TrueKNNError(rc, f"tknn_create_multi({list(device_ids)}, {mode}) failed")
        self._h, self.mode, self.n = h, mode, 0
        for name, v in options.items():
            self.set_option(name, v)

    def _check(self, rc):
        if rc != _lib.OK:
            raise TrueKNNError(rc, self._L.tknn_multi_last_error(self._h).decode())

    def set_option(self, name: str, value: int):
        self._check(self._L.tknn_multi_set_option(self._h, TrueKNN._OPTS[name], int(value)))

    @property
    def n_ranks(self) -> int:
        return int(self._L.tknn_multi_ranks(self._h))

    def rank(self, r: int) -> TrueKNN:
        return _RankView(self._L, C.c_void_p(self._L.tknn_multi_ctx(self._h, int(r))), self._device_ids[int(r)])

    def build(self, points, dim: int | None = None):
        points = np.ascontiguousarray(points, dtype=np.float32)
        stride = int(points.shape[1])
        if dim is None:
            dim = min(stride, 3)
        self._check(self._L.tknn_multi_build(self._h, _ptr(points), int(points.shape[0]), int(dim), stride))
        self.n = int(points.shape[0])
        return self

    def search(self, k: int, start_radius: float = 0.0, out=None):
        idx, dist = out if out is not None else (np.empty((self.n, k), np.int32), np.empty((self.n, k), np.float32))
        self._check(self._L.tknn_multi_search(self._h, int(k), C.c_float(start_radius), _ptr(idx), _ptr(dist)))
        return idx, dist

    def times(self) -> dict:
        t = (C.c_float * 4)()
        self._check(self._L.tknn_multi_get_times(self._h, t))
        return {"build_ms": t[0], "search_ms": t[1], "exchange_ms": t[2], "d2h_ms": t[3]}

    def close(self):
        if getattr(self, "_h", None):
            self._L.tknn_multi_destroy(self._h)
            self._h = None

    def __enter__(self):
        return self

    def __exit__(self, *exc):
        self.close()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


# ------------------------------------------------------------------------------------------------
# The sample's command line (hostCode.cpp:66-73) as a function.
# ------------------------------------------------------------------------------------------------
_FLOAT_RE = re.compile(r"[+-]?(?:\d+\.?\d*|\.\d+)(?:[eE][+-]?\d+)?")


def batch_to_offsets(batch, n: int, batch_size: int | None = None):
    """Cloud ids per point (torch_cluster's `batch`: non-decreasing, non-negative integers) -> the n_clouds + 1 segment
    offsets of tknn_build_segments, by bincount + cumsum on the batch's own device: uint64 numpy for numpy input, an
    int64 tensor for a tensor.  Cloud c is the points [offsets[c], offsets[c + 1]); ids that no point carries are empty
    clouds.  batch_size (optional): n_clouds, padding with trailing empty clouds.  Raises ValueError for a batch that is
    not 1-D of length n, not integer, negative or decreasing, for a batch_size below 1 and for an id >= batch_size."""
    if batch_size is not None and int(batch_size) < 1:
        raise ValueError(f"batch_size = {batch_size} must be >= 1")
    if _is_tensor(batch):
        import torch

        if batch.dim() != 1 or int(batch.shape[0]) != n:
            raise ValueError(f"batch must be 1-D with one entry per point ({n})")
        if batch.dtype.is_floating_point or batch.dtype == torch.bool:
            raise ValueError(f"batch must hold integer cloud ids, got {batch.dtype}")
        b = batch.to(torch.int64)
        if n == 0:
            return torch.zeros((1 if batch_size is None else int(batch_size) + 1,), dtype=torch.int64, device=b.device)
        if bool((b[0] < 0).item()) or (n > 1 and bool((b[1:] < b[:-1]).any().item())):
            raise ValueError("batch must be non-negative and non-decreasing (the points of a cloud are contiguous)")
        last = int(b[-1].item())
        if batch_size is not None and last >= int(batch_size):
            raise ValueError(f"batch holds cloud id {last} >= batch_size = {batch_size}")
        counts = torch.bincount(b, minlength=last + 1 if batch_size is None else int(batch_size))
        return torch.cat([torch.zeros((1,), dtype=torch.int64, device=b.device), torch.cumsum(counts, 0)]).contiguous()
    b = np.asarray(batch)
    if b.ndim != 1 or b.shape[0] != n:
        raise ValueError(f"batch must be 1-D with one entry per point ({n})")
    if not np.issubdtype(b.dtype, np.integer):
        raise ValueError(f"batch must hold integer cloud ids, got {b.dtype}")
    b = b.astype(np.int64)
    if n == 0:
        return np.zeros(1 if batch_size is None else int(batch_size) + 1, np.uint64)
    if b[0] < 0 or (n > 1 and bool((b[1:] < b[:-1]).any())):
        raise ValueError("batch must be non-negative and non-decreasing (the points of a cloud are contiguous)")
    if batch_size is not None and int(b[-1]) >= int(batch_size):
        raise ValueError(f"batch holds cloud id {int(b[-1])} >= batch_size = {batch_size}")
    counts = np.bincount(b, minlength=int(b[-1]) + 1 if batch_size is None else int(batch_size))
    return np.concatenate([[0], np.cumsum(counts)]).astype(np.uint64)


def fps_counts(sizes, ratio: float) -> np.ndarray:
    """Samples per cloud for a ratio, torch_cluster's rule: ceil(float32(n_s) * float32(ratio)), at most n_s, so an empty
    cloud gets 0.  ratio must lie in (0, 1]."""
    if not 0.0 < float(ratio) <= 1.0:
        raise ValueError(f"ratio = {ratio} must lie in (0, 1]")
    n = np.asarray(sizes, dtype=np.int64)
    return np.minimum(np.ceil(n.astype(np.float32) * np.float32(ratio)).astype(np.int64), n)


def fps_random_starts(offsets, like=None):
    """One uniformly drawn start per cloud, as a global index, from the global RNG of `like`'s framework: torch.randint
    on the tensor's device, numpy's global generator otherwise.  offsets: the n_clouds + 1 cloud offsets (numpy); an
    empty cloud gets its offset (it has no samples).  Returns int32 on `like`'s device, or numpy."""
    off = np.asarray(offsets, dtype=np.int64)
    sizes = np.maximum(np.diff(off), 1)
    if _is_tensor(like):
        import torch

        r = torch.randint(0, 2**62, (sizes.shape[0],), dtype=torch.int64, device=like.device)
        base = torch.as_tensor(off[:-1], device=like.device)
        return (base + r % torch.as_tensor(sizes, device=like.device)).to(torch.int32)
    return (off[:-1] + np.random.randint(0, sizes)).astype(np.int32)


def fps(src, batch=None, ratio: float = 0.5, random_start: bool = True, batch_size: int | None = None,
        device: int | None = None):
    """torch_cluster.fps(src, batch, ratio, random_start, batch_size) on the GPU, exact: farthest point sampling of every
    cloud, ceil(n_s * ratio) samples each (fps_counts).  Returns int64 global indices, concatenated cloud by cloud, each
    cloud's samples in the order they were picked.  random_start draws each cloud's first sample from the global RNG of
    the input's framework (fps_random_starts); otherwise it is the cloud's first point.  numpy in, numpy out; a CUDA
    tensor in, a tensor on its device out (device: the CUDA device for numpy input, default 0)."""
    n = int(src.shape[0])
    if n == 0:
        fps_counts([0], ratio)  # the same argument check
        return _zeros_like_rows(src, (0,), np.int64)
    with TrueKNN(_device_of(src, device)) as t:
        t.build(src, batch=batch, batch_size=batch_size)
        sizes = t.cloud_sizes()
        start = fps_random_starts(np.concatenate([[0], np.cumsum(sizes)]), src) if random_start else None
        idx, _ = t.fps(ratio=ratio, start=start)
    return _int64(idx)


def _voxel_args(points, size, start, end, all_columns=False):
    """Host-side checks of voxel_grid(): (points, dim, size, start, end) with size / start / end as float32 numpy of
    dim entries (scalars broadcast).  Raises ValueError for a shape, a non-finite value or a size <= 0.  all_columns:
    every column of points is a coordinate (torch_cluster's and PyG's signatures), so more than 3 is an error rather
    than columns skipped through the stride."""
    points = _arg(points, np.float32, "points")
    if points.ndim != 2 or int(points.shape[1]) < 2:
        raise ValueError("points must be [n, >= 2] (2-D or 3-D positions)")
    if all_columns and int(points.shape[1]) > 3:
        raise ValueError(f"pos has {int(points.shape[1])} columns: only 2-D and 3-D positions are supported")
    dim = min(int(points.shape[1]), 3)

    def axes(v, name):
        if v is None:
            return None
        if _is_tensor(v):
            v = v.detach().cpu().numpy()
        a = np.asarray(v, dtype=np.float32).reshape(-1)
        if a.shape[0] == 1:
            a = np.repeat(a, dim)
        if a.shape[0] != dim:
            raise ValueError(f"{name}: a scalar or {dim} values, got {a.shape[0]}")
        if not np.isfinite(a).all():
            raise ValueError(f"{name} must be finite")
        return np.ascontiguousarray(a)

    size = axes(size, "size")
    if size is None or not (size > 0).all():
        raise ValueError("size must be > 0 on every axis")
    return points, dim, size, axes(start, "start"), axes(end, "end")


def _device_of(a, device):
    return a.device.index if _is_tensor(a) else (device or 0)


def grid_cluster(pos, size, start=None, end=None, device: int | None = None):
    """torch_cluster.grid_cluster(pos, size, start, end) on the GPU, exact: the raw voxel id of every point (int64), by
    torch_cluster's rule in fp32 (TrueKNN.voxel_grid).  pos: [n, 2] or [n, 3] float32.  Differences from torch_cluster:
    only 2-D and 3-D positions (more columns raise ValueError rather than give other ids), and ids that do not fit in
    int64 (cell counts, their product, or points far outside [start, end]) raise TrueKNNError instead of overflowing
    silently.
    numpy in, numpy out; a CUDA tensor in, a tensor on its device out (device: the CUDA device for numpy input)."""
    return voxel_grid(pos, size, None, start, end, device)


def voxel_grid(pos, size, batch=None, start=None, end=None, device: int | None = None):
    """PyG's voxel_grid(pos, size, batch, start, end) on the GPU, exact: grid_cluster over [pos | batch] with size 1 for
    the cloud id column (which starts at 0 when start is given and ends at the largest cloud id).  Returns the raw int64
    ids; torch.unique(raw, sorted=True, return_inverse=True)[1] is the `cluster` of grid_sampling().  Same differences
    as grid_cluster()."""
    _voxel_args(pos, size, start, end, all_columns=True)  # argument errors before any device is touched
    with TrueKNN(_device_of(pos, device)) as t:
        raw, _, _ = t.voxel_grid(pos, size, start, end, batch=batch)
    return raw


def grid_sampling(pos, size, x=None, batch=None, reduce: str = "mean", device: int | None = None):
    """PyG's GridSampling(size) in one call: the voxel grid of voxel_grid(), then per voxel the mean position and x
    pooled with `reduce` ("mean" or "max").  Returns (pos_mean [nv, D] float32, x_pooled [nv, F] float32 or None,
    batch_out [nv] int64 or None: the cloud of each voxel, cluster [n] int64: the voxel of each point, PyG's
    consecutive_cluster ids).  Voxels are ordered by raw id, as in PyG.  Differences from PyG: the sums run in a fixed
    order without atomics, so every run gives the same bits; the position is always the mean (PyG pools it with
    `reduce` too); x must be float32; the overflow cases of grid_cluster() are rejected."""
    if reduce not in ("mean", "max"):
        raise ValueError(f"reduce must be 'mean' or 'max', got {reduce!r}")
    pos, _, _, _, _ = _voxel_args(pos, size, None, None, all_columns=True)
    with TrueKNN(_device_of(pos, device)) as t:
        _, cluster, _ = t.voxel_grid(pos, size, batch=batch)
        pos_mean = t.voxel_pool(pos, "mean")
        xp = t.voxel_pool(x, reduce) if x is not None else None
        batch_out = None
        if batch is not None:
            _, _, _, seg = t.voxel_members()
            batch_out = _int64(seg)
    return pos_mean, xp, batch_out, _int64(cluster)


def _int64(a):
    if _is_tensor(a):
        import torch

        return a.to(torch.int64)
    return a.astype(np.int64)


def _edges(query, nbr, query_row: int):
    """[2, E] int64 with the query (centre) ids in row query_row and their neighbours in the other: query_row 1 is
    torch_cluster's source_to_target flow of knn_graph / radius_graph, 0 the [y index, x index] rows of knn / radius."""
    rows = (nbr, query) if query_row == 1 else (query, nbr)
    if _is_tensor(query):
        import torch

        return torch.stack([_int64(r) for r in rows])
    return np.stack([_int64(r) for r in rows])


def _repeat_rows(like, m: int, counts):
    """The row id of every entry of m rows holding `counts` entries each (an int, or one count per row)."""
    rows = _arange_like(like, m)
    return rows.repeat_interleave(counts) if _is_tensor(rows) else np.repeat(rows, counts)


def _knn_edges(idx, k: int, query_row: int):
    """Edges of [m, k] neighbour rows, -1 slots dropped."""
    query = _repeat_rows(idx, int(idx.shape[0]), int(k))
    flat = idx.reshape(-1)
    keep = flat >= 0
    return _edges(query[keep], flat[keep], query_row)


def _csr_edges(offsets, idx, query_row: int, max_num_neighbors: int | None = None):
    """Edges of CSR neighbour rows (radius_search / radius_query); max_num_neighbors keeps the first entries of a row."""
    off = _int64(offsets)
    query = _repeat_rows(idx, int(offsets.shape[0]) - 1, off[1:] - off[:-1])
    if max_num_neighbors is not None:
        keep = _arange_like(idx, int(idx.shape[0])) - off[query] < int(max_num_neighbors)
        idx, query = idx[keep], query[keep]
    return _edges(query, idx, query_row)


def knn_graph(x, k: int, batch=None, device: int | None = None):
    """torch_cluster.knn_graph(x, k, batch) on the GPU, exact: the k nearest points of every point inside its own cloud.

    Returns edge_index [2, E] int64 (row 0 the neighbour, row 1 the centre), edges ordered by centre and then by
    (distance, index); a cloud of at most k points gives each of its points fewer than k edges.  Differences from
    torch_cluster: no `loop` option (a point is never its own neighbour) and no truncation of any kind.  numpy in, numpy
    out; a CUDA tensor in, a tensor on its device out (device: the CUDA device for numpy input, default 0).
    Only the first 2 or 3 columns of x are positions: columns beyond the third are ignored (they are skipped through
    the stride).  For neighbours over all columns (feature space, DGCNN) use feature_knn_graph()."""
    with TrueKNN(_device_of(x, device)) as t:
        idx, _ = t.build(x, batch=batch).search(int(k), indices_only=True)
    return _knn_edges(idx, k, 1)


def radius_graph(x, r: float, batch=None, device: int | None = None):
    """torch_cluster.radius_graph(x, r, batch) on the GPU, exact: every pair within the closed ball of radius r inside one
    cloud.  Returns edge_index [2, E] int64 (row 0 the neighbour, row 1 the centre), edges ordered by centre and then by
    (distance, index).  Differences from torch_cluster: no `loop` option (a point is never its own neighbour) and no
    max_num_neighbors truncation: every neighbour in the ball is returned."""
    with TrueKNN(_device_of(x, device)) as t:
        offsets, idx, _ = t.build(x, batch=batch).radius_search(float(r), indices_only=True)
    return _csr_edges(offsets, idx, 1)


def _bipartite_setup(x, y, batch_x, batch_y):
    """(batch_x, batch_y, batch_size) of knn() / radius(): both batches None (one cloud) or both filled in, a missing one
    with zeros; batch_size = max(batch_x.max(), batch_y.max()) + 1."""
    if batch_x is None and batch_y is None:
        return None, None, None
    batch_x = _zeros_like_rows(x, (int(x.shape[0]),), np.int64) if batch_x is None else batch_x
    batch_y = _zeros_like_rows(y, (int(y.shape[0]),), np.int64) if batch_y is None else batch_y
    top = max(int(b.max().item()) if _is_tensor(b) else int(np.max(b)) for b in (batch_x, batch_y))
    return batch_x, batch_y, top + 1


def knn(x, y, k: int, batch_x=None, batch_y=None, device: int | None = None):
    """torch_cluster.knn(x, y, k, batch_x, batch_y) on the GPU, exact: for every point of y, the k nearest points of x in
    the same cloud (tknn_query_segments).  Returns [2, E] int64 with row 0 the index into y (the query) and row 1 the
    index into x, torch_cluster's orientation for this call; edges are ordered by query and then by (distance, index).
    batch_size = max(batch_x.max(), batch_y.max()) + 1; a cloud present in only one of x and y gives no edges.  k is
    clamped to len(x); an empty x or y gives [2, 0].  A point of y is not excluded from its own neighbours: there is no
    self exclusion, as in torch_cluster.  numpy in, numpy out; a CUDA tensor in, a tensor on its device out (device:
    the CUDA device for numpy input, default 0).  Only the first 2 or 3 columns of x and y are positions: columns beyond
    the third are ignored.  For neighbours over all columns (feature space) use feature_knn()."""
    if int(x.shape[0]) == 0 or int(y.shape[0]) == 0:
        return _zeros_like_rows(x, (2, 0), np.int64)
    batch_x, batch_y, batch_size = _bipartite_setup(x, y, batch_x, batch_y)
    k = min(int(k), int(x.shape[0]))
    with TrueKNN(_device_of(x, device)) as t:
        t.build(x, batch=batch_x, batch_size=batch_size)
        idx, _ = t.query(y, k, batch=batch_y)
    return _knn_edges(idx, k, 0)


def feature_knn_graph(x, k: int, batch=None, device: int | None = None):
    """knn_graph() in feature space: the k nearest rows of every row of x ([n, F] float32, all F columns count) inside
    its own cloud, exact (tknn_feature_knn with self_ids = arange(n)).  Returns edge_index [2, E] int64 (row 0 the
    neighbour, row 1 the centre), edges ordered by centre and then by (d2, index); a point is never its own neighbour
    and a cloud of at most k points gives each of its points fewer than k edges.  numpy in, numpy out; a CUDA tensor
    in, a tensor on its device out (device: the CUDA device for numpy input, default 0)."""
    n = int(x.shape[0])
    if n == 0:
        return _zeros_like_rows(x, (2, 0), np.int64)
    k = int(k)
    self_ids = _arange_like(x, n, np.int32)
    with TrueKNN(_device_of(x, device)) as t:
        idx, _ = t.feature_knn(x, x, k, batch_x=batch, batch_y=batch, self_ids=self_ids, indices_only=True)
    return _knn_edges(idx, k, 1)


def feature_knn(x, y, k: int, batch_x=None, batch_y=None, device: int | None = None):
    """knn() in feature space: for every row of y, the k nearest rows of x in the same cloud over all F columns, exact
    (tknn_feature_knn).  Returns [2, E] int64 with row 0 the index into y (the query) and row 1 the index into x,
    edges ordered by query and then by (d2, index).  Batches as knn(); k is clamped to len(x); an empty x or y gives
    [2, 0]; no self exclusion, so DynamicEdgeConv's knn(x, x, k, b, b) is feature_knn(x, x, k, b, b).  numpy in, numpy
    out; a CUDA tensor in, a tensor on its device out (device: the CUDA device for numpy input, default 0)."""
    if int(x.shape[0]) == 0 or int(y.shape[0]) == 0:
        return _zeros_like_rows(x, (2, 0), np.int64)
    k = min(int(k), int(x.shape[0]))
    with TrueKNN(_device_of(x, device)) as t:
        idx, _ = t.feature_knn(x, y, k, batch_x=batch_x, batch_y=batch_y, indices_only=True)
    return _knn_edges(idx, k, 0)


def _positions(pos, name):
    """pos as [rows, 2|3] float32: PyG's knn_interpolate measures distances over every column, so other widths raise."""
    pos = _arg(pos, np.float32, name)
    if pos.ndim != 2 or int(pos.shape[1]) not in (2, 3):
        raise ValueError(f"{name} must be [n, 2] or [n, 3] (only 2-D and 3-D positions are supported), got "
                         f"{tuple(pos.shape)}")
    return pos


_KnnInterpolate = None


def _knn_interpolate_function():
    """The torch.autograd.Function of knn_interpolate(), made on first use (importing the package needs no torch)."""
    global _KnnInterpolate
    if _KnnInterpolate is None:
        import torch

        class KnnInterpolate(torch.autograd.Function):
            @staticmethod
            def forward(ctx, x, idx, d2, t):
                out, weight, den = t.interpolate(idx, d2, x)
                ctx.save_for_backward(idx, weight, den)
                ctx.n = int(x.shape[0])
                return out

            @staticmethod
            def backward(ctx, grad_out):
                idx, weight, den = ctx.saved_tensors
                with TrueKNN(grad_out.device.index) as t:
                    grad_x = t.interpolate_backward(idx, weight, den, grad_out.contiguous(), ctx.n)
                return grad_x, None, None, None

        _KnnInterpolate = KnnInterpolate
    return _KnnInterpolate


def knn_interpolate(x, pos_x, pos_y, batch_x=None, batch_y=None, k: int = 3, num_workers: int = 1,
                    device: int | None = None):
    """PyG's knn_interpolate(x, pos_x, pos_y, batch_x, batch_y, k) on the GPU, exact and deterministic: the feature
    propagation (upsampling) step of PointNet++.  For every point of pos_y, its k nearest points of pos_x in the same
    cloud (knn(), squared distances), then out = sum fl(x_j * w_j) / sum w_j with w_j = 1 / max(d2_j, 1e-16), each sum in
    neighbour order from +0 in fp32 (TrueKNN.interpolate).  x: [n, f] float32 with n = len(pos_x); positions: [*, 2] or
    [*, 3] float32 (other widths raise ValueError); batches as knn(); k is clamped to len(pos_x); num_workers is accepted
    and ignored.  Returns [len(pos_y), f] float32; a query whose cloud has no data point gets NaN, as in PyG.
    numpy in, numpy out (no autograd).  For a CUDA tensor x the result is differentiable with respect to x only, as in
    PyG: the backward pass (TrueKNN.interpolate_backward) sums in edge order without atomics, so x.grad has the same bits
    on every run; the positions get no gradient.  device: the CUDA device for numpy input (default 0)."""
    del num_workers
    x = _arg(x, np.float32, "x", ndim=2, cast=False, copy=True)
    pos_x, pos_y = _positions(pos_x, "pos_x"), _positions(pos_y, "pos_y")
    if int(pos_x.shape[1]) != int(pos_y.shape[1]):
        raise ValueError(f"pos_x has {int(pos_x.shape[1])} columns, pos_y {int(pos_y.shape[1])}")
    n, f, nq = int(x.shape[0]), int(x.shape[1]), int(pos_y.shape[0])
    if int(pos_x.shape[0]) != n:
        raise ValueError(f"x has {n} rows, pos_x {int(pos_x.shape[0])}")
    if int(k) < 1:
        raise ValueError(f"k = {k} must be >= 1")
    tensor = _is_tensor(x)
    if tensor:
        import torch

        if not x.is_cuda:
            raise ValueError("x must be a CUDA tensor or a numpy array")
        pos_x, pos_y = (torch.as_tensor(p, device=x.device) for p in (pos_x, pos_y))
    if nq == 0:
        return x[:0].clone() if tensor else np.zeros((0, f), np.float32)
    if n == 0:  # PyG: no neighbour, 0 / 0
        if tensor:
            return x.new_full((nq, f), float("nan")) + x.sum() * 0  # still part of x's graph
        return np.full((nq, f), np.nan, np.float32)
    batch_x, batch_y, batch_size = _bipartite_setup(pos_x, pos_y, batch_x, batch_y)
    k = min(int(k), n)
    with TrueKNN(_device_of(x, device), squared_dist=1) as t:
        if n == 1:  # a build needs two points; the feature-space search has the same d2 rule for 2 or 3 columns
            idx, d2 = t.feature_knn(pos_x, pos_y, 1, batch_x=batch_x, batch_y=batch_y)
        else:
            t.build(pos_x, batch=batch_x, batch_size=batch_size)
            idx, d2 = t.query(pos_y, k, batch=batch_y)
        if not tensor:
            out, _, _ = t.interpolate(idx, d2, x)
            return out
        return _knn_interpolate_function().apply(x, idx, d2, t)


def radius(x, y, r: float, batch_x=None, batch_y=None, max_num_neighbors: int | None = None, device: int | None = None):
    """torch_cluster.radius(x, y, r, batch_x, batch_y) on the GPU, exact: for every point of y, the points of x in the same
    cloud within the closed ball of radius r (tknn_radius_query_segments).  Returns [2, E] int64 with row 0 the index
    into y (the query) and row 1 the index into x; edges are ordered by query and then by (distance, index).  Batches,
    empty inputs and the missing self exclusion as knn().  max_num_neighbors=None returns the whole ball; an integer m
    keeps the first m entries of each sorted row, i.e. the m nearest.  This differs from torch_cluster, whose default
    is 32 and whose CUDA kernel keeps an unspecified m of the ball."""
    if int(x.shape[0]) == 0 or int(y.shape[0]) == 0:
        return _zeros_like_rows(x, (2, 0), np.int64)
    batch_x, batch_y, batch_size = _bipartite_setup(x, y, batch_x, batch_y)
    with TrueKNN(_device_of(x, device)) as t:
        t.build(x, batch=batch_x, batch_size=batch_size)
        offsets, idx, _ = t.radius_query(y, float(r), indices_only=True, batch=batch_y)
    return _csr_edges(offsets, idx, 0, max_num_neighbors)


def read_points(path: str, n: int, dim: int) -> np.ndarray:
    """Point-file grammar of the sample (hostCode.cpp:83-124): floats separated by ',' and/or blanks,
    lines read while n*dim floats are still owed (the last line read is consumed whole), then chunked
    by `dim`; dim 2 gives z = 0.  Fast path: a `.f32` file is raw little-endian float32 rows of `dim`."""
    if dim not in (2, 3):
        raise ValueError("dimension must be 2 or 3 (hostCode.cpp:114-124 creates no points otherwise)")
    if path.endswith(".f32"):
        flat = np.fromfile(path, dtype="<f4", count=n * dim)
    else:
        vals: list[float] = []
        owed = n * dim
        with open(path, "rb") as f:
            for line in f:
                if owed <= 0:
                    break
                # operator>> stops at the first token that is not a float; a ',' after a float is skipped
                pos, text = 0, line.decode("latin-1")
                ln = len(text)
                while True:
                    while pos < ln and text[pos].isspace():
                        pos += 1
                    if pos >= ln:
                        break
                    m = _FLOAT_RE.match(text, pos)
                    if not m:
                        break
                    vals.append(float(m.group(0)))
                    owed -= 1
                    pos = m.end()
                    if pos < ln and text[pos] == ",":
                        pos += 1
        flat = np.asarray(vals, dtype=np.float32)
    if flat.size % dim:
        raise ValueError(f"{flat.size} floats is not a multiple of dim={dim} (the reference throws std::out_of_range)")
    pts = flat.reshape(-1, dim)
    if dim == 2:
        pts = np.concatenate([pts, np.zeros((pts.shape[0], 1), np.float32)], axis=1)
    return np.ascontiguousarray(pts, dtype=np.float32)


def read_points_fast(path: str, n: int, dim: int) -> np.ndarray:
    """Same grammar as read_points, parsed in parallel by libtrueknn (tknn_read_points)."""
    L = _lib.load()
    cap = int(n) + 8
    m = C.c_uint64(0)
    for _ in range(2):
        out = np.empty((cap, 3), np.float32)
        rc = L.tknn_read_points(path.encode(), int(n), int(dim), C.c_void_p(out.ctypes.data), cap, C.byref(m))
        if rc == _lib.OK:
            return np.ascontiguousarray(out[: int(m.value)])
        # The last line read is consumed whole (hostCode.cpp:92), so a file with many floats per line yields more
        # than n rows: *n_out then names the row count needed — retry once with that capacity.
        if rc == _lib.EINVAL and int(m.value) > cap:
            cap = int(m.value)
            continue
        break
    raise ValueError(f"tknn_read_points({path!r}) failed with {_lib.ERROR_NAMES.get(rc, rc)}")


def write_neighbours(path: str, idx: np.ndarray, dist: np.ndarray, binary: bool = False):
    """`query,neighbourIndex,distance` lines (hostCode.cpp:316, commented out in the reference) or raw arrays."""
    L = _lib.load()
    idx = np.ascontiguousarray(idx, dtype=np.int32)
    dist = np.ascontiguousarray(dist, dtype=np.float32)
    rc = L.tknn_write_neighbours(path.encode(), C.c_void_p(idx.ctypes.data), C.c_void_p(dist.ctypes.data), idx.shape[0],
                                 idx.shape[1], 1 if binary else 0)
    if rc != _lib.OK:
        raise OSError(f"tknn_write_neighbours({path!r}) failed")


def write_neighbour_lists(path: str, offsets: np.ndarray, idx: np.ndarray, dist: np.ndarray | None, binary: bool = False):
    """The CSR rows of radius_search / radius_query: `query,neighbourIndex,distance` lines, or path.off.u64,
    path.idx.i32 and path.dist.f32 when binary (tknn_write_neighbour_lists)."""
    L = _lib.load()
    offsets = np.ascontiguousarray(offsets).view(np.uint64) if np.asarray(offsets).dtype == np.int64 else \
        np.ascontiguousarray(offsets, dtype=np.uint64)
    idx = np.ascontiguousarray(idx, dtype=np.int32)
    dist = None if dist is None else np.ascontiguousarray(dist, dtype=np.float32)
    rc = L.tknn_write_neighbour_lists(path.encode(), C.c_void_p(offsets.ctypes.data), C.c_void_p(idx.ctypes.data),
                                      None if dist is None else C.c_void_p(dist.ctypes.data), offsets.shape[0] - 1,
                                      1 if binary else 0)
    if rc != _lib.OK:
        raise OSError(f"tknn_write_neighbour_lists({path!r}) failed")


def run_sample(argv: list[str], device: int = 0, neighbours_path: str | None = None) -> dict:
    """`sample01-trueknn file n dim start_radius k outfile` (samples/s01-trueknn/README.md:7-14).

    Appends the total seconds (build + kNN) to `outfile` exactly like hostCode.cpp:346-356, and —
    what the reference leaves commented out at hostCode.cpp:312-319 — optionally writes the
    neighbours as `query,neighbourIndex,distance` lines to `neighbours_path`."""
    if len(argv) != 6:
        raise SystemExit("usage: trueknn <file> <n> <dim> <start radius> <k> <output file>")
    path, n, dim, r0, k, outfile = argv[0], int(argv[1]), int(argv[2]), float(argv[3]), int(argv[4]), argv[5]
    pts = read_points_fast(path, n, dim)
    with TrueKNN(device) as t:
        t0 = time.perf_counter()
        t.build(pts, dim=3)
        t1 = time.perf_counter()
        idx, dist = t.search(k, r0)
        t2 = time.perf_counter()
        st = t.stats()
    total = (t1 - t0) + (t2 - t1)
    with open(outfile, "a") as f:
        f.write(f"{total}\n")
    if neighbours_path:
        write_neighbours(neighbours_path, idx, dist)
    return {"build_s": t1 - t0, "knn_s": t2 - t1, "total_s": total, "rounds": st["rounds"], "idx": idx, "dist": dist,
            "stats": st}
