"""ctypes loader for libtrueknn.so (include/trueknn.h).

There is no CPU fallback: if the shared library is missing this raises, and if no CUDA device is
usable `tknn_create` fails and `TrueKNN(...)` raises.  The library is built in-tree by
`__graft_entry__.build()` (or `make -C owlraytracing_b200/csrc`).
"""
from __future__ import annotations

import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("TKNN_LIB_PATH") or os.path.join(_HERE, "lib", "libtrueknn.so")  # override: kernel A/B experiments

TKNN_MAX_ROUNDS = 48
TKNN_MAX_K = 512

OK, EINVAL, ENOMEM, ECUDA, ENCCL, ESTATE = 0, 1, 2, 3, 4, 5
ERROR_NAMES = {0: "TKNN_OK", 1: "TKNN_EINVAL", 2: "TKNN_ENOMEM", 3: "TKNN_ECUDA", 4: "TKNN_ENCCL", 5: "TKNN_ESTATE"}

(OPT_LEAF_SIZE, OPT_COUNTERS, OPT_LEAF_POLICY, OPT_SAMPLE_GROUPS, OPT_BLOCKS_PER_SM, OPT_SQUARED_DIST, OPT_RADIUS_QUANTILE,
 OPT_KEEP_SCRATCH, OPT_SPARSE_DIVISOR, OPT_APPROX_FILTER, OPT_OUTPUT_CHUNKS, OPT_FILE_ORDER_CHUNKS, OPT_MORTON_BITS,
 OPT_TIE_PRUNING, OPT_WARP_ROUND_MAX, OPT_CURVE, OPT_SPECULATIVE_MAX, OPT_SPARSE_TEAM, OPT_SORT_MODE, OPT_GRID,
 OPT_GRID_LEVEL, OPT_GRID_RADIUS_QUANTILE) = (1, 2, 3, 4, 5, 6, 7, 8, 9, 10, 11, 12, 13, 14, 15, 16, 17, 18, 19, 20, 21, 22)


class Stats(C.Structure):
    _fields_ = [
        ("n_points", C.c_uint64),
        ("n_leaves", C.c_uint32),
        ("n_nodes", C.c_uint32),
        ("build_ms", C.c_float),
        ("bounds_ms", C.c_float),
        ("morton_ms", C.c_float),
        ("sort_ms", C.c_float),
        ("leaves_ms", C.c_float),
        ("hierarchy_ms", C.c_float),
        ("refit_ms", C.c_float),
        ("h2d_ms", C.c_float),
        ("n_queries", C.c_uint64),
        ("k", C.c_int32),
        ("rounds", C.c_int32),
        ("start_radius", C.c_float),
        ("final_radius", C.c_float),
        ("estimate_ms", C.c_float),
        ("search_ms", C.c_float),
        ("d2h_ms", C.c_float),
        ("round_ms", C.c_float * TKNN_MAX_ROUNDS),
        ("kernel_ms", C.c_float * TKNN_MAX_ROUNDS),
        ("round_queries", C.c_uint64 * TKNN_MAX_ROUNDS),
        ("kernel_launches", C.c_uint32),
        ("build_launches", C.c_uint32),
        ("nodes_visited", C.c_uint64),
        ("points_tested", C.c_uint64),
        ("heap_inserts", C.c_uint64),
        ("warp_node_visits", C.c_uint64),
        ("warp_leaf_visits", C.c_uint64),
        ("warp_point_loads", C.c_uint64),
        ("filter_violations", C.c_uint64),
        ("h2d_bytes", C.c_uint64),
        ("d2h_bytes", C.c_uint64),
        ("grid_level", C.c_int32),
        ("grid_selected", C.c_int32),
        ("grid_max_cell", C.c_uint32),
        ("grid_split_cells", C.c_uint32),
        ("grid_ms", C.c_float),
        ("grid_rounds", C.c_uint32),
        ("grid_deferred", C.c_uint64),
        ("grid_phase_cycles", C.c_uint64 * 6),
        ("grid_insert_iters", C.c_uint64),
        ("grid_inserts", C.c_uint64),
    ]

    def as_dict(self) -> dict:
        d = {}
        for name, _ in self._fields_:
            v = getattr(self, name)
            if name in ("round_ms", "kernel_ms", "round_queries"):
                v = list(v)[: max(0, int(self.rounds))]
            elif name == "grid_phase_cycles":
                v = list(v)
            d[name] = v
        return d


class DistStats(C.Structure):
    """tknn_dist_stats (include/trueknn.h)."""
    _fields_ = [("n_ranks", C.c_int32), ("rank", C.c_int32), ("n_global", C.c_uint64), ("n_owned", C.c_uint64)] + [
        (name, C.c_float) for name in (
            "h2d_ms", "allgather_ms", "box_ms", "codes_ms", "splitters_ms", "bucket_ms", "exchange_ms", "lbvh_ms",
            "summaries_ms", "build_total_ms", "local_search_ms", "reach_ms", "exchange_out_ms", "remote_search_ms",
            "exchange_back_ms", "merge_ms", "finish_ms", "d2h_ms", "search_total_ms")] + [
        ("boundary_sent", C.c_uint64), ("boundary_received", C.c_uint64), ("bytes_sent_build", C.c_uint64),
        ("bytes_sent_search", C.c_uint64)]

    def as_dict(self) -> dict:
        return {name: getattr(self, name) for name, _ in self._fields_}


SHARD_QUERIES, PARTITION_POINTS = 1, 2
REDUCE_MEAN, REDUCE_MAX = 0, 1
UNIQUE_ID_BYTES = 128

# every symbol include/trueknn.h declares (tests check the library exports all of them)
EXPORTS = [
    "tknn_create", "tknn_destroy", "tknn_set_stream", "tknn_set_option", "tknn_build", "tknn_search",
    "tknn_search_shard", "tknn_shard_capacity", "tknn_query", "tknn_range_count", "tknn_estimate_start_radius",
    "tknn_brute_force", "tknn_merge_topk", "tknn_get_stats", "tknn_last_error", "tknn_version", "tknn_sort_pairs",
    "tknn_get_bvh", "tknn_generate_uniform", "tknn_measure_bandwidth", "tknn_morton_codes",
    "tknn_read_points", "tknn_write_neighbours", "tknn_reach_mask",
    "tknn_comm_unique_id", "tknn_comm_init", "tknn_get_dist_stats", "tknn_build_replicated", "tknn_partition_build",
    "tknn_partition_owned", "tknn_partition_search", "tknn_partition_verify", "tknn_create_multi", "tknn_multi_destroy",
    "tknn_multi_set_option", "tknn_multi_build", "tknn_multi_search", "tknn_multi_ranks", "tknn_multi_ctx",
    "tknn_multi_last_error", "tknn_multi_get_times", "tknn_measure_smem_bandwidth", "tknn_key_layout", "tknn_dbscan",
    "tknn_radius_search", "tknn_radius_query", "tknn_write_neighbour_lists", "tknn_build_segments",
    "tknn_query_segments", "tknn_radius_query_segments", "tknn_fps", "tknn_feature_knn",
    "tknn_voxel_grid", "tknn_voxel_members", "tknn_voxel_pool", "tknn_interpolate", "tknn_interpolate_backward",
]

_lib = None


def load() -> C.CDLL:
    """Load libtrueknn.so and declare the prototypes. Raises OSError when it was not built."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise OSError(
            f"{LIB_PATH} not found: build it with `python -c 'import __graft_entry__ as g; g.build()'` "
            "(there is no CPU fallback)")
    L = C.CDLL(LIB_PATH)
    vp, i32, u32, u64, f32 = C.c_void_p, C.c_int32, C.c_uint32, C.c_uint64, C.c_float
    L.tknn_version.restype = C.c_int
    L.tknn_last_error.restype = C.c_char_p
    L.tknn_last_error.argtypes = [vp]
    L.tknn_create.argtypes = [C.c_int, C.POINTER(vp)]
    L.tknn_destroy.argtypes = [vp]
    L.tknn_set_stream.argtypes = [vp, vp]
    L.tknn_set_option.argtypes = [vp, C.c_int, C.c_int64]
    L.tknn_build.argtypes = [vp, vp, u64, C.c_int, C.c_int]
    L.tknn_build_segments.argtypes = [vp, vp, u64, C.c_int, C.c_int, vp, u64]
    L.tknn_search.argtypes = [vp, C.c_int, f32, vp, vp]
    L.tknn_search_shard.argtypes = [vp, C.c_int, f32, C.c_int, C.c_int, vp, vp, vp, C.POINTER(u64)]
    L.tknn_key_layout.argtypes = [u64, C.c_int, C.c_int, C.POINTER(C.c_int), C.POINTER(C.c_int), C.POINTER(C.c_int)]
    L.tknn_shard_capacity.restype = u64
    L.tknn_shard_capacity.argtypes = [u64, C.c_int]
    L.tknn_query.argtypes = [vp, vp, u64, C.c_int, C.c_int, vp, vp, C.c_int, f32, vp, vp]
    L.tknn_range_count.argtypes = [vp, f32, vp]
    L.tknn_dbscan.argtypes = [vp, f32, C.c_int, vp, vp, C.POINTER(u64)]
    L.tknn_fps.argtypes = [vp, vp, u64, vp, vp, vp]
    L.tknn_feature_knn.argtypes = [vp, vp, u64, C.c_int, C.c_int, vp, vp, u64, C.c_int, vp, u64, vp, C.c_int, vp, vp]
    L.tknn_voxel_grid.argtypes = [vp, vp, u64, C.c_int, C.c_int, vp, u64, vp, vp, vp, vp, vp, C.POINTER(u64)]
    L.tknn_voxel_members.argtypes = [vp, vp, vp, vp, vp]
    L.tknn_voxel_pool.argtypes = [vp, vp, u64, C.c_int, C.c_int, C.c_int, vp]
    L.tknn_interpolate.argtypes = [vp, vp, vp, u64, C.c_int, vp, u64, C.c_int, C.c_int, vp, vp, vp]
    L.tknn_interpolate_backward.argtypes = [vp, vp, vp, vp, u64, C.c_int, vp, C.c_int, u64, C.c_int, vp]
    L.tknn_radius_search.argtypes = [vp, f32, vp, vp, vp, u64, C.POINTER(u64)]
    L.tknn_radius_query.argtypes = [vp, vp, u64, C.c_int, C.c_int, vp, f32, vp, vp, vp, u64, C.POINTER(u64)]
    L.tknn_query_segments.argtypes = [vp, vp, u64, C.c_int, C.c_int, vp, u64, vp, vp, C.c_int, f32, vp, vp]
    L.tknn_radius_query_segments.argtypes = [vp, vp, u64, C.c_int, C.c_int, vp, u64, vp, f32, vp, vp, vp, u64,
                                             C.POINTER(u64)]
    L.tknn_write_neighbour_lists.argtypes = [C.c_char_p, vp, vp, vp, u64, C.c_int]
    L.tknn_estimate_start_radius.argtypes = [vp, C.c_int, C.POINTER(f32)]
    L.tknn_brute_force.argtypes = [vp, vp, u64, C.c_int, vp, vp]
    L.tknn_merge_topk.argtypes = [vp, vp, vp, C.c_int, u64, C.c_int, vp, vp]
    L.tknn_get_stats.argtypes = [vp, C.POINTER(Stats)]
    L.tknn_sort_pairs.argtypes = [vp, vp, vp, u64]
    L.tknn_get_bvh.argtypes = [vp, vp, vp, vp]
    L.tknn_generate_uniform.argtypes = [vp, u64, u64, u64, vp]
    L.tknn_morton_codes.argtypes = [vp, vp, u64, C.c_int, C.c_int, vp, vp]
    L.tknn_reach_mask.argtypes = [vp, vp, u64, C.c_int, vp, vp, vp, C.c_int, C.c_int, C.c_int, vp]
    L.tknn_read_points.argtypes = [C.c_char_p, u64, C.c_int, vp, u64, C.POINTER(u64)]
    L.tknn_write_neighbours.argtypes = [C.c_char_p, vp, vp, u64, C.c_int, C.c_int]
    L.tknn_measure_bandwidth.argtypes = [vp, C.POINTER(C.c_double), C.POINTER(C.c_double), C.POINTER(C.c_int),
                                         C.POINTER(u64)]
    L.tknn_measure_smem_bandwidth.argtypes = [vp, C.POINTER(C.c_double), C.POINTER(C.c_double)]
    L.tknn_comm_unique_id.argtypes = [vp]
    L.tknn_comm_init.argtypes = [vp, C.c_int, C.c_int, vp]
    L.tknn_get_dist_stats.argtypes = [vp, C.POINTER(DistStats)]
    L.tknn_build_replicated.argtypes = [vp, vp, u64, u64, u64, C.c_int, C.c_int]
    L.tknn_partition_build.argtypes = [vp, vp, u64, u64, C.c_int, C.c_int]
    L.tknn_partition_owned.restype = u64
    L.tknn_partition_owned.argtypes = [vp]
    L.tknn_partition_search.argtypes = [vp, C.c_int, f32, vp, vp, vp, u64, C.POINTER(u64)]
    L.tknn_partition_verify.argtypes = [vp, C.c_int, C.c_int, vp, vp, vp, u64, C.POINTER(u64), C.POINTER(u64)]
    L.tknn_create_multi.argtypes = [C.POINTER(C.c_int), C.c_int, C.c_int, C.POINTER(vp)]
    L.tknn_multi_destroy.argtypes = [vp]
    L.tknn_multi_set_option.argtypes = [vp, C.c_int, C.c_int64]
    L.tknn_multi_build.argtypes = [vp, vp, u64, C.c_int, C.c_int]
    L.tknn_multi_search.argtypes = [vp, C.c_int, f32, vp, vp]
    L.tknn_multi_ranks.argtypes = [vp]
    L.tknn_multi_ctx.restype = vp
    L.tknn_multi_ctx.argtypes = [vp, C.c_int]
    L.tknn_multi_last_error.restype = C.c_char_p
    L.tknn_multi_last_error.argtypes = [vp]
    L.tknn_multi_get_times.argtypes = [vp, C.POINTER(f32)]
    _lib = L
    return L
