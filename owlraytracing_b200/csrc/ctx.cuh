// ctx.cuh — the context behind `tknn_ctx` and the internal entry points shared by the translation units of
// libtrueknn (trueknn.cu: single-GPU path and C ABI; dist.cu: the multi-GPU drivers).  Nothing here is exported.
#pragma once
#include "../../include/trueknn.h"

#include <cstdarg>
#include <cstdio>
#include <cstring>
#include <string>
#include <vector>

#include "common.cuh"

struct DevBuf {
  void* p = nullptr;
  size_t bytes = 0;
  template <typename T> T* as() const { return reinterpret_cast<T*>(p); }
};

namespace tknn { namespace dist { struct State; } }

struct tknn_ctx {
  int device = 0;
  int sm_count = 148;
  size_t l2_bytes = 0;
  cudaStream_t own_stream = nullptr, stream = nullptr, copy_stream = nullptr;
  std::string err;
  // options
  int leaf_size = 32, counters = 0, leaf_policy = 0, sample_groups = 128, blocks_per_sm = 0, squared = 0,
      radius_quantile = 990;
  // BVH
  uint64_t n = 0;
  uint32_t n_leaves = 0;
  bool ids_in_w = false;  // the BVH was built from float4 rows whose w holds caller-chosen ids (point-partitioned
                          // driver: GLOBAL ids, so local tie-breaks are global ones); row_mode 0 is unavailable then
  DevBuf pts, nodes, leaf_start, node_min_idx;
  float scene_box[6] = {0, 0, 0, 0, 0, 0};
  // search scratch (grown on demand, kept across searches)
  DevBuf queue_a, queue_b, unresolved, offsets, block_sums, scalars, stage_idx, stage_dist, sample;
  // build scratch, kept across builds (grow-only) unless keep_scratch == 0
  DevBuf b_in, b_keys_a, b_keys_b, b_vals_a, b_vals_b, b_sort_tmp, b_delta, b_ballots, b_leaf_key, b_child_info,
      b_parent_leaf, b_parent_node, b_arrive;
  // tknn_query scratch (grow-only; the reference has no analogue — it only queries its own points)
  DevBuf q_stage, q_keys_a, q_keys_b, q_vals_a, q_vals_b, q_sort_tmp, q_pts, q_sid_stage, q_sid_sorted, q_rad_stage,
      q_r2_sorted;
  // query sets of a segmented build (tknn_query_segments / tknn_radius_query_segments): the uploaded host offsets (u64,
  // n_segments + 1), the segment of every query row and of every sorted query position (u32)
  DevBuf q_seg_off, q_seg_row, q_seg_sorted;
  int keep_scratch = 1;
  int sparse_divisor = 8;
  int warp_round_max = 49152;  // rounds with at most this many active queries run one warp per query (0 = never)
  int sparse_team = 0;         // lanes per query in sparse rounds: 0 = the thread-per-query kernel (default: fastest), 4 / 8 / 16 = teams
  int speculative_max = 1 << 20;  // searches of at most this many queries launch round 2 without a host decision (0 = never)
  int approx_filter = 0;
  int tie_pruning = 0;        // 0 = auto (on when the build saw leaves of coincident points), 1 = on, 2 = off
  int morton_bits = 0;        // 0 = auto (packed sort: as many as fit beside the index, <= 13; pair sort: ceil(log2 n / 3) + 8 in [10, 21])
  int sort_mode = 0;          // 0 = packed (code, index) keys when they fit, 1 = (code, index) pairs (TKNN_OPT_SORT_MODE)
  int built_idx_bits = 0;     // index bits of the packed keys of the current BVH (0: pair sort)
  bool has_dup_leaves = false; // the build found a leaf of coincident points => tie-pruning kernel variant
  int built_morton_bits = 21; // what the current BVH was built with (queries are coded the same way)
  int curve = 1;              // space-filling curve of the next build: 1 = Hilbert (default), 0 = Morton
  int curve_levels = 0;       // > 0: Hilbert levels forced (experiments); 0 = ceil(log2 n / 3) + 2
  int built_curve = 0;        // Hilbert levels the current BVH's keys were made with (0 = Morton): queries are coded alike
  int output_chunks = 4;  // host-output pipelining: slices whose D2H overlaps the next slice's search (1 = off)
  int file_order_chunks = 0;  // same for tknn_search (file-order rows): slices by original index (1 = off; 0 = auto: 5 with
                              // distances, 2 indices-only; k > 24: 2 and 1 — the sweeps of profiles/r2_e2e_mailbox.txt, r2_e2e_cfg3.txt)
  DevBuf chunk_queue;
  // tknn_dbscan scratch (grow-only): union-find parents, per-root smallest original index and cluster id per position
  DevBuf db_parent, db_min_idx, db_pos_label, db_bits, db_core_stage;
  // tknn_radius_search / _query scratch (grow-only): counts and u64 offsets by position and by row, scan block sums, the
  // mailbox words, self positions, the unsorted rows, the long-row list and the long-row sort buffers (radius.cuh)
  DevBuf rl_cnt_pos, rl_cnt_row, rl_off_pos, rl_off_row, rl_sums, rl_stats, rl_pos_of, rl_self_pos, rl_keys, rl_long_pos,
      rl_long_len, rl_boff, rl_ka, rl_kb, rl_kc, rl_va, rl_vb, rl_vc, rl_row_of, rl_sort_tmp;
  // segmented build (tknn_build_segments with n_segments > 1; a later tknn_build clears it): the offsets (u64,
  // n_segments + 1), the segment of every position (u32; positions and indices of a segment share its offsets) and per
  // node the segment ranges of its two children (int4: lo0, hi0, lo1, hi1)
  bool segmented = false;
  uint64_t n_segments = 0;
  DevBuf seg_off, seg_of, node_seg;
  std::vector<uint64_t> seg_off_host;  // the same offsets on the host (tknn_fps sizes its tiers from them)
  // tknn_fps scratch (grow-only, fps.cuh): the segments of each tier, the tier of every segment, leaf flags, the grid
  // tier's compact leaf records (box, first position, key), D by position, position by index and the key slots
  DevBuf fps_segs, fps_slot_of_seg, fps_words, fps_leaf_lo, fps_leaf_hi, fps_leaf_first, fps_leaf_key, fps_D, fps_pos_of,
      fps_best;
  // tknn_feature_knn scratch (grow-only, features.cuh): staged host rows and self ids, the work list, the partial key
  // lists of a split call and the distances the merge writes when the caller asked for indices only.  It touches no
  // build state.
  DevBuf fk_x, fk_y, fk_sid, fk_items, fk_partial, fk_dist;
  // the clustering of the last tknn_voxel_grid (grow-only, voxel.cuh): staged rows and offsets, raw and dense ids by
  // point, the sort buffers, head words and their scan, members by sorted position, per voxel the offsets, lowest index,
  // cloud and long-voxel chunk offsets, the list of long voxels, the box / flag / count words, and the staging of host
  // pool rows and outputs.
  // Builds and searches never touch it.
  DevBuf vx_pts, vx_seg_off, vx_raw, vx_cluster, vx_keys_a, vx_keys_b, vx_vals_a, vx_vals_b, vx_sort_tmp, vx_words,
      vx_word_off, vx_members, vx_off, vx_first, vx_seg, vx_chunks, vx_chunk_off, vx_words_sc, vx_x, vx_out, vx_cs, vx_longs;
  bool vx_valid = false;  // a clustering exists
  uint64_t vx_n = 0, vx_nv = 0, vx_long_chunks = 0, vx_n_long = 0;
  // tknn_interpolate / _backward scratch (grow-only unless keep_scratch == 0, interpolate.cuh): staged host inputs and
  // outputs, and the backward's edge keys, values, sort buffers, per-row counts and run offsets.  It touches no build
  // state.
  DevBuf ip_idx, ip_w, ip_den, ip_x, ip_out, ip_wout, ip_dout, ip_keys_a, ip_keys_b, ip_vals_a, ip_vals_b, ip_sort_tmp,
      ip_cnt, ip_off;
  // cell grid over the sorted points (grid.cuh): runs per level-L cell and the table's frame; made by a plain build when
  // the cloud qualifies, and then round 1 of a dense kNN search with k <= 24 walks it instead of the LBVH
  int grid_mode = 0;        // TKNN_OPT_GRID: 0 = auto (occupancy decides), 1 = off, 2 = whenever the table is valid
  int grid_level = 0;       // TKNN_OPT_GRID_LEVEL: 0 = auto (floor(log2 n / 3)), else forced (1..8)
  bool grid_on = false;     // the current build's table serves dense kNN rounds
  int built_grid_level = 0;
  DevBuf grid_cells, grid_frame;
  // Mailbox: 16 words of mapped pinned host memory that a one-thread kernel fills (fetch_words): the small read-backs of a
  // search or build (unresolved count, radius, leaf count, flags) then never queue behind a bulk device->host copy on the
  // copy engine, and never pass through pageable staging.
  uint32_t* mailbox_h = nullptr;
  uint32_t* mailbox_d = nullptr;
  int mailbox_launches = 0;  // mailbox kernels since the counter was last folded into a launch count
  std::vector<cudaEvent_t> chunk_ev;
  cudaEvent_t ev[10] = {};
  std::vector<cudaEvent_t> round_ev;
  tknn_stats stats;
  tknn::dist::State* dist = nullptr;  // multi-GPU state (dist.cu), nullptr until tknn_comm_init
  tknn_ctx() { std::memset(&stats, 0, sizeof(stats)); }
};

namespace tknn {
namespace host {

int fail(tknn_ctx* c, int code, const char* fmt, ...);
int ensure(tknn_ctx* c, DevBuf& b, size_t bytes);
void release(DevBuf& b);
bool is_device_ptr(const void* p);

struct ScopedDevice {
  int prev = -1;
  explicit ScopedDevice(int d) { cudaGetDevice(&prev); if (prev != d) cudaSetDevice(d); else prev = -1; }
  ~ScopedDevice() { if (prev >= 0) cudaSetDevice(prev); }
};

inline unsigned blocks_for(uint64_t n, int threads) { return (unsigned)((n + threads - 1) / threads); }

// scalars layout (uint32 words unless noted)
enum { SC_GROUP_COUNTER = 0, SC_TOTAL = 1, SC_ERROR = 2, SC_QBAD = 3 /* non-finite query coordinate */, SC_BOUNDS = 4 /* 7 words */, SC_SCENE = 12 /* 6 floats */,
       SC_COUNTERS = 20 /* 8 x u64, 8-byte aligned */, SC_DUPLEAF = 40, SC_QUANTILE = 41 /* 2 floats: r, r * r */,
       SC_DBSCAN = 43 /* core points, other points */,
       SC_GRID = 45 /* largest cell, cells split into several runs */, SC_WORDS = 48 };

#define TK_CUDA(c, expr)                                                                            \
  do {                                                                                              \
    cudaError_t e__ = (expr);                                                                       \
    if (e__ != cudaSuccess) {                                                                       \
      cudaGetLastError();                                                                           \
      return ::tknn::host::fail((c), e__ == cudaErrorMemoryAllocation ? TKNN_ENOMEM : TKNN_ECUDA, "%s: %s (%s:%d)", #expr, \
                  cudaGetErrorString(e__), __FILE__, __LINE__);                                     \
    }                                                                                               \
  } while (0)

#define TK_TRY(expr)                 \
  do {                               \
    int rc__ = (expr);               \
    if (rc__ != TKNN_OK) return rc__; \
  } while (0)

// ---- internal entry points (trueknn.cu) used by the multi-GPU drivers (dist.cu) ----

// LBVH over n rows of `stride` floats on the DEVICE or HOST.  ids_in_w: rows are (x, y, z, id bits) and the id of
// every point is taken from its 4th float instead of its row number (requires stride >= 4, dim 3).
// seg_offsets (device, n_segments + 1 validated offsets, n_segments > 1) or nullptr: an unsegmented build.
int build_core(tknn_ctx* c, const float* xyz, uint64_t n, int dim, int stride, bool ids_in_w,
               const uint64_t* seg_offsets = nullptr, uint64_t n_segments = 0, uint64_t max_segment = 0);

// all-points search over sorted positions [q_begin, q_begin + nq); row_mode as in trav::Params
int search_range(tknn_ctx* c, int k, float start_radius, uint64_t q_begin, uint64_t nq, int row_mode, int32_t* qid_out,
                 int32_t* idx_out, float* dist_out, uint64_t rows);

// Exact tiled brute force of nq external queries (float4: x, y, z, id bits to exclude) against the context's sorted
// points; rows follow the query order; d_dist receives d2 when squared != 0.  Device arrays.
int brute_core(tknn_ctx* c, const float4* d_qpts, uint64_t nq, int k, const uint32_t* d_row_of, int32_t* d_idx, float* d_dist,
               int squared);

}  // namespace host
}  // namespace tknn

// dist.cu: frees the multi-GPU state of a context (communicator included); called by tknn_destroy
extern "C" void tknn_internal_free_dist(tknn_ctx* c);
// dist.cu: a plain tknn_build invalidates the partitioned state of the context
extern "C" void tknn_internal_dist_invalidate(tknn_ctx* c);
