// trueknn.cu — the C ABI of libtrueknn (include/trueknn.h) and the host-side round driver.
//
// Host logic replaced (reference file:line):
//   tknn_build   <- hostCode.cpp:165-175,199-212  + owl/UserGeomGroup.cpp:39-241 + owl/UserGeom.cu:172-232
//   tknn_search  <- hostCode.cpp:285-340 (round loop, termination scan, radius doubling, refits)
//   error model  <- owl/helper/cuda.h:22-59 / owl/helper/optix.h:34-55 (throw / exit) -> return codes
#include "../../include/trueknn.h"

#include <algorithm>
#include <cmath>
#include <cstdarg>
#include <cstdio>
#include <cstring>
#include <new>
#include <string>
#include <vector>

#include "brute.cuh"
#include "common.cuh"
#include "ctx.cuh"
#include "features.cuh"
#include "fps.cuh"
#include "frames.cuh"
#include "grid.cuh"
#include "interpolate.cuh"
#include "knn_grad.cuh"
#include "lbvh.cuh"
#include "radix_sort.cuh"
#include "radius.cuh"
#include "traverse.cuh"
#include "voxel.cuh"

using namespace tknn;

// ---------------------------------------------------------------------------------------------
// context helpers (declared in ctx.cuh)
// ---------------------------------------------------------------------------------------------
namespace tknn {
namespace host {

int fail(tknn_ctx* c, int code, const char* fmt, ...) {
  if (c) {
    char buf[512];
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(buf, sizeof(buf), fmt, ap);
    va_end(ap);
    c->err = buf;
  }
  return code;
}

int ensure(tknn_ctx* c, DevBuf& b, size_t bytes) {
  if (b.bytes >= bytes && b.p) return TKNN_OK;
  if (b.p) { cudaFree(b.p); b.p = nullptr; b.bytes = 0; }
  if (bytes == 0) bytes = 16;
  TK_CUDA(c, cudaMalloc(&b.p, bytes));
  b.bytes = bytes;
  return TKNN_OK;
}

void release(DevBuf& b) {
  if (b.p) cudaFree(b.p);
  b.p = nullptr;
  b.bytes = 0;
}

bool is_device_ptr(const void* p) {
  if (!p) return false;
  cudaPointerAttributes a;
  if (cudaPointerGetAttributes(&a, p) != cudaSuccess) { cudaGetLastError(); return false; }
  return a.type == cudaMemoryTypeDevice || a.type == cudaMemoryTypeManaged;
}

int ensure_round_events(tknn_ctx* c, size_t count) {
  while (c->round_ev.size() < count) {
    cudaEvent_t e;
    TK_CUDA(c, cudaEventCreate(&e));
    c->round_ev.push_back(e);
  }
  return TKNN_OK;
}

}  // namespace host
}  // namespace tknn

using namespace tknn::host;

namespace {

// exclusive scan of popc(words[0..nw)) into offsets, total into scalars[SC_TOTAL]
int popc_scan(tknn_ctx* c, const uint32_t* words, uint64_t nw, uint32_t* offsets, int* launches) {
  const uint32_t nb = (uint32_t)((nw + lbvh::SCAN_CHUNK - 1) / lbvh::SCAN_CHUNK);
  TK_TRY(ensure(c, c->block_sums, sizeof(uint32_t) * (size_t)(nb + 1)));
  uint32_t* sums = c->block_sums.as<uint32_t>();
  uint32_t* sc = c->scalars.as<uint32_t>();
  lbvh::popc_reduce_kernel<<<nb, lbvh::THREADS, 0, c->stream>>>(words, nw, sums);
  lbvh::scan_sums_kernel<<<1, lbvh::THREADS, 0, c->stream>>>(sums, nb, sc + SC_TOTAL);
  lbvh::popc_apply_kernel<<<nb, lbvh::THREADS, 0, c->stream>>>(words, nw, sums, offsets);
  if (launches) *launches += 3;
  return TKNN_OK;
}

// ---------------------------------------------------------------------------------------------
// the round driver (shared by search / shard / query / estimator)
// ---------------------------------------------------------------------------------------------
int fetch_words(tknn_ctx* c, const uint32_t* a, int na, const uint32_t* b, int nb, uint32_t* host_out);  // below

struct Job {
  const float4* queries = nullptr;
  const int32_t* self_ids = nullptr;
  const float* query_r2 = nullptr;
  const uint32_t* seg_of = nullptr;       // segmented build: the segment of every query position
  const uint32_t* first_queue = nullptr;  // optional explicit queue for round 1
  uint64_t n_queries = 0;                 // queries in round 1
  uint64_t q_begin = 0;
  int self_is_row = 0;
  int row_mode = 0;
  int k = 0;
  float start_radius = 0.f;  // > 0 or +inf; ignored while r_dev is set
  const float* r_dev = nullptr;  // {r, r * r} on the device (the estimator's output): round 1 reads r2 from there and the
                                 // host learns r with the first read-back it needs anyway
  float* r_host = nullptr;       // receives the radius round 1 ran with
  int squared = 0;
  int32_t* idx_out = nullptr;
  float* dist_out = nullptr;
  int32_t* qid_out = nullptr;
  bool record_stats = true;
  bool force_sparse = false;  // thread-per-query kernel from round 1 (the start-radius sample)
  bool grid = false;          // the queries are the built points: a dense round 1 may walk the cell grid (grid.cuh)
};

// block shape of a persistent traversal kernel: the warps-per-block that keeps the most warps resident per SM
// (227 KB shared memory, 64 K registers, 64 warps, 32 blocks); false when not even one warp fits
bool pick_shape(size_t per_warp, int num_regs, int* warps_out, int* bps_out) {
  const int regs_alloc = ((num_regs + 7) / 8) * 8;  // registers are allocated in units of 8 per thread
  const size_t sm_smem = 227 * 1024;
  int warps = 0, bps = 1, best = 0;
  for (int w = 8; w >= 1; --w) {
    const size_t need_b = per_warp * w + 1024;  // + per-block reservation
    if (need_b > sm_smem) continue;
    int b = (int)std::min<size_t>(sm_smem / need_b, (size_t)(64 / w));
    // registers: each of the 4 SM sub-partitions owns 16 K of them and the warps of successive blocks go to
    // the sub-partitions round-robin, so a block fits only while no sub-partition overflows (ncu: at 48
    // registers 224-thread blocks were limited to 5 per SM and 192-thread blocks to 6, not 6 and 7)
    {
      const int per_smsp = 16384 / (regs_alloc * 32);
      int load[4] = {0, 0, 0, 0}, next = 0, fit = 0;
      for (; fit < b; ++fit) {
        int trial[4] = {load[0], load[1], load[2], load[3]};
        for (int i = 0; i < w; ++i) ++trial[(next + i) & 3];
        if (std::max(std::max(trial[0], trial[1]), std::max(trial[2], trial[3])) > per_smsp) break;
        for (int i = 0; i < 4; ++i) load[i] = trial[i];
        next = (next + w) & 3;
      }
      b = fit;
    }
    b = std::min(b, 32);
    if (b * w > best) { best = b * w; warps = w; bps = b; }
  }
  *warps_out = warps;
  *bps_out = bps;
  return warps >= 1;
}

template <int MODE>
int launch_traverse(tknn_ctx* c, const trav::Params& P) {
  const int k = MODE == trav::MODE_KNN ? P.k : 0;
  const size_t per_warp = trav::smem_per_warp(k);
  // pick the kernel variant first: its register count enters the block-shape choice
  void (*kern)(const trav::Params) = nullptr;
  const bool ties = c->tie_pruning == 1 || (c->tie_pruning == 0 && c->has_dup_leaves);
  const int variant = MODE != trav::MODE_KNN ? 0 : (ties ? 2 : (c->approx_filter ? 1 : 0));
  const bool hp = MODE == trav::MODE_KNN && k > trav::LIST_MAX_K;
#define TK_PICK(CNT, VAR) (hp ? trav::traverse_kernel<MODE, CNT, VAR, true> : trav::traverse_kernel<MODE, CNT, VAR, false>)
#define TK_PICK_SEG(CNT, VAR) \
  (hp ? trav::traverse_kernel<MODE, CNT, VAR, true, true> : trav::traverse_kernel<MODE, CNT, VAR, false, true>)
  constexpr bool seg_mode = MODE == trav::MODE_KNN || MODE == trav::MODE_RANGE_COUNT || MODE == trav::MODE_RANGE_LIST_COUNT ||
                            MODE == trav::MODE_RANGE_LIST;
  if constexpr (seg_mode) {  // segmented build: the kernels with the per-lane segment cull
    if (c->segmented) {
      if constexpr (MODE == trav::MODE_KNN) {
        if (c->counters) kern = variant == 2 ? TK_PICK_SEG(true, 2) : variant == 1 ? TK_PICK_SEG(true, 1) : TK_PICK_SEG(true, 0);
        else kern = variant == 2 ? TK_PICK_SEG(false, 2) : variant == 1 ? TK_PICK_SEG(false, 1) : TK_PICK_SEG(false, 0);
      } else {
        kern = c->counters ? trav::traverse_kernel<MODE, true, 0, false, true> : trav::traverse_kernel<MODE, false, 0, false, true>;
      }
    }
  }
  if (!kern) {
    if constexpr (MODE >= trav::MODE_DBSCAN_CORE) {  // the DBSCAN passes: exact filter, no k-list (one variant each)
      kern = c->counters ? trav::traverse_kernel<MODE, true, 0, false> : trav::traverse_kernel<MODE, false, 0, false>;
    } else {
      if (c->counters) kern = variant == 2 ? TK_PICK(true, 2) : variant == 1 ? TK_PICK(true, 1) : TK_PICK(true, 0);
      else kern = variant == 2 ? TK_PICK(false, 2) : variant == 1 ? TK_PICK(false, 1) : TK_PICK(false, 0);
    }
  }
#undef TK_PICK
#undef TK_PICK_SEG
  cudaFuncAttributes fa;
  TK_CUDA(c, cudaFuncGetAttributes(&fa, kern));
  int warps = 0, bps = 1;
  if (!pick_shape(per_warp, fa.numRegs, &warps, &bps))
    return fail(c, TKNN_EINVAL, "k = %d needs %zu B of shared memory per warp", k, per_warp);
  const size_t smem = per_warp * warps;
  if (c->blocks_per_sm > 0) bps = c->blocks_per_sm;
  uint64_t grid = (uint64_t)c->sm_count * bps;
  const uint64_t need = ((uint64_t)P.n_groups + warps - 1) / warps;
  if (grid > need) grid = std::max<uint64_t>(1, need);
  TK_CUDA(c, cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  kern<<<(unsigned)grid, warps * 32, smem, c->stream>>>(P);
  TK_CUDA(c, cudaGetLastError());
  return TKNN_OK;
}

grid::GridParams grid_params(const tknn_ctx* c) {
  grid::GridParams G;
  G.cells = c->grid_cells.as<uint2>();
  G.frame = c->grid_frame.as<float>();
  G.level = c->built_grid_level;
  return G;
}

// dense kNN round (k <= 24, not final) on the cell grid of the current build (grid.cuh)
int launch_grid(tknn_ctx* c, const trav::Params& P) {
  void (*kern)(const trav::Params, const grid::GridParams) = c->counters ? grid::grid_knn_kernel<true> : grid::grid_knn_kernel<false>;
  const size_t per_warp = grid::smem_per_warp(P.k);
  cudaFuncAttributes fa;
  TK_CUDA(c, cudaFuncGetAttributes(&fa, kern));
  int warps = 0, bps = 1;
  if (!pick_shape(per_warp, fa.numRegs, &warps, &bps))
    return fail(c, TKNN_EINVAL, "k = %d needs %zu B of shared memory per warp", P.k, per_warp);
  const size_t smem = per_warp * warps;
  if (c->blocks_per_sm > 0) bps = c->blocks_per_sm;
  uint64_t grid = (uint64_t)c->sm_count * bps;
  const uint64_t need = ((uint64_t)P.n_groups + warps - 1) / warps;
  if (grid > need) grid = std::max<uint64_t>(1, need);
  TK_CUDA(c, cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  kern<<<(unsigned)grid, warps * 32, smem, c->stream>>>(P, grid_params(c));
  TK_CUDA(c, cudaGetLastError());
  return TKNN_OK;
}

// sparse kNN round (k <= 24, not final) on the cell grid: one thread per query (grid.cuh: grid_sparse_kernel)
int launch_grid_sparse(tknn_ctx* c, const trav::Params& P) {
  const size_t smem = trav::sparse_smem(P.k);
  const unsigned grid = (unsigned)((P.n_active + trav::SPARSE_THREADS - 1) / trav::SPARSE_THREADS);
  void (*kern)(const trav::Params, const grid::GridParams) =
      c->counters ? grid::grid_sparse_kernel<true> : grid::grid_sparse_kernel<false>;
  TK_CUDA(c, cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  kern<<<grid, trav::SPARSE_THREADS, smem, c->stream>>>(P, grid_params(c));
  TK_CUDA(c, cudaGetLastError());
  return TKNN_OK;
}

// thread-per-query variant for rounds whose active set is a small, spatially incoherent remainder
int launch_traverse_sparse(tknn_ctx* c, const trav::Params& P) {
  const size_t smem = trav::sparse_smem(P.k);
  if (smem > 200 * 1024) return TKNN_EINVAL;  // caller falls back to the cooperative kernel
  const unsigned grid = (unsigned)((P.n_active + trav::SPARSE_THREADS - 1) / trav::SPARSE_THREADS);
  void (*kern)(const trav::Params) =
      c->segmented ? (c->counters ? trav::traverse_sparse_kernel<true, true> : trav::traverse_sparse_kernel<false, true>)
                   : (c->counters ? trav::traverse_sparse_kernel<true> : trav::traverse_sparse_kernel<false>);
  TK_CUDA(c, cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  kern<<<grid, trav::SPARSE_THREADS, smem, c->stream>>>(P);
  TK_CUDA(c, cudaGetLastError());
  return TKNN_OK;
}

// warp-per-query (T = 32: tiny rounds, the start-radius sample, small query sets) or team-per-query (T = 4 / 8 / 16: sparse
// rounds) variant
template <int T>
int launch_traverse_team(tknn_ctx* c, const trav::Params& P) {
  const size_t smem = trav::warpq_smem(P.k, T);
  const uint64_t per_block = (uint64_t)trav::WQ_WARPS * (32 / T);
  const unsigned grid = (unsigned)((P.n_active + per_block - 1) / per_block);
  if (P.unresolved)  // the kernel ORs bits into the ballot words
    TK_CUDA(c, cudaMemsetAsync(P.unresolved, 0, sizeof(uint32_t) * (size_t)P.n_groups, c->stream));
  void (*kern)(const trav::Params) =
      c->segmented ? (c->counters ? trav::traverse_warp_kernel<true, T, true> : trav::traverse_warp_kernel<false, T, true>)
                   : (c->counters ? trav::traverse_warp_kernel<true, T> : trav::traverse_warp_kernel<false, T>);
  TK_CUDA(c, cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  kern<<<grid, trav::WQ_WARPS * 32, smem, c->stream>>>(P);
  TK_CUDA(c, cudaGetLastError());
  return TKNN_OK;
}

int launch_traverse_warp(tknn_ctx* c, const trav::Params& P) { return launch_traverse_team<32>(c, P); }

// sparse rounds: teams of c->sparse_team lanes per query, or (0) the thread-per-query kernel
int launch_traverse_sparse_round(tknn_ctx* c, const trav::Params& P) {
  const size_t team_smem = trav::warpq_smem(P.k, std::max(4, c->sparse_team));
  if (c->sparse_team == 0 || team_smem > 200 * 1024) return launch_traverse_sparse(c, P);
  switch (c->sparse_team) {
    case 4: return launch_traverse_team<4>(c, P);
    case 16: return launch_traverse_team<16>(c, P);
    default: return launch_traverse_team<8>(c, P);
  }
}

// the segment arrays of a segmented build (read by the SEG kernels only).  seg_of: the segment of every query position,
// c->seg_of when the queries are the built points, the sorted query segments of a staged query set otherwise.
void set_segments(const tknn_ctx* c, trav::Params& P, const uint32_t* seg_of) {
  if (!c->segmented) return;
  P.seg_of = seg_of;
  P.seg_off = c->seg_off.as<uint64_t>();
  P.node_seg = c->node_seg.as<int4>();
}

// One round = one traversal launch over the active queries; unresolved ones are compacted (order preserved) into the
// next round's queue and the radius doubles (hostCode.cpp:285-340 without the refits).
//
// Small searches are latency bound (cfg1: 100 K queries, 0.15 ms of kernels), so the common case makes NO host decision
// between its launches: round 1 reads its radius from the device (the estimator's output), the compaction runs
// unconditionally, and round 2 is launched SPECULATIVELY as the final, unbounded round of one warp per query over at most
// `cap` queue entries with the true count read on the device.  The host then reads {count, radius} once.  Only when more
// than `cap` queries were left (a far too small user radius) does the doubling loop continue for the rest.
int run_rounds(tknn_ctx* c, const Job& job, int* launches_io) {
  uint32_t* sc = c->scalars.as<uint32_t>();
  const uint64_t n0 = job.n_queries;
  const uint32_t g0 = (uint32_t)((n0 + 31) / 32);
  TK_TRY(ensure(c, c->unresolved, sizeof(uint32_t) * (size_t)(g0 + 1)));
  TK_TRY(ensure(c, c->offsets, sizeof(uint32_t) * (size_t)(g0 + 1)));

  const float diag = std::sqrt((c->scene_box[3] - c->scene_box[0]) * (c->scene_box[3] - c->scene_box[0]) +
                               (c->scene_box[4] - c->scene_box[1]) * (c->scene_box[4] - c->scene_box[1]) +
                               (c->scene_box[5] - c->scene_box[2]) * (c->scene_box[5] - c->scene_box[2]));
  float radius = job.r_dev ? 0.0f : job.start_radius;  // with r_dev: known after the first read-back
  bool radius_known = job.r_dev == nullptr;
  uint64_t active = n0;
  const uint32_t* queue = job.first_queue;
  DevBuf* qbuf = nullptr;  // which of queue_a / queue_b holds `queue` (nullptr: the caller's first queue, or none)
  int round = 0;
  int launches = 0;
  const uint64_t spec_cap = std::min<uint64_t>(n0, (uint64_t)std::max(0, c->warp_round_max));
  const bool speculate = c->speculative_max > 0 && n0 <= (uint64_t)c->speculative_max && spec_cap > 0;

  auto fill = [&](trav::Params& P, bool last) {
    std::memset(&P, 0, sizeof(P));
    P.nodes = c->nodes.as<Node>();
    P.node_min_idx = c->node_min_idx.as<int2>();
    P.pts = c->pts.as<float4>();
    P.queries = job.queries;
    P.queue = queue;
    P.self_ids = job.self_ids;
    P.query_r2 = job.query_r2;
    P.n_active = active;
    P.q_begin = job.q_begin;
    P.n_groups = (uint32_t)((active + 31) / 32);
    P.r2 = last ? INFINITY : radius * radius;
    P.k = job.k;
    P.self_is_row = job.self_is_row;
    P.row_mode = job.row_mode;
    P.final_round = last ? 1 : 0;
    P.squared = job.squared;
    P.error = sc + SC_ERROR;
    P.idx_out = job.idx_out;
    P.dist_out = job.dist_out;
    P.qid_out = job.qid_out;
    P.unresolved = last ? nullptr : c->unresolved.as<uint32_t>();
    P.group_counter = sc + SC_GROUP_COUNTER;
    P.counters = c->counters ? reinterpret_cast<unsigned long long*>(sc + SC_COUNTERS) : nullptr;
    set_segments(c, P, job.seg_of);
  };
  // {unresolved count, radius} in one read-back: the one host decision of a round (hostCode.cpp:310-330)
  auto read_back = [&](uint32_t* count) -> int {
    struct { uint32_t total; float r; } h = {0, 0.f};
    static_assert(sizeof(h) == 2 * sizeof(uint32_t), "mailbox layout");
    TK_TRY(fetch_words(c, sc + SC_TOTAL, 1, reinterpret_cast<const uint32_t*>(job.r_dev), radius_known ? 0 : 1,
                       reinterpret_cast<uint32_t*>(&h)));
    *count = h.total;
    if (!radius_known) { radius = h.r; radius_known = true; if (job.r_host) *job.r_host = h.r; }
    return TKNN_OK;
  };

  while (active > 0) {
    // a radius the host does not know yet (r_dev) is never treated as the last round: the estimator's fallback for a
    // degenerate sample is +inf, and a round at r2 = +inf resolves every query that has k neighbours at all
    const bool last = radius_known && (std::isinf(radius) || radius > 2.0f * diag || round >= TKNN_MAX_ROUNDS - 1);
    trav::Params P;
    fill(P, last);
    if (!radius_known) P.r2_dev = job.r_dev + 1;
    const bool timed = job.record_stats && round < TKNN_MAX_ROUNDS;
    if (timed) {
      TK_TRY(ensure_round_events(c, 4 * (round + 1)));
      TK_CUDA(c, cudaEventRecord(c->round_ev[4 * round], c->stream));
      c->stats.round_queries[round] = active;
    }
    TK_CUDA(c, cudaMemsetAsync(sc + SC_GROUP_COUNTER, 0, sizeof(uint32_t), c->stream));
    if (timed) TK_CUDA(c, cudaEventRecord(c->round_ev[4 * round + 2], c->stream));
    // sparse remainder (< 1/sparse_divisor of the round-1 queries, taken from a queue): one thread per query
    const bool sparse = trav::sparse_smem(job.k) <= 200 * 1024 &&
                        (job.force_sparse || (c->sparse_divisor > 0 && queue != nullptr && round > 0 &&
                                              active * (uint64_t)c->sparse_divisor <= n0));
    // one warp per query: small rounds; four times further for k > 24, where a private heap per THREAD is slow
    // (cfg3, 51 725 leftover queries: 3.6 ms on the thread-per-query kernel, profiles/r2_ab_opts.jsonl)
    bool tiny = c->warp_round_max > 0 && active <= (uint64_t)c->warp_round_max * (job.k > trav::LIST_MAX_K ? 4u : 1u);
    // the cell grid, never in a final round (a query it leaves unresolved, capped or underfilled, reaches an exact LBVH
    // round): the dense round 1 (its groups are 32 consecutive sorted queries, or a regular slice of them) and the sparse
    // rounds (one thread per query)
    const bool grid_ok = job.grid && c->grid_on && !c->segmented && !last && job.k <= trav::LIST_MAX_K;
    // A small sparse round still takes the grid when it holds more than three waves of the warp kernel's resident queries:
    // the grid kernel's time stays near the length of one query's walk (cfg2, 3 K to 97 K leftovers: 0.15 - 0.17 ms), while
    // the warp kernel's grows with its waves (0.08 ms at 3 K, 0.15 ms at 15 K, 0.24 ms at 30 K queries: the two cross near
    // 17 K, about three of its waves; DESIGN.md §3.2a).
    if (tiny && sparse && grid_ok) {
      int bps = 0;
      TK_CUDA(c, cudaOccupancyMaxActiveBlocksPerMultiprocessor(&bps, trav::traverse_warp_kernel<false, 32>, trav::WQ_WARPS * 32,
                                                              trav::warpq_smem(job.k)));
      if (active > 3ull * (uint64_t)bps * trav::WQ_WARPS * (uint64_t)c->sm_count) tiny = false;
    }
    // which rounds walked the grid (tknn_stats::grid_rounds), ORed over the slices of a sliced search
    if (!tiny && grid_ok && (sparse || round == 0) && round < 32) c->stats.grid_rounds |= 1u << round;
    if (tiny) TK_TRY(launch_traverse_warp(c, P));
    else if (sparse && grid_ok) TK_TRY(launch_grid_sparse(c, P));
    else if (sparse) TK_TRY(launch_traverse_sparse_round(c, P));
    else if (grid_ok && round == 0) TK_TRY(launch_grid(c, P));
    else TK_TRY(launch_traverse<trav::MODE_KNN>(c, P));
    if (timed) TK_CUDA(c, cudaEventRecord(c->round_ev[4 * round + 3], c->stream));
    ++launches;

    uint32_t next_active = 0;
    if (!last) {
      // order-preserving compaction of the unresolved queries (ballot words + prefix sums)
      TK_TRY(popc_scan(c, c->unresolved.as<uint32_t>(), P.n_groups, c->offsets.as<uint32_t>(), &launches));
      DevBuf& qout = (qbuf == &c->queue_a) ? c->queue_b : c->queue_a;
      if (speculate && round == 0) {
        // ---- no host decision: compact everything, run the final round over <= spec_cap entries, then look ----
        TK_TRY(ensure(c, qout, sizeof(uint32_t) * (size_t)n0));
        trav::compact_queue_kernel<<<blocks_for((uint64_t)P.n_groups * 32, 256), 256, 0, c->stream>>>(
            c->unresolved.as<uint32_t>(), c->offsets.as<uint32_t>(), P.n_groups, queue, job.q_begin, qout.as<uint32_t>());
        ++launches;
        if (timed) TK_CUDA(c, cudaEventRecord(c->round_ev[4 * round + 1], c->stream));
        queue = qout.as<uint32_t>();
        qbuf = &qout;
        active = spec_cap;
        trav::Params F;
        fill(F, true);
        F.n_active_dev = sc + SC_TOTAL;
        const bool timed2 = job.record_stats && round + 1 < TKNN_MAX_ROUNDS;
        if (timed2) {
          TK_TRY(ensure_round_events(c, 4 * (round + 2)));
          TK_CUDA(c, cudaEventRecord(c->round_ev[4 * (round + 1)], c->stream));
          TK_CUDA(c, cudaEventRecord(c->round_ev[4 * (round + 1) + 2], c->stream));
        }
        TK_TRY(launch_traverse_warp(c, F));
        ++launches;
        if (timed2) {
          TK_CUDA(c, cudaEventRecord(c->round_ev[4 * (round + 1) + 3], c->stream));
          TK_CUDA(c, cudaEventRecord(c->round_ev[4 * (round + 1) + 1], c->stream));
        }
        TK_TRY(read_back(&next_active));
        ++round;  // round 1 is done
        if (next_active > 0) {
          if (timed2) c->stats.round_queries[round] = std::min<uint64_t>(next_active, spec_cap);
          ++round;  // ... and so is the speculative final round
        }
        radius *= 2.0f;
        if (next_active <= spec_cap) { active = 0; break; }
        // more queries were left than the speculative round covered: the doubling loop takes the rest of the queue
        queue = queue + spec_cap;
        active = next_active - spec_cap;
        continue;
      }
      TK_TRY(read_back(&next_active));
      if (next_active > 0) {
        TK_TRY(ensure(c, qout, sizeof(uint32_t) * (size_t)next_active));
        trav::compact_queue_kernel<<<blocks_for((uint64_t)P.n_groups * 32, 256), 256, 0, c->stream>>>(
            c->unresolved.as<uint32_t>(), c->offsets.as<uint32_t>(), P.n_groups, queue, job.q_begin, qout.as<uint32_t>());
        ++launches;
        queue = qout.as<uint32_t>();
        qbuf = &qout;
      }
    }
    if (timed) TK_CUDA(c, cudaEventRecord(c->round_ev[4 * round + 1], c->stream));
    ++round;
    active = next_active;
    if (!last) radius *= 2.0f;
  }
  if (!radius_known && job.r_host) {  // a single final round ran on a device radius: fetch it for the statistics
    uint32_t dummy = 0;
    TK_TRY(read_back(&dummy));
  }
  if (job.record_stats) {
    c->stats.rounds = round;
    c->stats.final_radius = radius;
  }
  if (launches_io) *launches_io += launches;
  return TKNN_OK;
}

// Sampled k-th-neighbour distance -> start radius (role of Util/random_sample.py:5-32), entirely on the device: the
// sample queue is generated by a kernel, the sampled queries run one unbounded final round (one warp per query), and a
// one-block radix select leaves {r, r * r} at sc[SC_QUANTILE], r the quantile_pm per-mille quantile of the sampled k-th
// neighbour distances.  Nothing is copied and nothing waits: round 1 reads r2 from there (Job::r_dev).
int estimate_radius_device(tknn_ctx* c, const float4* queries, uint64_t q_begin, uint64_t nq, const int32_t* self_ids,
                           int self_is_row, const uint32_t* seg_of, int k, int quantile_pm, int* launches) {
  // sample_groups runs of 32 consecutive sorted positions: neighbouring queries walk nearly the same nodes and leaves
  const uint64_t groups = (nq + 31) / 32;
  const uint64_t sg = std::min<uint64_t>((uint64_t)std::max(1, c->sample_groups), groups);
  uint64_t m = sg * 32;  // only the last group of the range can be short, and only the last run can be that group
  if (groups * (sg - 1) / sg == groups - 1 && (nq & 31)) m -= 32 - (nq & 31);
  TK_TRY(ensure(c, c->sample, m * sizeof(uint32_t) + m * (size_t)k * (sizeof(int32_t) + sizeof(float))));
  uint32_t* dq = c->sample.as<uint32_t>();
  int32_t* di = reinterpret_cast<int32_t*>(dq + m);
  float* dd = reinterpret_cast<float*>(di + m * (size_t)k);
  trav::sample_queue_kernel<<<blocks_for(sg * 32, 256), 256, 0, c->stream>>>(groups, (uint32_t)sg, q_begin, nq, dq);
  Job job;
  job.queries = queries;
  job.self_ids = self_ids;
  job.seg_of = seg_of;
  job.first_queue = dq;
  job.n_queries = m;
  job.q_begin = q_begin;
  job.self_is_row = self_is_row;
  job.row_mode = 2;
  job.k = k;
  job.start_radius = INFINITY;
  job.squared = 0;
  job.idx_out = di;
  job.dist_out = dd;
  job.record_stats = false;
  job.force_sparse = true;
  const int saved = c->counters;
  c->counters = 0;
  int rc = run_rounds(c, job, launches);
  c->counters = saved;
  TK_TRY(rc);
  const int qpm = std::min(1000, std::max(0, quantile_pm));
  const uint32_t pos = (uint32_t)((double)(m - 1) * qpm / 1000.0);
  // a segmented build leaves the rows of segments with at most k points unfilled: the quantile ignores them
  trav::radius_quantile_kernel<<<1, 1024, 0, c->stream>>>(dd, (uint32_t)m, k, pos,
                                                          reinterpret_cast<float*>(c->scalars.as<uint32_t>() + SC_QUANTILE),
                                                          c->segmented ? qpm : -1);
  TK_CUDA(c, cudaGetLastError());
  if (launches) *launches += 2;
  return TKNN_OK;
}

int auto_morton_bits(uint64_t n) {
  int lg = 0;
  while (((uint64_t)1 << lg) < n) ++lg;
  return std::min(21, std::max(10, (lg + 2) / 3 + 8));
}

// Key layout of a build (TKNN_OPT_SORT_MODE, TKNN_OPT_MORTON_BITS).  Packed: the curve code sits above the point's index
// in one u64 and the sort moves keys only.  The code gets as many bits per axis as fit beside the index, at most 13
// (39 bits: five 8-bit passes) — 13 bits at 10 M points are cells 32x finer per axis than the mean point spacing, 12 bits
// at 100 M points 9x — and one bit per axis less where that saves a whole pass and still leaves log2(n)/3 + 4.  Points
// that share a cell are ordered by index: tree quality at the scale of one cell, never exactness.
// *idx_bits == 0: pair sort.
void key_layout(uint64_t n, int morton_bits, int sort_mode, int* mbits, int* idx_bits) {
  int lg = 0;
  while (((uint64_t)1 << lg) < n) ++lg;
  const int ib = std::max(1, lg), spacing = (lg + 2) / 3, fit = (64 - ib) / 3;
  *idx_bits = 0;
  if (morton_bits > 0) {
    *mbits = morton_bits;
    if (sort_mode == 0 && 3 * morton_bits + ib <= 64) *idx_bits = ib;
    return;
  }
  if (sort_mode == 0 && fit >= spacing + 3) {
    int b = std::min(13, fit);
    const int spare = 3 * b - 8 * ((3 * b - 1) / 8);  // code bits in the last, partial pass
    if (spare <= 3 && b - 1 >= spacing + 4) --b;
    *mbits = b;
    *idx_bits = ib;
    return;
  }
  *mbits = auto_morton_bits(n);
}

void choose_key_layout(const tknn_ctx* c, uint64_t n, int* mbits, int* idx_bits) {
  key_layout(n, c->morton_bits, c->sort_mode, mbits, idx_bits);
}

// Key layout of a segmented build: the segment id (*seg_bits = ceil(log2 n_segments) bits) above the curve code, and the
// code sized for the LARGEST segment, not for n (65 536 clouds of 64 points need few bits per axis).  Packed keys (code
// above the index) while the code keeps that segment's point spacing plus three bits per axis; else (code, index) pairs
// with the code cut to fit beside the segment id.
void segment_key_layout(const tknn_ctx* c, uint64_t n, uint64_t n_segments, uint64_t max_segment, int* mbits, int* idx_bits,
                        int* seg_bits) {
  int sb = 0, lg = 0, ls = 0;
  while (((uint64_t)1 << sb) < n_segments) ++sb;
  while (((uint64_t)1 << lg) < n) ++lg;
  const uint64_t ms = std::max<uint64_t>(2, max_segment);
  while (((uint64_t)1 << ls) < ms) ++ls;
  const int ib = std::max(1, lg), spacing = (ls + 2) / 3, fit = (64 - ib - sb) / 3;
  int want = 0, want_idx = 0;
  key_layout(ms, c->morton_bits, c->sort_mode, &want, &want_idx);
  *seg_bits = sb;
  if (c->sort_mode == 0 && (c->morton_bits > 0 ? c->morton_bits <= fit : fit >= spacing + 3)) {
    *mbits = std::min(want, fit);
    *idx_bits = ib;
    return;
  }
  *mbits = std::min(c->morton_bits > 0 ? c->morton_bits : auto_morton_bits(ms), (64 - sb) / 3);
  *idx_bits = 0;
}

// Hilbert levels of the key kernel (lbvh.cuh: morton_kernel): two levels below the one where a cell holds one point
int hilbert_levels(uint64_t n, int bits, int forced = 0) {
  if (forced > 0) return std::max(2, std::min(bits, forced));
  int lg = 0;
  while (((uint64_t)1 << lg) < n) ++lg;
  return std::max(2, std::min(bits, (lg + 2) / 3 + 2));
}

int check_ctx(tknn_ctx* c) { return c ? TKNN_OK : TKNN_EINVAL; }

// Reads n_segments + 1 offsets (host or device: one small read-back) into *off and checks that they start at 0, never
// decrease and end at `total` (named `total_name` in the message; a null total_name: they may end anywhere); `side`
// names the offsets in the message.
int read_offsets(tknn_ctx* c, const char* what, const char* side, const uint64_t* offsets, uint64_t n_segments,
                 uint64_t total, const char* total_name, std::vector<uint64_t>* off_out) {
  std::vector<uint64_t>& off = *off_out;
  off.assign(n_segments + 1, 0);
  TK_TRY(read_to_host(c, offsets, off.size(), off.data()));
  if (off[0] != 0) return fail(c, TKNN_EINVAL, "%s: %s offsets must start at 0", what, side);
  if (total_name && off[n_segments] != total)
    return fail(c, TKNN_EINVAL, "%s: %s offsets must end at %s = %llu", what, side, total_name, (unsigned long long)total);
  for (uint64_t s = 0; s < n_segments; ++s)
    if (off[s + 1] < off[s]) return fail(c, TKNN_EINVAL, "%s: %s offsets decrease at segment %llu", what, side, (unsigned long long)s);
  return TKNN_OK;
}

// the calls that do not restrict their neighbours to a segment yet refuse a segmented build rather than ignore it
int refuse_segmented(tknn_ctx* c, const char* what) {
  if (c->segmented) return fail(c, TKNN_ESTATE, "%s: segmented builds (tknn_build_segments) do not support it yet", what);
  return TKNN_OK;
}

// out[0 .. na) = a[0 .. na), out[na .. na + nb) = b[0 .. nb): the mailbox writer (ctx.cuh)
static __global__ void mailbox_kernel(const uint32_t* __restrict__ a, int na, const uint32_t* __restrict__ b, int nb,
                                      volatile uint32_t* out) {
  for (int i = 0; i < na; ++i) out[i] = a[i];
  for (int i = 0; i < nb; ++i) out[na + i] = b[i];
  __threadfence_system();
}

// Brings na + nb (<= 16) device words to the host and waits for the stream.  With host outputs the bulk result copies of
// the previous slice occupy the device->host copy engine for milliseconds; a 4-byte cudaMemcpyAsync on the compute stream
// would queue behind them and stall the round loop (measured: cfg2's four file-order slices searched in 15.2 ms with
// idx + dist copies in flight against 12.6 ms with half the bytes).  A kernel's stores to mapped host memory do not.
int fetch_words(tknn_ctx* c, const uint32_t* a, int na, const uint32_t* b, int nb, uint32_t* host_out) {
  if (na + nb > 16 || na < 0 || nb < 0) return fail(c, TKNN_EINVAL, "internal: mailbox overflow");
  if (c->mailbox_h) {
    mailbox_kernel<<<1, 1, 0, c->stream>>>(a, na, b, nb, c->mailbox_d);
    TK_CUDA(c, cudaGetLastError());
    ++c->mailbox_launches;
    TK_CUDA(c, cudaStreamSynchronize(c->stream));
    for (int i = 0; i < na + nb; ++i) host_out[i] = c->mailbox_h[i];
    return TKNN_OK;
  }
  if (na) TK_CUDA(c, cudaMemcpyAsync(host_out, a, na * sizeof(uint32_t), cudaMemcpyDeviceToHost, c->stream));
  if (nb) TK_CUDA(c, cudaMemcpyAsync(host_out + na, b, nb * sizeof(uint32_t), cudaMemcpyDeviceToHost, c->stream));
  TK_CUDA(c, cudaStreamSynchronize(c->stream));
  return TKNN_OK;
}

int read_error_flag(tknn_ctx* c) {
  uint32_t e[2] = {0, 0};  // SC_ERROR, SC_QBAD
  TK_TRY(fetch_words(c, c->scalars.as<uint32_t>() + SC_ERROR, 2, nullptr, 0, e));
  if (e[0]) return fail(c, TKNN_ECUDA, "traversal stack overflow (BVH deeper than %d)", STACK_DEPTH);
  if (e[1]) return fail(c, TKNN_EINVAL, "non-finite coordinate in the query points");
  return TKNN_OK;
}

int collect_counters(tknn_ctx* c) {
  if (!c->counters) return TKNN_OK;
  unsigned long long h[N_COUNTERS];
  TK_CUDA(c, cudaMemcpyAsync(h, c->scalars.as<uint32_t>() + SC_COUNTERS, sizeof(h), cudaMemcpyDeviceToHost, c->stream));
  TK_CUDA(c, cudaStreamSynchronize(c->stream));
  c->stats.nodes_visited = h[0];
  c->stats.points_tested = h[1];
  c->stats.heap_inserts = h[2];
  c->stats.warp_node_visits = h[3];
  c->stats.warp_leaf_visits = h[4];
  c->stats.warp_point_loads = h[5];
  c->stats.filter_violations = h[6];
  c->stats.grid_deferred = h[7];
  static_assert(grid::GRID_PHASES == 6 && grid::GRID_INSERT_SLOT < N_COUNTERS, "tknn_stats::grid_phase_cycles");
  for (int p = 0; p < grid::GRID_PHASES; ++p) c->stats.grid_phase_cycles[p] = h[grid::GRID_PHASE_SLOT + p];
  c->stats.grid_insert_iters = h[grid::GRID_INSERT_ITER_SLOT];
  c->stats.grid_inserts = h[grid::GRID_INSERT_SLOT];
  return TKNN_OK;
}

int finish_round_stats(tknn_ctx* c) {
  for (int r = 0; r < c->stats.rounds && r < TKNN_MAX_ROUNDS; ++r) {
    float ms = 0.f;
    TK_CUDA(c, cudaEventElapsedTime(&ms, c->round_ev[4 * r], c->round_ev[4 * r + 1]));
    c->stats.round_ms[r] = ms;
    TK_CUDA(c, cudaEventElapsedTime(&ms, c->round_ev[4 * r + 2], c->round_ev[4 * r + 3]));
    c->stats.kernel_ms[r] = ms;
  }
  return TKNN_OK;
}

void reset_search_stats(tknn_ctx* c) {
  tknn_stats& s = c->stats;
  s.n_queries = 0; s.k = 0; s.rounds = 0; s.start_radius = s.final_radius = 0.f;
  s.estimate_ms = s.search_ms = s.d2h_ms = 0.f;
  std::memset(s.round_ms, 0, sizeof(s.round_ms));
  std::memset(s.kernel_ms, 0, sizeof(s.kernel_ms));
  std::memset(s.round_queries, 0, sizeof(s.round_queries));
  s.kernel_launches = 0;
  s.nodes_visited = s.points_tested = s.heap_inserts = 0;
  s.warp_node_visits = s.warp_leaf_visits = s.warp_point_loads = s.filter_violations = 0;
  s.grid_rounds = 0;
  s.grid_deferred = 0;
  std::memset(s.grid_phase_cycles, 0, sizeof(s.grid_phase_cycles));
  s.grid_insert_iters = s.grid_inserts = 0;
  s.d2h_bytes = 0;
  c->mailbox_launches = 0;
}

}  // namespace

// all-points search over query positions [q_begin, q_begin + nq) of the sorted order
int tknn::host::search_range(tknn_ctx* c, int k, float start_radius, uint64_t q_begin, uint64_t nq, int row_mode, int32_t* qid_out,
                 int32_t* idx_out, float* dist_out, uint64_t rows) {
  if (c->n == 0) return fail(c, TKNN_ESTATE, "tknn_search before tknn_build");
  if (k < 1 || k > TKNN_MAX_K) return fail(c, TKNN_EINVAL, "k = %d outside [1, %d]", k, TKNN_MAX_K);
  if ((uint64_t)k > c->n - 1) return fail(c, TKNN_EINVAL, "k = %d > n - 1 = %llu: fewer than k neighbours exist", k,
                                          (unsigned long long)(c->n - 1));
  if (std::isnan(start_radius)) return fail(c, TKNN_EINVAL, "start_radius is NaN");
  if (!idx_out) return fail(c, TKNN_EINVAL, "null output array");
  if (c->ids_in_w && row_mode == 0)
    return fail(c, TKNN_ESTATE, "this BVH carries caller-chosen point ids (point-partitioned build): rows in build order do not exist");
  reset_search_stats(c);
  c->stats.n_queries = nq;
  c->stats.k = k;
  uint32_t* sc = c->scalars.as<uint32_t>();

  // dist_out == nullptr: indices only — the distances stay in device scratch and are never copied (half the
  // device->host bytes of a host-output call; a distance is recomputable from its index)
  const bool idx_dev = is_device_ptr(idx_out), dist_dev = !dist_out || is_device_ptr(dist_out);
  const bool qid_dev = qid_out ? is_device_ptr(qid_out) : true;
  int32_t* d_idx = idx_out;
  float* d_dist = dist_out;
  int32_t* d_qid = qid_out;
  const size_t out_elems = (size_t)rows * (size_t)k;
  if (!idx_dev || (qid_out && !qid_dev)) {
    TK_TRY(ensure(c, c->stage_idx, out_elems * sizeof(int32_t) + (qid_out ? rows * sizeof(int32_t) : 0)));
    if (!idx_dev) d_idx = c->stage_idx.as<int32_t>();
    if (qid_out && !qid_dev) d_qid = c->stage_idx.as<int32_t>() + out_elems;
  }
  if (!dist_dev || !dist_out) {
    TK_TRY(ensure(c, c->stage_dist, out_elems * sizeof(float)));
    d_dist = c->stage_dist.as<float>();
  }

  TK_CUDA(c, cudaMemsetAsync(sc + SC_ERROR, 0, 2 * sizeof(uint32_t), c->stream));
  TK_CUDA(c, cudaMemsetAsync(sc + SC_COUNTERS, 0, N_COUNTERS * sizeof(unsigned long long), c->stream));
  TK_CUDA(c, cudaEventRecord(c->ev[0], c->stream));
  int launches = 0;
  float r0 = start_radius;
  const bool estimated = nq > 0 && !(r0 > 0.0f);
  // round 1 on the cell grid (run_rounds: grid_ok) has its own start-radius quantile (TKNN_OPT_GRID_RADIUS_QUANTILE)
  const bool grid_round1 = c->grid_on && !c->segmented && k <= trav::LIST_MAX_K;
  if (estimated)
    TK_TRY(estimate_radius_device(c, c->pts.as<float4>(), q_begin, nq, nullptr, 1, c->seg_of.as<uint32_t>(), k,
                                  grid_round1 ? c->grid_radius_quantile : c->radius_quantile, &launches));
  TK_CUDA(c, cudaEventRecord(c->ev[1], c->stream));
  c->stats.start_radius = r0;

  Job job;
  if (estimated) {
    job.r_dev = reinterpret_cast<const float*>(sc + SC_QUANTILE);
    job.r_host = &c->stats.start_radius;
  }
  job.queries = c->pts.as<float4>();
  job.seg_of = c->seg_of.as<uint32_t>();
  job.n_queries = nq;
  job.q_begin = q_begin;
  job.self_is_row = 1;
  job.row_mode = row_mode;
  job.k = k;
  job.start_radius = r0;
  job.squared = c->squared;
  job.idx_out = d_idx;
  job.dist_out = d_dist;
  job.qid_out = d_qid;
  job.grid = true;

  // Compact rows (row_mode 1) are in Morton order, so a contiguous slice of the queries yields a
  // contiguous, FINAL slice of the output: with host outputs the shard is searched in chunks and each
  // chunk's device->host copy (copy stream) overlaps the search of the next one (compute stream).
  const uint64_t groups = (nq + 31) / 32;
  const bool host_out = !idx_dev || !dist_dev || (qid_out && !qid_dev);
  const int chunks = (row_mode == 1 && host_out && c->output_chunks > 1 && nq >= (1u << 18))
                         ? (int)std::min<uint64_t>((uint64_t)c->output_chunks, groups) : 1;
  // file-order slices: the device->host link moves the rows of a slice about as fast as a slice of that sparsity is
  // searched, so the step ends one slice-search after the link could have started: 5 slices with distances (cfg2: 21.2 /
  // 20.6 / 20.3 / 20.9 / 21.8 ms end to end with 3 / 4 / 5 / 6 / 8), 2 when only indices leave the device (17.9 / 16.5 / 16.9
  // ms with 1 / 2 / 3)
  // The heap kernel (k > 24) pays far more for a sparse slice (cfg3, k = 64: halves cost 1.7x per query, quarters 2.5x), so
  // there the search is the slower side from three slices on: 140.2 / 136.0 / 136.5 / 144.6 ms with 1 / 2 / 3 / 4 slices, and
  // 95.3 / 106.3 / 121.5 ms indices-only with 1 / 2 / 3 (profiles/r2_e2e_cfg3.txt).
  const bool heap_k = k > trav::LIST_MAX_K;
  const int fo_chunks = c->file_order_chunks > 0 ? c->file_order_chunks : (heap_k ? (dist_out ? 2 : 1) : (dist_out ? 5 : 2));
  if (chunks > 1) {
    while ((int)c->chunk_ev.size() < chunks) {
      cudaEvent_t e;
      TK_CUDA(c, cudaEventCreate(&e));
      c->chunk_ev.push_back(e);
    }
    for (int ci = 0; ci < chunks; ++ci) {
      const uint64_t g0 = groups * (uint64_t)ci / chunks, g1 = groups * (uint64_t)(ci + 1) / chunks;
      const uint64_t r_lo = g0 * 32, r_hi = std::min<uint64_t>(nq, g1 * 32);  // rows of this chunk
      if (r_hi <= r_lo) continue;
      Job cj = job;
      cj.q_begin = q_begin + r_lo;
      cj.n_queries = r_hi - r_lo;
      cj.idx_out = d_idx + r_lo * (uint64_t)k;
      cj.dist_out = d_dist + r_lo * (uint64_t)k;
      cj.qid_out = d_qid ? d_qid + r_lo : nullptr;
      cj.record_stats = (ci == 0);  // per-round figures describe the first chunk
      TK_TRY(run_rounds(c, cj, &launches));
      TK_CUDA(c, cudaEventRecord(c->chunk_ev[ci], c->stream));
      TK_CUDA(c, cudaStreamWaitEvent(c->copy_stream, c->chunk_ev[ci], 0));
      const size_t e0 = (size_t)r_lo * k, ne = (size_t)(r_hi - r_lo) * k;
      if (!idx_dev) {
        TK_CUDA(c, cudaMemcpyAsync(idx_out + e0, d_idx + e0, ne * sizeof(int32_t), cudaMemcpyDeviceToHost, c->copy_stream));
        c->stats.d2h_bytes += ne * sizeof(int32_t);
      }
      if (!dist_dev) {
        TK_CUDA(c, cudaMemcpyAsync(dist_out + e0, d_dist + e0, ne * sizeof(float), cudaMemcpyDeviceToHost, c->copy_stream));
        c->stats.d2h_bytes += ne * sizeof(float);
      }
      if (qid_out && !qid_dev) {
        TK_CUDA(c, cudaMemcpyAsync(qid_out + r_lo, d_qid + r_lo, (r_hi - r_lo) * sizeof(int32_t), cudaMemcpyDeviceToHost,
                                   c->copy_stream));
        c->stats.d2h_bytes += (r_hi - r_lo) * sizeof(int32_t);
      }
    }
    TK_CUDA(c, cudaEventRecord(c->ev[2], c->stream));
    // the caller's stream must not run ahead of the copies
    TK_CUDA(c, cudaEventRecord(c->chunk_ev[0], c->copy_stream));
    TK_CUDA(c, cudaStreamWaitEvent(c->stream, c->chunk_ev[0], 0));
  } else if (row_mode == 0 && host_out && fo_chunks > 1 && nq == c->n && nq >= (1u << 18)) {
    // File-order rows: slice the queries by ORIGINAL index so that each slice's rows are one contiguous,
    // final block of the output.  A slice is every C-th point of the cloud in Morton order, so its groups
    // are C times less dense in space (costlier per query) — the price of overlapping the result copy.
    const int fc = fo_chunks;
    while ((int)c->chunk_ev.size() < fc) {
      cudaEvent_t e;
      TK_CUDA(c, cudaEventCreate(&e));
      c->chunk_ev.push_back(e);
    }
    TK_TRY(ensure(c, c->chunk_queue, (size_t)nq * sizeof(uint32_t)));
    TK_TRY(ensure(c, c->unresolved, sizeof(uint32_t) * (size_t)(groups + 1)));
    TK_TRY(ensure(c, c->offsets, sizeof(uint32_t) * (size_t)(groups + 1)));
    for (int ci = 0; ci < fc; ++ci) {
      const uint64_t lo = nq * (uint64_t)ci / fc, hi = nq * (uint64_t)(ci + 1) / fc;
      if (hi <= lo) continue;
      uint32_t* cq = c->chunk_queue.as<uint32_t>() + lo;
      trav::index_range_flag_kernel<<<blocks_for(nq, 256), 256, 0, c->stream>>>(c->pts.as<float4>(), nq, (uint32_t)lo,
                                                                               (uint32_t)hi, c->unresolved.as<uint32_t>());
      TK_TRY(popc_scan(c, c->unresolved.as<uint32_t>(), groups, c->offsets.as<uint32_t>(), &launches));
      trav::compact_queue_kernel<<<blocks_for(groups * 32, 256), 256, 0, c->stream>>>(
          c->unresolved.as<uint32_t>(), c->offsets.as<uint32_t>(), (uint32_t)groups, nullptr, 0, cq);
      launches += 2;
      Job cj = job;
      cj.first_queue = cq;
      cj.n_queries = hi - lo;
      cj.record_stats = (ci == 0);
      TK_TRY(run_rounds(c, cj, &launches));
      TK_CUDA(c, cudaEventRecord(c->chunk_ev[ci], c->stream));
      TK_CUDA(c, cudaStreamWaitEvent(c->copy_stream, c->chunk_ev[ci], 0));
      const size_t e0 = (size_t)lo * k, ne = (size_t)(hi - lo) * k;
      if (!idx_dev) {
        TK_CUDA(c, cudaMemcpyAsync(idx_out + e0, d_idx + e0, ne * sizeof(int32_t), cudaMemcpyDeviceToHost, c->copy_stream));
        c->stats.d2h_bytes += ne * sizeof(int32_t);
      }
      if (!dist_dev) {
        TK_CUDA(c, cudaMemcpyAsync(dist_out + e0, d_dist + e0, ne * sizeof(float), cudaMemcpyDeviceToHost, c->copy_stream));
        c->stats.d2h_bytes += ne * sizeof(float);
      }
    }
    TK_CUDA(c, cudaEventRecord(c->ev[2], c->stream));
    TK_CUDA(c, cudaEventRecord(c->chunk_ev[0], c->copy_stream));
    TK_CUDA(c, cudaStreamWaitEvent(c->stream, c->chunk_ev[0], 0));
  } else {
    TK_TRY(run_rounds(c, job, &launches));
    TK_CUDA(c, cudaEventRecord(c->ev[2], c->stream));
    if (!idx_dev) {
      TK_CUDA(c, cudaMemcpyAsync(idx_out, d_idx, out_elems * sizeof(int32_t), cudaMemcpyDeviceToHost, c->stream));
      c->stats.d2h_bytes += out_elems * sizeof(int32_t);
    }
    if (!dist_dev) {
      TK_CUDA(c, cudaMemcpyAsync(dist_out, d_dist, out_elems * sizeof(float), cudaMemcpyDeviceToHost, c->stream));
      c->stats.d2h_bytes += out_elems * sizeof(float);
    }
    if (qid_out && !qid_dev) {
      TK_CUDA(c, cudaMemcpyAsync(qid_out, d_qid, rows * sizeof(int32_t), cudaMemcpyDeviceToHost, c->stream));
      c->stats.d2h_bytes += rows * sizeof(int32_t);
    }
  }
  TK_CUDA(c, cudaEventRecord(c->ev[3], c->stream));
  TK_CUDA(c, cudaStreamSynchronize(c->stream));
  TK_CUDA(c, cudaEventElapsedTime(&c->stats.estimate_ms, c->ev[0], c->ev[1]));
  TK_CUDA(c, cudaEventElapsedTime(&c->stats.search_ms, c->ev[0], c->ev[2]));
  TK_CUDA(c, cudaEventElapsedTime(&c->stats.d2h_ms, c->ev[2], c->ev[3]));
  if (start_radius > 0.0f) c->stats.estimate_ms = 0.f;
  c->stats.kernel_launches = (uint32_t)(launches + c->mailbox_launches + (c->mailbox_h ? 1 : 0));  // + the error-flag fetch below
  TK_TRY(finish_round_stats(c));
  TK_TRY(collect_counters(c));
  TK_TRY(read_error_flag(c));
  return TKNN_OK;
}

// ---------------------------------------------------------------------------------------------
// C ABI
// ---------------------------------------------------------------------------------------------
extern "C" {

int tknn_version(void) { return TKNN_VERSION; }

const char* tknn_last_error(const tknn_ctx* ctx) { return ctx ? ctx->err.c_str() : "null context"; }

int tknn_create(int device, tknn_ctx** out) {
  if (!out) return TKNN_EINVAL;
  *out = nullptr;
  int count = 0;
  cudaError_t e = cudaGetDeviceCount(&count);
  if (e != cudaSuccess || count <= 0) { cudaGetLastError(); return TKNN_ECUDA; }  // no CPU fallback
  if (device < 0 || device >= count) return TKNN_EINVAL;
  tknn_ctx* c = new (std::nothrow) tknn_ctx();
  if (!c) return TKNN_ENOMEM;
  c->device = device;
  ScopedDevice sd(device);
  cudaDeviceProp prop;
  if (cudaGetDeviceProperties(&prop, device) != cudaSuccess) { delete c; return TKNN_ECUDA; }
  if (prop.major < 10) { delete c; return TKNN_ECUDA; }  // sm_100a code only
  c->sm_count = prop.multiProcessorCount;
  c->l2_bytes = (size_t)prop.l2CacheSize;
  if (cudaStreamCreateWithFlags(&c->own_stream, cudaStreamNonBlocking) != cudaSuccess) { delete c; return TKNN_ECUDA; }
  c->stream = c->own_stream;
  if (cudaStreamCreateWithFlags(&c->copy_stream, cudaStreamNonBlocking) != cudaSuccess) { delete c; return TKNN_ECUDA; }
  for (auto& ev : c->ev)
    if (cudaEventCreate(&ev) != cudaSuccess) { delete c; return TKNN_ECUDA; }
  if (cudaMalloc(&c->scalars.p, SC_WORDS * sizeof(uint32_t)) != cudaSuccess) { delete c; return TKNN_ENOMEM; }
  c->scalars.bytes = SC_WORDS * sizeof(uint32_t);
  {  // the mailbox is an optimisation: without mapped memory fetch_words falls back to small copies
    void* h = nullptr;
    void* d = nullptr;
    if (cudaHostAlloc(&h, 16 * sizeof(uint32_t), cudaHostAllocMapped | cudaHostAllocPortable) == cudaSuccess &&
        cudaHostGetDevicePointer(&d, h, 0) == cudaSuccess) {
      c->mailbox_h = static_cast<uint32_t*>(h);
      c->mailbox_d = static_cast<uint32_t*>(d);
    } else {
      if (h) cudaFreeHost(h);
      cudaGetLastError();
    }
  }
  *out = c;
  return TKNN_OK;
}

int tknn_destroy(tknn_ctx* c) {
  if (!c) return TKNN_EINVAL;
  ScopedDevice sd(c->device);
  cudaStreamSynchronize(c->stream);
  tknn_internal_free_dist(c);
  for (DevBuf* b : {&c->pts, &c->nodes, &c->leaf_start, &c->node_min_idx, &c->queue_a, &c->queue_b, &c->unresolved, &c->offsets,
                    &c->block_sums, &c->scalars, &c->stage_idx, &c->stage_dist, &c->sample, &c->chunk_queue, &c->b_in, &c->b_keys_a,
                    &c->b_keys_b, &c->b_vals_a, &c->b_vals_b, &c->b_sort_tmp, &c->b_delta, &c->b_ballots, &c->b_leaf_key,
                    &c->b_child_info, &c->b_parent_leaf, &c->b_parent_node, &c->b_arrive, &c->q_stage, &c->q_keys_a, &c->q_keys_b,
                    &c->q_vals_a, &c->q_vals_b, &c->q_sort_tmp, &c->q_pts, &c->q_sid_stage, &c->q_sid_sorted, &c->q_rad_stage,
                    &c->q_r2_sorted, &c->db_parent, &c->db_min_idx, &c->db_pos_label, &c->db_bits, &c->db_core_stage,
                    &c->rl_cnt_pos, &c->rl_cnt_row, &c->rl_off_pos, &c->rl_off_row, &c->rl_sums, &c->rl_stats, &c->rl_pos_of,
                    &c->rl_self_pos, &c->rl_keys, &c->rl_long_pos, &c->rl_long_len, &c->rl_boff, &c->rl_ka, &c->rl_kb,
                    &c->rl_kc, &c->rl_va, &c->rl_vb, &c->rl_vc, &c->rl_row_of, &c->rl_sort_tmp, &c->seg_off, &c->seg_of, &c->node_seg,
                    &c->q_seg_off, &c->q_seg_row, &c->q_seg_sorted, &c->grid_cells, &c->grid_frame, &c->fps_segs,
                    &c->fps_slot_of_seg, &c->fps_words, &c->fps_leaf_lo, &c->fps_leaf_hi, &c->fps_leaf_first,
                    &c->fps_leaf_key, &c->fps_D, &c->fps_pos_of, &c->fps_best, &c->fk_x, &c->fk_y, &c->fk_sid,
                    &c->fk_items, &c->fk_partial, &c->fk_dist, &c->vx_pts, &c->vx_seg_off, &c->vx_raw,
                    &c->vx_cluster, &c->vx_keys_a, &c->vx_keys_b, &c->vx_vals_a, &c->vx_vals_b, &c->vx_sort_tmp, &c->vx_words,
                    &c->vx_word_off, &c->vx_members, &c->vx_off, &c->vx_first, &c->vx_seg, &c->vx_chunks, &c->vx_chunk_off,
                    &c->vx_words_sc, &c->vx_x, &c->vx_out, &c->vx_cs, &c->vx_longs, &c->ip_idx, &c->ip_w, &c->ip_den,
                    &c->ip_x, &c->ip_out, &c->ip_wout, &c->ip_dout, &c->ip_keys_a, &c->ip_keys_b, &c->ip_vals_a,
                    &c->ip_vals_b, &c->ip_sort_tmp, &c->ip_cnt, &c->ip_off, &c->kg_q, &c->kg_p, &c->kg_idx, &c->kg_g,
                    &c->kg_gq, &c->kg_gp, &c->kg_terms, &c->kg_keys_a, &c->kg_keys_b, &c->kg_vals_a, &c->kg_vals_b,
                    &c->kg_sort_tmp, &c->kg_cnt, &c->kg_off, &c->kg_x, &c->kg_seg_off, &c->kg_out, &c->kg_chunks,
                    &c->kg_chunk_off, &c->kg_longs, &c->kg_words, &c->kg_cs, &c->lf_pts, &c->lf_idx, &c->lf_eig,
                    &c->lf_frames})
    release(*b);
  for (auto& ev : c->ev) if (ev) cudaEventDestroy(ev);
  for (auto& ev : c->round_ev) cudaEventDestroy(ev);
  for (auto& ev : c->chunk_ev) cudaEventDestroy(ev);
  if (c->copy_stream) cudaStreamDestroy(c->copy_stream);
  if (c->own_stream) cudaStreamDestroy(c->own_stream);
  if (c->mailbox_h) cudaFreeHost(c->mailbox_h);
  delete c;
  return TKNN_OK;
}

int tknn_set_stream(tknn_ctx* c, void* cuda_stream) {
  TK_TRY(check_ctx(c));
  c->stream = cuda_stream ? reinterpret_cast<cudaStream_t>(cuda_stream) : c->own_stream;
  return TKNN_OK;
}

int tknn_set_option(tknn_ctx* c, int key, int64_t value) {
  TK_TRY(check_ctx(c));
  switch (key) {
    case TKNN_OPT_LEAF_SIZE:
      if (value < 2 || value > MAX_LEAF) return fail(c, TKNN_EINVAL, "leaf size %lld outside [2, %d]", (long long)value, MAX_LEAF);
      c->leaf_size = (int)value;
      return TKNN_OK;
    case TKNN_OPT_COUNTERS: c->counters = value ? 1 : 0; return TKNN_OK;
    case TKNN_OPT_LEAF_POLICY:
      if (value != 0 && value != 1) return fail(c, TKNN_EINVAL, "leaf policy must be 0 or 1");
      c->leaf_policy = (int)value;
      return TKNN_OK;
    case TKNN_OPT_SAMPLE_GROUPS:
      if (value < 1 || value > 65536) return fail(c, TKNN_EINVAL, "sample groups outside [1, 65536]");
      c->sample_groups = (int)value;
      return TKNN_OK;
    case TKNN_OPT_BLOCKS_PER_SM:
      if (value < 0 || value > 32) return fail(c, TKNN_EINVAL, "blocks per SM outside [0, 32]");
      c->blocks_per_sm = (int)value;
      return TKNN_OK;
    case TKNN_OPT_SQUARED_DIST: c->squared = value ? 1 : 0; return TKNN_OK;
    case TKNN_OPT_KEEP_SCRATCH: c->keep_scratch = value ? 1 : 0; return TKNN_OK;
    case TKNN_OPT_APPROX_FILTER: c->approx_filter = value ? 1 : 0; return TKNN_OK;
    case TKNN_OPT_TIE_PRUNING:
      if (value < 0 || value > 2) return fail(c, TKNN_EINVAL, "tie pruning must be 0 (auto), 1 (on) or 2 (off)");
      c->tie_pruning = (int)value;
      return TKNN_OK;
    case TKNN_OPT_MORTON_BITS:
      if (value != 0 && (value < 4 || value > 21)) return fail(c, TKNN_EINVAL, "morton bits per axis must be 0 (auto) or in [4, 21]");
      c->morton_bits = (int)value;
      return TKNN_OK;
    case TKNN_OPT_SPECULATIVE_MAX:
      if (value < 0 || value > (int64_t)1 << 30) return fail(c, TKNN_EINVAL, "speculative maximum outside [0, 2^30]");
      c->speculative_max = (int)value;
      return TKNN_OK;
    case TKNN_OPT_SORT_MODE:
      if (value != 0 && value != 1) return fail(c, TKNN_EINVAL, "sort mode must be 0 (packed keys when they fit) or 1 (pairs)");
      c->sort_mode = (int)value;
      return TKNN_OK;
    case TKNN_OPT_SPARSE_TEAM:
      if (value != 0 && value != 4 && value != 8 && value != 16) return fail(c, TKNN_EINVAL, "sparse team must be 0, 4, 8 or 16 lanes");
      c->sparse_team = (int)value;
      return TKNN_OK;
    case TKNN_OPT_CURVE:
      if (value != 0 && value != 1 && !(value >= 101 && value <= 121))
        return fail(c, TKNN_EINVAL, "curve must be 0 (Hilbert), 1 (Morton) or 100 + L (Hilbert on exactly L levels)");
      c->curve = value == 1 ? 0 : 1;  // internal: 1 = Hilbert
      c->curve_levels = value > 100 ? (int)value - 100 : 0;
      return TKNN_OK;
    case TKNN_OPT_FILE_ORDER_CHUNKS:
      if (value < 0 || value > 64) return fail(c, TKNN_EINVAL, "file-order chunks outside [0, 64]");
      c->file_order_chunks = (int)value;
      return TKNN_OK;
    case TKNN_OPT_OUTPUT_CHUNKS:
      if (value < 1 || value > 64) return fail(c, TKNN_EINVAL, "output chunks outside [1, 64]");
      c->output_chunks = (int)value;
      return TKNN_OK;
    case TKNN_OPT_SPARSE_DIVISOR:
      if (value < 0 || value > 1000000) return fail(c, TKNN_EINVAL, "sparse divisor outside [0, 1e6]");
      c->sparse_divisor = (int)value;
      return TKNN_OK;
    case TKNN_OPT_WARP_ROUND_MAX:
      if (value < 0 || value > (int64_t)1 << 30) return fail(c, TKNN_EINVAL, "warp round maximum outside [0, 2^30]");
      c->warp_round_max = (int)value;
      return TKNN_OK;
    case TKNN_OPT_GRID:
      if (value < 0 || value > 2) return fail(c, TKNN_EINVAL, "grid must be 0 (auto), 1 (off) or 2 (whenever the table is valid)");
      c->grid_mode = (int)value;
      return TKNN_OK;
    case TKNN_OPT_GRID_LEVEL:
      if (value < 0 || value > grid::MAX_LEVEL) return fail(c, TKNN_EINVAL, "grid level outside [0 (auto), %d]", grid::MAX_LEVEL);
      c->grid_level = (int)value;
      return TKNN_OK;
    case TKNN_OPT_RADIUS_QUANTILE:
      if (value < 0 || value > 1000) return fail(c, TKNN_EINVAL, "radius quantile outside [0, 1000] per mille");
      c->radius_quantile = (int)value;
      return TKNN_OK;
    case TKNN_OPT_GRID_RADIUS_QUANTILE:
      if (value < 0 || value > 1000) return fail(c, TKNN_EINVAL, "grid radius quantile outside [0, 1000] per mille");
      c->grid_radius_quantile = (int)value;
      return TKNN_OK;
    default: return fail(c, TKNN_EINVAL, "unknown option %d", key);
  }
}

int tknn_build(tknn_ctx* c, const float* xyz, uint64_t n, int dim, int stride_floats) {
  tknn_internal_dist_invalidate(c);
  return build_core(c, xyz, n, dim, stride_floats, false);
}

int tknn_build_segments(tknn_ctx* c, const float* xyz, uint64_t n, int dim, int stride_floats, const uint64_t* seg_offsets,
                        uint64_t n_segments) {
  TK_TRY(check_ctx(c));
  if (!seg_offsets) return fail(c, TKNN_EINVAL, "null segment offsets");
  if (n_segments < 1 || n_segments > (uint64_t)INT32_MAX)
    return fail(c, TKNN_EINVAL, "n_segments = %llu outside [1, 2^31 - 1]", (unsigned long long)n_segments);
  ScopedDevice sd(c->device);
  std::vector<uint64_t> off;
  TK_TRY(read_offsets(c, "tknn_build_segments", "segment", seg_offsets, n_segments, n, "n", &off));
  uint64_t max_segment = 0;
  for (uint64_t s = 0; s < n_segments; ++s) max_segment = std::max(max_segment, off[s + 1] - off[s]);
  if (n_segments == 1) return tknn_build(c, xyz, n, dim, stride_floats);  // one segment: an ordinary build
  tknn_internal_dist_invalidate(c);
  c->n = 0;  // the offsets of the previous build are overwritten: it is gone whatever happens below
  c->n_leaves = 0;
  c->segmented = false;
  TK_TRY(ensure(c, c->seg_off, off.size() * sizeof(uint64_t)));
  TK_CUDA(c, cudaMemcpyAsync(c->seg_off.p, off.data(), off.size() * sizeof(uint64_t), cudaMemcpyHostToDevice, c->stream));
  TK_CUDA(c, cudaStreamSynchronize(c->stream));
  c->seg_off_host = std::move(off);
  return build_core(c, xyz, n, dim, stride_floats, false, c->seg_off.as<uint64_t>(), n_segments, max_segment);
}

}  // extern "C"

// Level of the cell table: floor(log2(n) / 3), i.e. one to eight points per cell on a uniform cloud, at most the key's code
// bits per axis (a level-L cell must be a prefix of the key) and grid::MAX_LEVEL.  TKNN_OPT_GRID_LEVEL forces it.
static int grid_level_for(uint64_t n, int mbits, int forced) {
  int lg = 0;
  while (((uint64_t)2 << lg) <= n) ++lg;  // floor(log2 n)
  return std::max(1, std::min(std::min(forced > 0 ? forced : lg / 3, mbits), grid::MAX_LEVEL));
}

// The cell table of the current build (c->pts sorted, the scene bounds at SC_BOUNDS) and the decision to use it: every cell
// one contiguous run, and (auto) no cell fuller than grid::SELECT_MAX_CELL.
static int build_grid(tknn_ctx* c, uint64_t n, int mbits, int* launches) {
  uint32_t* sc = c->scalars.as<uint32_t>();
  cudaStream_t st = c->stream;
  const int L = grid_level_for(n, mbits, c->grid_level);
  const uint64_t n_cells = 1ull << (3 * L);
  TK_TRY(ensure(c, c->grid_cells, n_cells * sizeof(uint2)));
  TK_TRY(ensure(c, c->grid_frame, grid::frame_words(L) * sizeof(float)));
  TK_CUDA(c, cudaMemsetAsync(c->grid_cells.p, 0xff, n_cells * sizeof(uint2), st));
  TK_CUDA(c, cudaMemsetAsync(sc + SC_GRID, 0, 2 * sizeof(uint32_t), st));
  grid::fill_kernel<<<blocks_for(n, 256), 256, 0, st>>>(c->pts.as<float4>(), n, sc + SC_BOUNDS, L, c->grid_cells.as<uint2>(),
                                                         sc + SC_GRID + 1);
  grid::frame_kernel<<<blocks_for(3 * ((1ull << L) + 1), 256), 256, 0, st>>>(sc + SC_BOUNDS, L, c->grid_frame.as<float>());
  grid::occupancy_kernel<<<(unsigned)std::min<uint64_t>(blocks_for(n_cells, 256), (uint64_t)c->sm_count * 8), 256, 0, st>>>(
      c->grid_cells.as<uint2>(), n_cells, sc + SC_GRID);
  TK_CUDA(c, cudaGetLastError());
  *launches += 3;
  uint32_t h[2] = {0, 0};
  TK_TRY(fetch_words(c, sc + SC_GRID, 2, nullptr, 0, h));
  c->stats.grid_level = L;
  c->stats.grid_max_cell = h[0];
  c->stats.grid_split_cells = h[1];
  c->built_grid_level = L;
  c->grid_on = h[1] == 0 && (c->grid_mode == 2 || h[0] <= grid::SELECT_MAX_CELL);
  c->stats.grid_selected = c->grid_on ? 1 : 0;
  return TKNN_OK;
}

int tknn::host::build_core(tknn_ctx* c, const float* xyz, uint64_t n, int dim, int stride_floats, bool ids_in_w,
                           const uint64_t* seg_offsets, uint64_t n_segments, uint64_t max_segment) {
  TK_TRY(check_ctx(c));
  if (!xyz) return fail(c, TKNN_EINVAL, "null point array");
  if (ids_in_w && (dim != 3 || stride_floats < 4)) return fail(c, TKNN_EINVAL, "ids in w need dim 3 and stride >= 4");
  if (dim != 2 && dim != 3) return fail(c, TKNN_EINVAL, "dim = %d (must be 2 or 3, hostCode.cpp:114-124)", dim);
  if (stride_floats < dim) return fail(c, TKNN_EINVAL, "stride %d < dim %d", stride_floats, dim);
  if (n < 2) return fail(c, TKNN_EINVAL, "need at least 2 points (got %llu)", (unsigned long long)n);
  if (n > rsort::MAX_N) return fail(c, TKNN_EINVAL, "n = %llu exceeds %llu points per device", (unsigned long long)n,
                                    (unsigned long long)rsort::MAX_N);
  ScopedDevice sd(c->device);
  cudaStream_t st = c->stream;
  c->n = 0;
  c->n_leaves = 0;
  c->segmented = false;
  c->grid_on = false;
  const bool seg = seg_offsets != nullptr;
  tknn_stats& S = c->stats;
  std::memset(&S, 0, sizeof(S));
  c->mailbox_launches = 0;
  int launches = 0;

  // ---- stage the input ----
  DevBuf &keys_a = c->b_keys_a, &keys_b = c->b_keys_b, &vals_a = c->b_vals_a, &vals_b = c->b_vals_b,
         &sort_tmp = c->b_sort_tmp, &ballots = c->b_ballots, &leaf_key = c->b_leaf_key, &child_info = c->b_child_info,
         &parent_leaf = c->b_parent_leaf, &parent_node = c->b_parent_node, &arrive = c->b_arrive;
  ScratchScope scratch = build_scratch(c);
  // size-only allocations happen before the timed region (cudaMalloc is a synchronous host call)
  {
    const uint64_t nw0 = (n + 31) / 32;
    TK_TRY(reserve_stage(c, xyz, (size_t)n * stride_floats, c->b_in));
    TK_TRY(ensure(c, keys_a, n * sizeof(uint64_t)));
    TK_TRY(ensure(c, keys_b, n * sizeof(uint64_t)));
    TK_TRY(ensure(c, vals_a, n * sizeof(uint32_t)));
    TK_TRY(ensure(c, vals_b, n * sizeof(uint32_t)));
    TK_TRY(ensure(c, sort_tmp, rsort::temp_words(n) * sizeof(uint32_t)));
    TK_TRY(ensure(c, ballots, nw0 * sizeof(uint32_t)));
    TK_TRY(ensure(c, c->offsets, (nw0 + 1) * sizeof(uint32_t)));
    TK_TRY(ensure(c, c->block_sums, sizeof(uint32_t) * (size_t)(nw0 / lbvh::SCAN_CHUNK + 2)));
    TK_TRY(ensure(c, c->pts, n * sizeof(float4)));
    if (seg) TK_TRY(ensure(c, c->seg_of, n * sizeof(uint32_t)));
  }

  TK_CUDA(c, cudaEventRecord(c->ev[0], st));
  const float* d_xyz = nullptr;
  TK_TRY(stage_in(c, xyz, (size_t)n * stride_floats, c->b_in, &d_xyz));
  if (d_xyz != xyz) S.h2d_bytes = (size_t)n * stride_floats * sizeof(float);
  TK_CUDA(c, cudaEventRecord(c->ev[1], st));

  // ---- scene bounds ----
  uint32_t* sc = c->scalars.as<uint32_t>();
  const uint32_t binit[8] = {0xffffffffu, 0xffffffffu, 0xffffffffu, 0u, 0u, 0u, 0u, 0u};
  TK_CUDA(c, cudaMemcpyAsync(sc + SC_BOUNDS, binit, sizeof(binit), cudaMemcpyHostToDevice, st));
  {
    const unsigned nb = (unsigned)std::min<uint64_t>((uint64_t)c->sm_count * 8, blocks_for(n, lbvh::THREADS));
    lbvh::bounds_kernel<<<nb, lbvh::THREADS, 0, st>>>(d_xyz, n, dim, stride_floats, sc + SC_BOUNDS);
    ++launches;
  }
  TK_CUDA(c, cudaEventRecord(c->ev[2], st));

  // ---- Morton codes ----
  TK_TRY(ensure(c, keys_a, n * sizeof(uint64_t)));
  TK_TRY(ensure(c, keys_b, n * sizeof(uint64_t)));
  TK_TRY(ensure(c, vals_a, n * sizeof(uint32_t)));
  TK_TRY(ensure(c, vals_b, n * sizeof(uint32_t)));
  int mbits = 0, idx_bits = 0, seg_bits = 0;
  if (seg) segment_key_layout(c, n, n_segments, max_segment, &mbits, &idx_bits, &seg_bits);
  else choose_key_layout(c, n, &mbits, &idx_bits);
  const uint64_t curve_n = seg ? std::max<uint64_t>(2, max_segment) : n;  // the curve resolves the largest segment
  lbvh::morton_kernel<<<blocks_for(n, lbvh::THREADS), lbvh::THREADS, 0, st>>>(d_xyz, n, dim, stride_floats, sc + SC_BOUNDS, mbits,
                                                                             c->curve ? hilbert_levels(curve_n, mbits, c->curve_levels) : 0, idx_bits,
                                                                             keys_a.as<uint64_t>(), vals_a.as<uint32_t>());
  ++launches;
  if (seg) {  // the segment id above the code
    lbvh::segment_key_kernel<<<blocks_for(n, lbvh::THREADS), lbvh::THREADS, 0, st>>>(seg_offsets, n_segments, n, 3 * mbits + idx_bits,
                                                                                    keys_a.as<uint64_t>(), c->seg_of.as<uint32_t>());
    ++launches;
  }
  const int sort_passes = (3 * mbits + seg_bits + 7) / 8;
  TK_CUDA(c, cudaEventRecord(c->ev[3], st));

  // ---- onesweep radix sort ----
  TK_TRY(ensure(c, sort_tmp, rsort::temp_words(n) * sizeof(uint32_t)));
  bool sorted_in_b = false;
  if (idx_bits > 0)
    launches += rsort::sort_keys(keys_a.as<uint64_t>(), keys_b.as<uint64_t>(), n, sort_tmp.as<uint32_t>(), c->sm_count, st, idx_bits,
                                 sort_passes, &sorted_in_b);
  else
    launches += rsort::sort_pairs(keys_a.as<uint64_t>(), vals_a.as<uint32_t>(), keys_b.as<uint64_t>(), vals_b.as<uint32_t>(), n,
                                  sort_tmp.as<uint32_t>(), c->sm_count, st, sort_passes, &sorted_in_b);
  const uint64_t* skeys = sorted_in_b ? keys_b.as<uint64_t>() : keys_a.as<uint64_t>();
  const uint32_t* svals = idx_bits > 0 ? nullptr : (sorted_in_b ? vals_b.as<uint32_t>() : vals_a.as<uint32_t>());
  TK_CUDA(c, cudaGetLastError());
  TK_CUDA(c, cudaEventRecord(c->ev[4], st));

  // ---- leaf cut + point gather ----
  const uint64_t nw = (n + 31) / 32;
  TK_TRY(ensure(c, ballots, nw * sizeof(uint32_t)));
  TK_TRY(ensure(c, c->offsets, (nw + 1) * sizeof(uint32_t)));
  const uint64_t force_split = (n <= (uint64_t)c->leaf_size) ? n / 2 : 0;
  lbvh::leaf_flag_kernel<<<blocks_for(nw * 32, lbvh::THREADS), lbvh::THREADS, 0, st>>>(
      skeys, n, c->leaf_size, c->leaf_policy, force_split, ballots.as<uint32_t>());
  launches += 1;
  if (seg) {
    lbvh::segment_cut_kernel<<<blocks_for(n_segments, lbvh::THREADS), lbvh::THREADS, 0, st>>>(seg_offsets, n_segments, n,
                                                                                              ballots.as<uint32_t>());
    launches += 1;
  }
  TK_TRY(popc_scan(c, ballots.as<uint32_t>(), nw, c->offsets.as<uint32_t>(), &launches));
  uint32_t mb[2] = {0, 0};
  TK_TRY(fetch_words(c, sc + SC_TOTAL, 1, sc + SC_BOUNDS + 6, 1, mb));  // the leaf count sizes every later launch
  const uint32_t m = mb[0];
  const uint32_t bad[1] = {mb[1]};
  if (bad[0]) return fail(c, TKNN_EINVAL, "non-finite coordinate in the input points");
  if (m < 2) return fail(c, TKNN_ECUDA, "internal: leaf cut produced %u leaves", m);
  TK_TRY(ensure(c, c->leaf_start, (size_t)(m + 1) * sizeof(uint32_t)));
  TK_TRY(ensure(c, leaf_key, (size_t)m * sizeof(uint64_t)));
  TK_TRY(ensure(c, c->pts, n * sizeof(float4)));
  lbvh::leaf_emit_kernel<<<blocks_for(n, lbvh::THREADS), lbvh::THREADS, 0, st>>>(
      ballots.as<uint32_t>(), c->offsets.as<uint32_t>(), skeys, n, m, c->leaf_start.as<uint32_t>(),
      leaf_key.as<uint64_t>());
  lbvh::gather_points_kernel<<<blocks_for(n, lbvh::THREADS), lbvh::THREADS, 0, st>>>(d_xyz, dim, stride_floats, svals, skeys, idx_bits,
                                                                                   n, ids_in_w ? 1 : 0, c->pts.as<float4>());
  launches += 2;
  TK_CUDA(c, cudaEventRecord(c->ev[5], st));

  // ---- Karras hierarchy ----
  TK_TRY(ensure(c, c->nodes, (size_t)(m - 1) * sizeof(Node)));
  TK_TRY(ensure(c, c->node_min_idx, (size_t)(m - 1) * 2 * sizeof(int)));
  TK_TRY(ensure(c, child_info, (size_t)(m - 1) * sizeof(int4)));
  TK_TRY(ensure(c, parent_leaf, (size_t)m * sizeof(int32_t)));
  TK_TRY(ensure(c, parent_node, (size_t)m * sizeof(int32_t)));
  TK_TRY(ensure(c, arrive, (size_t)m * sizeof(uint32_t)));
  TK_CUDA(c, cudaMemsetAsync(arrive.p, 0, (size_t)m * sizeof(uint32_t), st));
  TK_CUDA(c, cudaMemsetAsync(sc + SC_DUPLEAF, 0, sizeof(uint32_t), st));
  lbvh::karras_kernel<<<blocks_for(m - 1, lbvh::THREADS), lbvh::THREADS, 0, st>>>(
      leaf_key.as<uint64_t>(), c->leaf_start.as<uint32_t>(), m, child_info.as<int4>(), parent_leaf.as<int32_t>(),
      parent_node.as<int32_t>());
  ++launches;
  if (seg) {
    TK_TRY(ensure(c, c->node_seg, (size_t)(m - 1) * sizeof(int4)));
    lbvh::node_segments_kernel<<<blocks_for(m - 1, lbvh::THREADS), lbvh::THREADS, 0, st>>>(
        leaf_key.as<uint64_t>(), c->leaf_start.as<uint32_t>(), m, c->seg_of.as<uint32_t>(), c->node_seg.as<int4>());
    ++launches;
  }
  TK_CUDA(c, cudaEventRecord(c->ev[6], st));

  // ---- bottom-up refit ----
  lbvh::refit_kernel<<<blocks_for(m, lbvh::THREADS), lbvh::THREADS, 0, st>>>(
      c->pts.as<float4>(), c->leaf_start.as<uint32_t>(), m, child_info.as<int4>(), parent_leaf.as<int32_t>(),
      parent_node.as<int32_t>(), arrive.as<uint32_t>(), c->nodes.as<Node>(), c->node_min_idx.as<int>(), sc + SC_DUPLEAF,
      (uint32_t)std::max(2, std::min(8, c->leaf_size)), reinterpret_cast<float*>(sc + SC_SCENE));
  ++launches;
  TK_CUDA(c, cudaGetLastError());
  TK_CUDA(c, cudaEventRecord(c->ev[7], st));
  uint32_t tail[7] = {0, 0, 0, 0, 0, 0, 0};
  TK_TRY(fetch_words(c, sc + SC_SCENE, 6, sc + SC_DUPLEAF, 1, tail));
  std::memcpy(c->scene_box, tail, 6 * sizeof(float));
  const uint32_t dupleaf = tail[6];

  // ---- cell grid: plain builds without coincident-point leaves (those take the tie-pruning LBVH kernel) ----
  TK_CUDA(c, cudaEventRecord(c->ev[8], st));
  if (!seg && dupleaf == 0 && c->grid_mode != 1) TK_TRY(build_grid(c, n, mbits, &launches));
  TK_CUDA(c, cudaEventRecord(c->ev[9], st));

  TK_CUDA(c, cudaEventElapsedTime(&S.h2d_ms, c->ev[0], c->ev[1]));
  TK_CUDA(c, cudaEventElapsedTime(&S.bounds_ms, c->ev[1], c->ev[2]));
  TK_CUDA(c, cudaEventElapsedTime(&S.morton_ms, c->ev[2], c->ev[3]));
  TK_CUDA(c, cudaEventElapsedTime(&S.sort_ms, c->ev[3], c->ev[4]));
  TK_CUDA(c, cudaEventElapsedTime(&S.leaves_ms, c->ev[4], c->ev[5]));
  TK_CUDA(c, cudaEventElapsedTime(&S.hierarchy_ms, c->ev[5], c->ev[6]));
  TK_CUDA(c, cudaEventElapsedTime(&S.refit_ms, c->ev[6], c->ev[7]));
  TK_CUDA(c, cudaEventElapsedTime(&S.grid_ms, c->ev[8], c->ev[9]));
  TK_CUDA(c, cudaEventElapsedTime(&S.build_ms, c->ev[1], c->ev[7]));
  S.build_ms += S.grid_ms;
  S.n_points = n;
  S.n_leaves = m;
  S.n_nodes = m - 1;
  c->built_morton_bits = mbits;
  c->built_idx_bits = idx_bits;
  c->built_curve = c->curve ? hilbert_levels(curve_n, mbits, c->curve_levels) : 0;
  c->has_dup_leaves = dupleaf != 0;
  S.build_launches = (uint32_t)(launches + c->mailbox_launches);
  c->n = n;
  c->n_leaves = m;
  c->ids_in_w = ids_in_w;
  c->segmented = seg;
  c->n_segments = seg ? n_segments : 1;
  return TKNN_OK;
}

extern "C" {

int tknn_search(tknn_ctx* c, int k, float start_radius, int32_t* idx_out, float* dist_out) {
  TK_TRY(check_ctx(c));
  ScopedDevice sd(c->device);
  return search_range(c, k, start_radius, 0, c->n, 0, nullptr, idx_out, dist_out, c->n);
}

int tknn_key_layout(uint64_t n, int morton_bits, int sort_mode, int* code_bits_per_axis, int* index_bits, int* sort_passes) {
  if (n < 2 || n > rsort::MAX_N || morton_bits < 0 || morton_bits > 21 || (morton_bits > 0 && morton_bits < 4) ||
      (sort_mode != 0 && sort_mode != 1) || !code_bits_per_axis || !index_bits || !sort_passes)
    return TKNN_EINVAL;
  key_layout(n, morton_bits, sort_mode, code_bits_per_axis, index_bits);
  *sort_passes = (3 * *code_bits_per_axis + 7) / 8;
  return TKNN_OK;
}

uint64_t tknn_shard_capacity(uint64_t n, int n_shards) {
  if (n_shards < 1) return 0;
  const uint64_t groups = (n + 31) / 32;
  return ((groups + n_shards - 1) / n_shards + 1) * 32;
}

int tknn_search_shard(tknn_ctx* c, int k, float start_radius, int shard, int n_shards, int32_t* qid_out, int32_t* idx_out,
                      float* dist_out, uint64_t* n_out) {
  TK_TRY(check_ctx(c));
  if (n_shards < 1 || shard < 0 || shard >= n_shards) return fail(c, TKNN_EINVAL, "shard %d of %d", shard, n_shards);
  if (!n_out) return fail(c, TKNN_EINVAL, "null n_out");
  TK_TRY(refuse_segmented(c, "tknn_search_shard"));
  ScopedDevice sd(c->device);
  const uint64_t groups = (c->n + 31) / 32;
  const uint64_t g0 = groups * (uint64_t)shard / (uint64_t)n_shards, g1 = groups * (uint64_t)(shard + 1) / (uint64_t)n_shards;
  const uint64_t q0 = g0 * 32, q1 = std::min<uint64_t>(c->n, g1 * 32);
  const uint64_t nq = q1 > q0 ? q1 - q0 : 0;
  *n_out = nq;
  if (nq == 0) {
    if (c->n == 0) return fail(c, TKNN_ESTATE, "tknn_search_shard before tknn_build");
    reset_search_stats(c);
    return TKNN_OK;
  }
  return search_range(c, k, start_radius, q0, nq, 1, qid_out, idx_out, dist_out, nq);
}

int tknn_estimate_start_radius(tknn_ctx* c, int k, float* radius_out) {
  TK_TRY(check_ctx(c));
  if (!radius_out) return fail(c, TKNN_EINVAL, "null radius_out");
  if (c->n == 0) return fail(c, TKNN_ESTATE, "tknn_estimate_start_radius before tknn_build");
  if (k < 1 || k > TKNN_MAX_K || (uint64_t)k > c->n - 1) return fail(c, TKNN_EINVAL, "k = %d invalid for n = %llu", k,
                                                                     (unsigned long long)c->n);
  ScopedDevice sd(c->device);
  int launches = 0;
  TK_TRY(estimate_radius_device(c, c->pts.as<float4>(), 0, c->n, nullptr, 1, c->seg_of.as<uint32_t>(), k, c->radius_quantile,
                                &launches));
  uint32_t rb = 0;
  TK_TRY(fetch_words(c, c->scalars.as<uint32_t>() + SC_QUANTILE, 1, nullptr, 0, &rb));
  std::memcpy(radius_out, &rb, sizeof(float));
  return TKNN_OK;
}

}  // extern "C"

namespace {
// Query offsets of the _segments calls (host or device): n_segments + 1 entries that start at 0, never decrease and end at
// nq, with n_segments the segment count of the last build.  Device offsets cost one small read-back.
int check_query_offsets(tknn_ctx* c, const char* what, const uint64_t* q_seg_offsets, uint64_t n_segments, uint64_t nq) {
  if (!q_seg_offsets) return fail(c, TKNN_EINVAL, "%s: null query segment offsets", what);
  if (n_segments != c->n_segments)
    return fail(c, TKNN_EINVAL, "%s: n_segments = %llu, the last build has %llu", what, (unsigned long long)n_segments,
                (unsigned long long)c->n_segments);
  std::vector<uint64_t> off;
  return read_offsets(c, what, "query segment", q_seg_offsets, n_segments, nq, "nq", &off);
}

// The query staging of tknn_query and tknn_radius_query: host inputs are copied to the device, the queries are sorted on
// the DATA's space-filling curve so that groups of 32 are spatially coherent, and gathered into c->q_pts (x, y, z, query
// row bits); self ids and radius caps follow into that order.  Sets SC_ERROR / SC_QBAD (a non-finite query coordinate).
// q_seg_offsets (validated, host or device; segmented builds only): the query segment id goes above the curve code as in
// the build, so each segment's queries stay contiguous in the sorted order, and *seg_sorted_out receives the segment of
// every sorted position.
int stage_queries(tknn_ctx* c, const float* queries, uint64_t nq, int dim, int stride_floats, const int32_t* self_ids,
                  const float* init_radius2, const int32_t** sid_sorted_out, const float** r2_sorted_out, int* launches,
                  const uint64_t* q_seg_offsets = nullptr, uint64_t n_segments = 0, const uint32_t** seg_sorted_out = nullptr) {
  cudaStream_t st = c->stream;
  uint32_t* sc = c->scalars.as<uint32_t>();
  DevBuf &keys_a = c->q_keys_a, &keys_b = c->q_keys_b, &vals_a = c->q_vals_a, &vals_b = c->q_vals_b,
         &sort_tmp = c->q_sort_tmp, &qpts = c->q_pts, &sid_sorted = c->q_sid_sorted, &r2_sorted = c->q_r2_sorted;
  *sid_sorted_out = nullptr;
  *r2_sorted_out = nullptr;
  if (seg_sorted_out) *seg_sorted_out = nullptr;
  const float *d_q = nullptr, *d_rad = nullptr;
  const int32_t* d_sid = nullptr;
  TK_TRY(stage_in(c, queries, (size_t)nq * stride_floats, c->q_stage, &d_q));
  TK_TRY(stage_in(c, self_ids, nq, c->q_sid_stage, &d_sid));
  TK_TRY(stage_in(c, init_radius2, nq, c->q_rad_stage, &d_rad));
  const bool seg = q_seg_offsets != nullptr;
  const uint64_t* d_qoff = nullptr;
  if (seg) {
    TK_TRY(ensure(c, c->q_seg_row, nq * sizeof(uint32_t)));
    TK_TRY(ensure(c, c->q_seg_sorted, nq * sizeof(uint32_t)));
    TK_TRY(stage_in(c, q_seg_offsets, n_segments + 1, c->q_seg_off, &d_qoff));
  }
  // Morton-sort the queries on the DATA's grid so that groups of 32 are spatially coherent
  TK_TRY(ensure(c, keys_a, nq * sizeof(uint64_t)));
  TK_TRY(ensure(c, keys_b, nq * sizeof(uint64_t)));
  TK_TRY(ensure(c, vals_a, nq * sizeof(uint32_t)));
  TK_TRY(ensure(c, vals_b, nq * sizeof(uint32_t)));
  TK_TRY(ensure(c, sort_tmp, rsort::temp_words(nq) * sizeof(uint32_t)));
  TK_TRY(ensure(c, qpts, nq * sizeof(float4)));
  TK_CUDA(c, cudaMemsetAsync(sc + SC_ERROR, 0, 2 * sizeof(uint32_t), st));
  const int qbits = c->built_morton_bits;
  lbvh::morton_kernel<<<blocks_for(nq, lbvh::THREADS), lbvh::THREADS, 0, st>>>(d_q, nq, dim, stride_floats, sc + SC_BOUNDS, qbits,
                                                                              c->built_curve, 0, keys_a.as<uint64_t>(), vals_a.as<uint32_t>());
  ++*launches;
  int seg_bits = 0;
  if (seg) {  // the segment id above the code (3 * qbits + seg_bits <= 64: the build's key layout fits it too)
    while (((uint64_t)1 << seg_bits) < n_segments) ++seg_bits;
    lbvh::segment_key_kernel<<<blocks_for(nq, lbvh::THREADS), lbvh::THREADS, 0, st>>>(d_qoff, n_segments, nq, 3 * qbits,
                                                                                     keys_a.as<uint64_t>(), c->q_seg_row.as<uint32_t>());
    ++*launches;
  }
  bool q_in_b = false;
  *launches += rsort::sort_pairs(keys_a.as<uint64_t>(), vals_a.as<uint32_t>(), keys_b.as<uint64_t>(), vals_b.as<uint32_t>(), nq,
                                sort_tmp.as<uint32_t>(), c->sm_count, st, (3 * qbits + seg_bits + 7) / 8, &q_in_b);
  const uint32_t* qorder = q_in_b ? vals_b.as<uint32_t>() : vals_a.as<uint32_t>();
  lbvh::gather_points_kernel<<<blocks_for(nq, lbvh::THREADS), lbvh::THREADS, 0, st>>>(d_q, dim, stride_floats,
                                                                                    qorder, nullptr, 0, nq, 0, qpts.as<float4>(), sc + SC_QBAD);
  TK_CUDA(c, cudaGetLastError());
  ++*launches;
  if (d_sid) {
    TK_TRY(ensure(c, sid_sorted, nq * sizeof(int32_t)));
    brute::gather_i32_kernel<<<blocks_for(nq, 256), 256, 0, st>>>(d_sid, qorder, nq, sid_sorted.as<int32_t>());
    *sid_sorted_out = sid_sorted.as<int32_t>();
    ++*launches;
  }
  if (d_rad) {
    TK_TRY(ensure(c, r2_sorted, nq * sizeof(float)));
    brute::gather_r2_kernel<<<blocks_for(nq, 256), 256, 0, st>>>(d_rad, qorder, nq, r2_sorted.as<float>());
    *r2_sorted_out = r2_sorted.as<float>();
    ++*launches;
  }
  if (seg) {  // segment ids are < 2^31: the i32 gather moves them unchanged
    brute::gather_i32_kernel<<<blocks_for(nq, 256), 256, 0, st>>>(c->q_seg_row.as<int32_t>(), qorder, nq,
                                                                  c->q_seg_sorted.as<int32_t>());
    *seg_sorted_out = c->q_seg_sorted.as<uint32_t>();
    ++*launches;
  }
  return TKNN_OK;
}


// tknn_query and tknn_query_segments after their state checks.  segments: the call carries query segment offsets, which
// are validated here; on a segmented build they restrict query segment s to data segment s, on a plain build (one
// segment) the call is tknn_query.
int query_core(tknn_ctx* c, const char* what, const float* queries, uint64_t nq, int dim, int stride_floats,
               bool segments, const uint64_t* q_seg_offsets, uint64_t n_segments, const int32_t* self_ids,
               const float* init_radius2, int k, float start_radius, int32_t* idx_out, float* dist_out) {
  if (!queries && nq) return fail(c, TKNN_EINVAL, "null query array");
  if (dim != 2 && dim != 3) return fail(c, TKNN_EINVAL, "dim = %d (must be 2 or 3)", dim);
  if (stride_floats < dim) return fail(c, TKNN_EINVAL, "stride %d < dim %d", stride_floats, dim);
  if (k < 1 || k > TKNN_MAX_K) return fail(c, TKNN_EINVAL, "k = %d outside [1, %d]", k, TKNN_MAX_K);
  if ((uint64_t)k > c->n) return fail(c, TKNN_EINVAL, "k = %d > n = %llu", k, (unsigned long long)c->n);
  if (nq > rsort::MAX_N) return fail(c, TKNN_EINVAL, "too many queries");
  if (nq && (!idx_out || !dist_out)) return fail(c, TKNN_EINVAL, "null output array");
  if (std::isnan(start_radius)) return fail(c, TKNN_EINVAL, "start_radius is NaN");
  ScopedDevice sd(c->device);
  if (segments) TK_TRY(check_query_offsets(c, what, q_seg_offsets, n_segments, nq));
  if (!c->segmented) q_seg_offsets = nullptr;
  reset_search_stats(c);
  c->stats.n_queries = nq;
  c->stats.k = k;
  if (nq == 0) return TKNN_OK;
  cudaStream_t st = c->stream;
  uint32_t* sc = c->scalars.as<uint32_t>();

  // scratch lives in the context (grow-only): a call allocates nothing once the buffers have reached their size
  ScratchScope scratch = query_scratch(c);
  TK_CUDA(c, cudaEventRecord(c->ev[0], st));
  int launches = 0;
  const int32_t* d_sid_sorted = nullptr;
  const float* d_r2_sorted = nullptr;
  const uint32_t* d_seg_sorted = nullptr;
  TK_TRY(stage_queries(c, queries, nq, dim, stride_floats, self_ids, init_radius2, &d_sid_sorted, &d_r2_sorted, &launches,
                       q_seg_offsets, n_segments, &d_seg_sorted));

  int32_t* d_idx = nullptr;
  float* d_dist = nullptr;
  const size_t out_elems = (size_t)nq * k;
  TK_TRY(out_view(c, idx_out, out_elems, c->stage_idx, &d_idx));
  TK_TRY(out_view(c, dist_out, out_elems, c->stage_dist, &d_dist));

  TK_CUDA(c, cudaMemsetAsync(sc + SC_COUNTERS, 0, N_COUNTERS * sizeof(unsigned long long), st));
  float r0 = start_radius;
  // a query set can hold fewer than k reachable neighbours only through self exclusion / radius caps
  const bool may_underfill = (uint64_t)k > c->n - (self_ids ? 1 : 0);
  bool estimated = false;
  if (!(r0 > 0.0f)) {
    if (init_radius2 || may_underfill) r0 = INFINITY;
    else { TK_TRY(estimate_radius_device(c, c->q_pts.as<float4>(), 0, nq, d_sid_sorted, 0, d_seg_sorted, k, c->radius_quantile, &launches)); estimated = true; }
  }
  TK_CUDA(c, cudaEventRecord(c->ev[1], st));
  c->stats.start_radius = r0;
  Job job;
  if (estimated) {
    job.r_dev = reinterpret_cast<const float*>(sc + SC_QUANTILE);
    job.r_host = &c->stats.start_radius;
  }
  job.queries = c->q_pts.as<float4>();
  job.self_ids = d_sid_sorted;
  job.query_r2 = d_r2_sorted;
  job.seg_of = d_seg_sorted;
  job.n_queries = nq;
  job.q_begin = 0;
  job.self_is_row = 0;
  job.row_mode = 0;
  job.k = k;
  job.start_radius = r0;
  job.squared = c->squared;
  job.idx_out = d_idx;
  job.dist_out = d_dist;
  TK_TRY(run_rounds(c, job, &launches));
  TK_CUDA(c, cudaEventRecord(c->ev[2], st));
  TK_TRY(copy_back(c, idx_out, d_idx, out_elems, &c->stats.d2h_bytes));
  TK_TRY(copy_back(c, dist_out, d_dist, out_elems, &c->stats.d2h_bytes));
  TK_CUDA(c, cudaEventRecord(c->ev[3], st));
  TK_CUDA(c, cudaStreamSynchronize(st));
  TK_CUDA(c, cudaEventElapsedTime(&c->stats.search_ms, c->ev[0], c->ev[2]));
  TK_CUDA(c, cudaEventElapsedTime(&c->stats.d2h_ms, c->ev[2], c->ev[3]));
  c->stats.kernel_launches = (uint32_t)(launches + c->mailbox_launches + (c->mailbox_h ? 1 : 0));  // + the error-flag fetch below
  TK_TRY(finish_round_stats(c));
  TK_TRY(collect_counters(c));
  TK_TRY(read_error_flag(c));
  return TKNN_OK;
}

}  // namespace

extern "C" {

int tknn_query(tknn_ctx* c, const float* queries, uint64_t nq, int dim, int stride_floats, const int32_t* self_ids,
               const float* init_radius2, int k, float start_radius, int32_t* idx_out, float* dist_out) {
  TK_TRY(check_ctx(c));
  if (c->n == 0) return fail(c, TKNN_ESTATE, "tknn_query before tknn_build");
  TK_TRY(refuse_segmented(c, "tknn_query"));
  return query_core(c, "tknn_query", queries, nq, dim, stride_floats, false, nullptr, 0, self_ids, init_radius2, k,
                    start_radius, idx_out, dist_out);
}

int tknn_query_segments(tknn_ctx* c, const float* queries, uint64_t nq, int dim, int stride_floats,
                        const uint64_t* q_seg_offsets, uint64_t n_segments, const int32_t* self_ids,
                        const float* init_radius2, int k, float start_radius, int32_t* idx_out, float* dist_out) {
  TK_TRY(check_ctx(c));
  if (c->n == 0) return fail(c, TKNN_ESTATE, "tknn_query_segments before tknn_build");
  if (c->ids_in_w) return fail(c, TKNN_ESTATE, "this BVH carries caller-chosen point ids (point-partitioned build)");
  return query_core(c, "tknn_query_segments", queries, nq, dim, stride_floats, true, q_seg_offsets, n_segments, self_ids,
                    init_radius2, k, start_radius, idx_out, dist_out);
}

int tknn_range_count(tknn_ctx* c, float radius, uint32_t* count_out) {
  TK_TRY(check_ctx(c));
  if (c->n == 0) return fail(c, TKNN_ESTATE, "tknn_range_count before tknn_build");
  if (!count_out) return fail(c, TKNN_EINVAL, "null output array");
  if (!(radius >= 0.0f)) return fail(c, TKNN_EINVAL, "radius must be >= 0");
  ScopedDevice sd(c->device);
  reset_search_stats(c);
  c->stats.n_queries = c->n;
  uint32_t* sc = c->scalars.as<uint32_t>();
  uint32_t* d_out = nullptr;
  TK_TRY(out_view(c, count_out, c->n, c->stage_idx, &d_out));
  trav::Params P;
  std::memset(&P, 0, sizeof(P));
  P.nodes = c->nodes.as<Node>();
  P.node_min_idx = c->node_min_idx.as<int2>();
  P.pts = c->pts.as<float4>();
  P.queries = c->pts.as<float4>();
  P.n_active = c->n;
  P.n_groups = (uint32_t)((c->n + 31) / 32);
  P.r2 = radius * radius;
  P.k = 0;
  P.self_is_row = 1;
  P.final_round = 1;
  P.error = sc + SC_ERROR;
  P.count_out = d_out;
  P.group_counter = sc + SC_GROUP_COUNTER;
  P.counters = c->counters ? reinterpret_cast<unsigned long long*>(sc + SC_COUNTERS) : nullptr;
  set_segments(c, P, c->seg_of.as<uint32_t>());
  TK_CUDA(c, cudaMemsetAsync(sc + SC_ERROR, 0, 2 * sizeof(uint32_t), c->stream));
  TK_CUDA(c, cudaMemsetAsync(sc + SC_COUNTERS, 0, N_COUNTERS * sizeof(unsigned long long), c->stream));
  TK_CUDA(c, cudaMemsetAsync(sc + SC_GROUP_COUNTER, 0, sizeof(uint32_t), c->stream));
  TK_CUDA(c, cudaEventRecord(c->ev[0], c->stream));
  TK_TRY(launch_traverse<trav::MODE_RANGE_COUNT>(c, P));
  TK_CUDA(c, cudaEventRecord(c->ev[2], c->stream));
  TK_TRY(copy_back(c, count_out, d_out, c->n, &c->stats.d2h_bytes));
  TK_CUDA(c, cudaStreamSynchronize(c->stream));
  TK_CUDA(c, cudaEventElapsedTime(&c->stats.search_ms, c->ev[0], c->ev[2]));
  c->stats.rounds = 1;
  c->stats.kernel_launches = 1;
  c->stats.start_radius = c->stats.final_radius = radius;
  TK_TRY(collect_counters(c));
  TK_TRY(read_error_flag(c));
  return TKNN_OK;
}

// Four phases, all on the device (dbscan.cuh): core test + queue split, link, labelling, border.  The only host read-back is
// the queue sizes and C at the end: the link and border passes take their query counts from the device.
int tknn_dbscan(tknn_ctx* c, float eps, int min_pts, int32_t* label_out, uint8_t* core_out, uint64_t* n_clusters_out) {
  TK_TRY(check_ctx(c));
  if (c->n == 0) return fail(c, TKNN_ESTATE, "tknn_dbscan before tknn_build");
  if (c->ids_in_w) return fail(c, TKNN_ESTATE, "this BVH carries caller-chosen point ids (point-partitioned build)");
  TK_TRY(refuse_segmented(c, "tknn_dbscan"));
  if (!(eps >= 0.0f)) return fail(c, TKNN_EINVAL, "eps must be >= 0");
  if (min_pts < 1) return fail(c, TKNN_EINVAL, "min_pts = %d must be >= 1", min_pts);
  if (!label_out) return fail(c, TKNN_EINVAL, "null label array");
  if (c->n > (uint64_t)INT32_MAX) return fail(c, TKNN_EINVAL, "tknn_dbscan supports at most 2^31 - 1 points");
  ScopedDevice sd(c->device);
  reset_search_stats(c);
  const uint64_t n = c->n;
  const uint32_t n_groups = (uint32_t)((n + 31) / 32);
  cudaStream_t st = c->stream;
  uint32_t* sc = c->scalars.as<uint32_t>();
  TK_TRY(ensure(c, c->unresolved, sizeof(uint32_t) * (size_t)(n_groups + 1)));
  TK_TRY(ensure(c, c->offsets, sizeof(uint32_t) * (size_t)(n_groups + 1)));
  TK_TRY(ensure(c, c->queue_a, sizeof(uint32_t) * n));
  TK_TRY(ensure(c, c->queue_b, sizeof(uint32_t) * n));
  TK_TRY(ensure(c, c->db_parent, sizeof(int) * n));
  TK_TRY(ensure(c, c->db_min_idx, sizeof(int) * n));
  TK_TRY(ensure(c, c->db_pos_label, sizeof(int32_t) * n));
  TK_TRY(ensure(c, c->db_bits, sizeof(uint32_t) * (size_t)n_groups));
  int32_t* d_label = nullptr;
  uint8_t* d_core = nullptr;
  TK_TRY(out_view(c, label_out, n, c->stage_idx, &d_label));
  TK_TRY(out_view(c, core_out, n, c->db_core_stage, &d_core));
  uint32_t* core_words = c->unresolved.as<uint32_t>();
  uint32_t* core_q = c->queue_a.as<uint32_t>();
  uint32_t* other_q = c->queue_b.as<uint32_t>();
  int* parent = c->db_parent.as<int>();
  int* min_idx = c->db_min_idx.as<int>();
  int32_t* pos_label = c->db_pos_label.as<int32_t>();
  uint32_t* cluster_bits = c->db_bits.as<uint32_t>();
  int launches = 0;
  TK_TRY(ensure_round_events(c, 16));
  cudaEvent_t* ev = c->round_ev.data();  // phase r: [4r] start, [4r + 1] end, [4r + 2 / + 3] its traversal kernel

  trav::Params P;
  std::memset(&P, 0, sizeof(P));
  P.nodes = c->nodes.as<Node>();
  P.node_min_idx = c->node_min_idx.as<int2>();
  P.pts = c->pts.as<float4>();
  P.queries = c->pts.as<float4>();
  P.r2 = eps * eps;
  P.k = min_pts;
  P.final_round = 1;
  P.error = sc + SC_ERROR;
  P.group_counter = sc + SC_GROUP_COUNTER;
  P.counters = c->counters ? reinterpret_cast<unsigned long long*>(sc + SC_COUNTERS) : nullptr;
  P.core_words = core_words;
  P.n_core_words = n_groups;
  const unsigned blocks = blocks_for(n, dbscan::THREADS);
  TK_CUDA(c, cudaMemsetAsync(sc + SC_ERROR, 0, 2 * sizeof(uint32_t), st));
  TK_CUDA(c, cudaMemsetAsync(sc + SC_COUNTERS, 0, N_COUNTERS * sizeof(unsigned long long), st));
  TK_CUDA(c, cudaEventRecord(c->ev[0], st));

  // 1. core test over every position, then the core / non-core queues
  TK_CUDA(c, cudaEventRecord(ev[0], st));
  TK_CUDA(c, cudaMemsetAsync(sc + SC_GROUP_COUNTER, 0, sizeof(uint32_t), st));
  P.n_active = n;
  P.n_groups = n_groups;
  P.unresolved = core_words;
  TK_CUDA(c, cudaEventRecord(ev[2], st));
  TK_TRY(launch_traverse<trav::MODE_DBSCAN_CORE>(c, P));
  TK_CUDA(c, cudaEventRecord(ev[3], st));
  TK_TRY(popc_scan(c, core_words, n_groups, c->offsets.as<uint32_t>(), &launches));
  dbscan::split_queues_kernel<<<blocks, dbscan::THREADS, 0, st>>>(core_words, c->offsets.as<uint32_t>(), n, core_q, other_q, parent,
                                                                  min_idx, sc + SC_DBSCAN);
  TK_CUDA(c, cudaGetLastError());
  TK_CUDA(c, cudaEventRecord(ev[1], st));
  P.unresolved = nullptr;

  // 2. link: the core queue, its length read on the device
  TK_CUDA(c, cudaEventRecord(ev[4], st));
  TK_CUDA(c, cudaMemsetAsync(sc + SC_GROUP_COUNTER, 0, sizeof(uint32_t), st));
  P.queue = core_q;
  P.n_active_dev = sc + SC_DBSCAN;
  P.uf_parent = parent;
  TK_CUDA(c, cudaEventRecord(ev[6], st));
  TK_TRY(launch_traverse<trav::MODE_DBSCAN_LINK>(c, P));
  TK_CUDA(c, cudaEventRecord(ev[7], st));
  TK_CUDA(c, cudaEventRecord(ev[5], st));

  // 3. labelling: roots, the smallest original index per cluster, dense ids from a popc scan of one bit per cluster
  TK_CUDA(c, cudaEventRecord(ev[8], st));
  TK_CUDA(c, cudaEventRecord(ev[10], st));  // no traversal kernel in this phase
  TK_CUDA(c, cudaEventRecord(ev[11], st));
  TK_CUDA(c, cudaMemsetAsync(cluster_bits, 0, sizeof(uint32_t) * (size_t)n_groups, st));
  dbscan::flatten_kernel<<<blocks, dbscan::THREADS, 0, st>>>(core_words, P.pts, n, parent, min_idx);
  dbscan::mark_kernel<<<blocks, dbscan::THREADS, 0, st>>>(core_words, n, parent, min_idx, cluster_bits);
  TK_CUDA(c, cudaGetLastError());
  TK_TRY(popc_scan(c, cluster_bits, n_groups, c->offsets.as<uint32_t>(), &launches));  // C -> sc[SC_TOTAL]
  dbscan::label_core_kernel<<<blocks, dbscan::THREADS, 0, st>>>(core_words, P.pts, n, parent, min_idx, cluster_bits,
                                                                c->offsets.as<uint32_t>(), pos_label, d_label, d_core);
  TK_CUDA(c, cudaGetLastError());
  TK_CUDA(c, cudaEventRecord(ev[9], st));

  // 4. border: the non-core queue
  TK_CUDA(c, cudaEventRecord(ev[12], st));
  TK_CUDA(c, cudaMemsetAsync(sc + SC_GROUP_COUNTER, 0, sizeof(uint32_t), st));
  P.queue = other_q;
  P.n_active_dev = sc + SC_DBSCAN + 1;
  P.uf_parent = nullptr;
  P.pos_label = pos_label;
  P.label_out = d_label;
  P.core_out = d_core;
  TK_CUDA(c, cudaEventRecord(ev[14], st));
  TK_TRY(launch_traverse<trav::MODE_DBSCAN_BORDER>(c, P));
  TK_CUDA(c, cudaEventRecord(ev[15], st));
  TK_CUDA(c, cudaEventRecord(ev[13], st));
  TK_CUDA(c, cudaEventRecord(c->ev[2], st));
  launches += 3 /* traversals */ + 4 /* split, flatten, mark, label */;

  TK_TRY(copy_back(c, label_out, d_label, n, &c->stats.d2h_bytes));
  TK_TRY(copy_back(c, core_out, d_core, n, &c->stats.d2h_bytes));
  uint32_t rb[3] = {0, 0, 0};  // core points, other points, clusters
  TK_TRY(fetch_words(c, sc + SC_DBSCAN, 2, sc + SC_TOTAL, 1, rb));  // synchronises the stream
  TK_CUDA(c, cudaEventElapsedTime(&c->stats.search_ms, c->ev[0], c->ev[2]));
  c->stats.n_queries = n;
  c->stats.k = min_pts;
  c->stats.rounds = 4;
  c->stats.start_radius = c->stats.final_radius = eps;
  c->stats.round_queries[0] = n;
  c->stats.round_queries[1] = c->stats.round_queries[2] = rb[0];
  c->stats.round_queries[3] = rb[1];
  c->stats.kernel_launches = (uint32_t)(launches + c->mailbox_launches + (c->mailbox_h ? 1 : 0));  // + the error-flag fetch
  TK_TRY(finish_round_stats(c));
  if (n_clusters_out) *n_clusters_out = rb[2];
  TK_TRY(collect_counters(c));
  TK_TRY(read_error_flag(c));
  return TKNN_OK;
}

// Farthest point sampling (fps.cuh).  The host reads the offsets, counts and starts (host copies, or one read-back of each
// for device arrays), splits the segments into the block tier (at most fps::BLOCK_CAP points) and the grid tier, and runs
// both on the stream, one after the other.
int tknn_fps(tknn_ctx* c, const uint64_t* sample_offsets, uint64_t n_segments, const int32_t* start_ids, int32_t* idx_out,
             float* dist_out) {
  TK_TRY(check_ctx(c));
  if (c->n == 0) return fail(c, TKNN_ESTATE, "tknn_fps before tknn_build");
  if (c->ids_in_w) return fail(c, TKNN_ESTATE, "this BVH carries caller-chosen point ids (point-partitioned build)");
  if (!sample_offsets) return fail(c, TKNN_EINVAL, "tknn_fps: null sample offsets");
  if (!idx_out) return fail(c, TKNN_EINVAL, "tknn_fps: null idx_out");
  if (c->n > (uint64_t)INT32_MAX) return fail(c, TKNN_EINVAL, "tknn_fps supports at most 2^31 - 1 points");
  if (n_segments != c->n_segments)
    return fail(c, TKNN_EINVAL, "tknn_fps: n_segments = %llu, the last build has %llu", (unsigned long long)n_segments,
                (unsigned long long)c->n_segments);
  ScopedDevice sd(c->device);
  cudaStream_t st = c->stream;
  const uint64_t S = n_segments;
  const std::vector<uint64_t> off = c->segmented ? c->seg_off_host : std::vector<uint64_t>{0, c->n};
  std::vector<uint64_t> soff;  // the sample total is free
  TK_TRY(read_offsets(c, "tknn_fps", "sample", sample_offsets, S, 0, nullptr, &soff));
  std::vector<int32_t> starts(S);
  if (start_ids) TK_TRY(read_to_host(c, start_ids, S, starts.data()));
  std::vector<fps::Seg> small, large;
  std::vector<uint32_t> slot_of_seg;
  uint32_t small_max = 0, large_max_m = 0;
  uint64_t small_samples = 0, large_samples = 0;
  for (uint64_t s = 0; s < S; ++s) {
    const uint64_t ns = off[s + 1] - off[s], m = soff[s + 1] - soff[s];
    if (m > ns)
      return fail(c, TKNN_EINVAL, "tknn_fps: %llu samples of segment %llu, which has %llu points", (unsigned long long)m,
                  (unsigned long long)s, (unsigned long long)ns);
    if (!start_ids) starts[s] = (int32_t)off[s];
    if (m > 0 && (starts[s] < 0 || (uint64_t)starts[s] < off[s] || (uint64_t)starts[s] >= off[s + 1]))
      return fail(c, TKNN_EINVAL, "tknn_fps: start %d outside segment %llu = [%llu, %llu)", starts[s], (unsigned long long)s,
                  (unsigned long long)off[s], (unsigned long long)off[s + 1]);
  }
  for (uint64_t s = 0; s < S; ++s) {
    const uint64_t ns = off[s + 1] - off[s], m = soff[s + 1] - soff[s];
    if (m == 0) continue;
    const fps::Seg sg = {(uint32_t)off[s], (uint32_t)ns, (uint32_t)soff[s], (uint32_t)m, (uint32_t)starts[s], 0, 0, 0};
    if (ns <= (uint64_t)fps::BLOCK_CAP) {
      small.push_back(sg);
      small_max = std::max(small_max, (uint32_t)ns);
      small_samples += m;
    } else {
      if (slot_of_seg.empty()) slot_of_seg.assign(S, fps::NO_SLOT);
      slot_of_seg[s] = (uint32_t)large.size();
      large.push_back(sg);
      large_max_m = std::max(large_max_m, (uint32_t)m);
      large_samples += m;
    }
  }
  const uint64_t total = soff[S];
  if (!large.empty()) {
    int coop = 0;
    TK_CUDA(c, cudaDeviceGetAttribute(&coop, cudaDevAttrCooperativeLaunch, c->device));
    if (!coop) return fail(c, TKNN_ECUDA, "tknn_fps: the device does not support cooperative launches (needed by clouds above %d points)",
                           fps::BLOCK_CAP);
  }

  reset_search_stats(c);
  int32_t* d_idx = nullptr;
  float* d_dist = nullptr;
  TK_TRY(out_view(c, idx_out, std::max<uint64_t>(total, 1), c->stage_idx, &d_idx));
  TK_TRY(out_view(c, dist_out, std::max<uint64_t>(total, 1), c->stage_dist, &d_dist));
  TK_TRY(ensure(c, c->fps_segs, sizeof(fps::Seg) * (small.size() + large.size())));
  fps::Seg* d_small = c->fps_segs.as<fps::Seg>();
  fps::Seg* d_large = d_small + small.size();
  if (!small.empty())
    TK_CUDA(c, cudaMemcpyAsync(d_small, small.data(), sizeof(fps::Seg) * small.size(), cudaMemcpyHostToDevice, st));
  if (!large.empty())
    TK_CUDA(c, cudaMemcpyAsync(d_large, large.data(), sizeof(fps::Seg) * large.size(), cudaMemcpyHostToDevice, st));
  TK_TRY(ensure_round_events(c, 8));
  cudaEvent_t* ev = c->round_ev.data();  // tier r: [4r] start, [4r + 1] end, [4r + 2 / + 3] its sampling kernel
  uint32_t* sc = c->scalars.as<uint32_t>();
  unsigned long long* counters = reinterpret_cast<unsigned long long*>(sc + SC_COUNTERS);
  int launches = 0;
  TK_CUDA(c, cudaMemsetAsync(counters, 0, N_COUNTERS * sizeof(unsigned long long), st));
  TK_CUDA(c, cudaEventRecord(c->ev[0], st));

  // block tier: one CTA per segment, sized for the largest one (about BLOCK_TARGET_PER points per thread)
  TK_CUDA(c, cudaEventRecord(ev[0], st));
  TK_CUDA(c, cudaEventRecord(ev[2], st));
  if (!small.empty()) {
    const uint32_t per = (small_max + fps::BLOCK_TARGET_PER - 1) / fps::BLOCK_TARGET_PER;
    const unsigned threads = std::min(1024u, std::max(32u, (per + 31u) / 32u * 32u));
    const size_t smem = sizeof(float4) * small_max + 2 * WARP * (sizeof(uint64_t) + sizeof(uint32_t));
    TK_CUDA(c, cudaFuncSetAttribute(fps::fps_block_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    fps::fps_block_kernel<<<(unsigned)small.size(), threads, smem, st>>>(c->pts.as<float4>(), d_small, small_max, d_idx, d_dist,
                                                                         c->squared);
    TK_CUDA(c, cudaGetLastError());
    ++launches;
  }
  TK_CUDA(c, cudaEventRecord(ev[3], st));
  TK_CUDA(c, cudaEventRecord(ev[1], st));

  // grid tier: compact leaf records of the large segments, then the cooperative kernel
  TK_CUDA(c, cudaEventRecord(ev[4], st));
  if (large.empty()) {
    TK_CUDA(c, cudaEventRecord(ev[6], st));
    TK_CUDA(c, cudaEventRecord(ev[7], st));
  } else {
    const uint32_t nl = c->n_leaves, n_words = (nl + 31) / 32, L = (uint32_t)large.size();
    const uint64_t n = c->n;
    TK_TRY(ensure(c, c->fps_slot_of_seg, sizeof(uint32_t) * S));
    TK_TRY(ensure(c, c->fps_words, sizeof(uint32_t) * n_words));
    TK_TRY(ensure(c, c->offsets, sizeof(uint32_t) * (size_t)(n_words + 1)));
    TK_TRY(ensure(c, c->fps_leaf_lo, sizeof(float4) * nl));
    TK_TRY(ensure(c, c->fps_leaf_hi, sizeof(float4) * nl));
    TK_TRY(ensure(c, c->fps_leaf_first, sizeof(uint32_t) * nl));
    TK_TRY(ensure(c, c->fps_leaf_key, sizeof(uint64_t) * nl));
    TK_TRY(ensure(c, c->fps_D, sizeof(float) * n));
    TK_TRY(ensure(c, c->fps_pos_of, sizeof(uint32_t) * n));
    TK_TRY(ensure(c, c->fps_best, sizeof(uint64_t) * 3 * (size_t)L));
    TK_CUDA(c, cudaMemcpyAsync(c->fps_slot_of_seg.p, slot_of_seg.data(), sizeof(uint32_t) * S, cudaMemcpyHostToDevice, st));
    const uint32_t* seg_of = c->segmented ? c->seg_of.as<uint32_t>() : nullptr;
    uint32_t* words = c->fps_words.as<uint32_t>();
    fps::leaf_flag_kernel<<<blocks_for(nl, fps::INIT_THREADS), fps::INIT_THREADS, 0, st>>>(
        c->leaf_start.as<uint32_t>(), nl, seg_of, c->fps_slot_of_seg.as<uint32_t>(), words);
    TK_CUDA(c, cudaGetLastError());
    TK_TRY(popc_scan(c, words, n_words, c->offsets.as<uint32_t>(), &launches));  // compact leaf count -> sc[SC_TOTAL]
    fps::leaf_init_kernel<<<blocks_for((uint64_t)nl * WARP, fps::INIT_THREADS), fps::INIT_THREADS, 0, st>>>(
        c->pts.as<float4>(), c->leaf_start.as<uint32_t>(), nl, seg_of, c->fps_slot_of_seg.as<uint32_t>(), words,
        c->offsets.as<uint32_t>(), c->fps_leaf_lo.as<float4>(), c->fps_leaf_hi.as<float4>(), c->fps_leaf_first.as<uint32_t>(),
        c->fps_leaf_key.as<uint64_t>(), c->fps_D.as<float>(), c->fps_pos_of.as<uint32_t>());
    fps::slot_init_kernel<<<blocks_for(L, fps::INIT_THREADS), fps::INIT_THREADS, 0, st>>>(d_large, L, c->fps_best.as<uint64_t>(),
                                                                                          d_idx, d_dist);
    TK_CUDA(c, cudaGetLastError());
    launches += 3;
    fps::GridParams P;
    P.pts = c->pts.as<float4>();
    P.leaf_lo = c->fps_leaf_lo.as<float4>();
    P.leaf_hi = c->fps_leaf_hi.as<float4>();
    P.leaf_first = c->fps_leaf_first.as<uint32_t>();
    P.leaf_key = c->fps_leaf_key.as<uint64_t>();
    P.D = c->fps_D.as<float>();
    P.pos_of = c->fps_pos_of.as<uint32_t>();
    P.segs = d_large;
    P.n_slots = L;
    P.max_m = large_max_m;
    P.n_leaves = sc + SC_TOTAL;
    P.best = c->fps_best.as<uint64_t>();
    P.idx_out = d_idx;
    P.dist_out = d_dist;
    P.squared = c->squared;
    P.counters = counters;
    void (*kernel)(const fps::GridParams) = c->counters ? fps::fps_grid_kernel<true> : fps::fps_grid_kernel<false>;
    int per_sm = 0;
    TK_CUDA(c, cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, kernel, fps::GRID_THREADS, 0));
    if (per_sm < 1) return fail(c, TKNN_ECUDA, "tknn_fps: the grid-tier kernel cannot be resident on an SM");
    // every block must be resident for the grid barrier: at most what the occupancy calculator allows, and two blocks per
    // SM at most, since a barrier over more blocks costs more than their extra warps hide
    const unsigned grid_blocks = (unsigned)(std::min(per_sm, 2) * c->sm_count);
    void* args[] = {&P};
    TK_CUDA(c, cudaEventRecord(ev[6], st));
    TK_CUDA(c, cudaLaunchCooperativeKernel((const void*)kernel, dim3(grid_blocks), dim3(fps::GRID_THREADS), args, 0, st));
    TK_CUDA(c, cudaEventRecord(ev[7], st));
    ++launches;
  }
  TK_CUDA(c, cudaEventRecord(ev[5], st));
  TK_CUDA(c, cudaEventRecord(c->ev[2], st));

  TK_TRY(copy_back(c, idx_out, d_idx, total, &c->stats.d2h_bytes));
  TK_TRY(copy_back(c, dist_out, d_dist, total, &c->stats.d2h_bytes));
  TK_CUDA(c, cudaStreamSynchronize(st));
  TK_CUDA(c, cudaEventElapsedTime(&c->stats.search_ms, c->ev[0], c->ev[2]));
  c->stats.n_queries = total;
  c->stats.rounds = 2;
  c->stats.round_queries[0] = small_samples;
  c->stats.round_queries[1] = large_samples;
  c->stats.kernel_launches = (uint32_t)launches;
  TK_TRY(finish_round_stats(c));
  TK_TRY(collect_counters(c));
  return TKNN_OK;
}

}  // extern "C"

namespace {

template <int QT>
int launch_feature_knn(tknn_ctx* c, const feat::Params& P, uint32_t n_items) {
  const size_t smem = feat::smem_bytes<QT>(P.k);
  TK_CUDA(c, cudaFuncSetAttribute(feat::feature_knn_kernel<QT>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  feat::feature_knn_kernel<QT><<<n_items, QT * 4, smem, c->stream>>>(P);
  TK_CUDA(c, cudaGetLastError());
  return TKNN_OK;
}

// Partial key lists of a split call are bounded to this many bytes (splits x nq x k x 8 B)
constexpr uint64_t FEATURE_PARTIAL_BYTES = 1ull << 29;

}  // namespace

extern "C" {

int tknn_feature_knn(tknn_ctx* c, const float* x, uint64_t n, int f, int x_stride_floats, const uint64_t* x_seg_offsets,
                     const float* y, uint64_t nq, int y_stride_floats, const uint64_t* y_seg_offsets, uint64_t n_segments,
                     const int32_t* self_ids, int k, int32_t* idx_out, float* dist_out) {
  TK_TRY(check_ctx(c));
  const char* what = "tknn_feature_knn";
  if (!x || !y || !idx_out) return fail(c, TKNN_EINVAL, "%s: null x, y or idx_out", what);
  if (f < 1 || f > 1024) return fail(c, TKNN_EINVAL, "%s: f = %d outside [1, 1024]", what, f);
  if (x_stride_floats < f || y_stride_floats < f)
    return fail(c, TKNN_EINVAL, "%s: strides %d / %d below f = %d", what, x_stride_floats, y_stride_floats, f);
  if (n >= (1ull << 31) || nq >= (1ull << 31)) return fail(c, TKNN_EINVAL, "%s: n and nq must be below 2^31", what);
  if (k < 1 || k > TKNN_MAX_K || (uint64_t)k > n)
    return fail(c, TKNN_EINVAL, "%s: k = %d outside [1, min(n = %llu, %d)]", what, k, (unsigned long long)n, TKNN_MAX_K);
  if ((x_seg_offsets == nullptr) != (y_seg_offsets == nullptr))
    return fail(c, TKNN_EINVAL, "%s: give both segment offset arrays or neither", what);
  if (!x_seg_offsets && n_segments != 1)
    return fail(c, TKNN_EINVAL, "%s: n_segments = %llu without offsets (must be 1)", what, (unsigned long long)n_segments);
  if (n_segments < 1 || n_segments >= (1ull << 31))
    return fail(c, TKNN_EINVAL, "%s: n_segments = %llu outside [1, 2^31 - 1]", what, (unsigned long long)n_segments);
  ScopedDevice sd(c->device);
  cudaStream_t st = c->stream;
  std::vector<uint64_t> xo{0, n}, yo{0, nq};
  if (x_seg_offsets) {
    TK_TRY(read_offsets(c, what, "data segment", x_seg_offsets, n_segments, n, "n", &xo));
    TK_TRY(read_offsets(c, what, "query segment", y_seg_offsets, n_segments, nq, "nq", &yo));
  }
  reset_search_stats(c);
  c->stats.n_queries = nq;
  c->stats.k = k;
  if (nq == 0) return TKNN_OK;

  // work list: (segment, tile of QT query rows, split of the segment's data rows); splits only when the tiles alone
  // leave the GPU idle (few queries against big clouds), at least 4 data tiles each, the partial lists bounded
  const int QT = feat::query_tile(k);
  uint64_t tiles = 0, max_n = 0, pairs = 0;
  for (uint64_t s = 0; s < n_segments; ++s) {
    const uint64_t ns = xo[s + 1] - xo[s], ms = yo[s + 1] - yo[s];
    tiles += (ms + QT - 1) / QT;
    if (ms) max_n = std::max(max_n, ns);
    pairs += ns * ms;
  }
  const uint64_t target = (uint64_t)c->sm_count * 2;
  uint64_t splits = 1;
  if (tiles < target) {
    splits = (target + tiles - 1) / tiles;
    splits = std::min<uint64_t>(splits, std::max<uint64_t>(1, max_n / (4 * feat::PT)));
    splits = std::min<uint64_t>(splits, 256);
    splits = std::min<uint64_t>(splits, std::max<uint64_t>(1, FEATURE_PARTIAL_BYTES / (nq * (uint64_t)k * sizeof(uint64_t))));
  }
  std::vector<feat::Item> items;
  items.reserve(tiles * splits);
  for (uint64_t s = 0; s < n_segments; ++s) {
    const uint64_t ns = xo[s + 1] - xo[s];
    const uint64_t chunk = ((ns + splits - 1) / splits + feat::PT - 1) / feat::PT * feat::PT;
    for (uint64_t q0 = yo[s]; q0 < yo[s + 1]; q0 += QT)
      for (uint64_t sp = 0; sp < splits; ++sp) {
        const uint64_t a = std::min(xo[s] + sp * chunk, xo[s + 1]), b = std::min(a + chunk, xo[s + 1]);
        items.push_back({(uint32_t)q0, (uint32_t)std::min<uint64_t>(QT, yo[s + 1] - q0), (uint32_t)a, (uint32_t)b,
                         (uint32_t)sp, 0, 0, 0});
      }
  }

  // inputs: host rows are staged (y aliasing x is staged once), device rows are read in place
  const float *d_x = nullptr, *d_y = nullptr;
  const int32_t* d_sid = nullptr;
  const bool same = y == x && y_stride_floats == x_stride_floats && nq == n;
  TK_TRY(stage_in(c, x, (size_t)(n - 1) * x_stride_floats + f, c->fk_x, &d_x));
  if (same) d_y = d_x;
  else TK_TRY(stage_in(c, y, (size_t)(nq - 1) * y_stride_floats + f, c->fk_y, &d_y));
  TK_TRY(stage_in(c, self_ids, nq, c->fk_sid, &d_sid));
  TK_TRY(ensure(c, c->fk_items, items.size() * sizeof(feat::Item)));
  TK_CUDA(c, cudaMemcpyAsync(c->fk_items.p, items.data(), items.size() * sizeof(feat::Item), cudaMemcpyHostToDevice, st));
  const size_t out_elems = (size_t)nq * k;
  int32_t* d_idx = nullptr;
  float* d_dist = nullptr;
  TK_TRY(out_view(c, idx_out, out_elems, c->stage_idx, &d_idx));
  TK_TRY(out_view(c, dist_out, out_elems, c->stage_dist, &d_dist));
  if (splits > 1) {
    TK_TRY(ensure(c, c->fk_partial, splits * out_elems * sizeof(uint64_t)));
    if (!d_dist) {  // the merge writes distances unconditionally
      TK_TRY(ensure(c, c->fk_dist, out_elems * sizeof(float)));
    }
  }
  TK_TRY(ensure_round_events(c, 8));
  cudaEvent_t* ev = c->round_ev.data();  // round r: [4r] start, [4r + 1] end, [4r + 2 / + 3] its kernel
  uint32_t* sc = c->scalars.as<uint32_t>();
  int launches = 0;
  TK_CUDA(c, cudaEventRecord(c->ev[0], st));
  TK_CUDA(c, cudaEventRecord(ev[0], st));
  TK_CUDA(c, cudaMemsetAsync(sc + SC_ERROR, 0, 2 * sizeof(uint32_t), st));
  {
    const unsigned blocks = (unsigned)std::min<uint64_t>((uint64_t)c->sm_count * 8, std::max<uint64_t>(1, (n * f + 255) / 256));
    feat::finite_kernel<<<blocks, 256, 0, st>>>(d_x, n, f, x_stride_floats, sc + SC_QBAD);
    ++launches;
    if (!same) {
      const unsigned qblocks = (unsigned)std::min<uint64_t>((uint64_t)c->sm_count * 8, std::max<uint64_t>(1, (nq * f + 255) / 256));
      feat::finite_kernel<<<qblocks, 256, 0, st>>>(d_y, nq, f, y_stride_floats, sc + SC_QBAD);
      ++launches;
    }
    TK_CUDA(c, cudaGetLastError());
  }
  feat::Params P;
  P.x = d_x;
  P.y = d_y;
  P.sid = d_sid;
  P.items = c->fk_items.as<feat::Item>();
  P.f = f;
  P.x_stride = x_stride_floats;
  P.y_stride = y_stride_floats;
  P.k = k;
  P.squared = c->squared;
  P.nq = (uint32_t)nq;
  P.idx_out = d_idx;
  P.dist_out = d_dist;
  P.partial = splits > 1 ? c->fk_partial.as<uint64_t>() : nullptr;
  TK_CUDA(c, cudaEventRecord(ev[2], st));
  if (QT == 64) TK_TRY(launch_feature_knn<64>(c, P, (uint32_t)items.size()));
  else TK_TRY(launch_feature_knn<32>(c, P, (uint32_t)items.size()));
  ++launches;
  TK_CUDA(c, cudaEventRecord(ev[3], st));
  TK_CUDA(c, cudaEventRecord(ev[1], st));
  if (splits > 1) {
    float* m_dist = d_dist ? d_dist : c->fk_dist.as<float>();
    const size_t smem = (size_t)k * 32 * sizeof(uint64_t);
    TK_CUDA(c, cudaEventRecord(ev[4], st));
    TK_CUDA(c, cudaEventRecord(ev[6], st));
    TK_CUDA(c, cudaFuncSetAttribute(brute::merge_keys_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    brute::merge_keys_kernel<<<(unsigned)((nq + 31) / 32), 32, smem, st>>>(c->fk_partial.as<uint64_t>(), (int)splits,
                                                                          (uint32_t)nq, k, nullptr, c->squared, d_idx, m_dist);
    TK_CUDA(c, cudaGetLastError());
    ++launches;
    TK_CUDA(c, cudaEventRecord(ev[7], st));
    TK_CUDA(c, cudaEventRecord(ev[5], st));
  }
  TK_CUDA(c, cudaEventRecord(c->ev[2], st));
  TK_TRY(copy_back(c, idx_out, d_idx, out_elems, &c->stats.d2h_bytes));
  TK_TRY(copy_back(c, dist_out, d_dist, out_elems, &c->stats.d2h_bytes));
  TK_CUDA(c, cudaEventRecord(c->ev[3], st));
  TK_CUDA(c, cudaStreamSynchronize(st));
  TK_CUDA(c, cudaEventElapsedTime(&c->stats.search_ms, c->ev[0], c->ev[2]));
  TK_CUDA(c, cudaEventElapsedTime(&c->stats.d2h_ms, c->ev[2], c->ev[3]));
  c->stats.rounds = splits > 1 ? 2 : 1;
  c->stats.round_queries[0] = nq;
  if (splits > 1) c->stats.round_queries[1] = nq;
  c->stats.points_tested = pairs;
  c->stats.kernel_launches = (uint32_t)(launches + (c->mailbox_h ? 1 : 0));  // + the error-flag fetch below
  TK_TRY(finish_round_stats(c));
  uint32_t e[2] = {0, 0};
  TK_TRY(fetch_words(c, sc + SC_ERROR, 2, nullptr, 0, e));
  if (e[1]) return fail(c, TKNN_EINVAL, "%s: non-finite value in the first %d columns of x or y", what, f);
  return TKNN_OK;
}

}  // extern "C"

namespace {

// Long rows are radix-sorted in batches of at most this many entries (40 B of device scratch per entry).
constexpr uint64_t RADIUS_LONG_BATCH = 1ull << 26;

// exclusive u64 scan of counts[0 .. m) into off[0 .. m] (off[m] = total, also written to *total)
int scan_counts(tknn_ctx* c, const uint32_t* counts, uint64_t m, uint64_t* off, uint64_t* total, int* launches) {
  const uint64_t nb = std::max<uint64_t>(1, (m + radius::SCAN_CHUNK - 1) / radius::SCAN_CHUNK);
  TK_TRY(ensure(c, c->rl_sums, sizeof(uint64_t) * nb));
  uint64_t* sums = c->rl_sums.as<uint64_t>();
  radius::scan_reduce_kernel<<<(unsigned)nb, radius::THREADS, 0, c->stream>>>(counts, m, sums);
  radius::scan_sums_kernel<<<1, radius::THREADS, 0, c->stream>>>(sums, nb, total);
  radius::scan_apply_kernel<<<(unsigned)nb, radius::THREADS, 0, c->stream>>>(counts, m, sums, total, off);
  TK_CUDA(c, cudaGetLastError());
  *launches += 3;
  return TKNN_OK;
}

// The pipeline of radius.cuh over nq staged query positions (qpts: x, y, z, output row bits).  self_sorted: the excluded
// data index per position (query form) or nullptr with self_is_row (all-points form: the point itself).  seg_of: the
// segment of every position on a segmented build (set_segments).  The caller has recorded c->ev[0] and cleared
// SC_ERROR / SC_QBAD; launches counts its own kernels so far.
int radius_core(tknn_ctx* c, const float4* qpts, uint64_t nq, const int32_t* self_sorted, int self_is_row,
                const uint32_t* seg_of, float radius, uint64_t* offsets_out, int32_t* idx_out, float* dist_out,
                uint64_t capacity, uint64_t* total_out, int launches) {
  cudaStream_t st = c->stream;
  uint32_t* sc = c->scalars.as<uint32_t>();
  const uint64_t n = c->n;
  const bool fill_rows = idx_out != nullptr;
  ScratchScope scratch = radius_list_scratch(c);
  TK_TRY(ensure_round_events(c, 12));
  cudaEvent_t* ev = c->round_ev.data();  // phase r: [4r] start, [4r + 1] end, [4r + 2 / + 3] its kernels

  TK_TRY(ensure(c, c->rl_cnt_pos, sizeof(uint32_t) * nq));
  TK_TRY(ensure(c, c->rl_cnt_row, sizeof(uint32_t) * nq));
  TK_TRY(ensure(c, c->rl_off_pos, sizeof(uint64_t) * (nq + 1)));
  uint64_t* off_row = nullptr;
  TK_TRY(out_view(c, offsets_out, nq + 1, c->rl_off_row, &off_row));
  TK_TRY(ensure(c, c->rl_stats, sizeof(uint64_t) * 4));
  TK_TRY(ensure(c, c->rl_long_pos, sizeof(uint32_t) * nq));
  TK_TRY(ensure(c, c->rl_long_len, sizeof(uint32_t) * nq));
  uint32_t* cnt_pos = c->rl_cnt_pos.as<uint32_t>();
  uint32_t* cnt_row = c->rl_cnt_row.as<uint32_t>();
  uint64_t* off_pos = c->rl_off_pos.as<uint64_t>();
  uint64_t* rstats = c->rl_stats.as<uint64_t>();  // row total, position total, long rows, long-row entries
  uint32_t* long_pos = c->rl_long_pos.as<uint32_t>();
  const int32_t* self_pos = nullptr;
  if (self_sorted) {
    TK_TRY(ensure(c, c->rl_pos_of, sizeof(int32_t) * n));
    TK_TRY(ensure(c, c->rl_self_pos, sizeof(int32_t) * nq));
    self_pos = c->rl_self_pos.as<int32_t>();
  }

  trav::Params P;
  std::memset(&P, 0, sizeof(P));
  P.nodes = c->nodes.as<Node>();
  P.node_min_idx = c->node_min_idx.as<int2>();
  P.pts = c->pts.as<float4>();
  P.queries = qpts;
  P.n_active = nq;
  P.n_groups = (uint32_t)((nq + 31) / 32);
  P.r2 = radius * radius;
  P.k = 0;
  P.self_is_row = self_is_row;
  P.self_pos = self_pos;
  P.final_round = 1;
  P.squared = c->squared;
  P.error = sc + SC_ERROR;
  P.group_counter = sc + SC_GROUP_COUNTER;
  P.counters = c->counters ? reinterpret_cast<unsigned long long*>(sc + SC_COUNTERS) : nullptr;
  set_segments(c, P, seg_of);
  TK_CUDA(c, cudaMemsetAsync(sc + SC_COUNTERS, 0, N_COUNTERS * sizeof(unsigned long long), st));

  // 1. count (minus self, by position and by row), both scans, the long-row list; one read-back
  TK_CUDA(c, cudaEventRecord(ev[0], st));
  if (self_sorted) {
    radius::inverse_kernel<<<blocks_for(n, 256), 256, 0, st>>>(P.pts, n, c->rl_pos_of.as<int32_t>());
    radius::self_pos_kernel<<<blocks_for(nq, 256), 256, 0, st>>>(self_sorted, nq, c->rl_pos_of.as<int32_t>(), n,
                                                                 c->rl_self_pos.as<int32_t>());
    TK_CUDA(c, cudaGetLastError());
    launches += 2;
  }
  TK_CUDA(c, cudaMemsetAsync(sc + SC_GROUP_COUNTER, 0, sizeof(uint32_t), st));
  P.count_out = cnt_pos;
  P.count_row = cnt_row;
  TK_CUDA(c, cudaEventRecord(ev[2], st));
  TK_TRY(launch_traverse<trav::MODE_RANGE_LIST_COUNT>(c, P));
  TK_CUDA(c, cudaEventRecord(ev[3], st));
  TK_TRY(scan_counts(c, cnt_row, nq, off_row, rstats, &launches));
  TK_TRY(scan_counts(c, cnt_pos, nq, off_pos, rstats + 1, &launches));
  TK_CUDA(c, cudaMemsetAsync(rstats + 2, 0, 2 * sizeof(uint64_t), st));
  radius::long_rows_kernel<<<blocks_for(nq, 256), 256, 0, st>>>(cnt_pos, nq, long_pos, c->rl_long_len.as<uint32_t>(),
                                                                 reinterpret_cast<unsigned long long*>(rstats + 2));
  TK_CUDA(c, cudaGetLastError());
  launches += 2;  // the traversal, long_rows_kernel
  TK_CUDA(c, cudaEventRecord(ev[1], st));
  uint64_t rb[4] = {0, 0, 0, 0};
  TK_TRY(fetch_words(c, reinterpret_cast<const uint32_t*>(rstats), 8, nullptr, 0, reinterpret_cast<uint32_t*>(rb)));
  const uint64_t total = rb[0], n_long = rb[2];
  if (rb[1] != total) return fail(c, TKNN_ECUDA, "internal: row and position totals differ");
  if (total_out) *total_out = total;
  TK_TRY(copy_back(c, offsets_out, off_row, nq + 1, &c->stats.d2h_bytes));
  const bool write_rows = fill_rows && capacity >= total;

  // 2. fill: the unsorted rows in position order
  TK_CUDA(c, cudaEventRecord(ev[4], st));
  TK_CUDA(c, cudaEventRecord(ev[6], st));
  int32_t* d_idx = nullptr;
  float* d_dist = nullptr;
  if (write_rows && total) {
    TK_TRY(ensure(c, c->rl_keys, sizeof(uint64_t) * total));
    TK_TRY(out_view(c, idx_out, total, c->stage_idx, &d_idx));
    TK_TRY(out_view(c, dist_out, total, c->stage_dist, &d_dist));
    TK_CUDA(c, cudaMemsetAsync(sc + SC_GROUP_COUNTER, 0, sizeof(uint32_t), st));
    P.list_off = off_pos;
    P.list_keys = c->rl_keys.as<uint64_t>();
    TK_TRY(launch_traverse<trav::MODE_RANGE_LIST>(c, P));
    ++launches;
  }
  TK_CUDA(c, cudaEventRecord(ev[7], st));
  TK_CUDA(c, cudaEventRecord(ev[5], st));

  // 3. order: short rows one warp each in shared memory, long rows by the radix sort in batches
  TK_CUDA(c, cudaEventRecord(ev[8], st));
  TK_CUDA(c, cudaEventRecord(ev[10], st));
  if (write_rows && total) {
    const uint64_t* keys = c->rl_keys.as<uint64_t>();
    radius::sort_rows_warp_kernel<<<blocks_for(nq, radius::SORT_WARPS), radius::SORT_WARPS * 32, 0, st>>>(
        keys, off_pos, cnt_pos, qpts, nq, off_row, c->squared, d_idx, d_dist);
    TK_CUDA(c, cudaGetLastError());
    ++launches;
    if (n_long) {
      // the long rows in position order (the list was appended in any order), their lengths and global prefix
      std::vector<uint32_t> hpos(n_long), hlen(n_long), lp(n_long);
      std::vector<uint64_t> order(n_long), boff(n_long + 1);
      TK_CUDA(c, cudaMemcpyAsync(hpos.data(), long_pos, sizeof(uint32_t) * n_long, cudaMemcpyDeviceToHost, st));
      TK_CUDA(c, cudaMemcpyAsync(hlen.data(), c->rl_long_len.p, sizeof(uint32_t) * n_long, cudaMemcpyDeviceToHost, st));
      TK_CUDA(c, cudaStreamSynchronize(st));
      for (uint64_t r = 0; r < n_long; ++r) order[r] = r;
      std::sort(order.begin(), order.end(), [&](uint64_t a, uint64_t b) { return hpos[a] < hpos[b]; });
      boff[0] = 0;
      for (uint64_t r = 0; r < n_long; ++r) {
        lp[r] = hpos[order[r]];
        const uint64_t len = hlen[order[r]];
        if (len > rsort::MAX_N)
          return fail(c, TKNN_EINVAL, "a row of %llu entries exceeds the sort's limit", (unsigned long long)len);
        boff[r + 1] = boff[r] + len;
      }
      TK_TRY(ensure(c, c->rl_boff, sizeof(uint64_t) * (n_long + 1)));
      TK_CUDA(c, cudaMemcpyAsync(long_pos, lp.data(), sizeof(uint32_t) * n_long, cudaMemcpyHostToDevice, st));
      TK_CUDA(c, cudaMemcpyAsync(c->rl_boff.p, boff.data(), sizeof(uint64_t) * (n_long + 1), cudaMemcpyHostToDevice, st));
      uint64_t batch_max = 0;  // entries of the largest batch
      std::vector<uint64_t> firsts;
      for (uint64_t r = 0; r < n_long;) {
        uint64_t e = r + 1;
        while (e < n_long && boff[e + 1] - boff[r] <= RADIUS_LONG_BATCH) ++e;
        firsts.push_back(r);
        batch_max = std::max(batch_max, boff[e] - boff[r]);
        r = e;
      }
      firsts.push_back(n_long);
      TK_TRY(ensure(c, c->rl_ka, sizeof(uint64_t) * batch_max));
      TK_TRY(ensure(c, c->rl_kb, sizeof(uint64_t) * batch_max));
      TK_TRY(ensure(c, c->rl_kc, sizeof(uint64_t) * batch_max));
      TK_TRY(ensure(c, c->rl_va, sizeof(uint32_t) * batch_max));
      TK_TRY(ensure(c, c->rl_vb, sizeof(uint32_t) * batch_max));
      TK_TRY(ensure(c, c->rl_vc, sizeof(uint32_t) * batch_max));
      TK_TRY(ensure(c, c->rl_row_of, sizeof(uint32_t) * batch_max));
      TK_TRY(ensure(c, c->rl_sort_tmp, sizeof(uint32_t) * rsort::temp_words(batch_max)));
      uint64_t *ka = c->rl_ka.as<uint64_t>(), *kb = c->rl_kb.as<uint64_t>(), *kc = c->rl_kc.as<uint64_t>();
      uint32_t *va = c->rl_va.as<uint32_t>(), *vb = c->rl_vb.as<uint32_t>(), *vc = c->rl_vc.as<uint32_t>();
      uint32_t* row_of = c->rl_row_of.as<uint32_t>();
      const uint64_t* d_boff = c->rl_boff.as<uint64_t>();
      for (size_t b = 0; b + 1 < firsts.size(); ++b) {
        const uint32_t first = (uint32_t)firsts[b], rows = (uint32_t)(firsts[b + 1] - firsts[b]);
        const uint64_t e = boff[firsts[b + 1]] - boff[first];
        radius::long_gather_kernel<<<rows, radius::THREADS, 0, st>>>(keys, off_pos, long_pos, d_boff, first, ka, va, row_of);
        // by key (all 64 bits: 8 passes, so the result is back in ka / va) ...
        bool in_b = false;
        launches += 1 + rsort::sort_pairs(ka, va, kb, vb, e, c->rl_sort_tmp.as<uint32_t>(), c->sm_count, st, rsort::PASSES, &in_b);
        if (in_b) return fail(c, TKNN_ECUDA, "internal: odd key-sort pass count");
        // ... then stably by the row's rank in the batch
        radius::long_rowkey_kernel<<<blocks_for(e, 256), 256, 0, st>>>(va, row_of, e, kb, vb);
        const int row_bits = rows > 1 ? 32 - __builtin_clz(rows - 1) : 1;
        launches += 1 + rsort::sort_pairs(kb, vb, kc, vc, e, c->rl_sort_tmp.as<uint32_t>(), c->sm_count, st,
                                          (row_bits + 7) / 8, &in_b);
        radius::long_emit_kernel<<<blocks_for(e, 256), 256, 0, st>>>(ka, in_b ? kc : kb, in_b ? vc : vb, e, long_pos, d_boff,
                                                                     first, qpts, off_row, c->squared, d_idx, d_dist);
        TK_CUDA(c, cudaGetLastError());
        ++launches;
      }
    }
  }
  TK_CUDA(c, cudaEventRecord(ev[11], st));
  TK_CUDA(c, cudaEventRecord(ev[9], st));
  TK_CUDA(c, cudaEventRecord(c->ev[2], st));
  if (write_rows && total) {
    TK_TRY(copy_back(c, idx_out, d_idx, total, &c->stats.d2h_bytes));
    TK_TRY(copy_back(c, dist_out, d_dist, total, &c->stats.d2h_bytes));
  }
  TK_CUDA(c, cudaStreamSynchronize(st));
  TK_CUDA(c, cudaEventElapsedTime(&c->stats.search_ms, c->ev[0], c->ev[2]));
  c->stats.n_queries = nq;
  c->stats.rounds = 3;
  c->stats.start_radius = c->stats.final_radius = radius;
  c->stats.round_queries[0] = nq;
  c->stats.round_queries[1] = write_rows ? nq : 0;
  c->stats.round_queries[2] = write_rows ? n_long : 0;
  c->stats.kernel_launches = (uint32_t)(launches + c->mailbox_launches + (c->mailbox_h ? 1 : 0));  // + the error-flag fetch
  TK_TRY(finish_round_stats(c));
  TK_TRY(collect_counters(c));
  TK_TRY(read_error_flag(c));
  if (fill_rows && !write_rows)
    return fail(c, TKNN_EINVAL, "capacity %llu < %llu entries", (unsigned long long)capacity, (unsigned long long)total);
  return TKNN_OK;
}

// checks shared by both forms; nq = 0 (query form) writes offsets_out[0] = 0 and a zero total
int radius_args(tknn_ctx* c, const char* what, float radius, uint64_t* offsets_out) {
  TK_TRY(check_ctx(c));
  if (c->n == 0) return fail(c, TKNN_ESTATE, "%s before tknn_build", what);
  if (c->ids_in_w) return fail(c, TKNN_ESTATE, "this BVH carries caller-chosen point ids (point-partitioned build)");
  if (!(radius >= 0.0f)) return fail(c, TKNN_EINVAL, "radius must be >= 0");
  if (!offsets_out) return fail(c, TKNN_EINVAL, "null offsets array");
  if (c->n > (uint64_t)INT32_MAX) return fail(c, TKNN_EINVAL, "%s supports at most 2^31 - 1 points", what);
  return TKNN_OK;
}

// tknn_radius_query and tknn_radius_query_segments after radius_args; segments as in query_core
int radius_query_core(tknn_ctx* c, const char* what, const float* queries, uint64_t nq, int dim, int stride_floats,
                      bool segments, const uint64_t* q_seg_offsets, uint64_t n_segments, const int32_t* self_ids,
                      float radius, uint64_t* offsets_out, int32_t* idx_out, float* dist_out, uint64_t capacity,
                      uint64_t* total_out) {
  if (!queries && nq) return fail(c, TKNN_EINVAL, "null query array");
  if (dim != 2 && dim != 3) return fail(c, TKNN_EINVAL, "dim = %d (must be 2 or 3)", dim);
  if (stride_floats < dim) return fail(c, TKNN_EINVAL, "stride %d < dim %d", stride_floats, dim);
  if (nq > rsort::MAX_N) return fail(c, TKNN_EINVAL, "too many queries");
  ScopedDevice sd(c->device);
  if (segments) TK_TRY(check_query_offsets(c, what, q_seg_offsets, n_segments, nq));
  if (!c->segmented) q_seg_offsets = nullptr;
  reset_search_stats(c);
  if (nq == 0) {
    if (total_out) *total_out = 0;
    return zero_fill(c, offsets_out, 1);
  }
  TK_CUDA(c, cudaEventRecord(c->ev[0], c->stream));
  ScratchScope scratch = query_scratch(c);
  int launches = 0;
  const int32_t* d_sid_sorted = nullptr;
  const float* d_r2_sorted = nullptr;
  const uint32_t* d_seg_sorted = nullptr;
  TK_TRY(stage_queries(c, queries, nq, dim, stride_floats, self_ids, nullptr, &d_sid_sorted, &d_r2_sorted, &launches,
                       q_seg_offsets, n_segments, &d_seg_sorted));
  return radius_core(c, c->q_pts.as<float4>(), nq, d_sid_sorted, 0, d_seg_sorted, radius, offsets_out, idx_out, dist_out,
                     capacity, total_out, launches);
}

}  // namespace

extern "C" {

int tknn_radius_search(tknn_ctx* c, float radius, uint64_t* offsets_out, int32_t* idx_out, float* dist_out,
                       uint64_t capacity, uint64_t* total_out) {
  TK_TRY(radius_args(c, "tknn_radius_search", radius, offsets_out));
  ScopedDevice sd(c->device);
  reset_search_stats(c);
  uint32_t* sc = c->scalars.as<uint32_t>();
  TK_CUDA(c, cudaEventRecord(c->ev[0], c->stream));
  TK_CUDA(c, cudaMemsetAsync(sc + SC_ERROR, 0, 2 * sizeof(uint32_t), c->stream));
  return radius_core(c, c->pts.as<float4>(), c->n, nullptr, 1, c->seg_of.as<uint32_t>(), radius, offsets_out, idx_out,
                     dist_out, capacity, total_out, 0);
}

int tknn_radius_query(tknn_ctx* c, const float* queries, uint64_t nq, int dim, int stride_floats, const int32_t* self_ids,
                      float radius, uint64_t* offsets_out, int32_t* idx_out, float* dist_out, uint64_t capacity,
                      uint64_t* total_out) {
  TK_TRY(radius_args(c, "tknn_radius_query", radius, offsets_out));
  TK_TRY(refuse_segmented(c, "tknn_radius_query"));
  return radius_query_core(c, "tknn_radius_query", queries, nq, dim, stride_floats, false, nullptr, 0, self_ids, radius,
                           offsets_out, idx_out, dist_out, capacity, total_out);
}

int tknn_radius_query_segments(tknn_ctx* c, const float* queries, uint64_t nq, int dim, int stride_floats,
                               const uint64_t* q_seg_offsets, uint64_t n_segments, const int32_t* self_ids, float radius,
                               uint64_t* offsets_out, int32_t* idx_out, float* dist_out, uint64_t capacity,
                               uint64_t* total_out) {
  TK_TRY(radius_args(c, "tknn_radius_query_segments", radius, offsets_out));
  return radius_query_core(c, "tknn_radius_query_segments", queries, nq, dim, stride_floats, true, q_seg_offsets,
                           n_segments, self_ids, radius, offsets_out, idx_out, dist_out, capacity, total_out);
}

int tknn_brute_force(tknn_ctx* c, const int32_t* query_ids, uint64_t nq, int k, int32_t* idx_out, float* dist_out) {
  TK_TRY(check_ctx(c));
  if (c->n == 0) return fail(c, TKNN_ESTATE, "tknn_brute_force before tknn_build");
  TK_TRY(refuse_segmented(c, "tknn_brute_force"));
  if (k < 1 || k > TKNN_MAX_K || (uint64_t)k > c->n - 1) return fail(c, TKNN_EINVAL, "k = %d invalid for n = %llu", k,
                                                                     (unsigned long long)c->n);
  if (nq == 0) return TKNN_OK;
  if (!query_ids || !idx_out || !dist_out) return fail(c, TKNN_EINVAL, "null array");
  if (nq > (1u << 20)) return fail(c, TKNN_EINVAL, "at most 2^20 brute-force queries per call");
  if (c->ids_in_w) return fail(c, TKNN_ESTATE, "this BVH carries caller-chosen point ids: use tknn_partition_verify");
  ScopedDevice sd(c->device);
  cudaStream_t st = c->stream;
  std::vector<int32_t> ids(nq);
  TK_TRY(read_to_host(c, query_ids, nq, ids.data()));
  std::vector<uint32_t> perm(nq);
  for (uint32_t i = 0; i < nq; ++i) perm[i] = i;
  std::sort(perm.begin(), perm.end(), [&](uint32_t a, uint32_t b) { return ids[a] < ids[b]; });
  std::vector<int32_t> sorted(nq);
  for (uint32_t i = 0; i < nq; ++i) sorted[i] = ids[perm[i]];
  for (uint32_t i = 0; i < nq; ++i) {
    if (sorted[i] < 0 || (uint64_t)sorted[i] >= c->n) return fail(c, TKNN_EINVAL, "query id %d out of range", sorted[i]);
    if (i && sorted[i] == sorted[i - 1]) return fail(c, TKNN_EINVAL, "duplicate query id %d", sorted[i]);
  }
  DevBuf d_ids, d_perm, qpts, o_idx, o_dist;
  ScratchScope scratch({&d_ids, &d_perm, &qpts, &o_idx, &o_dist});
  TK_TRY(ensure(c, d_ids, nq * sizeof(int32_t)));
  TK_TRY(ensure(c, d_perm, nq * sizeof(uint32_t)));
  TK_TRY(ensure(c, qpts, nq * sizeof(float4)));
  TK_CUDA(c, cudaMemcpyAsync(d_ids.p, sorted.data(), nq * sizeof(int32_t), cudaMemcpyHostToDevice, st));
  TK_CUDA(c, cudaMemcpyAsync(d_perm.p, perm.data(), nq * sizeof(uint32_t), cudaMemcpyHostToDevice, st));
  int32_t* d_idx = nullptr;
  float* d_dist = nullptr;
  TK_TRY(out_view(c, idx_out, nq * k, o_idx, &d_idx));
  TK_TRY(out_view(c, dist_out, nq * k, o_dist, &d_dist));
  brute::lookup_queries_kernel<<<blocks_for(c->n, 256), 256, 0, st>>>(c->pts.as<float4>(), c->n, d_ids.as<int32_t>(),
                                                                       (uint32_t)nq, qpts.as<float4>());
  TK_TRY(brute_core(c, qpts.as<float4>(), nq, k, d_perm.as<uint32_t>(), d_idx, d_dist, 0));
  TK_TRY(copy_back(c, idx_out, d_idx, nq * k));
  TK_TRY(copy_back(c, dist_out, d_dist, nq * k));
  TK_CUDA(c, cudaStreamSynchronize(st));
  return TKNN_OK;
}

}  // extern "C"

// Exact tiled brute force of external queries (x, y, z, id to exclude) against the sorted points: one warp per
// (32 queries, split of the point range), then a per-query merge of the splits.  Fills the grid twice over.
int tknn::host::brute_core(tknn_ctx* c, const float4* d_qpts, uint64_t nq, int k, const uint32_t* d_row_of, int32_t* d_idx,
                           float* d_dist, int squared) {
  if (nq == 0) return TKNN_OK;
  cudaStream_t st = c->stream;
  const uint64_t groups = (nq + 31) / 32;
  int splits = (int)std::max<uint64_t>(1, std::min<uint64_t>(256, ((uint64_t)c->sm_count * 64 + groups - 1) / groups));
  splits = (int)std::max<uint64_t>(1, std::min<uint64_t>((uint64_t)splits, (c->n + 1023) / 1024));
  DevBuf partial;
  ScratchScope scratch({&partial});
  TK_TRY(ensure(c, partial, (size_t)splits * nq * k * sizeof(uint64_t)));
  const size_t smem = 32 * sizeof(float4) + (size_t)k * 32 * sizeof(uint64_t);
  cudaError_t e = cudaFuncSetAttribute(brute::brute_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
  if (e == cudaSuccess) e = cudaFuncSetAttribute(brute::merge_keys_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
  if (e == cudaSuccess) {
    dim3 grid((unsigned)groups, (unsigned)splits);
    brute::brute_kernel<<<grid, 32, smem, st>>>(c->pts.as<float4>(), c->n, d_qpts, (uint32_t)nq, k, splits, partial.as<uint64_t>());
    brute::merge_keys_kernel<<<(unsigned)groups, 32, smem, st>>>(partial.as<uint64_t>(), splits, (uint32_t)nq, k, d_row_of, squared,
                                                                 d_idx, d_dist);
    e = cudaGetLastError();
  }
  if (e == cudaSuccess) e = cudaStreamSynchronize(st);  // `partial` is released on return
  if (e != cudaSuccess) { cudaGetLastError(); return fail(c, TKNN_ECUDA, "brute force: %s", cudaGetErrorString(e)); }
  return TKNN_OK;
}

extern "C" {

int tknn_merge_topk(tknn_ctx* c, const int32_t* idx_parts, const float* d2_parts, int parts, uint64_t nq, int k,
                    int32_t* idx_out, float* dist_out) {
  TK_TRY(check_ctx(c));
  if (parts < 1 || k < 1 || k > TKNN_MAX_K) return fail(c, TKNN_EINVAL, "bad parts / k");
  if (nq == 0) return TKNN_OK;
  if (!idx_parts || !d2_parts || !idx_out || !dist_out) return fail(c, TKNN_EINVAL, "null array");
  if (!is_device_ptr(idx_parts) || !is_device_ptr(d2_parts) || !is_device_ptr(idx_out) || !is_device_ptr(dist_out))
    return fail(c, TKNN_EINVAL, "tknn_merge_topk takes device arrays");
  ScopedDevice sd(c->device);
  const size_t smem = (size_t)k * 32 * sizeof(uint64_t);
  TK_CUDA(c, cudaFuncSetAttribute(brute::merge_lists_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  brute::merge_lists_kernel<<<(unsigned)((nq + 31) / 32), 32, smem, c->stream>>>(idx_parts, d2_parts, parts, (uint32_t)nq, k,
                                                                               c->squared, idx_out, dist_out);
  TK_CUDA(c, cudaGetLastError());
  TK_CUDA(c, cudaStreamSynchronize(c->stream));
  return TKNN_OK;
}

int tknn_get_stats(const tknn_ctx* c, tknn_stats* out) {
  if (!c || !out) return TKNN_EINVAL;
  *out = c->stats;
  return TKNN_OK;
}

int tknn_sort_pairs(tknn_ctx* c, uint64_t* keys, uint32_t* values, uint64_t n) {
  TK_TRY(check_ctx(c));
  if (n == 0) return TKNN_OK;
  if (!keys) return fail(c, TKNN_EINVAL, "null array");
  if (n > rsort::MAX_N) return fail(c, TKNN_EINVAL, "n too large");
  ScopedDevice sd(c->device);
  cudaStream_t st = c->stream;
  DevBuf ka, kb, va, vb, tmp;
  ScratchScope scratch({&ka, &kb, &va, &vb, &tmp});
  uint64_t* dk = nullptr;
  uint32_t* dv = nullptr;  // values == nullptr: keys only
  TK_TRY(stage_in(c, keys, n, ka, &dk));
  TK_TRY(stage_in(c, values, n, va, &dv));
  TK_TRY(ensure(c, kb, n * sizeof(uint64_t)));
  if (values) TK_TRY(ensure(c, vb, n * sizeof(uint32_t)));
  TK_TRY(ensure(c, tmp, rsort::temp_words(n) * sizeof(uint32_t)));
  if (values) rsort::sort_pairs(dk, dv, kb.as<uint64_t>(), vb.as<uint32_t>(), n, tmp.as<uint32_t>(), c->sm_count, st);
  else rsort::sort_keys(dk, kb.as<uint64_t>(), n, tmp.as<uint32_t>(), c->sm_count, st, 0, rsort::PASSES);
  TK_CUDA(c, cudaGetLastError());
  TK_TRY(copy_back(c, keys, dk, n));
  TK_TRY(copy_back(c, values, dv, n));
  TK_CUDA(c, cudaStreamSynchronize(st));
  return TKNN_OK;
}

int tknn_get_bvh(const tknn_ctx* c, void* nodes_out, void* points_out, uint32_t* leaf_start_out) {
  if (!c) return TKNN_EINVAL;
  if (c->n == 0) return TKNN_ESTATE;
  ScopedDevice sd(c->device);
  cudaStreamSynchronize(c->stream);
  if (nodes_out && cudaMemcpy(nodes_out, c->nodes.p, (size_t)(c->n_leaves - 1) * sizeof(Node), cudaMemcpyDefault) != cudaSuccess)
    return TKNN_ECUDA;
  if (points_out && cudaMemcpy(points_out, c->pts.p, c->n * sizeof(float4), cudaMemcpyDefault) != cudaSuccess) return TKNN_ECUDA;
  if (leaf_start_out &&
      cudaMemcpy(leaf_start_out, c->leaf_start.p, (size_t)(c->n_leaves + 1) * sizeof(uint32_t), cudaMemcpyDefault) != cudaSuccess)
    return TKNN_ECUDA;
  return TKNN_OK;
}

int tknn_morton_codes(tknn_ctx* c, const float* xyz, uint64_t n, int dim, int stride_floats, const float* box6,
                      uint64_t* codes_out) {
  TK_TRY(check_ctx(c));
  if (n == 0) return TKNN_OK;
  if (!xyz || !box6 || !codes_out) return fail(c, TKNN_EINVAL, "null array");
  if (dim != 2 && dim != 3) return fail(c, TKNN_EINVAL, "dim = %d (must be 2 or 3)", dim);
  if (stride_floats < dim) return fail(c, TKNN_EINVAL, "stride %d < dim %d", stride_floats, dim);
  ScopedDevice sd(c->device);
  cudaStream_t st = c->stream;
  float hbox[6];
  TK_TRY(read_to_host(c, box6, 6, hbox));
  // same order-preserving encoding the builder's bounds kernel produces
  auto enc = [](float f) { uint32_t b; std::memcpy(&b, &f, 4); return (b & 0x80000000u) ? ~b : (b | 0x80000000u); };
  uint32_t ob[8] = {enc(hbox[0]), enc(hbox[1]), enc(hbox[2]), enc(hbox[3]), enc(hbox[4]), enc(hbox[5]), 0u, 0u};
  DevBuf in, keys, vals, dob;
  ScratchScope scratch({&in, &keys, &vals, &dob});
  const float* d_xyz = nullptr;
  uint64_t* d_keys = nullptr;
  TK_TRY(stage_in(c, xyz, (size_t)n * stride_floats, in, &d_xyz));
  TK_TRY(out_view(c, codes_out, n, keys, &d_keys));
  TK_TRY(ensure(c, vals, n * sizeof(uint32_t)));
  TK_TRY(ensure(c, dob, sizeof(ob)));
  TK_CUDA(c, cudaMemcpyAsync(dob.p, ob, sizeof(ob), cudaMemcpyHostToDevice, st));
  lbvh::morton_kernel<<<blocks_for(n, lbvh::THREADS), lbvh::THREADS, 0, st>>>(d_xyz, n, dim, stride_floats, dob.as<uint32_t>(), 21,
                                                                             0, 0, d_keys, vals.as<uint32_t>());
  TK_CUDA(c, cudaGetLastError());
  TK_TRY(copy_back(c, codes_out, d_keys, n));
  TK_CUDA(c, cudaStreamSynchronize(st));
  return TKNN_OK;
}

int tknn_reach_mask(tknn_ctx* c, const float* xyz, uint64_t n, int stride_floats, const float* reach2, const float* box6,
                    const float* summaries, int n_ranks, int cell_bits, int self_rank, uint32_t* mask_out) {
  TK_TRY(check_ctx(c));
  if (n == 0) return TKNN_OK;
  if (!xyz || !reach2 || !box6 || !summaries || !mask_out) return fail(c, TKNN_EINVAL, "null array");
  if (n_ranks < 1 || n_ranks > 32 || cell_bits < 1 || cell_bits > 5 || stride_floats < 3)
    return fail(c, TKNN_EINVAL, "n_ranks in [1,32], cell_bits in [1,5], stride >= 3");
  if (!is_device_ptr(xyz) || !is_device_ptr(reach2) || !is_device_ptr(box6) || !is_device_ptr(summaries) ||
      !is_device_ptr(mask_out))
    return fail(c, TKNN_EINVAL, "tknn_reach_mask takes device arrays");
  ScopedDevice sd(c->device);
  brute::reach_mask_kernel<<<blocks_for(n, 256), 256, 0, c->stream>>>(xyz, n, stride_floats, reach2, box6, summaries, n_ranks,
                                                                     cell_bits, self_rank, mask_out);
  TK_CUDA(c, cudaGetLastError());
  TK_CUDA(c, cudaStreamSynchronize(c->stream));
  return TKNN_OK;
}

int tknn_generate_uniform(tknn_ctx* c, uint64_t seed, uint64_t first, uint64_t n, float* xyz_out) {
  TK_TRY(check_ctx(c));
  if (n == 0) return TKNN_OK;
  if (!xyz_out) return fail(c, TKNN_EINVAL, "null output array");
  ScopedDevice sd(c->device);
  DevBuf tmp;
  ScratchScope scratch({&tmp});
  float* d = nullptr;
  TK_TRY(out_view(c, xyz_out, 3 * n, tmp, &d));
  brute::generate_uniform_kernel<<<blocks_for(3 * n, 256), 256, 0, c->stream>>>(seed, first, n, d);
  cudaError_t e = cudaGetLastError();
  if (e == cudaSuccess && d != xyz_out) e = cudaMemcpyAsync(xyz_out, d, 3 * n * sizeof(float), cudaMemcpyDeviceToHost, c->stream);
  if (e == cudaSuccess) e = cudaStreamSynchronize(c->stream);
  if (e != cudaSuccess) return fail(c, TKNN_ECUDA, "generate_uniform: %s", cudaGetErrorString(e));
  return TKNN_OK;
}

int tknn_measure_bandwidth(tknn_ctx* c, double* l2_gbs, double* hbm_gbs, int* sm_count, uint64_t* l2_bytes) {
  TK_TRY(check_ctx(c));
  ScopedDevice sd(c->device);
  if (sm_count) *sm_count = c->sm_count;
  if (l2_bytes) *l2_bytes = c->l2_bytes;
  cudaStream_t st = c->stream;
  DevBuf buf;
  ScratchScope scratch({&buf});
  const size_t big = (size_t)2 << 30;  // HBM-sized: 2 GiB >> L2
  TK_TRY(ensure(c, buf, big));
  cudaError_t e = cudaMemsetAsync(buf.p, 1, big, st);
  uint32_t* sink = c->scalars.as<uint32_t>() + SC_WORDS - 1;
  const unsigned grid = (unsigned)c->sm_count * 16;
  float ms = 0.f;
  auto run = [&](size_t bytes, int passes, double* out) {
    const uint64_t words = bytes / 16;
    brute::read_probe_kernel<<<grid, 256, 0, st>>>(buf.as<uint4>(), words, 1, sink);  // warm
    double best = 0;
    for (int rep = 0; rep < 5; ++rep) {
      cudaEventRecord(c->ev[0], st);
      brute::read_probe_kernel<<<grid, 256, 0, st>>>(buf.as<uint4>(), words, passes, sink);
      cudaEventRecord(c->ev[1], st);
      cudaEventSynchronize(c->ev[1]);
      cudaEventElapsedTime(&ms, c->ev[0], c->ev[1]);
      const double gbs = (double)bytes * passes / (ms * 1e-3) / 1e9;
      if (gbs > best) best = gbs;
    }
    if (out) *out = best;
  };
  if (e == cudaSuccess) {
    run((size_t)32 << 20, 64, l2_gbs);  // 32 MiB stays L2-resident
    run(big, 1, hbm_gbs);
    e = cudaGetLastError();
  }
  if (e != cudaSuccess) return fail(c, TKNN_ECUDA, "measure_bandwidth: %s", cudaGetErrorString(e));
  return TKNN_OK;
}

// Aggregate shared-memory bandwidth in GB/s of bytes delivered to lanes: conflict-free LDS.128 (the 128 B/clk/SM
// crossbar) and warp-broadcast LDS.128 (the traversal kernel's leaf filter).  Best of 5 runs of ~1 ms each.
int tknn_measure_smem_bandwidth(tknn_ctx* c, double* conflict_free_gbs, double* broadcast_gbs) {
  TK_TRY(check_ctx(c));
  ScopedDevice sd(c->device);
  cudaStream_t st = c->stream;
  uint32_t* sink = c->scalars.as<uint32_t>() + SC_WORDS - 1;
  const unsigned grid = (unsigned)c->sm_count * 8;
  const int iters = 2048;
  for (int mode = 0; mode < 2; ++mode) {
    double best = 0;
    brute::smem_probe_kernel<<<grid, 256, 0, st>>>(64, mode, 264, sink);  // warm
    for (int rep = 0; rep < 5; ++rep) {
      float ms = 0.f;
      TK_CUDA(c, cudaEventRecord(c->ev[0], st));
      brute::smem_probe_kernel<<<grid, 256, 0, st>>>(iters, mode, 264, sink);
      TK_CUDA(c, cudaEventRecord(c->ev[1], st));
      TK_CUDA(c, cudaEventSynchronize(c->ev[1]));
      TK_CUDA(c, cudaEventElapsedTime(&ms, c->ev[0], c->ev[1]));
      const double gbs = (double)grid * 256 * iters * 8 * 16 / (ms * 1e-3) / 1e9;
      if (gbs > best) best = gbs;
    }
    if (mode == 0 && conflict_free_gbs) *conflict_free_gbs = best;
    if (mode == 1 && broadcast_gbs) *broadcast_gbs = best;
  }
  TK_CUDA(c, cudaGetLastError());
  return TKNN_OK;
}

}  // extern "C"

// ---------------------------------------------------------------------------------------------
// voxel-grid clustering and pooling (voxel.cuh, DESIGN.md §3.9)
// ---------------------------------------------------------------------------------------------
namespace {

constexpr double VOXEL_I64 = 9223372036854775808.0;  // 2^63
constexpr uint64_t VOXEL_CS_FLOATS = 1ull << 22;     // chunk results of one pooling pass (16 MB)

inline float voxel_unordered(uint32_t o) { uint32_t b = (o & 0x80000000u) ? (o & 0x7fffffffu) : ~o; float v; std::memcpy(&v, &b, 4); return v; }

inline bool fits_i64(__int128 v) { return v >= -(__int128)VOXEL_I64 && v < (__int128)VOXEL_I64; }

// (int64) q when q lies in int64's range (truncation toward zero), else false
inline bool voxel_trunc(float q, int64_t* t) {
  if (!(q >= -(float)VOXEL_I64 && q < (float)VOXEL_I64)) return false;  // also NaN
  *t = (int64_t)q;
  return true;
}

unsigned voxel_blocks(tknn_ctx* c, uint64_t work) {
  return (unsigned)std::max<uint64_t>(1, std::min<uint64_t>((work + voxel::THREADS - 1) / voxel::THREADS, (uint64_t)c->sm_count * 16));
}

// The chunk layout of the pooling of voxel.cuh over the runs [vox_off[v], vox_off[v + 1]) of `members` entries in all,
// v < *nv_dev <= bound (device words): chunks[v] and their scan chunk_off (bound + 1), the long runs listed in longs,
// and in words[0, 2) the number of long-run chunks (u64), in words[2] the number of long runs.  Launches only: the
// caller reads the words back.
int pool_layout(tknn_ctx* c, const uint64_t* vox_off, const uint32_t* nv_dev, uint64_t bound, uint64_t members,
                DevBuf& chunks, DevBuf& chunk_off, DevBuf& longs, uint32_t* words, int* launches) {
  TK_TRY(ensure(c, chunks, bound * sizeof(uint32_t)));
  TK_TRY(ensure(c, chunk_off, (bound + 1) * sizeof(uint64_t)));
  TK_TRY(ensure(c, longs, (std::min(bound, members / (voxel::LONG_VOXEL + 1)) + 1) * sizeof(uint32_t)));
  TK_CUDA(c, cudaMemsetAsync(words + 2, 0, sizeof(uint32_t), c->stream));
  voxel::long_chunks_kernel<<<blocks_for(bound, voxel::THREADS), voxel::THREADS, 0, c->stream>>>(
      vox_off, nv_dev, bound, chunks.as<uint32_t>(), longs.as<uint32_t>(), words + 2);
  TK_CUDA(c, cudaGetLastError());
  ++*launches;
  return scan_counts(c, chunks.as<uint32_t>(), bound, chunk_off.as<uint64_t>(), reinterpret_cast<uint64_t*>(words),
                     launches);
}

template <int R, bool IDENT>
void launch_pool(tknn_ctx* c, const voxel::PoolParams& P, const uint32_t* longs, uint64_t n_long, int* launches) {
  cudaStream_t st = c->stream;
  if (P.n_chunks) {  // the chunks of a sum and of a mean are the same
    voxel::chunk_kernel<R == voxel::R_MAX ? voxel::R_MAX : voxel::R_MEAN, IDENT>
        <<<voxel_blocks(c, P.n_chunks * P.cb), voxel::THREADS, 0, st>>>(P);
    ++*launches;
  }
  voxel::voxel_kernel<R, IDENT><<<voxel_blocks(c, P.nv * P.cb), voxel::THREADS, 0, st>>>(P);
  ++*launches;
  if (n_long) {
    voxel::fold_kernel<R, IDENT><<<voxel_blocks(c, n_long * P.cb * 32), voxel::THREADS, 0, st>>>(P, longs, n_long);
    ++*launches;
  }
}

// The column passes of the pooling over a layout of pool_layout: P holds x, stride, f, members (nullptr: member j is
// row j), vox_off, chunk_off, nv, n_chunks and out; the columns run in passes so that the chunk results in cs stay
// bounded.  reduce: voxel::R_MEAN / R_MAX / R_SUM.
int pool_columns(tknn_ctx* c, voxel::PoolParams P, int reduce, const uint32_t* longs, uint64_t n_long, DevBuf& cs,
                 int* launches) {
  const uint64_t chunks = P.n_chunks;
  const int f = P.f;
  const int cb = chunks ? (int)std::min<uint64_t>((uint64_t)f, std::max<uint64_t>(1, VOXEL_CS_FLOATS / chunks)) : f;
  if (chunks) TK_TRY(ensure(c, cs, chunks * (uint64_t)cb * sizeof(float)));
  P.cs = cs.as<float>();
  const bool ident = P.members == nullptr;
  for (int c0 = 0; c0 < f; c0 += cb) {
    P.c0 = c0;
    P.cb = std::min(cb, f - c0);
    if (reduce == voxel::R_MAX) launch_pool<voxel::R_MAX, false>(c, P, longs, n_long, launches);
    else if (reduce == voxel::R_MEAN && !ident) launch_pool<voxel::R_MEAN, false>(c, P, longs, n_long, launches);
    else if (reduce == voxel::R_MEAN) launch_pool<voxel::R_MEAN, true>(c, P, longs, n_long, launches);
    else if (!ident) launch_pool<voxel::R_SUM, false>(c, P, longs, n_long, launches);
    else launch_pool<voxel::R_SUM, true>(c, P, longs, n_long, launches);
    TK_CUDA(c, cudaGetLastError());
  }
  return TKNN_OK;
}

}  // namespace

extern "C" {

int tknn_voxel_grid(tknn_ctx* c, const float* points, uint64_t n, int dim, int stride_floats, const uint64_t* seg_offsets,
                    uint64_t n_segments, const float* size, const float* start, const float* end, int64_t* raw_out,
                    int32_t* cluster_out, uint64_t* n_voxels_out) {
  TK_TRY(check_ctx(c));
  const char* what = "tknn_voxel_grid";
  if (!size || !n_voxels_out || (!points && n)) return fail(c, TKNN_EINVAL, "%s: null points, size or n_voxels_out", what);
  if (dim != 2 && dim != 3) return fail(c, TKNN_EINVAL, "%s: dim = %d (must be 2 or 3)", what, dim);
  if (stride_floats < dim) return fail(c, TKNN_EINVAL, "%s: stride %d below dim = %d", what, stride_floats, dim);
  if (n > rsort::MAX_N) return fail(c, TKNN_EINVAL, "%s: n = %llu exceeds %llu", what, (unsigned long long)n, (unsigned long long)rsort::MAX_N);
  if (!seg_offsets && n_segments != 1)
    return fail(c, TKNN_EINVAL, "%s: n_segments = %llu without offsets (must be 1)", what, (unsigned long long)n_segments);
  if (n_segments < 1 || n_segments >= (1ull << 24))
    return fail(c, TKNN_EINVAL, "%s: n_segments = %llu outside [1, 2^24 - 1]", what, (unsigned long long)n_segments);
  for (int d = 0; d < dim; ++d) {
    if (!std::isfinite(size[d]) || !(size[d] > 0.f)) return fail(c, TKNN_EINVAL, "%s: size[%d] = %g must be finite and > 0", what, d, size[d]);
    if ((start && !std::isfinite(start[d])) || (end && !std::isfinite(end[d])))
      return fail(c, TKNN_EINVAL, "%s: non-finite start or end in column %d", what, d);
  }
  ScopedDevice sd(c->device);
  cudaStream_t st = c->stream;
  std::vector<uint64_t> off{0, n};
  if (seg_offsets) TK_TRY(read_offsets(c, what, "segment", seg_offsets, n_segments, n, "n", &off));
  c->vx_valid = false;  // the previous clustering is gone whatever happens below
  c->vx_n = c->vx_nv = c->vx_long_chunks = c->vx_n_long = 0;
  if (n == 0) {
    c->vx_valid = true;
    *n_voxels_out = 0;
    return TKNN_OK;
  }
  const bool batched = seg_offsets != nullptr;
  const float* d_pts = nullptr;
  TK_TRY(stage_in(c, points, (size_t)(n - 1) * stride_floats + dim, c->vx_pts, &d_pts));
  if (batched) {
    TK_TRY(ensure(c, c->vx_seg_off, off.size() * sizeof(uint64_t)));
    TK_CUDA(c, cudaMemcpyAsync(c->vx_seg_off.p, off.data(), off.size() * sizeof(uint64_t), cudaMemcpyHostToDevice, st));
  }

  // 1. exact column box and the non-finite flag
  TK_TRY(ensure(c, c->vx_words_sc, 16 * sizeof(uint32_t)));
  uint32_t* w = c->vx_words_sc.as<uint32_t>();  // [0, 4) min, [4, 8) max, 8 flag, [10, 12) long chunks (u64), 12 long voxels
  TK_CUDA(c, cudaMemsetAsync(w, 0xff, 4 * sizeof(uint32_t), st));
  TK_CUDA(c, cudaMemsetAsync(w + 4, 0, 12 * sizeof(uint32_t), st));
  voxel::box_kernel<<<voxel_blocks(c, n), voxel::THREADS, 0, st>>>(d_pts, n, dim, stride_floats, w, w + 8);
  TK_CUDA(c, cudaGetLastError());
  uint32_t box[9];
  TK_TRY(fetch_words(c, w, 9, nullptr, 0, box));
  if (box[8]) return fail(c, TKNN_EINVAL, "%s: non-finite coordinate", what);

  // 2. per column start / size / multiplier and the bound [lo, hi] of every raw id (the ids of the box's corners)
  voxel::RawParams P{};
  P.p = d_pts;
  P.n = n;
  P.dim = dim;
  P.stride = stride_floats;
  P.seg_off = batched ? c->vx_seg_off.as<uint64_t>() : nullptr;
  P.n_seg = (uint32_t)n_segments;
  uint64_t s_first = 0, s_last = 0;
  if (batched) {
    while (off[s_first + 1] == 0) ++s_first;
    s_last = n_segments - 1;
    while (off[s_last] == n) --s_last;
  }
  const int cols = dim + (batched ? 1 : 0);
  __int128 m = 1, lo = 0, hi = 0;
  for (int d = 0; d < cols; ++d) {
    const bool id = d == dim;
    const float mn = id ? (float)s_first : voxel_unordered(box[d]), mx = id ? (float)s_last : voxel_unordered(box[4 + d]);
    const float s0 = id ? (start ? 0.f : mn) : (start ? start[d] : mn);
    const float e0 = id ? mx : (end ? end[d] : mx);
    const float sz = id ? 1.f : size[d];
    int64_t cnt, tlo, thi;
    const float span = e0 - s0;  // IEEE single: the host evaluates the formula as the device does
    if (!voxel_trunc(span / sz, &cnt)) return fail(c, TKNN_EINVAL, "%s: the cell count of column %d overflows int64", what, d);
    const float qlo = (mn - s0) / sz, qhi = (mx - s0) / sz;
    if (!voxel_trunc(qlo, &tlo) || !voxel_trunc(qhi, &thi))
      return fail(c, TKNN_EINVAL, "%s: a cell index of column %d overflows int64 (points far outside [start, end])", what, d);
    const __int128 a = (__int128)tlo * m, b = (__int128)thi * m;
    lo += std::min(a, b);
    hi += std::max(a, b);
    if (!fits_i64(a) || !fits_i64(b) || !fits_i64(lo) || !fits_i64(hi))
      return fail(c, TKNN_EINVAL, "%s: a raw voxel id overflows int64 (points far outside [start, end])", what);
    P.start[d] = s0;
    P.size[d] = sz;
    P.mult[d] = (long long)m;
    m *= (__int128)cnt + 1;
    if (!fits_i64(m)) return fail(c, TKNN_EINVAL, "%s: the product of the cell counts overflows int64", what);
  }
  P.lo = (long long)lo;
  const uint64_t range = (uint64_t)(int64_t)hi - (uint64_t)(int64_t)lo;
  const int bits = range ? 64 - __builtin_clzll(range) : 0;
  const bool packed = bits + voxel::IDX_BITS <= 64;
  const int passes = (bits + 7) / 8;

  // 3. raw ids and sort keys, the sort
  TK_TRY(ensure(c, c->vx_raw, n * sizeof(int64_t)));
  TK_TRY(ensure(c, c->vx_keys_a, n * sizeof(uint64_t)));
  TK_TRY(ensure(c, c->vx_keys_b, n * sizeof(uint64_t)));
  if (!packed) {
    TK_TRY(ensure(c, c->vx_vals_a, n * sizeof(uint32_t)));
    TK_TRY(ensure(c, c->vx_vals_b, n * sizeof(uint32_t)));
  }
  TK_TRY(ensure(c, c->vx_sort_tmp, rsort::temp_words(n) * sizeof(uint32_t)));
  P.packed = packed;
  P.raw = c->vx_raw.as<long long>();
  P.keys = c->vx_keys_a.as<uint64_t>();
  P.vals = packed ? nullptr : c->vx_vals_a.as<uint32_t>();
  voxel::raw_kernel<<<blocks_for(n, voxel::THREADS), voxel::THREADS, 0, st>>>(P);
  TK_CUDA(c, cudaGetLastError());
  int launches = 0;
  bool in_b = false;
  if (passes > 0) {
    if (packed)
      launches += rsort::sort_keys(c->vx_keys_a.as<uint64_t>(), c->vx_keys_b.as<uint64_t>(), n, c->vx_sort_tmp.as<uint32_t>(),
                                   c->sm_count, st, voxel::IDX_BITS, passes, &in_b);
    else
      launches += rsort::sort_pairs(c->vx_keys_a.as<uint64_t>(), c->vx_vals_a.as<uint32_t>(), c->vx_keys_b.as<uint64_t>(),
                                    c->vx_vals_b.as<uint32_t>(), n, c->vx_sort_tmp.as<uint32_t>(), c->sm_count, st, passes,
                                    &in_b);
    TK_CUDA(c, cudaGetLastError());
  }
  const uint64_t* keys = in_b ? c->vx_keys_b.as<uint64_t>() : c->vx_keys_a.as<uint64_t>();
  const uint32_t* vals = packed ? nullptr : (in_b ? c->vx_vals_b.as<uint32_t>() : c->vx_vals_a.as<uint32_t>());

  // 4. heads, their ranks, labels, long-voxel chunk layout
  const uint64_t nw = (n + 31) / 32;
  TK_TRY(ensure(c, c->vx_words, nw * sizeof(uint32_t)));
  TK_TRY(ensure(c, c->vx_word_off, nw * sizeof(uint32_t)));
  TK_TRY(ensure(c, c->vx_members, n * sizeof(uint32_t)));
  TK_TRY(ensure(c, c->vx_cluster, n * sizeof(int32_t)));
  TK_TRY(ensure(c, c->vx_off, (n + 1) * sizeof(uint64_t)));
  TK_TRY(ensure(c, c->vx_first, n * sizeof(int32_t)));
  TK_TRY(ensure(c, c->vx_seg, n * sizeof(int32_t)));
  voxel::heads_kernel<<<blocks_for(n, voxel::THREADS), voxel::THREADS, 0, st>>>(keys, n, packed ? voxel::IDX_BITS : 0,
                                                                                 c->vx_words.as<uint32_t>());
  TK_CUDA(c, cudaGetLastError());
  TK_TRY(popc_scan(c, c->vx_words.as<uint32_t>(), nw, c->vx_word_off.as<uint32_t>(), &launches));  // nv -> sc[SC_TOTAL]
  voxel::LabelParams Lp{keys, vals, n, c->vx_words.as<uint32_t>(), c->vx_word_off.as<uint32_t>(), P.seg_off, P.n_seg,
                        c->vx_members.as<uint32_t>(), c->vx_cluster.as<int32_t>(), c->vx_off.as<uint64_t>(),
                        c->vx_first.as<int32_t>(), c->vx_seg.as<int32_t>()};
  voxel::label_kernel<<<blocks_for(n, voxel::THREADS), voxel::THREADS, 0, st>>>(Lp);
  uint32_t* sc = c->scalars.as<uint32_t>();
  TK_TRY(pool_layout(c, c->vx_off.as<uint64_t>(), sc + SC_TOTAL, n, n, c->vx_chunks, c->vx_chunk_off, c->vx_longs, w + 10,
                     &launches));
  if (raw_out) TK_CUDA(c, cudaMemcpyAsync(raw_out, c->vx_raw.p, n * sizeof(int64_t), cudaMemcpyDefault, st));
  if (cluster_out) TK_CUDA(c, cudaMemcpyAsync(cluster_out, c->vx_cluster.p, n * sizeof(int32_t), cudaMemcpyDefault, st));
  uint32_t h[4];
  TK_TRY(fetch_words(c, w + 10, 3, sc + SC_TOTAL, 1, h));  // synchronises the stream
  c->vx_long_chunks = (uint64_t)h[0] | ((uint64_t)h[1] << 32);
  c->vx_n_long = h[2];
  c->vx_nv = h[3];
  c->vx_n = n;
  c->vx_valid = true;
  *n_voxels_out = c->vx_nv;
  return TKNN_OK;
}

int tknn_voxel_members(tknn_ctx* c, uint64_t* offsets_out, int32_t* members_out, int32_t* first_out, int32_t* seg_out) {
  TK_TRY(check_ctx(c));
  if (!c->vx_valid) return fail(c, TKNN_ESTATE, "tknn_voxel_members before tknn_voxel_grid");
  ScopedDevice sd(c->device);
  cudaStream_t st = c->stream;
  const uint64_t n = c->vx_n, nv = c->vx_nv;
  const uint64_t zero = 0;
  if (offsets_out)
    TK_CUDA(c, cudaMemcpyAsync(offsets_out, n ? c->vx_off.p : (const void*)&zero, (nv + 1) * sizeof(uint64_t), cudaMemcpyDefault, st));
  if (n) {
    if (members_out) TK_CUDA(c, cudaMemcpyAsync(members_out, c->vx_members.p, n * sizeof(int32_t), cudaMemcpyDefault, st));
    if (first_out) TK_CUDA(c, cudaMemcpyAsync(first_out, c->vx_first.p, nv * sizeof(int32_t), cudaMemcpyDefault, st));
    if (seg_out) TK_CUDA(c, cudaMemcpyAsync(seg_out, c->vx_seg.p, nv * sizeof(int32_t), cudaMemcpyDefault, st));
  }
  TK_CUDA(c, cudaStreamSynchronize(st));
  return TKNN_OK;
}

int tknn_voxel_pool(tknn_ctx* c, const float* x, uint64_t n, int f, int stride_floats, int reduce, float* out) {
  TK_TRY(check_ctx(c));
  const char* what = "tknn_voxel_pool";
  if (!c->vx_valid) return fail(c, TKNN_ESTATE, "%s before tknn_voxel_grid", what);
  if (n != c->vx_n)
    return fail(c, TKNN_EINVAL, "%s: n = %llu, the clustering has %llu points", what, (unsigned long long)n, (unsigned long long)c->vx_n);
  if (f < 1 || f > 1024) return fail(c, TKNN_EINVAL, "%s: f = %d outside [1, 1024]", what, f);
  if (stride_floats < f) return fail(c, TKNN_EINVAL, "%s: stride %d below f = %d", what, stride_floats, f);
  if (reduce != TKNN_REDUCE_MEAN && reduce != TKNN_REDUCE_MAX) return fail(c, TKNN_EINVAL, "%s: unknown reduce %d", what, reduce);
  const uint64_t nv = c->vx_nv;
  if (nv == 0) return TKNN_OK;
  if (!x || !out) return fail(c, TKNN_EINVAL, "%s: null x or out", what);
  ScopedDevice sd(c->device);
  cudaStream_t st = c->stream;
  const float* d_x = nullptr;
  float* d_out = nullptr;
  TK_TRY(stage_in(c, x, (size_t)(n - 1) * stride_floats + f, c->vx_x, &d_x));
  TK_TRY(out_view(c, out, nv * (size_t)f, c->vx_out, &d_out));
  uint32_t* w = c->vx_words_sc.as<uint32_t>();
  const bool mx = reduce == TKNN_REDUCE_MAX;
  if (mx) {
    TK_CUDA(c, cudaMemsetAsync(w + 8, 0, sizeof(uint32_t), st));
    feat::finite_kernel<<<voxel_blocks(c, n * (uint64_t)f), 256, 0, st>>>(d_x, n, f, stride_floats, w + 8);
    TK_CUDA(c, cudaGetLastError());
  }
  voxel::PoolParams P{d_x, stride_floats, f, 0, f, c->vx_members.as<uint32_t>(), c->vx_off.as<uint64_t>(),
                      c->vx_chunk_off.as<uint64_t>(), nv, c->vx_long_chunks, nullptr, d_out};
  int launches = 0;
  TK_TRY(pool_columns(c, P, mx ? voxel::R_MAX : voxel::R_MEAN, c->vx_longs.as<uint32_t>(), c->vx_n_long, c->vx_cs,
                      &launches));
  TK_TRY(copy_back(c, out, d_out, nv * (size_t)f));
  if (mx) {
    uint32_t bad = 0;
    TK_TRY(fetch_words(c, w + 8, 1, nullptr, 0, &bad));
    if (bad) return fail(c, TKNN_EINVAL, "%s: non-finite value in the first %d columns of x", what, f);
  } else {
    TK_CUDA(c, cudaStreamSynchronize(st));
  }
  return TKNN_OK;
}

}  // extern "C"

// ---------------------------------------------------------------------------------------------
// k-NN interpolation and its backward pass (interpolate.cuh, DESIGN.md §3.10)
// ---------------------------------------------------------------------------------------------
namespace {

unsigned interp_blocks(tknn_ctx* c, uint64_t threads) {
  return (unsigned)std::max<uint64_t>(1, std::min<uint64_t>((threads + interp::THREADS - 1) / interp::THREADS,
                                                            (uint64_t)c->sm_count * 16));
}

int interpolate_core(tknn_ctx* c, const int32_t* idx, const float* d2, uint64_t nq, int k, const float* x, uint64_t n,
                     int f, int x_stride, float* out, float* weight_out, float* den_out) {
  const char* what = "tknn_interpolate";
  cudaStream_t st = c->stream;
  const size_t slots = (size_t)nq * k;
  ScratchScope scratch = interp_scratch(c);
  const int32_t* d_idx = nullptr;
  const float *d_d2 = nullptr, *d_x = nullptr;
  TK_TRY(stage_in(c, idx, slots, c->ip_idx, &d_idx));
  TK_TRY(stage_in(c, d2, slots, c->ip_w, &d_d2));
  if (n) TK_TRY(stage_in(c, x, (size_t)(n - 1) * x_stride + f, c->ip_x, &d_x));
  float *d_out = nullptr, *d_w = nullptr, *d_den = nullptr;
  TK_TRY(out_view(c, out, (size_t)nq * f, c->ip_out, &d_out));
  TK_TRY(out_view(c, weight_out, slots, c->ip_wout, &d_w));
  TK_TRY(out_view(c, den_out, nq, c->ip_dout, &d_den));
  TK_TRY(ensure_round_events(c, 4));
  cudaEvent_t* ev = c->round_ev.data();
  uint32_t* sc = c->scalars.as<uint32_t>();
  TK_CUDA(c, cudaEventRecord(c->ev[0], st));
  TK_CUDA(c, cudaEventRecord(ev[0], st));
  TK_CUDA(c, cudaMemsetAsync(sc + SC_QBAD, 0, sizeof(uint32_t), st));
  interp::FwdParams P{d_idx, d_d2, d_x, nq, (uint32_t)n, k, f, x_stride, d_out, d_w, d_den, sc + SC_QBAD};
  const int G = interp::group_of(f);
  const unsigned blocks = interp_blocks(c, nq * (uint64_t)G);
  TK_CUDA(c, cudaEventRecord(ev[2], st));
  switch (G) {
    case 4: interp::forward_kernel<4><<<blocks, interp::THREADS, 0, st>>>(P); break;
    case 8: interp::forward_kernel<8><<<blocks, interp::THREADS, 0, st>>>(P); break;
    case 16: interp::forward_kernel<16><<<blocks, interp::THREADS, 0, st>>>(P); break;
    default: interp::forward_kernel<32><<<blocks, interp::THREADS, 0, st>>>(P); break;
  }
  TK_CUDA(c, cudaGetLastError());
  TK_CUDA(c, cudaEventRecord(ev[3], st));
  TK_CUDA(c, cudaEventRecord(ev[1], st));
  TK_CUDA(c, cudaEventRecord(c->ev[2], st));
  TK_TRY(copy_back(c, out, d_out, (size_t)nq * f));
  TK_TRY(copy_back(c, weight_out, d_w, slots));
  TK_TRY(copy_back(c, den_out, d_den, nq));
  TK_CUDA(c, cudaEventRecord(c->ev[3], st));
  uint32_t bad = 0;
  TK_TRY(fetch_words(c, sc + SC_QBAD, 1, nullptr, 0, &bad));  // synchronises the stream
  TK_CUDA(c, cudaEventElapsedTime(&c->stats.search_ms, c->ev[0], c->ev[2]));
  TK_CUDA(c, cudaEventElapsedTime(&c->stats.d2h_ms, c->ev[2], c->ev[3]));
  c->stats.rounds = 1;
  c->stats.round_queries[0] = nq;
  c->stats.kernel_launches = 1 + (c->mailbox_h ? 1 : 0);
  TK_TRY(finish_round_stats(c));
  if (bad) return fail(c, TKNN_EINVAL, "%s: an idx entry lies outside {-1} and [0, n = %llu)", what, (unsigned long long)n);
  return TKNN_OK;
}

int interpolate_backward_core(tknn_ctx* c, const int32_t* idx, const float* weight, const float* den, uint64_t nq, int k,
                              const float* grad_out, int g_stride, uint64_t n, int f, float* grad_x) {
  const char* what = "tknn_interpolate_backward";
  cudaStream_t st = c->stream;
  const uint64_t edges = nq * (uint64_t)k;
  ScratchScope scratch = interp_scratch(c);
  const int32_t* d_idx = nullptr;
  const float *d_w = nullptr, *d_den = nullptr, *d_g = nullptr;
  TK_TRY(stage_in(c, idx, edges, c->ip_idx, &d_idx));
  TK_TRY(stage_in(c, weight, edges, c->ip_w, &d_w));
  TK_TRY(stage_in(c, den, nq, c->ip_den, &d_den));
  TK_TRY(stage_in(c, grad_out, (size_t)(nq - 1) * g_stride + f, c->ip_x, &d_g));
  float* d_gx = nullptr;
  if (n) TK_TRY(out_view(c, grad_x, (size_t)n * f, c->ip_out, &d_gx));
  TK_TRY(ensure(c, c->ip_keys_a, edges * sizeof(uint64_t)));
  TK_TRY(ensure(c, c->ip_keys_b, edges * sizeof(uint64_t)));
  TK_TRY(ensure(c, c->ip_vals_a, edges * sizeof(uint32_t)));
  TK_TRY(ensure(c, c->ip_vals_b, edges * sizeof(uint32_t)));
  TK_TRY(ensure(c, c->ip_sort_tmp, rsort::temp_words(edges) * sizeof(uint32_t)));
  TK_TRY(ensure(c, c->ip_cnt, n * sizeof(uint32_t)));
  TK_TRY(ensure(c, c->ip_off, (n + 1) * sizeof(uint64_t)));
  TK_TRY(ensure_round_events(c, 12));
  cudaEvent_t* ev = c->round_ev.data();  // phase r: [4r] start, [4r + 1] end, [4r + 2 / + 3] its kernels
  uint32_t* sc = c->scalars.as<uint32_t>();
  int launches = 0;
  TK_CUDA(c, cudaEventRecord(c->ev[0], st));

  // 1. edge keys and per-row counts
  TK_CUDA(c, cudaEventRecord(ev[0], st));
  TK_CUDA(c, cudaMemsetAsync(sc + SC_QBAD, 0, sizeof(uint32_t), st));
  if (n) TK_CUDA(c, cudaMemsetAsync(c->ip_cnt.p, 0, n * sizeof(uint32_t), st));
  TK_CUDA(c, cudaEventRecord(ev[2], st));
  interp::edge_kernel<<<interp_blocks(c, edges), interp::THREADS, 0, st>>>(
      d_idx, edges, (uint32_t)n, c->ip_keys_a.as<uint64_t>(), c->ip_vals_a.as<uint32_t>(),
      c->ip_cnt.as<uint32_t>(), sc + SC_QBAD);
  TK_CUDA(c, cudaGetLastError());
  ++launches;
  TK_CUDA(c, cudaEventRecord(ev[3], st));
  TK_CUDA(c, cudaEventRecord(ev[1], st));

  // 2. stable sort of the edges by data row: keys 0 .. n need bits(n) bits
  const int passes = n ? (64 - __builtin_clzll(n) + 7) / 8 : 0;
  bool in_b = false;
  TK_CUDA(c, cudaEventRecord(ev[4], st));
  TK_CUDA(c, cudaEventRecord(ev[6], st));
  if (passes > 0) {
    launches += rsort::sort_pairs(c->ip_keys_a.as<uint64_t>(), c->ip_vals_a.as<uint32_t>(), c->ip_keys_b.as<uint64_t>(),
                                  c->ip_vals_b.as<uint32_t>(), edges, c->ip_sort_tmp.as<uint32_t>(), c->sm_count, st, passes,
                                  &in_b);
    TK_CUDA(c, cudaGetLastError());
  }
  TK_CUDA(c, cudaEventRecord(ev[7], st));
  TK_CUDA(c, cudaEventRecord(ev[5], st));

  // 3. run offsets, 4. column sums in edge order
  TK_CUDA(c, cudaEventRecord(ev[8], st));
  if (n) {
    uint64_t* off = c->ip_off.as<uint64_t>();
    TK_TRY(scan_counts(c, c->ip_cnt.as<uint32_t>(), n, off, off + n, &launches));
    const int G = interp::group_of(f);
    interp::BwdParams P{in_b ? c->ip_vals_b.as<uint32_t>() : c->ip_vals_a.as<uint32_t>(), off, d_w, d_den, d_g,
                        (uint32_t)n, k, f, g_stride, (f + G - 1) / G, d_gx};
    const unsigned blocks = interp_blocks(c, n * (uint64_t)P.blocks * G);
    TK_CUDA(c, cudaEventRecord(ev[10], st));
    switch (G) {
      case 4: interp::colsum_kernel<4><<<blocks, interp::THREADS, 0, st>>>(P); break;
      case 8: interp::colsum_kernel<8><<<blocks, interp::THREADS, 0, st>>>(P); break;
      case 16: interp::colsum_kernel<16><<<blocks, interp::THREADS, 0, st>>>(P); break;
      default: interp::colsum_kernel<32><<<blocks, interp::THREADS, 0, st>>>(P); break;
    }
    TK_CUDA(c, cudaGetLastError());
    ++launches;
    TK_CUDA(c, cudaEventRecord(ev[11], st));
  } else {
    TK_CUDA(c, cudaEventRecord(ev[10], st));
    TK_CUDA(c, cudaEventRecord(ev[11], st));
  }
  TK_CUDA(c, cudaEventRecord(ev[9], st));
  TK_CUDA(c, cudaEventRecord(c->ev[2], st));
  if (n) TK_TRY(copy_back(c, grad_x, d_gx, (size_t)n * f));
  TK_CUDA(c, cudaEventRecord(c->ev[3], st));
  uint32_t bad = 0;
  TK_TRY(fetch_words(c, sc + SC_QBAD, 1, nullptr, 0, &bad));  // synchronises the stream
  TK_CUDA(c, cudaEventElapsedTime(&c->stats.search_ms, c->ev[0], c->ev[2]));
  TK_CUDA(c, cudaEventElapsedTime(&c->stats.d2h_ms, c->ev[2], c->ev[3]));
  c->stats.rounds = 3;
  c->stats.round_queries[0] = nq;
  c->stats.round_queries[1] = edges;
  c->stats.round_queries[2] = n;
  c->stats.kernel_launches = (uint32_t)(launches + (c->mailbox_h ? 1 : 0));
  TK_TRY(finish_round_stats(c));
  if (bad) return fail(c, TKNN_EINVAL, "%s: an idx entry lies outside {-1} and [0, n = %llu)", what, (unsigned long long)n);
  return TKNN_OK;
}

int interp_args(tknn_ctx* c, const char* what, uint64_t nq, int k, uint64_t n, int f, int stride, const char* stride_name) {
  if (k < 1 || k > TKNN_MAX_K) return fail(c, TKNN_EINVAL, "%s: k = %d outside [1, %d]", what, k, TKNN_MAX_K);
  if (f < 1) return fail(c, TKNN_EINVAL, "%s: f = %d below 1", what, f);
  if (stride < f) return fail(c, TKNN_EINVAL, "%s: %s = %d below f = %d", what, stride_name, stride, f);
  if (n >= (1ull << 31) || nq >= (1ull << 31)) return fail(c, TKNN_EINVAL, "%s: n and nq must be below 2^31", what);
  return TKNN_OK;
}

}  // namespace

extern "C" {

int tknn_interpolate(tknn_ctx* c, const int32_t* idx, const float* d2, uint64_t nq, int k, const float* x, uint64_t n,
                     int f, int x_stride_floats, float* out, float* weight_out, float* den_out) {
  TK_TRY(check_ctx(c));
  const char* what = "tknn_interpolate";
  TK_TRY(interp_args(c, what, nq, k, n, f, x_stride_floats, "x_stride_floats"));
  if (nq > 0 && (!idx || !d2 || !out || (n > 0 && !x)))
    return fail(c, TKNN_EINVAL, "%s: null idx, d2, x or out", what);
  ScopedDevice sd(c->device);
  reset_search_stats(c);
  c->stats.n_queries = nq;
  c->stats.k = k;
  if (nq == 0) return TKNN_OK;
  return interpolate_core(c, idx, d2, nq, k, x, n, f, x_stride_floats, out, weight_out, den_out);
}

int tknn_interpolate_backward(tknn_ctx* c, const int32_t* idx, const float* weight, const float* den, uint64_t nq, int k,
                              const float* grad_out, int g_stride_floats, uint64_t n, int f, float* grad_x) {
  TK_TRY(check_ctx(c));
  const char* what = "tknn_interpolate_backward";
  TK_TRY(interp_args(c, what, nq, k, n, f, g_stride_floats, "g_stride_floats"));
  if (nq * (uint64_t)k > rsort::MAX_N)
    return fail(c, TKNN_EINVAL, "%s: nq * k = %llu edges exceed the sort's %llu", what,
                (unsigned long long)(nq * (uint64_t)k), (unsigned long long)rsort::MAX_N);
  if (nq > 0 && (!idx || !weight || !den || !grad_out || (n > 0 && !grad_x)))
    return fail(c, TKNN_EINVAL, "%s: null idx, weight, den, grad_out or grad_x", what);
  ScopedDevice sd(c->device);
  reset_search_stats(c);
  c->stats.n_queries = nq;
  c->stats.k = k;
  if (nq == 0) {  // no edge: every row of grad_x is +0
    if (n && grad_x) TK_TRY(zero_fill(c, grad_x, (size_t)n * f));
    return TKNN_OK;
  }
  return interpolate_backward_core(c, idx, weight, den, nq, k, grad_out, g_stride_floats, n, f, grad_x);
}

}  // extern "C"

// ---------------------------------------------------------------------------------------------
// gradients of kNN squared distances and segment reductions (knn_grad.cuh, voxel.cuh's pooling, DESIGN.md §3.11)
// ---------------------------------------------------------------------------------------------
namespace {

unsigned kgrad_blocks(tknn_ctx* c, uint64_t threads) {
  return (unsigned)std::max<uint64_t>(1, std::min<uint64_t>((threads + kgrad::THREADS - 1) / kgrad::THREADS,
                                                            (uint64_t)c->sm_count * 16));
}

// Uploads nv (< 2^32) to words[3] and lays out the chunks of the nv runs of vox_off (pool_layout); returns the chunk
// totals through *long_chunks / *n_long.  `extra` (device word or nullptr) is read back in the same transfer.
int kgrad_layout(tknn_ctx* c, const uint64_t* vox_off, uint64_t nv, uint64_t members, const uint32_t* extra,
                 uint64_t* long_chunks, uint64_t* n_long, uint32_t* extra_out, int* launches) {
  TK_TRY(ensure(c, c->kg_words, 4 * sizeof(uint32_t)));
  uint32_t* w = c->kg_words.as<uint32_t>();  // [0, 2) long-run chunks (u64), 2 long runs, 3 nv
  const uint32_t nv32 = (uint32_t)nv;
  TK_CUDA(c, cudaMemcpyAsync(w + 3, &nv32, sizeof(uint32_t), cudaMemcpyHostToDevice, c->stream));
  TK_TRY(pool_layout(c, vox_off, w + 3, nv, members, c->kg_chunks, c->kg_chunk_off, c->kg_longs, w, launches));
  uint32_t h[4] = {0, 0, 0, 0};
  TK_TRY(fetch_words(c, w, 3, extra, extra ? 1 : 0, h));  // synchronises the stream
  *long_chunks = (uint64_t)h[0] | ((uint64_t)h[1] << 32);
  *n_long = h[2];
  if (extra_out) *extra_out = h[3];
  return TKNN_OK;
}

template <int D>
void launch_terms(tknn_ctx* c, const kgrad::Params& P) {
  kgrad::terms_kernel<D><<<kgrad_blocks(c, P.nq), kgrad::THREADS, 0, c->stream>>>(P);
}

int knn_backward_core(tknn_ctx* c, const float* queries, uint64_t nq, int q_stride, const float* points, uint64_t n,
                      int p_stride, int dim, const int32_t* idx, int k, const float* grad_d2, float* grad_q,
                      float* grad_p) {
  const char* what = "tknn_knn_backward";
  cudaStream_t st = c->stream;
  const uint64_t edges = nq * (uint64_t)k;
  const bool want_p = grad_p && n > 0;
  ScratchScope scratch = knn_grad_scratch(c);
  const float *d_q = nullptr, *d_p = nullptr, *d_g = nullptr;
  const int32_t* d_idx = nullptr;
  TK_TRY(stage_in(c, queries, (size_t)(nq - 1) * q_stride + dim, c->kg_q, &d_q));
  if (n) TK_TRY(stage_in(c, points, (size_t)(n - 1) * p_stride + dim, c->kg_p, &d_p));
  TK_TRY(stage_in(c, idx, edges, c->kg_idx, &d_idx));
  TK_TRY(stage_in(c, grad_d2, edges, c->kg_g, &d_g));
  float *d_gq = nullptr, *d_gp = nullptr;
  TK_TRY(out_view(c, grad_q, (size_t)nq * dim, c->kg_gq, &d_gq));
  if (want_p) {
    TK_TRY(out_view(c, grad_p, (size_t)n * dim, c->kg_gp, &d_gp));
    TK_TRY(ensure(c, c->kg_terms, edges * dim * sizeof(float)));
    TK_TRY(ensure(c, c->kg_keys_a, edges * sizeof(uint64_t)));
    TK_TRY(ensure(c, c->kg_keys_b, edges * sizeof(uint64_t)));
    TK_TRY(ensure(c, c->kg_vals_a, edges * sizeof(uint32_t)));
    TK_TRY(ensure(c, c->kg_vals_b, edges * sizeof(uint32_t)));
    TK_TRY(ensure(c, c->kg_sort_tmp, rsort::temp_words(edges) * sizeof(uint32_t)));
    TK_TRY(ensure(c, c->kg_cnt, n * sizeof(uint32_t)));
    TK_TRY(ensure(c, c->kg_off, (n + 1) * sizeof(uint64_t)));
  }
  TK_TRY(ensure_round_events(c, 12));
  cudaEvent_t* ev = c->round_ev.data();  // phase r: [4r] start, [4r + 1] end, [4r + 2 / + 3] its kernels
  uint32_t* sc = c->scalars.as<uint32_t>();
  int launches = 0;
  TK_CUDA(c, cudaEventRecord(c->ev[0], st));

  // 1. terms and grad_q; edge keys and per-row counts
  TK_CUDA(c, cudaEventRecord(ev[0], st));
  TK_CUDA(c, cudaMemsetAsync(sc + SC_QBAD, 0, sizeof(uint32_t), st));
  if (want_p) TK_CUDA(c, cudaMemsetAsync(c->kg_cnt.p, 0, n * sizeof(uint32_t), st));
  TK_CUDA(c, cudaEventRecord(ev[2], st));
  const kgrad::Params P{d_q, d_p, d_idx, d_g, nq, (uint32_t)n, k, q_stride, p_stride, d_gq,
                        want_p ? c->kg_terms.as<float>() : nullptr, sc + SC_QBAD};
  if (dim == 2) launch_terms<2>(c, P);
  else launch_terms<3>(c, P);
  TK_CUDA(c, cudaGetLastError());
  ++launches;
  if (want_p) {
    interp::edge_kernel<<<interp_blocks(c, edges), interp::THREADS, 0, st>>>(
        d_idx, edges, (uint32_t)n, c->kg_keys_a.as<uint64_t>(), c->kg_vals_a.as<uint32_t>(), c->kg_cnt.as<uint32_t>(),
        sc + SC_QBAD);
    TK_CUDA(c, cudaGetLastError());
    ++launches;
  }
  TK_CUDA(c, cudaEventRecord(ev[3], st));
  TK_CUDA(c, cudaEventRecord(ev[1], st));

  // 2. stable sort of the edges by data row: keys 0 .. n need bits(n) bits
  bool in_b = false;
  TK_CUDA(c, cudaEventRecord(ev[4], st));
  TK_CUDA(c, cudaEventRecord(ev[6], st));
  if (want_p) {
    const int passes = (64 - __builtin_clzll(n) + 7) / 8;
    launches += rsort::sort_pairs(c->kg_keys_a.as<uint64_t>(), c->kg_vals_a.as<uint32_t>(), c->kg_keys_b.as<uint64_t>(),
                                  c->kg_vals_b.as<uint32_t>(), edges, c->kg_sort_tmp.as<uint32_t>(), c->sm_count, st,
                                  passes, &in_b);
    TK_CUDA(c, cudaGetLastError());
  }
  TK_CUDA(c, cudaEventRecord(ev[7], st));
  TK_CUDA(c, cudaEventRecord(ev[5], st));

  // 3. run offsets, the chunk layout of the runs, the chunked sums of term_p
  TK_CUDA(c, cudaEventRecord(ev[8], st));
  TK_CUDA(c, cudaEventRecord(ev[10], st));
  uint32_t bad = 0;
  if (want_p) {
    uint64_t* off = c->kg_off.as<uint64_t>();
    TK_TRY(scan_counts(c, c->kg_cnt.as<uint32_t>(), n, off, off + n, &launches));
    uint64_t long_chunks = 0, n_long = 0;
    TK_TRY(kgrad_layout(c, off, n, edges, sc + SC_QBAD, &long_chunks, &n_long, &bad, &launches));
    if (bad) return fail(c, TKNN_EINVAL, "%s: an idx entry lies outside {-1} and [0, n = %llu)", what, (unsigned long long)n);
    const voxel::PoolParams Pp{c->kg_terms.as<float>(), dim, dim, 0, dim, in_b ? c->kg_vals_b.as<uint32_t>() : c->kg_vals_a.as<uint32_t>(),
                               off, c->kg_chunk_off.as<uint64_t>(), n, long_chunks, nullptr, d_gp};
    TK_TRY(pool_columns(c, Pp, voxel::R_SUM, c->kg_longs.as<uint32_t>(), n_long, c->kg_cs, &launches));
  }
  TK_CUDA(c, cudaEventRecord(ev[11], st));
  TK_CUDA(c, cudaEventRecord(ev[9], st));
  TK_CUDA(c, cudaEventRecord(c->ev[2], st));
  TK_TRY(copy_back(c, grad_q, d_gq, (size_t)nq * dim));
  if (want_p) TK_TRY(copy_back(c, grad_p, d_gp, (size_t)n * dim));
  TK_CUDA(c, cudaEventRecord(c->ev[3], st));
  TK_TRY(fetch_words(c, sc + SC_QBAD, 1, nullptr, 0, &bad));  // synchronises the stream
  TK_CUDA(c, cudaEventElapsedTime(&c->stats.search_ms, c->ev[0], c->ev[2]));
  TK_CUDA(c, cudaEventElapsedTime(&c->stats.d2h_ms, c->ev[2], c->ev[3]));
  c->stats.rounds = 3;
  c->stats.round_queries[0] = nq;
  c->stats.round_queries[1] = want_p ? edges : 0;
  c->stats.round_queries[2] = want_p ? n : 0;
  c->stats.kernel_launches = (uint32_t)(launches + c->mailbox_launches);
  TK_TRY(finish_round_stats(c));
  if (bad) return fail(c, TKNN_EINVAL, "%s: an idx entry lies outside {-1} and [0, n = %llu)", what, (unsigned long long)n);
  return TKNN_OK;
}

}  // namespace

extern "C" {

int tknn_knn_backward(tknn_ctx* c, const float* queries, uint64_t nq, int q_stride_floats, const float* points, uint64_t n,
                      int p_stride_floats, int dim, const int32_t* idx, int k, const float* grad_d2, float* grad_q_out,
                      float* grad_p_out) {
  TK_TRY(check_ctx(c));
  const char* what = "tknn_knn_backward";
  if (dim != 2 && dim != 3) return fail(c, TKNN_EINVAL, "%s: dim = %d (must be 2 or 3)", what, dim);
  if (q_stride_floats < dim || p_stride_floats < dim)
    return fail(c, TKNN_EINVAL, "%s: strides %d and %d must be at least dim = %d", what, q_stride_floats, p_stride_floats, dim);
  if (k < 1 || k > TKNN_MAX_K) return fail(c, TKNN_EINVAL, "%s: k = %d outside [1, %d]", what, k, TKNN_MAX_K);
  if (n >= (1ull << 31) || nq >= (1ull << 31)) return fail(c, TKNN_EINVAL, "%s: n and nq must be below 2^31", what);
  if (nq * (uint64_t)k > rsort::MAX_N)
    return fail(c, TKNN_EINVAL, "%s: nq * k = %llu edges exceed the sort's %llu", what,
                (unsigned long long)(nq * (uint64_t)k), (unsigned long long)rsort::MAX_N);
  if (!grad_q_out && !grad_p_out) return TKNN_OK;
  if (nq > 0 && (!queries || !idx || !grad_d2 || (n > 0 && !points)))
    return fail(c, TKNN_EINVAL, "%s: null queries, idx, grad_d2 or points", what);
  ScopedDevice sd(c->device);
  reset_search_stats(c);
  c->stats.n_queries = nq;
  c->stats.k = k;
  if (nq == 0) {  // no edge: every row of grad_p is +0
    if (n && grad_p_out) TK_TRY(zero_fill(c, grad_p_out, (size_t)n * dim));
    return TKNN_OK;
  }
  return knn_backward_core(c, queries, nq, q_stride_floats, points, n, p_stride_floats, dim, idx, k, grad_d2, grad_q_out,
                           grad_p_out);
}

int tknn_segment_reduce(tknn_ctx* c, const float* x, uint64_t n, int f, int stride_floats, const uint64_t* seg_offsets,
                        uint64_t n_segments, int reduce, float* out) {
  TK_TRY(check_ctx(c));
  const char* what = "tknn_segment_reduce";
  if (f < 1 || f > 1024) return fail(c, TKNN_EINVAL, "%s: f = %d outside [1, 1024]", what, f);
  if (stride_floats < f) return fail(c, TKNN_EINVAL, "%s: stride %d below f = %d", what, stride_floats, f);
  if (reduce != TKNN_REDUCE_SUM && reduce != TKNN_REDUCE_MEAN) return fail(c, TKNN_EINVAL, "%s: unknown reduce %d", what, reduce);
  if (!seg_offsets && n_segments != 1)
    return fail(c, TKNN_EINVAL, "%s: n_segments = %llu without offsets (must be 1)", what, (unsigned long long)n_segments);
  if (n_segments < 1 || n_segments > (uint64_t)INT32_MAX)
    return fail(c, TKNN_EINVAL, "%s: n_segments = %llu outside [1, 2^31 - 1]", what, (unsigned long long)n_segments);
  if (!out || (n > 0 && !x)) return fail(c, TKNN_EINVAL, "%s: null x or out", what);
  ScopedDevice sd(c->device);
  cudaStream_t st = c->stream;
  std::vector<uint64_t> off{0, n};
  if (seg_offsets) TK_TRY(read_offsets(c, what, "segment", seg_offsets, n_segments, n, "n", &off));
  if (n == 0) return zero_fill(c, out, (size_t)n_segments * f);  // every segment is empty
  ScratchScope scratch = knn_grad_scratch(c);
  const float* d_x = nullptr;
  float* d_out = nullptr;
  TK_TRY(stage_in(c, x, (size_t)(n - 1) * stride_floats + f, c->kg_x, &d_x));
  TK_TRY(out_view(c, out, (size_t)n_segments * f, c->kg_out, &d_out));
  TK_TRY(ensure(c, c->kg_seg_off, off.size() * sizeof(uint64_t)));
  TK_CUDA(c, cudaMemcpyAsync(c->kg_seg_off.p, off.data(), off.size() * sizeof(uint64_t), cudaMemcpyHostToDevice, st));
  const uint64_t* d_off = c->kg_seg_off.as<uint64_t>();
  int launches = 0;
  uint64_t long_chunks = 0, n_long = 0;
  TK_TRY(kgrad_layout(c, d_off, n_segments, n, nullptr, &long_chunks, &n_long, nullptr, &launches));
  const voxel::PoolParams P{d_x, stride_floats, f, 0, f, nullptr, d_off, c->kg_chunk_off.as<uint64_t>(), n_segments,
                            long_chunks, nullptr, d_out};
  TK_TRY(pool_columns(c, P, reduce == TKNN_REDUCE_SUM ? voxel::R_SUM : voxel::R_MEAN, c->kg_longs.as<uint32_t>(), n_long,
                      c->kg_cs, &launches));
  TK_TRY(copy_back(c, out, d_out, (size_t)n_segments * f));
  TK_CUDA(c, cudaStreamSynchronize(st));
  return TKNN_OK;
}

}  // extern "C"

// ---------------------------------------------------------------------------------------------
// surface normals and local frames (frames.cuh, DESIGN.md §3.12)
// ---------------------------------------------------------------------------------------------
namespace {

int local_frames_core(tknn_ctx* c, const float* points, uint64_t n, int stride, const int32_t* idx, uint64_t m, int k,
                      int disambiguate, float* eigvals, float* frames_out) {
  const char* what = "tknn_local_frames";
  cudaStream_t st = c->stream;
  ScratchScope scratch = frames_scratch(c);
  const float* d_p = nullptr;
  const int32_t* d_idx = nullptr;
  if (n) TK_TRY(stage_in(c, points, (size_t)(n - 1) * stride + 3, c->lf_pts, &d_p));
  TK_TRY(stage_in(c, idx, (size_t)m * k, c->lf_idx, &d_idx));
  float *d_eig = nullptr, *d_frames = nullptr;
  TK_TRY(out_view(c, eigvals, (size_t)m * 3, c->lf_eig, &d_eig));
  TK_TRY(out_view(c, frames_out, (size_t)m * 9, c->lf_frames, &d_frames));
  TK_TRY(ensure_round_events(c, 4));
  cudaEvent_t* ev = c->round_ev.data();
  uint32_t* sc = c->scalars.as<uint32_t>();
  TK_CUDA(c, cudaEventRecord(c->ev[0], st));
  TK_CUDA(c, cudaEventRecord(ev[0], st));
  TK_CUDA(c, cudaMemsetAsync(sc + SC_QBAD, 0, sizeof(uint32_t), st));
  const frames::Params P{d_p, d_idx, m, (uint32_t)n, k, stride, disambiguate, d_eig, d_frames, sc + SC_QBAD};
  const unsigned blocks = (unsigned)std::max<uint64_t>(
      1, std::min<uint64_t>((m + frames::THREADS - 1) / frames::THREADS, (uint64_t)c->sm_count * 16));
  TK_CUDA(c, cudaEventRecord(ev[2], st));
  frames::frames_kernel<<<blocks, frames::THREADS, 0, st>>>(P);
  TK_CUDA(c, cudaGetLastError());
  TK_CUDA(c, cudaEventRecord(ev[3], st));
  TK_CUDA(c, cudaEventRecord(ev[1], st));
  TK_CUDA(c, cudaEventRecord(c->ev[2], st));
  TK_TRY(copy_back(c, eigvals, d_eig, (size_t)m * 3));
  TK_TRY(copy_back(c, frames_out, d_frames, (size_t)m * 9));
  TK_CUDA(c, cudaEventRecord(c->ev[3], st));
  uint32_t bad = 0;
  TK_TRY(fetch_words(c, sc + SC_QBAD, 1, nullptr, 0, &bad));  // synchronises the stream
  TK_CUDA(c, cudaEventElapsedTime(&c->stats.search_ms, c->ev[0], c->ev[2]));
  TK_CUDA(c, cudaEventElapsedTime(&c->stats.d2h_ms, c->ev[2], c->ev[3]));
  c->stats.rounds = 1;
  c->stats.round_queries[0] = m;
  c->stats.kernel_launches = (uint32_t)(1 + c->mailbox_launches);
  TK_TRY(finish_round_stats(c));
  if (bad) return fail(c, TKNN_EINVAL, "%s: an idx entry lies outside {-1} and [0, n = %llu)", what, (unsigned long long)n);
  return TKNN_OK;
}

}  // namespace

extern "C" {

int tknn_local_frames(tknn_ctx* c, const float* points, uint64_t n, int stride_floats, const int32_t* idx, uint64_t m,
                      int k, int disambiguate, float* eigvals_out, float* frames_out) {
  TK_TRY(check_ctx(c));
  const char* what = "tknn_local_frames";
  if (k < 1 || k > TKNN_MAX_K) return fail(c, TKNN_EINVAL, "%s: k = %d outside [1, %d]", what, k, TKNN_MAX_K);
  if (stride_floats < 3) return fail(c, TKNN_EINVAL, "%s: stride %d below 3", what, stride_floats);
  if (n >= (1ull << 31) || m >= (1ull << 31)) return fail(c, TKNN_EINVAL, "%s: n and m must be below 2^31", what);
  if (disambiguate != 0 && disambiguate != 1)
    return fail(c, TKNN_EINVAL, "%s: disambiguate = %d (must be 0 or 1)", what, disambiguate);
  const bool work = m > 0 && (eigvals_out || frames_out);
  if (work && (!idx || (n > 0 && !points))) return fail(c, TKNN_EINVAL, "%s: null idx or points", what);
  ScopedDevice sd(c->device);
  reset_search_stats(c);
  c->stats.n_queries = m;
  c->stats.k = k;
  if (!work) return TKNN_OK;
  return local_frames_core(c, points, n, stride_floats, idx, m, k, disambiguate, eigvals_out, frames_out);
}

}  // extern "C"
