// dist.cu — the multi-GPU drivers of libtrueknn, inside the library and behind the C ABI (include/trueknn.h,
// "multi-GPU"): query-sharded search over a replicated LBVH and point-partitioned search over Morton-range
// ownership, one rank per GPU, NCCL over NVLink 5 / NVSwitch.
//
// Reference pattern superseded: OWL's replicate-and-split multi-GPU model — every object replicated on every device
// of the context's device list, the identical launch issued on each, results in page-interleaved managed memory
// (owl/RayGen.cpp:150-200, owl/Context.cpp:75-120, owl/Buffer.cpp:307-353) — which TrueKNN never uses
// (samples/s01-trueknn/hostCode.cpp:141 creates a 1-device context) and which cannot hold more than 2^29 primitives
// per accel (owl/UserGeomGroup.cpp:87-117).  The reference has no communication backend at all.
//
// Per-rank pipeline of the point-partitioned variant (all device-side; the host only sizes buffers):
//   build   global box (bounds kernel + all-reduce) -> 63-bit Morton codes on the global grid -> histogram of the top
//           24 code bits + all-reduce -> cell-aligned splitters (host scan of the histogram) -> destination rank per
//           point, ONE onesweep pass on it, packed (x, y, z, global id) rows -> all-to-all -> local LBVH whose point
//           ids ARE the global ids (so local (d2, id) tie-breaks are the global ones) -> per-cell boxes + all-gather
//   search  local all-points search (d2 kept) -> reach test against the peers' cell boxes + compaction of the boundary
//           queries -> all-to-all -> remote search capped at the asker's k-th d2 -> all-to-all back -> 2-way merges
//           on (d2, global id) -> sqrt
#include <dlfcn.h>
#include <nccl.h>

#include <algorithm>
#include <atomic>
#include <chrono>
#include <cmath>
#include <condition_variable>
#include <mutex>
#include <new>
#include <thread>

#include "brute.cuh"
#include "ctx.cuh"
#include "lbvh.cuh"
#include "radix_sort.cuh"

using namespace tknn;
using namespace tknn::host;

namespace tknn {
namespace dist {

// ---------------------------------------------------------------------------------------------
// NCCL, loaded at first use.  libtrueknn.so does not link libnccl: a process that already carries an NCCL (PyTorch
// bundles its own under the same soname) must keep exactly that one, and the single-GPU path needs none.
// ---------------------------------------------------------------------------------------------
struct NcclApi {
  void* handle = nullptr;
  ncclResult_t (*GetUniqueId)(ncclUniqueId*) = nullptr;
  ncclResult_t (*CommInitRank)(ncclComm_t*, int, ncclUniqueId, int) = nullptr;
  ncclResult_t (*CommInitAll)(ncclComm_t*, int, const int*) = nullptr;
  ncclResult_t (*CommDestroy)(ncclComm_t) = nullptr;
  ncclResult_t (*AllReduce)(const void*, void*, size_t, ncclDataType_t, ncclRedOp_t, ncclComm_t, cudaStream_t) = nullptr;
  ncclResult_t (*AllGather)(const void*, void*, size_t, ncclDataType_t, ncclComm_t, cudaStream_t) = nullptr;
  ncclResult_t (*Send)(const void*, size_t, ncclDataType_t, int, ncclComm_t, cudaStream_t) = nullptr;
  ncclResult_t (*Recv)(void*, size_t, ncclDataType_t, int, ncclComm_t, cudaStream_t) = nullptr;
  ncclResult_t (*GroupStart)() = nullptr;
  ncclResult_t (*GroupEnd)() = nullptr;
  const char* (*GetErrorString)(ncclResult_t) = nullptr;
  std::string error;
};

static NcclApi* nccl_api() {
  static NcclApi api;
  static std::once_flag once;
  std::call_once(once, [] {
    const char* names[] = {"libnccl.so.2", "libnccl.so"};
    for (const char* nm : names) {
      api.handle = dlopen(nm, RTLD_NOW | RTLD_LOCAL);
      if (api.handle) break;
    }
    if (!api.handle) { api.error = std::string("cannot load libnccl.so.2: ") + (dlerror() ? dlerror() : "?"); return; }
#define TK_SYM(field, name)                                                        \
  api.field = reinterpret_cast<decltype(api.field)>(dlsym(api.handle, name));      \
  if (!api.field && api.error.empty()) api.error = std::string("libnccl lacks ") + name;
    TK_SYM(GetUniqueId, "ncclGetUniqueId")
    TK_SYM(CommInitRank, "ncclCommInitRank")
    TK_SYM(CommInitAll, "ncclCommInitAll")
    TK_SYM(CommDestroy, "ncclCommDestroy")
    TK_SYM(AllReduce, "ncclAllReduce")
    TK_SYM(AllGather, "ncclAllGather")
    TK_SYM(Send, "ncclSend")
    TK_SYM(Recv, "ncclRecv")
    TK_SYM(GroupStart, "ncclGroupStart")
    TK_SYM(GroupEnd, "ncclGroupEnd")
    TK_SYM(GetErrorString, "ncclGetErrorString")
#undef TK_SYM
  });
  return &api;
}

#define TK_NCCL(c, expr)                                                                                      \
  do {                                                                                                        \
    ncclResult_t r__ = (expr);                                                                                \
    if (r__ != ncclSuccess)                                                                                   \
      return fail((c), TKNN_ENCCL, "%s: %s (%s:%d)", #expr, nccl_api()->GetErrorString(r__), __FILE__, __LINE__); \
  } while (0)

// ---------------------------------------------------------------------------------------------
// small kernels of the drivers
// ---------------------------------------------------------------------------------------------
constexpr int CELL_BITS = 24;                 // splitters fall on boundaries of the 256^3 grid of the global cube
constexpr int CELL_SHIFT = 63 - CELL_BITS;
constexpr size_t N_CELLS = (size_t)1 << CELL_BITS;
constexpr int SUMMARY_AXIS_BITS = 3;          // partition summaries live on the 8 x 8 x 8 grid (512 boxes per rank)
constexpr int SUMMARY_BOXES = 1 << (3 * SUMMARY_AXIS_BITS);
constexpr int MAX_RANKS = 32;

struct Splitters {
  uint32_t cell[MAX_RANKS];  // cell[r - 1] = first cell of rank r (r = 1 .. n_ranks - 1)
};

static __global__ void __launch_bounds__(256) cell_hist_kernel(const uint64_t* __restrict__ codes, uint64_t n,
                                                               uint32_t* __restrict__ hist) {
  const uint64_t i = (uint64_t)blockIdx.x * 256 + threadIdx.x;
  if (i < n) atomicAdd(&hist[(uint32_t)(codes[i] >> CELL_SHIFT)], 1u);
}

// sums[b] = number of points in cells [b * SPLIT_BLOCK, (b + 1) * SPLIT_BLOCK): the host finds the block each splitter
// falls into from these 4096 sums and reads back only those blocks instead of the whole 64 MB histogram
constexpr int SPLIT_BLOCK = 4096;
static __global__ void __launch_bounds__(256) cell_block_sums_kernel(const uint32_t* __restrict__ hist, uint64_t* __restrict__ sums) {
  __shared__ uint64_t s_w[8];
  const uint32_t* h = hist + (size_t)blockIdx.x * SPLIT_BLOCK;
  uint64_t v = 0;
  for (int i = threadIdx.x; i < SPLIT_BLOCK; i += 256) v += h[i];
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(FULL_MASK, v, o);
  if ((threadIdx.x & 31) == 0) s_w[threadIdx.x >> 5] = v;
  __syncthreads();
  if (threadIdx.x == 0) {
    uint64_t t = 0;
    for (int w = 0; w < 8; ++w) t += s_w[w];
    sums[blockIdx.x] = t;
  }
}

// keys[i] <- destination rank of point i (in place over its Morton code); counts[r] += points going to rank r
static __global__ void __launch_bounds__(256) dest_kernel(uint64_t* __restrict__ keys, uint64_t n, Splitters sp, int n_ranks,
                                                          uint32_t* __restrict__ counts) {
  __shared__ uint32_t s_cnt[MAX_RANKS];
  if (threadIdx.x < MAX_RANKS) s_cnt[threadIdx.x] = 0;
  __syncthreads();
  const uint64_t i = (uint64_t)blockIdx.x * 256 + threadIdx.x;
  if (i < n) {
    const uint32_t cell = (uint32_t)(keys[i] >> CELL_SHIFT);
    int d = 0;
    for (int r = 0; r < n_ranks - 1; ++r) d += (sp.cell[r] <= cell) ? 1 : 0;
    keys[i] = (uint64_t)d;
    atomicAdd(&s_cnt[d], 1u);
  }
  __syncthreads();
  if (threadIdx.x < n_ranks && s_cnt[threadIdx.x]) atomicAdd(&counts[threadIdx.x], s_cnt[threadIdx.x]);
}

// rows[j] = (x, y, z, bits(first + order[j])): the points in destination order, carrying their global ids
static __global__ void __launch_bounds__(256) pack_rows_kernel(const float* __restrict__ xyz, int dim, int stride,
                                                               const uint32_t* __restrict__ order, uint64_t n, uint32_t first,
                                                               float4* __restrict__ rows) {
  const uint64_t j = (uint64_t)blockIdx.x * 256 + threadIdx.x;
  if (j >= n) return;
  const uint32_t src = order[j];
  const float* p = xyz + (uint64_t)src * (uint64_t)stride;
  rows[j] = make_float4(p[0], p[1], dim > 2 ? p[2] : 0.0f, __uint_as_float(first + src));
}

// pad rows of `stride` floats to a dense [n][3] block (the replicated build's all-gather moves xyz only)
static __global__ void __launch_bounds__(256) dense_xyz_kernel(const float* __restrict__ xyz, int dim, int stride, uint64_t n,
                                                               float* __restrict__ out) {
  const uint64_t i = (uint64_t)blockIdx.x * 256 + threadIdx.x;
  if (i >= n) return;
  const float* p = xyz + i * (uint64_t)stride;
  out[3 * i] = p[0];
  out[3 * i + 1] = p[1];
  out[3 * i + 2] = dim > 2 ? p[2] : 0.0f;
}

// Tight box of this rank's points inside every top-level cell of the GLOBAL grid (same quantiser as morton_kernel).
// boxes: [512][6] order-preserving uints (min xyz, max xyz), initialised to (~0, ~0, ~0, 0, 0, 0).
// The points are Morton-sorted on (nearly) the same grid, so a cell is one long run of consecutive points: a warp
// walks CELL_RUN consecutive points (coalesced, 32 per step), every lane accumulating a private box that it flushes
// with atomics only when its cell changes; at the end a warp whose lanes all sit in one cell reduces with shuffles and
// issues ONE set of six atomics.  (The first version issued six atomics per warp of 32 points onto the same few
// addresses: 53 ms for 250 M points; profiles/r2_bench_cfg5_2B_n8.json.)
constexpr int CELL_RUN = 2048;
__device__ __forceinline__ void flush_cell_box(uint32_t* __restrict__ boxes, uint32_t cell, const float lo[3], const float hi[3]) {
#pragma unroll
  for (int a = 0; a < 3; ++a) {
    atomicMin(&boxes[cell * 6 + a], float_to_ordered(lo[a]));
    atomicMax(&boxes[cell * 6 + 3 + a], float_to_ordered(hi[a]));
  }
}

static __global__ void __launch_bounds__(256) cell_boxes_kernel(const float4* __restrict__ pts, uint64_t n,
                                                                const float* __restrict__ box6, uint32_t* __restrict__ boxes) {
  const int lane = threadIdx.x & 31;
  const uint64_t warp_id = ((uint64_t)blockIdx.x * 256 + threadIdx.x) >> 5;
  const uint64_t begin = warp_id * CELL_RUN;
  if (begin >= n) return;
  const uint64_t end = begin + CELL_RUN < n ? begin + CELL_RUN : n;
  const float lx = box6[0], ly = box6[1], lz = box6[2];
  const float ext = fmaxf(fmaxf(box6[3] - lx, box6[4] - ly), fmaxf(box6[5] - lz, FLT_MIN));
  const float scale = 2097152.0f / ext;
  uint32_t cur = 0xffffffffu;  // no cell yet
  float lo[3] = {INFINITY, INFINITY, INFINITY}, hi[3] = {-INFINITY, -INFINITY, -INFINITY};
  for (uint64_t i = begin + lane; i < end; i += 32) {
    const float4 p = __ldg(&pts[i]);
    const uint32_t cx = (uint32_t)fminf(fmaxf((p.x - lx) * scale, 0.0f), 2097151.0f) >> (21 - SUMMARY_AXIS_BITS);
    const uint32_t cy = (uint32_t)fminf(fmaxf((p.y - ly) * scale, 0.0f), 2097151.0f) >> (21 - SUMMARY_AXIS_BITS);
    const uint32_t cz = (uint32_t)fminf(fmaxf((p.z - lz) * scale, 0.0f), 2097151.0f) >> (21 - SUMMARY_AXIS_BITS);
    uint32_t cell = 0;
#pragma unroll
    for (int b = 0; b < SUMMARY_AXIS_BITS; ++b)
      cell |= ((cx >> b) & 1u) << (3 * b + 2) | ((cy >> b) & 1u) << (3 * b + 1) | ((cz >> b) & 1u) << (3 * b);
    if (cell != cur) {
      if (cur != 0xffffffffu) flush_cell_box(boxes, cur, lo, hi);
      cur = cell;
      lo[0] = hi[0] = p.x; lo[1] = hi[1] = p.y; lo[2] = hi[2] = p.z;
    } else {
      lo[0] = fminf(lo[0], p.x); lo[1] = fminf(lo[1], p.y); lo[2] = fminf(lo[2], p.z);
      hi[0] = fmaxf(hi[0], p.x); hi[1] = fmaxf(hi[1], p.y); hi[2] = fmaxf(hi[2], p.z);
    }
  }
  // the run is over: one set of atomics per warp when every lane ended in the same cell (lanes without a point agree)
  const uint32_t c0 = __shfl_sync(FULL_MASK, cur, 0);
  if (__all_sync(FULL_MASK, cur == c0 || cur == 0xffffffffu) && c0 != 0xffffffffu) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1)
#pragma unroll
      for (int a = 0; a < 3; ++a) {
        lo[a] = fminf(lo[a], __shfl_xor_sync(FULL_MASK, lo[a], o));
        hi[a] = fmaxf(hi[a], __shfl_xor_sync(FULL_MASK, hi[a], o));
      }
    if (lane == 0) flush_cell_box(boxes, c0, lo, hi);
  } else if (cur != 0xffffffffu) {
    flush_cell_box(boxes, cur, lo, hi);
  }
}

// ordered uints -> floats; an untouched cell becomes an inverted box (+inf, -inf), which no ball reaches
static __global__ void boxes_to_float_kernel(const uint32_t* __restrict__ boxes, int n_boxes, float* __restrict__ out) {
  const int b = blockIdx.x * blockDim.x + threadIdx.x;
  if (b >= n_boxes) return;
  const bool empty = boxes[b * 6] == 0xffffffffu;
  for (int a = 0; a < 3; ++a) {
    out[b * 6 + a] = empty ? INFINITY : ordered_to_float(boxes[b * 6 + a]);
    out[b * 6 + 3 + a] = empty ? -INFINITY : ordered_to_float(boxes[b * 6 + 3 + a]);
  }
}

// ordered box words -> 6 floats (global box)
static __global__ void box_to_float_kernel(const uint32_t* __restrict__ ob, float* __restrict__ out) {
  if (threadIdx.x < 6) out[threadIdx.x] = ordered_to_float(ob[threadIdx.x]);
}

// Which remote ranks can each owned query's ball (q, d_k) reach?  mask[i] (bit s = rank s) + per-rank counts.
// Row i of the local result belongs to sorted point i (row_mode 1, q_begin 0).
static __global__ void __launch_bounds__(256) reach_kernel(const float4* __restrict__ pts, uint64_t n, const int32_t* __restrict__ idx,
                                                           const float* __restrict__ d2, int k, const float* __restrict__ box6,
                                                           const float* __restrict__ summ, int n_ranks, int self_rank,
                                                           uint32_t* __restrict__ mask_out, uint32_t* __restrict__ counts) {
  const uint64_t i = (uint64_t)blockIdx.x * 256 + threadIdx.x;
  uint32_t mask = 0;
  if (i < n) {
    const float4 p = __ldg(&pts[i]);
    const uint64_t last = i * (uint64_t)k + (uint64_t)(k - 1);
    const float r2 = idx[last] >= 0 ? d2[last] : INFINITY;  // unfilled list: unbounded ball
    mask = brute::reach_mask_of(p.x, p.y, p.z, r2, box6, summ, n_ranks, SUMMARY_AXIS_BITS, self_rank);
    mask_out[i] = mask;
  }
  for (int s = 0; s < n_ranks; ++s) {
    const uint32_t b = __ballot_sync(FULL_MASK, (mask >> s) & 1u);
    if (b && (threadIdx.x & 31) == 0) atomicAdd(&counts[s], (uint32_t)__popc(b));
  }
}

// Boundary queries grouped by destination rank: rows_out[pos] = local row, payload[pos] = (x, y, z, d_k^2).
// cursor[s] starts at the first slot of rank s; order inside a rank's block is arbitrary (answers return in it).
static __global__ void __launch_bounds__(256) boundary_scatter_kernel(const float4* __restrict__ pts, uint64_t n,
                                                                      const int32_t* __restrict__ idx, const float* __restrict__ d2,
                                                                      int k, const uint32_t* __restrict__ mask_in, int n_ranks,
                                                                      uint32_t* __restrict__ cursor, uint32_t* __restrict__ rows_out,
                                                                      float4* __restrict__ payload) {
  const uint64_t i = (uint64_t)blockIdx.x * 256 + threadIdx.x;
  const uint32_t mask = i < n ? mask_in[i] : 0u;
  if (!__any_sync(FULL_MASK, mask != 0u)) return;
  const int lane = threadIdx.x & 31;
  float4 row = make_float4(0.f, 0.f, 0.f, 0.f);
  if (mask) {
    const float4 p = __ldg(&pts[i]);
    const uint64_t last = i * (uint64_t)k + (uint64_t)(k - 1);
    row = make_float4(p.x, p.y, p.z, idx[last] >= 0 ? d2[last] : INFINITY);
  }
  for (int s = 0; s < n_ranks; ++s) {
    const uint32_t b = __ballot_sync(FULL_MASK, (mask >> s) & 1u);
    if (!b) continue;
    uint32_t base = 0;
    if (lane == __ffs(b) - 1) base = atomicAdd(&cursor[s], (uint32_t)__popc(b));
    base = __shfl_sync(FULL_MASK, base, __ffs(b) - 1);
    if ((mask >> s) & 1u) {
      const uint32_t pos = base + __popc(b & ((1u << lane) - 1u));
      rows_out[pos] = (uint32_t)i;
      payload[pos] = row;
    }
  }
}

static __global__ void __launch_bounds__(256) column_w_kernel(const float4* __restrict__ rows, uint64_t n, float* __restrict__ out) {
  const uint64_t i = (uint64_t)blockIdx.x * 256 + threadIdx.x;
  if (i < n) out[i] = rows[i].w;
}

__device__ __forceinline__ uint64_t list_key(int id, float d2) { return id < 0 ? ~0ull : make_key(d2, id); }

// 2-way merge on (d2, global id): own list of row rows[j] with the answer of one remote rank, smallest k kept, in
// place.  The point sets of two ranks are disjoint, so there are no duplicates to drop.  Both lists ascend and end
// in -1 / FLT_MAX sentinels.  One thread per boundary query of ONE destination rank (rows are distinct within it).
static __global__ void __launch_bounds__(128) merge_reply_kernel(const uint32_t* __restrict__ rows, uint64_t m,
                                                                 const int32_t* __restrict__ r_idx, const float* __restrict__ r_d2,
                                                                 int k, int32_t* __restrict__ idx, float* __restrict__ d2) {
  const uint64_t j = (uint64_t)blockIdx.x * 128 + threadIdx.x;
  if (j >= m) return;
  int32_t* ai = idx + (uint64_t)rows[j] * k;
  float* ad = d2 + (uint64_t)rows[j] * k;
  const int32_t* bi = r_idx + j * (uint64_t)k;
  const float* bd = r_d2 + j * (uint64_t)k;
  if (bi[0] < 0) return;  // nothing came back
  // how many of the k smallest come from the own list?
  int ta = 0, tb = 0;
  for (int t = 0; t < k; ++t) {
    const uint64_t ka = list_key(ai[ta], ad[ta]);
    const uint64_t kb = tb < k ? list_key(bi[tb], bd[tb]) : ~0ull;
    if (kb < ka) ++tb; else ++ta;
  }
  if (tb == 0) return;
  // merge from the back: the write position ta + tb - 1 never runs ahead of the own read position ta - 1
  int ia = ta - 1, ib = tb - 1;
  for (int w = k - 1; w >= 0 && ib >= 0; --w) {
    const uint64_t kb = list_key(bi[ib], bd[ib]);
    if (ia >= 0 && list_key(ai[ia], ad[ia]) > kb) {
      ai[w] = ai[ia]; ad[w] = ad[ia]; --ia;
    } else {
      ai[w] = bi[ib]; ad[w] = bd[ib]; --ib;
    }
  }
}

// d2 -> distance in place.  Every rank owns more than k points, so every list is full: there are no -1 / FLT_MAX
// sentinels to preserve and the index array need not be read.  n4 float4 + a scalar tail.
static __global__ void __launch_bounds__(256) sqrt_rows_kernel(float* __restrict__ d, uint64_t n, int vec) {
  const uint64_t i = (uint64_t)blockIdx.x * 256 + threadIdx.x;
  const uint64_t n4 = vec ? n / 4 : 0;
  if (i < n4) {
    float4 v = reinterpret_cast<float4*>(d)[i];
    v.x = __fsqrt_rn(v.x); v.y = __fsqrt_rn(v.y); v.z = __fsqrt_rn(v.z); v.w = __fsqrt_rn(v.w);
    reinterpret_cast<float4*>(d)[i] = v;
  }
  if (i < n - n4 * 4) d[n4 * 4 + i] = __fsqrt_rn(d[n4 * 4 + i]);
}

// min / max / sum of n_parts blocks of `count` u32 words into the first block (in-process transport)
static __global__ void __launch_bounds__(256) reduce_parts_kernel(uint32_t* __restrict__ parts, size_t count, int n_parts, int op,
                                                                  uint32_t* __restrict__ out) {
  const size_t i = (size_t)blockIdx.x * 256 + threadIdx.x;
  if (i >= count) return;
  uint32_t v = parts[i];
  for (int p = 1; p < n_parts; ++p) {
    const uint32_t w = parts[(size_t)p * count + i];
    v = op == 0 ? min(v, w) : (op == 1 ? max(v, w) : v + w);
  }
  out[i] = v;
}

// result rows -> the owner GPU's slice of the file-order arrays, through peer pointers (P2P stores over NVLink)
struct PeerTable {
  int32_t* idx[MAX_RANKS];
  float* dist[MAX_RANKS];
};
static __global__ void __launch_bounds__(256) scatter_rows_kernel(const int32_t* __restrict__ qid, const int32_t* __restrict__ idx,
                                                                  const float* __restrict__ dist, uint64_t m, int k,
                                                                  uint64_t rows_per_owner, PeerTable peers) {
  const uint64_t t = (uint64_t)blockIdx.x * 256 + threadIdx.x;
  if (t >= m * (uint64_t)k) return;
  const uint64_t j = t / (uint64_t)k;
  const int i = (int)(t - j * (uint64_t)k);
  const uint64_t row = (uint64_t)(uint32_t)qid[j];
  const int owner = (int)(row / rows_per_owner);
  const uint64_t local = row - (uint64_t)owner * rows_per_owner;
  peers.idx[owner][local * k + i] = idx[t];
  peers.dist[owner][local * k + i] = dist[t];
}

static __global__ void __launch_bounds__(256) sample_rows_kernel(const float4* __restrict__ pts, const int32_t* __restrict__ gid,
                                                                 const int32_t* __restrict__ idx, const float* __restrict__ dist,
                                                                 uint64_t n_rows, int samples, int k, float4* __restrict__ q_out,
                                                                 int32_t* __restrict__ idx_out, float* __restrict__ dist_out) {
  const int t = blockIdx.x * 256 + threadIdx.x;
  if (t >= samples) return;
  const uint64_t r = n_rows * (uint64_t)t / (uint64_t)samples;
  float4 p = pts[r];
  p.w = __int_as_float(gid[r]);  // == the id already stored in w; taken from the result to check that too
  q_out[t] = p;
  for (int i = 0; i < k; ++i) {
    idx_out[(uint64_t)t * k + i] = idx[r * (uint64_t)k + i];
    dist_out[(uint64_t)t * k + i] = dist[r * (uint64_t)k + i];
  }
}

// ---------------------------------------------------------------------------------------------
// transports
// ---------------------------------------------------------------------------------------------
struct Comm {
  int rank = 0, n = 1;
  virtual ~Comm() {}
  // u32 words, in place on the device; op 0 = min, 1 = max, 2 = sum
  virtual int all_reduce_u32(tknn_ctx* c, uint32_t* buf, size_t count, int op) = 0;
  // recv holds n blocks of `bytes`; block r comes from rank r's `send`
  virtual int all_gather(tknn_ctx* c, const void* send, void* recv, size_t bytes) = 0;
  // rows of row_bytes; counts and offsets in rows, host arrays of n
  virtual int all_to_all_v(tknn_ctx* c, const void* send, const uint64_t* scnt, const uint64_t* soff, void* recv,
                           const uint64_t* rcnt, const uint64_t* roff, size_t row_bytes) = 0;
  // every rank has finished its device work up to here (host rendezvous where ranks share a process)
  virtual int barrier(tknn_ctx* c) = 0;
};

// host rendezvous of the rank threads of one process
struct HostBarrier {
  std::mutex mu;
  std::condition_variable cv;
  int n = 1, waiting = 0;
  uint64_t phase = 0;
  void arrive() {
    std::unique_lock<std::mutex> lk(mu);
    const uint64_t ph = phase;
    if (++waiting == n) { waiting = 0; ++phase; cv.notify_all(); }
    else cv.wait(lk, [&] { return phase != ph; });
  }
};

struct NcclComm : Comm {
  ncclComm_t comm = nullptr;
  HostBarrier* hb = nullptr;  // set when the ranks are threads of one process (tknn_create_multi)
  ~NcclComm() override { if (comm) nccl_api()->CommDestroy(comm); }
  // rank threads of one process: do not leave a collective in flight while a sibling thread may cudaMalloc
  int settle(tknn_ctx* c) {
    if (hb) TK_CUDA(c, cudaStreamSynchronize(c->stream));
    return TKNN_OK;
  }
  int all_reduce_u32(tknn_ctx* c, uint32_t* buf, size_t count, int op) override {
    NcclApi* A = nccl_api();
    TK_NCCL(c, A->AllReduce(buf, buf, count, ncclUint32, op == 0 ? ncclMin : (op == 1 ? ncclMax : ncclSum), comm, c->stream));
    return settle(c);
  }
  int all_gather(tknn_ctx* c, const void* send, void* recv, size_t bytes) override {
    NcclApi* A = nccl_api();
    TK_NCCL(c, A->AllGather(send, recv, bytes, ncclUint8, comm, c->stream));
    return settle(c);
  }
  int all_to_all_v(tknn_ctx* c, const void* send, const uint64_t* scnt, const uint64_t* soff, void* recv, const uint64_t* rcnt,
                   const uint64_t* roff, size_t row_bytes) override {
    NcclApi* A = nccl_api();
    const char* s = static_cast<const char*>(send);
    char* r = static_cast<char*>(recv);
    if (scnt[rank]) TK_CUDA(c, cudaMemcpyAsync(r + roff[rank] * row_bytes, s + soff[rank] * row_bytes, scnt[rank] * row_bytes,
                                               cudaMemcpyDeviceToDevice, c->stream));
    TK_NCCL(c, A->GroupStart());
    for (int p = 0; p < n; ++p) {
      if (p == rank) continue;
      if (scnt[p]) TK_NCCL(c, A->Send(s + soff[p] * row_bytes, scnt[p] * row_bytes, ncclUint8, p, comm, c->stream));
      if (rcnt[p]) TK_NCCL(c, A->Recv(r + roff[p] * row_bytes, rcnt[p] * row_bytes, ncclUint8, p, comm, c->stream));
    }
    TK_NCCL(c, A->GroupEnd());
    return settle(c);
  }
  int barrier(tknn_ctx* c) override {
    TK_CUDA(c, cudaStreamSynchronize(c->stream));
    if (hb) hb->arrive();
    return TKNN_OK;
  }
};

// In-process transport: the ranks are threads of one process (possibly several on ONE device, which NCCL refuses).
// A collective is: finish my device work, publish my buffers, rendezvous, copy my inbound pieces from the peers'
// buffers (device-to-device, or peer copies between devices), finish, rendezvous again (buffers reusable).
struct LocalHub {
  HostBarrier hb;
  const void* send[MAX_RANKS];
  const uint64_t* scnt[MAX_RANKS];
  const uint64_t* soff[MAX_RANKS];
};

struct LocalComm : Comm {
  LocalHub* hub = nullptr;
  DevBuf tmp;
  ~LocalComm() override { release(tmp); }
  int all_gather(tknn_ctx* c, const void* send, void* recv, size_t bytes) override {
    TK_CUDA(c, cudaStreamSynchronize(c->stream));
    hub->send[rank] = send;
    hub->hb.arrive();
    for (int p = 0; p < n; ++p)
      TK_CUDA(c, cudaMemcpyAsync(static_cast<char*>(recv) + (size_t)p * bytes, hub->send[p], bytes, cudaMemcpyDefault, c->stream));
    TK_CUDA(c, cudaStreamSynchronize(c->stream));
    hub->hb.arrive();
    return TKNN_OK;
  }
  int all_reduce_u32(tknn_ctx* c, uint32_t* buf, size_t count, int op) override {
    TK_TRY(ensure(c, tmp, (size_t)n * count * sizeof(uint32_t)));
    TK_TRY(all_gather(c, buf, tmp.p, count * sizeof(uint32_t)));
    reduce_parts_kernel<<<blocks_for(count, 256), 256, 0, c->stream>>>(tmp.as<uint32_t>(), count, n, op, buf);
    TK_CUDA(c, cudaGetLastError());
    return TKNN_OK;
  }
  int all_to_all_v(tknn_ctx* c, const void* send, const uint64_t* scnt, const uint64_t* soff, void* recv, const uint64_t* rcnt,
                   const uint64_t* roff, size_t row_bytes) override {
    TK_CUDA(c, cudaStreamSynchronize(c->stream));
    hub->send[rank] = send;
    hub->scnt[rank] = scnt;
    hub->soff[rank] = soff;
    hub->hb.arrive();
    int rc = TKNN_OK;
    for (int p = 0; p < n && rc == TKNN_OK; ++p) {
      const uint64_t cnt = hub->scnt[p][rank];
      if (cnt != rcnt[p]) { rc = fail(c, TKNN_ENCCL, "all_to_all_v: rank %d sends %llu rows, %llu expected", p,
                                      (unsigned long long)cnt, (unsigned long long)rcnt[p]); break; }
      if (!cnt) continue;
      const char* src = static_cast<const char*>(hub->send[p]) + hub->soff[p][rank] * row_bytes;
      if (cudaMemcpyAsync(static_cast<char*>(recv) + roff[p] * row_bytes, src, cnt * row_bytes, cudaMemcpyDefault, c->stream) !=
          cudaSuccess) { cudaGetLastError(); rc = fail(c, TKNN_ECUDA, "all_to_all_v: peer copy failed"); }
    }
    if (cudaStreamSynchronize(c->stream) != cudaSuccess && rc == TKNN_OK) { cudaGetLastError(); rc = fail(c, TKNN_ECUDA, "all_to_all_v: sync failed"); }
    hub->hb.arrive();
    return rc;
  }
  int barrier(tknn_ctx* c) override {
    TK_CUDA(c, cudaStreamSynchronize(c->stream));
    hub->hb.arrive();
    return TKNN_OK;
  }
};

// ---------------------------------------------------------------------------------------------
// per-rank state
// ---------------------------------------------------------------------------------------------
struct State {
  Comm* comm = nullptr;
  bool partition_built = false;
  uint64_t n_global = 0;
  DevBuf small;        // counts matrices and other tiny exchanges (16 KB)
  DevBuf gbox;         // 8 ordered words | 6 floats (global box)
  DevBuf hist, summ, summ_mine, boxes_ord;
  DevBuf rows_send, rows_recv;                 // build: packed (x, y, z, gid) rows
  DevBuf full_xyz, dense_local;                // replicated build
  DevBuf mask, brows, payload, recv_q, cap;    // search: boundary queries
  DevBuf ans_idx, ans_d2, back_idx, back_d2;   // search: answers
  DevBuf out_gid, out_idx, out_d2;             // search: device staging for host outputs
  DevBuf ver;                                  // verification scratch
  std::vector<cudaEvent_t> ev;
  tknn_dist_stats stats;
  State() { std::memset(&stats, 0, sizeof(stats)); }
};

static void free_state(State* S) {
  if (!S) return;
  for (DevBuf* b : {&S->small, &S->gbox, &S->hist, &S->summ, &S->summ_mine, &S->boxes_ord, &S->rows_send, &S->rows_recv,
                    &S->full_xyz, &S->dense_local, &S->mask, &S->brows, &S->payload, &S->recv_q, &S->cap, &S->ans_idx, &S->ans_d2,
                    &S->back_idx, &S->back_d2, &S->out_gid, &S->out_idx, &S->out_d2, &S->ver})
    release(*b);
  for (auto e : S->ev) cudaEventDestroy(e);
  delete S->comm;
  delete S;
}

static int mark(tknn_ctx* c, State* S, int i) {
  while ((int)S->ev.size() <= i) {
    cudaEvent_t e;
    TK_CUDA(c, cudaEventCreate(&e));
    S->ev.push_back(e);
  }
  TK_CUDA(c, cudaEventRecord(S->ev[i], c->stream));
  return TKNN_OK;
}
static float between(State* S, int a, int b) {
  float ms = 0.f;
  if (cudaEventElapsedTime(&ms, S->ev[a], S->ev[b]) != cudaSuccess) { cudaGetLastError(); return 0.f; }
  return ms;
}

static int need_comm(tknn_ctx* c) {
  if (!c) return TKNN_EINVAL;
  if (!c->dist || !c->dist->comm) return fail(c, TKNN_ESTATE, "no communicator: call tknn_comm_init (or use tknn_create_multi) first");
  return TKNN_OK;
}

// counts matrix: M[p][q] = rows rank p sends to rank q; rcnt[p] = M[p][me]
static int exchange_counts(tknn_ctx* c, State* S, const uint64_t* scnt, uint64_t* rcnt) {
  Comm* cm = S->comm;
  const int n = cm->n;
  TK_TRY(ensure(c, S->small, 16384));
  uint64_t* d = S->small.as<uint64_t>();  // [n] mine | [n][n] all
  TK_CUDA(c, cudaMemcpyAsync(d, scnt, n * sizeof(uint64_t), cudaMemcpyHostToDevice, c->stream));
  TK_TRY(cm->all_gather(c, d, d + MAX_RANKS, n * sizeof(uint64_t)));
  std::vector<uint64_t> M((size_t)n * n);
  TK_CUDA(c, cudaMemcpyAsync(M.data(), d + MAX_RANKS, M.size() * sizeof(uint64_t), cudaMemcpyDeviceToHost, c->stream));
  TK_CUDA(c, cudaStreamSynchronize(c->stream));
  for (int p = 0; p < n; ++p) rcnt[p] = M[(size_t)p * n + cm->rank];
  return TKNN_OK;
}

// Argument checks are local, collectives are not: a rank that returned early would leave its peers waiting in the
// next collective.  Every rank contributes its verdict; all return together.
static int agree(tknn_ctx* c, State* S, int local_rc) {
  TK_TRY(ensure(c, S->small, 16384));
  uint32_t* d_flag = S->small.as<uint32_t>() + 2176;
  const uint32_t mine = local_rc != TKNN_OK ? 1u : 0u;
  TK_CUDA(c, cudaMemcpyAsync(d_flag, &mine, sizeof(uint32_t), cudaMemcpyHostToDevice, c->stream));
  TK_TRY(S->comm->all_reduce_u32(c, d_flag, 1, 1));
  uint32_t any = 0;
  TK_CUDA(c, cudaMemcpyAsync(&any, d_flag, sizeof(uint32_t), cudaMemcpyDeviceToHost, c->stream));
  TK_CUDA(c, cudaStreamSynchronize(c->stream));
  if (local_rc != TKNN_OK) return local_rc;
  if (any) return fail(c, TKNN_EINVAL, "another rank rejected its arguments");
  return TKNN_OK;
}

static void prefix(const uint64_t* cnt, uint64_t* off, int n, uint64_t* total) {
  uint64_t acc = 0;
  for (int p = 0; p < n; ++p) { off[p] = acc; acc += cnt[p]; }
  *total = acc;
}

// ---------------------------------------------------------------------------------------------
// TKNN_SHARD_QUERIES: replicated build from per-rank slices
// ---------------------------------------------------------------------------------------------
static int build_replicated(tknn_ctx* c, const float* xyz_local, uint64_t n_local, uint64_t first, uint64_t n_total, int dim,
                            int stride) {
  TK_TRY(need_comm(c));
  State* S = c->dist;
  Comm* cm = S->comm;
  const uint64_t per = (n_total + cm->n - 1) / cm->n;  // slices are ceil(n / N) rows, the last one shorter
  const uint64_t want_first = std::min<uint64_t>(n_total, per * (uint64_t)cm->rank);
  const uint64_t want_n = std::min<uint64_t>(n_total, want_first + per) - want_first;
  int ok = TKNN_OK;
  if (!xyz_local && n_local) ok = fail(c, TKNN_EINVAL, "null point array");
  else if (dim != 2 && dim != 3) ok = fail(c, TKNN_EINVAL, "dim = %d (must be 2 or 3)", dim);
  else if (stride < dim) ok = fail(c, TKNN_EINVAL, "stride %d < dim %d", stride, dim);
  else if (n_total < 2 || n_total > rsort::MAX_N) ok = fail(c, TKNN_EINVAL, "2 <= n_total <= 2^30 - 1 points per replica");
  else if (first != want_first || n_local != want_n)
    ok = fail(c, TKNN_EINVAL, "rank %d must hold rows [%llu, %llu) of the cloud (got [%llu, %llu))", cm->rank,
              (unsigned long long)want_first, (unsigned long long)(want_first + want_n), (unsigned long long)first,
              (unsigned long long)(first + n_local));
  ScopedDevice sd(c->device);
  TK_TRY(agree(c, S, ok));
  cudaStream_t st = c->stream;
  std::memset(&S->stats, 0, sizeof(S->stats));
  S->stats.n_ranks = cm->n;
  S->stats.rank = cm->rank;
  S->stats.n_global = n_total;
  TK_TRY(ensure(c, S->dense_local, std::max<uint64_t>(per, 1) * 3 * sizeof(float)));
  TK_TRY(ensure(c, S->full_xyz, per * cm->n * 3 * sizeof(float)));
  const bool dev_in = is_device_ptr(xyz_local);
  if (!dev_in && n_local) TK_TRY(ensure(c, c->b_in, n_local * (uint64_t)stride * sizeof(float)));
  TK_TRY(mark(c, S, 0));
  const float* d_local = xyz_local;
  if (!dev_in && n_local) {
    TK_CUDA(c, cudaMemcpyAsync(c->b_in.p, xyz_local, n_local * (uint64_t)stride * sizeof(float), cudaMemcpyHostToDevice, st));
    d_local = c->b_in.as<float>();
  }
  TK_TRY(mark(c, S, 1));
  if (n_local) {
    dense_xyz_kernel<<<blocks_for(n_local, 256), 256, 0, st>>>(d_local, dim, stride, n_local, S->dense_local.as<float>());
    TK_CUDA(c, cudaGetLastError());
  }
  TK_TRY(cm->all_gather(c, S->dense_local.p, S->full_xyz.p, per * 3 * sizeof(float)));
  TK_TRY(mark(c, S, 2));
  TK_TRY(build_core(c, S->full_xyz.as<float>(), n_total, 3, 3, false));
  S->stats.h2d_ms = between(S, 0, 1);
  S->stats.allgather_ms = between(S, 1, 2);
  S->stats.lbvh_ms = c->stats.build_ms;
  S->stats.build_total_ms = S->stats.h2d_ms + S->stats.allgather_ms + c->stats.build_ms;
  S->stats.bytes_sent_build = per * 3 * sizeof(float) * (uint64_t)(cm->n - 1);
  c->stats.h2d_bytes = dev_in ? 0 : n_local * (uint64_t)stride * sizeof(float);
  c->stats.h2d_ms = S->stats.h2d_ms;
  S->partition_built = false;
  return TKNN_OK;
}

// ---------------------------------------------------------------------------------------------
// TKNN_PARTITION_POINTS: build
// ---------------------------------------------------------------------------------------------
static int partition_build(tknn_ctx* c, const float* xyz_local, uint64_t n_local, uint64_t first_index, int dim, int stride) {
  TK_TRY(need_comm(c));
  State* S = c->dist;
  Comm* cm = S->comm;
  const int n = cm->n;
  int ok = TKNN_OK;
  if (!xyz_local && n_local) ok = fail(c, TKNN_EINVAL, "null point array");
  else if (dim != 2 && dim != 3) ok = fail(c, TKNN_EINVAL, "dim = %d (must be 2 or 3)", dim);
  else if (stride < dim) ok = fail(c, TKNN_EINVAL, "stride %d < dim %d", stride, dim);
  else if (n_local > rsort::MAX_N) ok = fail(c, TKNN_EINVAL, "more than 2^30 - 1 points on one rank");
  else if (first_index + n_local > (1ull << 31)) ok = fail(c, TKNN_EINVAL, "global point indices must stay below 2^31");
  ScopedDevice sd(c->device);
  cudaStream_t st = c->stream;
  S->partition_built = false;
  TK_TRY(agree(c, S, ok));
  std::memset(&S->stats, 0, sizeof(S->stats));
  S->stats.n_ranks = n;
  S->stats.rank = cm->rank;
  uint32_t* sc = c->scalars.as<uint32_t>();

  // ---- allocations whose size is known up front (cudaMalloc is a synchronous host call) ----
  const uint64_t nl = std::max<uint64_t>(n_local, 1);
  const bool dev_in = is_device_ptr(xyz_local);
  if (!dev_in) TK_TRY(ensure(c, c->b_in, nl * (uint64_t)stride * sizeof(float)));
  TK_TRY(ensure(c, c->b_keys_a, nl * sizeof(uint64_t)));
  TK_TRY(ensure(c, c->b_keys_b, nl * sizeof(uint64_t)));
  TK_TRY(ensure(c, c->b_vals_a, nl * sizeof(uint32_t)));
  TK_TRY(ensure(c, c->b_vals_b, nl * sizeof(uint32_t)));
  TK_TRY(ensure(c, c->b_sort_tmp, rsort::temp_words(nl) * sizeof(uint32_t)));
  TK_TRY(ensure(c, S->hist, N_CELLS * sizeof(uint32_t)));
  TK_TRY(ensure(c, S->gbox, 64));
  TK_TRY(ensure(c, S->small, 16384));
  TK_TRY(ensure(c, S->rows_send, nl * sizeof(float4)));
  TK_TRY(ensure(c, S->boxes_ord, SUMMARY_BOXES * 6 * sizeof(uint32_t)));
  TK_TRY(ensure(c, S->summ_mine, SUMMARY_BOXES * 6 * sizeof(float)));
  TK_TRY(ensure(c, S->summ, (size_t)n * SUMMARY_BOXES * 6 * sizeof(float)));

  TK_TRY(mark(c, S, 0));
  const float* d_xyz = xyz_local;
  if (!dev_in && n_local) {
    TK_CUDA(c, cudaMemcpyAsync(c->b_in.p, xyz_local, n_local * (uint64_t)stride * sizeof(float), cudaMemcpyHostToDevice, st));
    d_xyz = c->b_in.as<float>();
  }
  TK_TRY(mark(c, S, 1));

  // ---- global box + global point count ----
  uint32_t* ob = S->gbox.as<uint32_t>();  // [0..2] min, [3..5] max, [6] bad flag, [7] unused; then 6 floats at +8
  float* gbox_f = reinterpret_cast<float*>(ob + 8);
  const uint32_t binit[8] = {0xffffffffu, 0xffffffffu, 0xffffffffu, 0u, 0u, 0u, 0u, 0u};
  TK_CUDA(c, cudaMemcpyAsync(ob, binit, sizeof(binit), cudaMemcpyHostToDevice, st));
  if (n_local) {
    const unsigned nb = (unsigned)std::min<uint64_t>((uint64_t)c->sm_count * 8, blocks_for(n_local, lbvh::THREADS));
    lbvh::bounds_kernel<<<nb, lbvh::THREADS, 0, st>>>(d_xyz, n_local, dim, stride, ob);
    TK_CUDA(c, cudaGetLastError());
  }
  TK_TRY(cm->all_reduce_u32(c, ob, 3, 0));
  TK_TRY(cm->all_reduce_u32(c, ob + 3, 4, 1));
  box_to_float_kernel<<<1, 32, 0, st>>>(ob, gbox_f);
  uint32_t* d_cnt = S->small.as<uint32_t>() + 2240;  // the point count as two 16-bit halves: their sums cannot wrap
  const uint32_t cnt_words[2] = {(uint32_t)(n_local & 0xffffu), (uint32_t)(n_local >> 16)};
  TK_CUDA(c, cudaMemcpyAsync(d_cnt, cnt_words, sizeof(cnt_words), cudaMemcpyHostToDevice, st));
  TK_TRY(cm->all_reduce_u32(c, d_cnt, 2, 2));
  uint32_t h_box[8];
  uint32_t h_total[2] = {0, 0};
  TK_CUDA(c, cudaMemcpyAsync(h_box, ob, sizeof(h_box), cudaMemcpyDeviceToHost, st));
  TK_CUDA(c, cudaMemcpyAsync(h_total, d_cnt, sizeof(h_total), cudaMemcpyDeviceToHost, st));
  TK_CUDA(c, cudaStreamSynchronize(st));
  if (h_box[6]) return fail(c, TKNN_EINVAL, "non-finite coordinate in the input points");
  const uint64_t n_global = (uint64_t)h_total[0] + ((uint64_t)h_total[1] << 16);
  if (n_global >= (1ull << 31)) return fail(c, TKNN_EINVAL, "the global cloud must hold fewer than 2^31 points");
  if (n_global < 2) return fail(c, TKNN_EINVAL, "need at least 2 points");
  S->n_global = n_global;
  S->stats.n_global = n_global;
  TK_TRY(mark(c, S, 2));

  // ---- Morton codes on the global grid, cell histogram ----
  uint64_t* keys = c->b_keys_a.as<uint64_t>();
  uint32_t* vals = c->b_vals_a.as<uint32_t>();
  TK_CUDA(c, cudaMemsetAsync(S->hist.p, 0, N_CELLS * sizeof(uint32_t), st));
  if (n_local) {
    lbvh::morton_kernel<<<blocks_for(n_local, lbvh::THREADS), lbvh::THREADS, 0, st>>>(d_xyz, n_local, dim, stride, ob, 21, 0, 0, keys, vals);
    cell_hist_kernel<<<blocks_for(n_local, 256), 256, 0, st>>>(keys, n_local, S->hist.as<uint32_t>());
    TK_CUDA(c, cudaGetLastError());
  }
  TK_TRY(cm->all_reduce_u32(c, S->hist.as<uint32_t>(), N_CELLS, 2));
  TK_TRY(mark(c, S, 3));

  // ---- splitters: rank r starts at the first cell whose exclusive prefix reaches r * N / n_ranks ----
  Splitters sp;
  {
    // two levels: 4096 block sums on the device, then only the blocks a splitter falls into are read back
    constexpr size_t NB = N_CELLS / SPLIT_BLOCK;
    TK_TRY(ensure(c, S->ver, NB * sizeof(uint64_t)));
    cell_block_sums_kernel<<<(unsigned)NB, 256, 0, st>>>(S->hist.as<uint32_t>(), S->ver.as<uint64_t>());
    TK_CUDA(c, cudaGetLastError());
    std::vector<uint64_t> bs(NB);
    TK_CUDA(c, cudaMemcpyAsync(bs.data(), S->ver.p, NB * sizeof(uint64_t), cudaMemcpyDeviceToHost, st));
    TK_CUDA(c, cudaStreamSynchronize(st));
    std::vector<uint32_t> blk(SPLIT_BLOCK);
    uint64_t acc = 0;    // points in the blocks before `b`
    size_t b = 0;
    for (int r = 1; r < n; ++r) {
      const uint64_t target = n_global * (uint64_t)r / (uint64_t)n;
      while (b < NB && acc + bs[b] < target) { acc += bs[b]; ++b; }  // P(first cell of block b + 1) < target: not in block b
      // rank r starts at the first cell whose exclusive prefix reaches the target: it lies in block b (or is its first cell)
      if (b >= NB) { sp.cell[r - 1] = (uint32_t)N_CELLS; continue; }
      TK_CUDA(c, cudaMemcpyAsync(blk.data(), S->hist.as<uint32_t>() + b * SPLIT_BLOCK, SPLIT_BLOCK * sizeof(uint32_t),
                                 cudaMemcpyDeviceToHost, st));
      TK_CUDA(c, cudaStreamSynchronize(st));
      uint64_t a2 = acc;
      size_t cell = 0;
      while (cell < (size_t)SPLIT_BLOCK && a2 < target) { a2 += blk[cell]; ++cell; }
      if (a2 < target) { sp.cell[r - 1] = (uint32_t)N_CELLS; continue; }  // cannot happen: the block holds the target
      sp.cell[r - 1] = (uint32_t)(b * SPLIT_BLOCK + cell);
    }
    for (int i = n - 1; i < MAX_RANKS; ++i) sp.cell[i] = 0xffffffffu;
  }
  TK_TRY(mark(c, S, 4));

  // ---- destination ranks, one onesweep pass on them, packed rows ----
  uint32_t* d_counts = S->small.as<uint32_t>() + 2112;  // n_ranks words
  TK_CUDA(c, cudaMemsetAsync(d_counts, 0, MAX_RANKS * sizeof(uint32_t), st));
  uint64_t scnt[MAX_RANKS] = {0}, soff[MAX_RANKS], rcnt[MAX_RANKS] = {0}, roff[MAX_RANKS], stotal = 0, rtotal = 0;
  if (n_local) {
    dest_kernel<<<blocks_for(n_local, 256), 256, 0, st>>>(keys, n_local, sp, n, d_counts);
    bool in_b = false;
    rsort::sort_pairs(keys, vals, c->b_keys_b.as<uint64_t>(), c->b_vals_b.as<uint32_t>(), n_local, c->b_sort_tmp.as<uint32_t>(),
                      c->sm_count, st, 1, &in_b);
    const uint32_t* order = in_b ? c->b_vals_b.as<uint32_t>() : vals;
    pack_rows_kernel<<<blocks_for(n_local, 256), 256, 0, st>>>(d_xyz, dim, stride, order, n_local, (uint32_t)first_index,
                                                              S->rows_send.as<float4>());
    TK_CUDA(c, cudaGetLastError());
  }
  {
    uint32_t hc[MAX_RANKS];
    TK_CUDA(c, cudaMemcpyAsync(hc, d_counts, MAX_RANKS * sizeof(uint32_t), cudaMemcpyDeviceToHost, st));
    TK_CUDA(c, cudaStreamSynchronize(st));
    for (int p = 0; p < n; ++p) scnt[p] = hc[p];
  }
  prefix(scnt, soff, n, &stotal);
  if (stotal != n_local) return fail(c, TKNN_ECUDA, "internal: destination counts %llu != %llu", (unsigned long long)stotal,
                                     (unsigned long long)n_local);
  TK_TRY(mark(c, S, 5));

  // ---- all-to-all of the rows ----
  TK_TRY(exchange_counts(c, S, scnt, rcnt));
  prefix(rcnt, roff, n, &rtotal);
  const uint64_t n_owned = rtotal;
  S->stats.n_owned = n_owned;
  // every rank must learn whether ANY rank cannot go on, or the next collective would hang
  uint32_t* d_flag = S->small.as<uint32_t>() + 2176;
  const uint32_t too_few = n_owned < 2 ? 1u : 0u;
  TK_CUDA(c, cudaMemcpyAsync(d_flag, &too_few, sizeof(uint32_t), cudaMemcpyHostToDevice, st));
  TK_TRY(cm->all_reduce_u32(c, d_flag, 1, 1));
  uint32_t any_few = 0;
  TK_CUDA(c, cudaMemcpyAsync(&any_few, d_flag, sizeof(uint32_t), cudaMemcpyDeviceToHost, st));
  TK_CUDA(c, cudaStreamSynchronize(st));
  if (any_few) return fail(c, TKNN_EINVAL, "a rank would own fewer than 2 points (this rank: %llu): use fewer ranks for this cloud",
                           (unsigned long long)n_owned);
  if (n_owned > rsort::MAX_N) return fail(c, TKNN_EINVAL, "this rank would own more than 2^30 - 1 points");
  TK_TRY(ensure(c, S->rows_recv, n_owned * sizeof(float4)));
  TK_TRY(cm->all_to_all_v(c, S->rows_send.p, scnt, soff, S->rows_recv.p, rcnt, roff, sizeof(float4)));
  for (int p = 0; p < n; ++p)
    if (p != cm->rank) S->stats.bytes_sent_build += scnt[p] * sizeof(float4);
  TK_TRY(mark(c, S, 6));

  // ---- local LBVH; point ids = global ids ----
  TK_TRY(build_core(c, S->rows_recv.as<float>(), n_owned, 3, 4, true));
  TK_TRY(mark(c, S, 7));

  // ---- partition summaries ----
  {
    std::vector<uint32_t> init((size_t)SUMMARY_BOXES * 6);
    for (int b = 0; b < SUMMARY_BOXES; ++b)
      for (int a = 0; a < 6; ++a) init[(size_t)b * 6 + a] = a < 3 ? 0xffffffffu : 0u;
    TK_CUDA(c, cudaMemcpyAsync(S->boxes_ord.p, init.data(), init.size() * sizeof(uint32_t), cudaMemcpyHostToDevice, st));
    cell_boxes_kernel<<<blocks_for((n_owned + CELL_RUN - 1) / CELL_RUN * 32, 256), 256, 0, st>>>(c->pts.as<float4>(), n_owned, gbox_f,
                                                                                          S->boxes_ord.as<uint32_t>());
    boxes_to_float_kernel<<<blocks_for(SUMMARY_BOXES, 128), 128, 0, st>>>(S->boxes_ord.as<uint32_t>(), SUMMARY_BOXES,
                                                                       S->summ_mine.as<float>());
    TK_CUDA(c, cudaGetLastError());
    TK_CUDA(c, cudaStreamSynchronize(st));  // `init` leaves scope
  }
  TK_TRY(cm->all_gather(c, S->summ_mine.p, S->summ.p, SUMMARY_BOXES * 6 * sizeof(float)));
  TK_TRY(mark(c, S, 8));
  TK_CUDA(c, cudaStreamSynchronize(st));
  release(S->rows_send);  // the staging rows are not needed again (the local BVH holds the points)
  release(S->rows_recv);

  tknn_dist_stats& T = S->stats;
  T.h2d_ms = between(S, 0, 1);
  T.box_ms = between(S, 1, 2);
  T.codes_ms = between(S, 2, 3);
  T.splitters_ms = between(S, 3, 4);
  T.bucket_ms = between(S, 4, 5);
  T.exchange_ms = between(S, 5, 6);
  T.lbvh_ms = between(S, 6, 7);
  T.summaries_ms = between(S, 7, 8);
  T.build_total_ms = between(S, 0, 8);
  S->partition_built = true;
  return TKNN_OK;
}

// ---------------------------------------------------------------------------------------------
// TKNN_PARTITION_POINTS: search
// ---------------------------------------------------------------------------------------------
static int partition_search(tknn_ctx* c, int k, float start_radius, int32_t* gid_out, int32_t* idx_out, float* dist_out,
                            uint64_t capacity, uint64_t* n_out) {
  TK_TRY(need_comm(c));
  State* S = c->dist;
  Comm* cm = S->comm;
  const int n = cm->n;
  if (!S->partition_built || c->n == 0) return fail(c, TKNN_ESTATE, "tknn_partition_search before tknn_partition_build");
  if (!gid_out || !idx_out || !dist_out || !n_out) return fail(c, TKNN_EINVAL, "null output array");
  const uint64_t m = c->n;
  if (capacity < m) return fail(c, TKNN_EINVAL, "output capacity %llu < %llu owned rows", (unsigned long long)capacity,
                                (unsigned long long)m);
  if (k < 1 || k > TKNN_MAX_K) return fail(c, TKNN_EINVAL, "k = %d outside [1, %d]", k, TKNN_MAX_K);
  ScopedDevice sd(c->device);
  cudaStream_t st = c->stream;
  // a rank owning <= k points could not fill its local lists, nor answer with k: every rank must agree to stop
  {
    TK_TRY(ensure(c, S->small, 16384));
    uint32_t* d_flag = S->small.as<uint32_t>() + 2176;
    const uint32_t few = m <= (uint64_t)k ? 1u : 0u;
    TK_CUDA(c, cudaMemcpyAsync(d_flag, &few, sizeof(uint32_t), cudaMemcpyHostToDevice, st));
    TK_TRY(cm->all_reduce_u32(c, d_flag, 1, 1));
    uint32_t any = 0;
    TK_CUDA(c, cudaMemcpyAsync(&any, d_flag, sizeof(uint32_t), cudaMemcpyDeviceToHost, st));
    TK_CUDA(c, cudaStreamSynchronize(st));
    if (any) return fail(c, TKNN_EINVAL, "k = %d: a rank owns no more than k points (this rank: %llu) — use fewer ranks", k,
                         (unsigned long long)m);
  }
  const bool gid_dev = is_device_ptr(gid_out), idx_dev = is_device_ptr(idx_out), dist_dev = is_device_ptr(dist_out);
  int32_t* d_gid = gid_out;
  int32_t* d_idx = idx_out;
  float* d_d2 = dist_out;
  const size_t elems = (size_t)m * k;
  if (!gid_dev) { TK_TRY(ensure(c, S->out_gid, m * sizeof(int32_t))); d_gid = S->out_gid.as<int32_t>(); }
  if (!idx_dev) { TK_TRY(ensure(c, S->out_idx, elems * sizeof(int32_t))); d_idx = S->out_idx.as<int32_t>(); }
  if (!dist_dev) { TK_TRY(ensure(c, S->out_d2, elems * sizeof(float))); d_d2 = S->out_d2.as<float>(); }
  TK_TRY(ensure(c, S->mask, m * sizeof(uint32_t)));
  uint32_t* d_counts = S->small.as<uint32_t>() + 2112;
  uint32_t* d_cursor = S->small.as<uint32_t>() + 2144;
  const float* gbox_f = reinterpret_cast<const float*>(S->gbox.as<uint32_t>() + 8);
  tknn_dist_stats& T = S->stats;
  T.boundary_sent = T.boundary_received = T.bytes_sent_search = 0;

  // ---- 1. local all-points search, squared distances, compact rows in sorted order ----
  TK_TRY(mark(c, S, 10));
  const int user_squared = c->squared;
  c->squared = 1;
  const int rc_local = search_range(c, k, start_radius, 0, m, 1, d_gid, d_idx, d_d2, m);
  c->squared = user_squared;
  TK_TRY(rc_local);
  const tknn_stats local_stats = c->stats;
  TK_TRY(mark(c, S, 11));

  uint64_t scnt[MAX_RANKS] = {0}, soff[MAX_RANKS], rcnt[MAX_RANKS] = {0}, roff[MAX_RANKS], stotal = 0, rtotal = 0;
  if (n > 1) {
    // ---- 2. which remote ranks can each ball reach; boundary queries grouped by destination ----
    TK_CUDA(c, cudaMemsetAsync(d_counts, 0, MAX_RANKS * sizeof(uint32_t), st));
    reach_kernel<<<blocks_for(m, 256), 256, 0, st>>>(c->pts.as<float4>(), m, d_idx, d_d2, k, gbox_f, S->summ.as<float>(), n, cm->rank,
                                                    S->mask.as<uint32_t>(), d_counts);
    TK_CUDA(c, cudaGetLastError());
    uint32_t hc[MAX_RANKS];
    TK_CUDA(c, cudaMemcpyAsync(hc, d_counts, MAX_RANKS * sizeof(uint32_t), cudaMemcpyDeviceToHost, st));
    TK_CUDA(c, cudaStreamSynchronize(st));
    for (int p = 0; p < n; ++p) scnt[p] = hc[p];
    prefix(scnt, soff, n, &stotal);
    TK_TRY(ensure(c, S->brows, std::max<uint64_t>(stotal, 1) * sizeof(uint32_t)));
    TK_TRY(ensure(c, S->payload, std::max<uint64_t>(stotal, 1) * sizeof(float4)));
    uint32_t cur[MAX_RANKS];
    for (int p = 0; p < MAX_RANKS; ++p) cur[p] = p < n ? (uint32_t)soff[p] : 0u;
    TK_CUDA(c, cudaMemcpyAsync(d_cursor, cur, sizeof(cur), cudaMemcpyHostToDevice, st));
    if (stotal) {
      boundary_scatter_kernel<<<blocks_for(m, 256), 256, 0, st>>>(c->pts.as<float4>(), m, d_idx, d_d2, k, S->mask.as<uint32_t>(), n,
                                                                 d_cursor, S->brows.as<uint32_t>(), S->payload.as<float4>());
      TK_CUDA(c, cudaGetLastError());
    }
    TK_TRY(mark(c, S, 12));

    // ---- 3. boundary queries out ----
    TK_TRY(exchange_counts(c, S, scnt, rcnt));
    prefix(rcnt, roff, n, &rtotal);
    TK_TRY(ensure(c, S->recv_q, std::max<uint64_t>(rtotal, 1) * sizeof(float4)));
    TK_TRY(cm->all_to_all_v(c, S->payload.p, scnt, soff, S->recv_q.p, rcnt, roff, sizeof(float4)));
    T.boundary_sent = stotal;
    T.boundary_received = rtotal;
    TK_TRY(mark(c, S, 13));

    // ---- 4. remote search: closed cap at the asker's k-th d2; the answers carry global ids already ----
    TK_TRY(ensure(c, S->ans_idx, std::max<uint64_t>(rtotal, 1) * k * sizeof(int32_t)));
    TK_TRY(ensure(c, S->ans_d2, std::max<uint64_t>(rtotal, 1) * k * sizeof(float)));
    TK_TRY(ensure(c, S->cap, std::max<uint64_t>(rtotal, 1) * sizeof(float)));
    if (rtotal) {
      column_w_kernel<<<blocks_for(rtotal, 256), 256, 0, st>>>(S->recv_q.as<float4>(), rtotal, S->cap.as<float>());
      TK_CUDA(c, cudaGetLastError());
      c->squared = 1;
      const int rc_q = tknn_query(c, S->recv_q.as<float>(), rtotal, 3, 4, nullptr, S->cap.as<float>(), k, 0.0f, S->ans_idx.as<int32_t>(),
                                  S->ans_d2.as<float>());
      c->squared = user_squared;
      TK_TRY(rc_q);
    }
    TK_TRY(mark(c, S, 14));

    // ---- 5. answers back along the same routes ----
    TK_TRY(ensure(c, S->back_idx, std::max<uint64_t>(stotal, 1) * k * sizeof(int32_t)));
    TK_TRY(ensure(c, S->back_d2, std::max<uint64_t>(stotal, 1) * k * sizeof(float)));
    TK_TRY(cm->all_to_all_v(c, S->ans_idx.p, rcnt, roff, S->back_idx.p, scnt, soff, (size_t)k * sizeof(int32_t)));
    TK_TRY(cm->all_to_all_v(c, S->ans_d2.p, rcnt, roff, S->back_d2.p, scnt, soff, (size_t)k * sizeof(float)));
    for (int p = 0; p < n; ++p)
      if (p != cm->rank) T.bytes_sent_search += scnt[p] * sizeof(float4) + rcnt[p] * (uint64_t)k * 8;
    TK_TRY(mark(c, S, 15));

    // ---- 6. merge, one destination rank at a time (a row appears at most once per rank) ----
    for (int p = 0; p < n; ++p) {
      if (p == cm->rank || scnt[p] == 0) continue;
      merge_reply_kernel<<<blocks_for(scnt[p], 128), 128, 0, st>>>(S->brows.as<uint32_t>() + soff[p], scnt[p],
                                                                  S->back_idx.as<int32_t>() + soff[p] * k,
                                                                  S->back_d2.as<float>() + soff[p] * k, k, d_idx, d_d2);
    }
    TK_CUDA(c, cudaGetLastError());
  } else {
    for (int i = 12; i <= 15; ++i) TK_TRY(mark(c, S, i));
  }
  TK_TRY(mark(c, S, 16));
  if (!user_squared) {
    const int vec = (reinterpret_cast<uintptr_t>(d_d2) & 15u) == 0;  // caller-provided arrays may be unaligned
    sqrt_rows_kernel<<<blocks_for(vec ? elems / 4 + 4 : elems, 256), 256, 0, st>>>(d_d2, elems, vec);
    TK_CUDA(c, cudaGetLastError());
  }
  TK_TRY(mark(c, S, 17));
  uint64_t d2h = 0;
  if (!gid_dev) { TK_CUDA(c, cudaMemcpyAsync(gid_out, d_gid, m * sizeof(int32_t), cudaMemcpyDeviceToHost, st)); d2h += m * 4; }
  if (!idx_dev) { TK_CUDA(c, cudaMemcpyAsync(idx_out, d_idx, elems * sizeof(int32_t), cudaMemcpyDeviceToHost, st)); d2h += elems * 4; }
  if (!dist_dev) { TK_CUDA(c, cudaMemcpyAsync(dist_out, d_d2, elems * sizeof(float), cudaMemcpyDeviceToHost, st)); d2h += elems * 4; }
  TK_TRY(mark(c, S, 18));
  TK_CUDA(c, cudaStreamSynchronize(st));
  *n_out = m;
  T.local_search_ms = between(S, 10, 11);
  T.reach_ms = between(S, 11, 12);
  T.exchange_out_ms = between(S, 12, 13);
  T.remote_search_ms = between(S, 13, 14);
  T.exchange_back_ms = between(S, 14, 15);
  T.merge_ms = between(S, 15, 16);
  T.finish_ms = between(S, 16, 17);
  T.d2h_ms = between(S, 17, 18);
  T.search_total_ms = between(S, 10, 17);
  // the context's search statistics describe the local search (rounds, radius, per-round times) with the whole time
  c->stats = local_stats;
  c->stats.search_ms = T.search_total_ms;
  c->stats.d2h_ms = T.d2h_ms;
  c->stats.d2h_bytes = d2h;
  return TKNN_OK;
}

// ---------------------------------------------------------------------------------------------
// TKNN_PARTITION_POINTS: distributed brute-force verification of sampled rows
// ---------------------------------------------------------------------------------------------
static int partition_verify(tknn_ctx* c, int k, int samples, const int32_t* gid, const int32_t* idx, const float* dist,
                            uint64_t n_rows, uint64_t* n_checked, uint64_t* n_bad) {
  TK_TRY(need_comm(c));
  State* S = c->dist;
  Comm* cm = S->comm;
  const int n = cm->n;
  if (!S->partition_built) return fail(c, TKNN_ESTATE, "tknn_partition_verify before tknn_partition_build");
  if (!gid || !idx || !dist) return fail(c, TKNN_EINVAL, "null array");
  if (n_rows != c->n) return fail(c, TKNN_EINVAL, "n_rows %llu != %llu owned rows", (unsigned long long)n_rows, (unsigned long long)c->n);
  if (samples < 1 || samples > 65536 || (uint64_t)samples > n_rows) return fail(c, TKNN_EINVAL, "samples outside [1, min(65536, rows)]");
  if (k < 1 || k > TKNN_MAX_K) return fail(c, TKNN_EINVAL, "bad k");
  ScopedDevice sd(c->device);
  cudaStream_t st = c->stream;
  const size_t SQ = (size_t)samples, ALL = SQ * n;
  // layout of the scratch: q_mine[S] | q_all[ALL] | res_idx[S*k] | res_dist[S*k] | part_idx[ALL*k] | part_d2[ALL*k] |
  //                        gath_idx[n*ALL*k] | gath_d2[n*ALL*k] | mine_idx[n*S*k] | mine_d2[n*S*k] | out_idx[S*k] | out_d2[S*k]
  size_t off = 0;
  auto take = [&](size_t bytes) { const size_t o = off; off += (bytes + 255) / 256 * 256; return o; };
  const size_t o_qm = take(SQ * sizeof(float4)), o_qa = take(ALL * sizeof(float4)), o_ri = take(SQ * k * 4), o_rd = take(SQ * k * 4),
               o_pi = take(ALL * k * 4), o_pd = take(ALL * k * 4), o_gi = take((size_t)n * ALL * k * 4), o_gd = take((size_t)n * ALL * k * 4),
               o_mi = take((size_t)n * SQ * k * 4), o_md = take((size_t)n * SQ * k * 4), o_oi = take(SQ * k * 4), o_od = take(SQ * k * 4);
  TK_TRY(ensure(c, S->ver, off));
  char* base = S->ver.as<char>();
  float4* q_mine = reinterpret_cast<float4*>(base + o_qm);
  float4* q_all = reinterpret_cast<float4*>(base + o_qa);
  int32_t* res_idx = reinterpret_cast<int32_t*>(base + o_ri);
  float* res_dist = reinterpret_cast<float*>(base + o_rd);
  int32_t* part_idx = reinterpret_cast<int32_t*>(base + o_pi);
  float* part_d2 = reinterpret_cast<float*>(base + o_pd);
  int32_t* gath_idx = reinterpret_cast<int32_t*>(base + o_gi);
  float* gath_d2 = reinterpret_cast<float*>(base + o_gd);
  int32_t* mine_idx = reinterpret_cast<int32_t*>(base + o_mi);
  float* mine_d2 = reinterpret_cast<float*>(base + o_md);
  int32_t* out_idx = reinterpret_cast<int32_t*>(base + o_oi);
  float* out_d2 = reinterpret_cast<float*>(base + o_od);

  // the sampled rows of the result (query point, its global id, its answer)
  std::vector<int32_t> h_ridx(SQ * k);
  std::vector<float> h_rdist(SQ * k);
  std::vector<float4> h_q(SQ);
  if (is_device_ptr(gid) && is_device_ptr(idx) && is_device_ptr(dist)) {
    sample_rows_kernel<<<blocks_for(SQ, 256), 256, 0, st>>>(c->pts.as<float4>(), gid, idx, dist, n_rows, samples, k, q_mine, res_idx, res_dist);
    TK_CUDA(c, cudaGetLastError());
    TK_CUDA(c, cudaMemcpyAsync(h_ridx.data(), res_idx, SQ * k * 4, cudaMemcpyDeviceToHost, st));
    TK_CUDA(c, cudaMemcpyAsync(h_rdist.data(), res_dist, SQ * k * 4, cudaMemcpyDeviceToHost, st));
    TK_CUDA(c, cudaStreamSynchronize(st));
  } else if (!is_device_ptr(gid) && !is_device_ptr(idx) && !is_device_ptr(dist)) {
    for (size_t t = 0; t < SQ; ++t) {
      const uint64_t r = n_rows * (uint64_t)t / (uint64_t)samples;
      TK_CUDA(c, cudaMemcpyAsync(&h_q[t], c->pts.as<float4>() + r, sizeof(float4), cudaMemcpyDeviceToHost, st));
      std::memcpy(&h_ridx[t * k], idx + r * (uint64_t)k, (size_t)k * 4);
      std::memcpy(&h_rdist[t * k], dist + r * (uint64_t)k, (size_t)k * 4);
    }
    TK_CUDA(c, cudaStreamSynchronize(st));
    for (size_t t = 0; t < SQ; ++t) {
      const uint64_t r = n_rows * (uint64_t)t / (uint64_t)samples;
      std::memcpy(&h_q[t].w, &gid[r], 4);
    }
    TK_CUDA(c, cudaMemcpyAsync(q_mine, h_q.data(), SQ * sizeof(float4), cudaMemcpyHostToDevice, st));
  } else {
    return fail(c, TKNN_EINVAL, "gid / idx / dist must all be host or all be device arrays");
  }
  // every rank brute-forces ALL sampled queries against its own points
  TK_TRY(cm->all_gather(c, q_mine, q_all, SQ * sizeof(float4)));
  TK_TRY(brute_core(c, q_all, ALL, k, nullptr, part_idx, part_d2, 1));
  TK_TRY(cm->all_gather(c, part_idx, gath_idx, ALL * k * 4));
  TK_TRY(cm->all_gather(c, part_d2, gath_d2, ALL * k * 4));
  // my samples' partial lists, one block per answering rank: [n][S][k]
  for (int p = 0; p < n; ++p) {
    TK_CUDA(c, cudaMemcpyAsync(mine_idx + (size_t)p * SQ * k, gath_idx + ((size_t)p * ALL + (size_t)cm->rank * SQ) * k, SQ * k * 4,
                               cudaMemcpyDeviceToDevice, st));
    TK_CUDA(c, cudaMemcpyAsync(mine_d2 + (size_t)p * SQ * k, gath_d2 + ((size_t)p * ALL + (size_t)cm->rank * SQ) * k, SQ * k * 4,
                               cudaMemcpyDeviceToDevice, st));
  }
  const size_t smem = (size_t)k * 32 * sizeof(uint64_t);
  TK_CUDA(c, cudaFuncSetAttribute(brute::merge_lists_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  brute::merge_lists_kernel<<<blocks_for(SQ, 32), 32, smem, st>>>(mine_idx, mine_d2, n, (uint32_t)SQ, k, 1, out_idx, out_d2);
  TK_CUDA(c, cudaGetLastError());
  std::vector<int32_t> h_oidx(SQ * k);
  std::vector<float> h_od2(SQ * k);
  TK_CUDA(c, cudaMemcpyAsync(h_oidx.data(), out_idx, SQ * k * 4, cudaMemcpyDeviceToHost, st));
  TK_CUDA(c, cudaMemcpyAsync(h_od2.data(), out_d2, SQ * k * 4, cudaMemcpyDeviceToHost, st));
  TK_CUDA(c, cudaStreamSynchronize(st));
  uint32_t bad = 0;
  long long first_bad = -1;
  for (size_t t = 0; t < SQ; ++t) {
    bool ok = true;
    for (int i = 0; i < k && ok; ++i) {
      const int32_t wi = h_oidx[t * k + i];
      const float wd = wi >= 0 ? (c->squared ? h_od2[t * k + i] : sqrtf(h_od2[t * k + i])) : FLT_MAX;
      ok = h_ridx[t * k + i] == wi && h_rdist[t * k + i] == wd;
    }
    if (!ok) { ++bad; if (first_bad < 0) first_bad = (long long)t; }
  }
  uint32_t* d_sum = S->small.as<uint32_t>() + 2200;
  const uint32_t mine[2] = {(uint32_t)SQ, bad};
  TK_CUDA(c, cudaMemcpyAsync(d_sum, mine, sizeof(mine), cudaMemcpyHostToDevice, st));
  TK_TRY(cm->all_reduce_u32(c, d_sum, 2, 2));
  uint32_t tot[2] = {0, 0};
  TK_CUDA(c, cudaMemcpyAsync(tot, d_sum, sizeof(tot), cudaMemcpyDeviceToHost, st));
  TK_CUDA(c, cudaStreamSynchronize(st));
  if (n_checked) *n_checked = tot[0];
  if (n_bad) *n_bad = tot[1];
  if (bad) fail(c, TKNN_OK, "verify: %u of %zu sampled rows differ from the distributed brute force (first: sample %lld)", bad, SQ, first_bad);
  return TKNN_OK;
}

}  // namespace dist
}  // namespace tknn

using namespace tknn::dist;

// ---------------------------------------------------------------------------------------------
// (a) one process, all devices
// ---------------------------------------------------------------------------------------------
struct tknn_multi {
  int n = 0, mode = 0;
  std::vector<tknn_ctx*> ctx;
  std::vector<int> devices;
  LocalHub* hub = nullptr;     // in-process transport (repeated device ids)
  HostBarrier* hb = nullptr;   // rendezvous of the rank threads
  uint64_t n_points = 0;
  std::vector<DevBuf> file_idx, file_dist;  // per rank: its slice of the file-order result arrays
  std::string err;
  float times[4] = {0, 0, 0, 0};
};

namespace {

template <typename F>
int run_ranks(tknn_multi* m, F&& body) {
  std::vector<int> rc(m->n, TKNN_OK);
  std::vector<std::thread> th;
  th.reserve(m->n);
  for (int r = 0; r < m->n; ++r) th.emplace_back([&, r] { rc[r] = body(r); });
  for (auto& t : th) t.join();
  for (int r = 0; r < m->n; ++r)
    if (rc[r] != TKNN_OK) {
      m->err = "rank " + std::to_string(r) + ": " + m->ctx[r]->err;
      return rc[r];
    }
  return TKNN_OK;
}

double now_ms() {
  return std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now().time_since_epoch()).count();
}

}  // namespace

extern "C" {

int tknn_comm_unique_id(void* id128_out) {
  if (!id128_out) return TKNN_EINVAL;
  NcclApi* A = nccl_api();
  if (!A->error.empty()) return TKNN_ENCCL;
  ncclUniqueId id;
  if (A->GetUniqueId(&id) != ncclSuccess) return TKNN_ENCCL;
  static_assert(sizeof(id) == TKNN_UNIQUE_ID_BYTES, "ncclUniqueId size");
  std::memcpy(id128_out, &id, sizeof(id));
  return TKNN_OK;
}

int tknn_comm_init(tknn_ctx* c, int n_ranks, int rank, const void* id128) {
  if (!c) return TKNN_EINVAL;
  if (!id128 || n_ranks < 1 || n_ranks > MAX_RANKS || rank < 0 || rank >= n_ranks)
    return fail(c, TKNN_EINVAL, "tknn_comm_init: 1 <= n_ranks <= %d, 0 <= rank < n_ranks, id not null", MAX_RANKS);
  NcclApi* A = nccl_api();
  if (!A->error.empty()) return fail(c, TKNN_ENCCL, "%s", A->error.c_str());
  ScopedDevice sd(c->device);
  if (c->dist) { free_state(c->dist); c->dist = nullptr; }
  State* S = new (std::nothrow) State();
  if (!S) return TKNN_ENOMEM;
  NcclComm* cm = new (std::nothrow) NcclComm();
  if (!cm) { delete S; return TKNN_ENOMEM; }
  cm->rank = rank;
  cm->n = n_ranks;
  S->comm = cm;
  c->dist = S;
  ncclUniqueId id;
  std::memcpy(&id, id128, sizeof(id));
  TK_NCCL(c, A->CommInitRank(&cm->comm, n_ranks, id, rank));
  return TKNN_OK;
}

int tknn_get_dist_stats(const tknn_ctx* c, tknn_dist_stats* out) {
  if (!c || !out) return TKNN_EINVAL;
  if (!c->dist) return TKNN_ESTATE;
  *out = c->dist->stats;
  return TKNN_OK;
}

int tknn_build_replicated(tknn_ctx* c, const float* xyz_local, uint64_t n_local, uint64_t first, uint64_t n_total, int dim,
                          int stride_floats) {
  return build_replicated(c, xyz_local, n_local, first, n_total, dim, stride_floats);
}

int tknn_partition_build(tknn_ctx* c, const float* xyz_local, uint64_t n_local, uint64_t first_index, int dim, int stride_floats) {
  return partition_build(c, xyz_local, n_local, first_index, dim, stride_floats);
}

uint64_t tknn_partition_owned(const tknn_ctx* c) { return (c && c->dist && c->dist->partition_built) ? c->n : 0; }

int tknn_partition_search(tknn_ctx* c, int k, float start_radius, int32_t* gid_out, int32_t* idx_out, float* dist_out,
                          uint64_t capacity, uint64_t* n_out) {
  if (c && c->segmented) return fail(c, TKNN_ESTATE, "tknn_partition_search: segmented builds (tknn_build_segments) do not support it yet");
  return partition_search(c, k, start_radius, gid_out, idx_out, dist_out, capacity, n_out);
}

int tknn_partition_verify(tknn_ctx* c, int k, int samples, const int32_t* gid, const int32_t* idx, const float* dist, uint64_t n_rows,
                          uint64_t* n_checked, uint64_t* n_bad) {
  if (c && c->segmented) return fail(c, TKNN_ESTATE, "tknn_partition_verify: segmented builds (tknn_build_segments) do not support it yet");
  return partition_verify(c, k, samples, gid, idx, dist, n_rows, n_checked, n_bad);
}

// called by tknn_build and tknn_build_segments (trueknn.cu): a plain build replaces whatever a partitioned build left in the context
void tknn_internal_dist_invalidate(tknn_ctx* c) {
  if (c && c->dist) c->dist->partition_built = false;
}

// called by tknn_destroy (trueknn.cu)
void tknn_internal_free_dist(tknn_ctx* c) {
  if (c && c->dist) { free_state(c->dist); c->dist = nullptr; }
}

// ---- one process, all devices ----
int tknn_create_multi(const int* device_ids, int n_devices, int mode, tknn_multi** out) {
  if (!out) return TKNN_EINVAL;
  *out = nullptr;
  if (!device_ids || n_devices < 1 || n_devices > MAX_RANKS) return TKNN_EINVAL;
  if (mode != TKNN_SHARD_QUERIES && mode != TKNN_PARTITION_POINTS) return TKNN_EINVAL;
  tknn_multi* m = new (std::nothrow) tknn_multi();
  if (!m) return TKNN_ENOMEM;
  m->n = n_devices;
  m->mode = mode;
  m->devices.assign(device_ids, device_ids + n_devices);
  m->file_idx.resize(n_devices);
  m->file_dist.resize(n_devices);
  for (int r = 0; r < n_devices; ++r) {
    tknn_ctx* c = nullptr;
    const int rc = tknn_create(device_ids[r], &c);
    if (rc != TKNN_OK) { tknn_multi_destroy(m); return rc; }
    m->ctx.push_back(c);
  }
  bool distinct = true;
  for (int a = 0; a < n_devices; ++a)
    for (int b = a + 1; b < n_devices; ++b) distinct = distinct && device_ids[a] != device_ids[b];
  // peer access between distinct devices: result rows are stored straight into the owner's arrays
  for (int a = 0; a < n_devices; ++a)
    for (int b = 0; b < n_devices; ++b) {
      if (device_ids[a] == device_ids[b]) continue;
      ScopedDevice sd(device_ids[a]);
      const cudaError_t e = cudaDeviceEnablePeerAccess(device_ids[b], 0);
      if (e != cudaSuccess && e != cudaErrorPeerAccessAlreadyEnabled) {
        cudaGetLastError();
        tknn_multi_destroy(m);
        return TKNN_ECUDA;
      }
      cudaGetLastError();
    }
  m->hb = new HostBarrier();
  m->hb->n = n_devices;
  std::vector<ncclComm_t> comms(n_devices, nullptr);
  if (distinct && n_devices > 1) {
    NcclApi* A = nccl_api();
    if (!A->error.empty() || A->CommInitAll(comms.data(), n_devices, device_ids) != ncclSuccess) {
      tknn_multi_destroy(m);
      return TKNN_ENCCL;
    }
  } else {
    m->hub = new LocalHub();
    m->hub->hb.n = n_devices;
  }
  for (int r = 0; r < n_devices; ++r) {
    State* S = new State();
    if (m->hub) {
      LocalComm* lc = new LocalComm();
      lc->hub = m->hub;
      S->comm = lc;
    } else {
      NcclComm* nc = new NcclComm();
      nc->comm = comms[r];
      nc->hb = m->hb;
      S->comm = nc;
    }
    S->comm->rank = r;
    S->comm->n = n_devices;
    m->ctx[r]->dist = S;
  }
  *out = m;
  return TKNN_OK;
}

int tknn_multi_destroy(tknn_multi* m) {
  if (!m) return TKNN_EINVAL;
  for (size_t r = 0; r < m->ctx.size(); ++r) {
    ScopedDevice sd(m->devices[r]);
    release(m->file_idx[r]);
    release(m->file_dist[r]);
    tknn_destroy(m->ctx[r]);
  }
  delete m->hub;
  delete m->hb;
  delete m;
  return TKNN_OK;
}

int tknn_multi_ranks(const tknn_multi* m) { return m ? m->n : 0; }
tknn_ctx* tknn_multi_ctx(tknn_multi* m, int rank) { return (m && rank >= 0 && rank < m->n) ? m->ctx[rank] : nullptr; }
const char* tknn_multi_last_error(const tknn_multi* m) { return m ? m->err.c_str() : "null handle"; }

int tknn_multi_set_option(tknn_multi* m, int key, int64_t value) {
  if (!m) return TKNN_EINVAL;
  for (int r = 0; r < m->n; ++r) {
    const int rc = tknn_set_option(m->ctx[r], key, value);
    if (rc != TKNN_OK) { m->err = m->ctx[r]->err; return rc; }
  }
  return TKNN_OK;
}

int tknn_multi_get_times(const tknn_multi* m, float* ms4) {
  if (!m || !ms4) return TKNN_EINVAL;
  std::memcpy(ms4, m->times, sizeof(m->times));
  return TKNN_OK;
}

int tknn_multi_build(tknn_multi* m, const float* xyz, uint64_t n, int dim, int stride_floats) {
  if (!m) return TKNN_EINVAL;
  if (!xyz || (dim != 2 && dim != 3) || stride_floats < dim) { m->err = "tknn_multi_build: bad arguments"; return TKNN_EINVAL; }
  if (n < 2 || n >= (1ull << 31)) { m->err = "tknn_multi_build: 2 <= n < 2^31"; return TKNN_EINVAL; }
  if (is_device_ptr(xyz)) { m->err = "tknn_multi_build takes a host array (each rank uploads its slice)"; return TKNN_EINVAL; }
  m->n_points = 0;
  const uint64_t per = (n + m->n - 1) / m->n;
  const double t0 = now_ms();
  const int rc = run_ranks(m, [&](int r) {
    const uint64_t first = std::min<uint64_t>(n, per * (uint64_t)r);
    const uint64_t cnt = std::min<uint64_t>(n, first + per) - first;
    const float* slice = xyz + first * (uint64_t)stride_floats;
    if (m->mode == TKNN_SHARD_QUERIES) return build_replicated(m->ctx[r], slice, cnt, first, n, dim, stride_floats);
    return partition_build(m->ctx[r], slice, cnt, first, dim, stride_floats);
  });
  m->times[0] = (float)(now_ms() - t0);
  if (rc == TKNN_OK) m->n_points = n;
  return rc;
}

int tknn_multi_search(tknn_multi* m, int k, float start_radius, int32_t* idx_out, float* dist_out) {
  if (!m) return TKNN_EINVAL;
  if (m->n_points == 0) { m->err = "tknn_multi_search before tknn_multi_build"; return TKNN_ESTATE; }
  if (!idx_out || !dist_out) { m->err = "null output array"; return TKNN_EINVAL; }
  if (is_device_ptr(idx_out) || is_device_ptr(dist_out)) { m->err = "tknn_multi_search writes host arrays"; return TKNN_EINVAL; }
  if (k < 1 || k > TKNN_MAX_K || (uint64_t)k > m->n_points - 1) { m->err = "k outside [1, min(n - 1, 512)]"; return TKNN_EINVAL; }
  const uint64_t n = m->n_points;
  const uint64_t per = (n + m->n - 1) / m->n;  // owner of file-order row i = i / per
  // every rank's slice of the file-order arrays, allocated before any rank starts storing into its peers'
  for (int r = 0; r < m->n; ++r) {
    ScopedDevice sd(m->devices[r]);
    int rc = ensure(m->ctx[r], m->file_idx[r], per * (uint64_t)k * sizeof(int32_t));
    if (rc == TKNN_OK) rc = ensure(m->ctx[r], m->file_dist[r], per * (uint64_t)k * sizeof(float));
    if (rc != TKNN_OK) { m->err = m->ctx[r]->err; return rc; }
  }
  PeerTable peers;
  std::memset(&peers, 0, sizeof(peers));
  for (int r = 0; r < m->n; ++r) { peers.idx[r] = m->file_idx[r].as<int32_t>(); peers.dist[r] = m->file_dist[r].as<float>(); }
  std::vector<double> t_search(m->n, 0.0), t_exch(m->n, 0.0), t_copy(m->n, 0.0);
  const double t0 = now_ms();
  const int rc = run_ranks(m, [&](int r) -> int {
    tknn_ctx* c = m->ctx[r];
    State* S = c->dist;
    ScopedDevice sd(c->device);
    uint64_t rows = 0;
    int32_t *d_qid = nullptr, *d_idx = nullptr;
    float* d_dist = nullptr;
    if (m->mode == TKNN_SHARD_QUERIES) {
      const uint64_t cap = tknn_shard_capacity(n, m->n);
      TK_TRY(ensure(c, S->out_gid, cap * sizeof(int32_t)));
      TK_TRY(ensure(c, S->out_idx, cap * (uint64_t)k * sizeof(int32_t)));
      TK_TRY(ensure(c, S->out_d2, cap * (uint64_t)k * sizeof(float)));
      d_qid = S->out_gid.as<int32_t>(); d_idx = S->out_idx.as<int32_t>(); d_dist = S->out_d2.as<float>();
      TK_TRY(tknn_search_shard(c, k, start_radius, r, m->n, d_qid, d_idx, d_dist, &rows));
    } else {
      const uint64_t cap = c->n;
      TK_TRY(ensure(c, S->out_gid, cap * sizeof(int32_t)));
      TK_TRY(ensure(c, S->out_idx, cap * (uint64_t)k * sizeof(int32_t)));
      TK_TRY(ensure(c, S->out_d2, cap * (uint64_t)k * sizeof(float)));
      d_qid = S->out_gid.as<int32_t>(); d_idx = S->out_idx.as<int32_t>(); d_dist = S->out_d2.as<float>();
      TK_TRY(partition_search(c, k, start_radius, d_qid, d_idx, d_dist, cap, &rows));
    }
    TK_TRY(S->comm->barrier(c));
    t_search[r] = now_ms() - t0;
    // rows -> their owners' slices of the file-order arrays (peer stores), then everyone waits for everyone
    if (rows) {
      scatter_rows_kernel<<<blocks_for(rows * (uint64_t)k, 256), 256, 0, c->stream>>>(d_qid, d_idx, d_dist, rows, k, per, peers);
      TK_CUDA(c, cudaGetLastError());
    }
    TK_TRY(S->comm->barrier(c));
    t_exch[r] = now_ms() - t0;
    const uint64_t first = std::min<uint64_t>(n, per * (uint64_t)r);
    const uint64_t cnt = std::min<uint64_t>(n, first + per) - first;
    if (cnt) {
      TK_CUDA(c, cudaMemcpyAsync(idx_out + first * (uint64_t)k, m->file_idx[r].p, cnt * (uint64_t)k * sizeof(int32_t),
                                 cudaMemcpyDeviceToHost, c->stream));
      TK_CUDA(c, cudaMemcpyAsync(dist_out + first * (uint64_t)k, m->file_dist[r].p, cnt * (uint64_t)k * sizeof(float),
                                 cudaMemcpyDeviceToHost, c->stream));
      TK_CUDA(c, cudaStreamSynchronize(c->stream));
    }
    t_copy[r] = now_ms() - t0;
    return TKNN_OK;
  });
  if (rc == TKNN_OK) {
    m->times[1] = (float)*std::max_element(t_search.begin(), t_search.end());
    m->times[2] = (float)(*std::max_element(t_exch.begin(), t_exch.end()) - m->times[1]);
    m->times[3] = (float)(*std::max_element(t_copy.begin(), t_copy.end()) - m->times[1] - m->times[2]);
  }
  return rc;
}

}  // extern "C"
