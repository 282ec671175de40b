// radius.cuh — the kernels of tknn_radius_search / tknn_radius_query around the two traversal passes of traverse.cuh.
//
// Pipeline (positions = sorted positions of the query points: the BVH's own order in the all-points form, the Morton
// order of tknn_query's staging for a separate query set; rows = build order or query order):
//   1. count   traverse_kernel<MODE_RANGE_LIST_COUNT>: ball size minus self, by position and by row.
//   2. scan    exclusive u64 scans of both count arrays (scan_reduce_kernel, scan_sums_kernel, scan_apply_kernel):
//              position offsets for the key scratch, row offsets for the caller; long_rows_kernel lists the rows that
//              do not fit the shared-memory sort.
//   3. fill    traverse_kernel<MODE_RANGE_LIST>: the keys make_key(d2, index) of every row, unsorted, in position order
//              (neighbouring lanes write neighbouring rows).
//   4. order   short rows: sort_rows_warp_kernel, one warp per row, a bitonic sort in shared memory; long rows:
//              rsort::sort_pairs by key, then stably by row (long_* kernels), in batches.  Both write the sorted row to
//              the caller's row offset, split into index and distance.
// The final order depends only on the set of keys in a row, never on traversal or scheduling order.
#pragma once
#include "common.cuh"

namespace tknn {
namespace radius {

constexpr int THREADS = 256;
constexpr int SCAN_ITEMS = 8;
constexpr int SCAN_CHUNK = THREADS * SCAN_ITEMS;  // counts per block of the u64 scan
// Rows of at most SHORT_MAX keys are sorted by one warp in shared memory (8 KB a warp, 4 warps a block); longer rows go
// through the radix sort.
#ifndef TKNN_RADIUS_SHORT_MAX
#define TKNN_RADIUS_SHORT_MAX 1024
#endif
constexpr int SHORT_MAX = TKNN_RADIUS_SHORT_MAX;
constexpr int SORT_WARPS = 4;

// ---- exclusive u64 scan of u32 counts ------------------------------------------------------------------------------
__device__ __forceinline__ uint64_t block_exclusive_scan_u64(uint64_t v, uint64_t* s_warp, uint64_t* total) {
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  uint64_t x = v;
#pragma unroll
  for (int o = 1; o < 32; o <<= 1) {
    const uint64_t y = __shfl_up_sync(FULL_MASK, x, o);
    if (lane >= o) x += y;
  }
  if (lane == 31) s_warp[warp] = x;
  __syncthreads();
  if (warp == 0) {
    uint64_t w = lane < THREADS / 32 ? s_warp[lane] : 0;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
      const uint64_t y = __shfl_up_sync(FULL_MASK, w, o);
      if (lane >= o) w += y;
    }
    if (lane < THREADS / 32) s_warp[lane] = w;  // inclusive over warps
  }
  __syncthreads();
  const uint64_t before = warp ? s_warp[warp - 1] : 0;
  if (total) *total = s_warp[THREADS / 32 - 1];
  __syncthreads();
  return before + x - v;
}

// sums[b] = sum of counts[b * SCAN_CHUNK .. + SCAN_CHUNK)
static __global__ void __launch_bounds__(THREADS) scan_reduce_kernel(const uint32_t* __restrict__ counts, uint64_t n,
                                                                     uint64_t* __restrict__ sums) {
  __shared__ uint64_t s_warp[THREADS / 32];
  const uint64_t base = (uint64_t)blockIdx.x * SCAN_CHUNK + (uint64_t)threadIdx.x * SCAN_ITEMS;
  uint64_t v = 0;
#pragma unroll
  for (int i = 0; i < SCAN_ITEMS; ++i)
    if (base + i < n) v += counts[base + i];
  uint64_t total;
  block_exclusive_scan_u64(v, s_warp, &total);
  if (threadIdx.x == 0) sums[blockIdx.x] = total;
}

// one block: sums[0 .. nb) -> exclusive prefix in place; the grand total to *total_out
static __global__ void __launch_bounds__(THREADS) scan_sums_kernel(uint64_t* __restrict__ sums, uint64_t nb,
                                                                   uint64_t* __restrict__ total_out) {
  __shared__ uint64_t s_warp[THREADS / 32];
  uint64_t carry = 0;
  for (uint64_t b0 = 0; b0 < nb; b0 += THREADS) {
    const uint64_t i = b0 + threadIdx.x;
    const uint64_t v = i < nb ? sums[i] : 0;
    uint64_t tile;
    const uint64_t ex = block_exclusive_scan_u64(v, s_warp, &tile);
    if (i < nb) sums[i] = carry + ex;
    carry += tile;
  }
  if (threadIdx.x == 0) *total_out = carry;
}

// off[i] = sum of counts[0 .. i) for i in [0, n]
static __global__ void __launch_bounds__(THREADS) scan_apply_kernel(const uint32_t* __restrict__ counts, uint64_t n,
                                                                    const uint64_t* __restrict__ sums,
                                                                    const uint64_t* __restrict__ total,
                                                                    uint64_t* __restrict__ off) {
  __shared__ uint64_t s_warp[THREADS / 32];
  const uint64_t base = (uint64_t)blockIdx.x * SCAN_CHUNK + (uint64_t)threadIdx.x * SCAN_ITEMS;
  uint64_t v = 0;
#pragma unroll
  for (int i = 0; i < SCAN_ITEMS; ++i)
    if (base + i < n) v += counts[base + i];
  uint64_t run = sums[blockIdx.x] + block_exclusive_scan_u64(v, s_warp, nullptr);
#pragma unroll
  for (int i = 0; i < SCAN_ITEMS; ++i)  // the second read of the chunk hits L1
    if (base + i < n) {
      off[base + i] = run;
      run += counts[base + i];
    }
  if (blockIdx.x == 0 && threadIdx.x == 0) off[n] = *total;
}

// ---- self exclusion by position --------------------------------------------------------------------------------------
// pos_of[index] = position of the data point with that original index
static __global__ void inverse_kernel(const float4* __restrict__ pts, uint64_t n, int32_t* __restrict__ pos_of) {
  const uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) pos_of[(uint32_t)__float_as_int(pts[i].w)] = (int32_t)i;
}

// self_pos[q] = position of the data point self_sorted[q], or -1 (no exclusion: -1 or an id outside [0, n))
static __global__ void self_pos_kernel(const int32_t* __restrict__ self_sorted, uint64_t nq, const int32_t* __restrict__ pos_of,
                                       uint64_t n, int32_t* __restrict__ self_pos) {
  const uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= nq) return;
  const int32_t s = self_sorted[i];
  self_pos[i] = (s >= 0 && (uint64_t)s < n) ? pos_of[s] : -1;
}

// Rows longer than SHORT_MAX: (position, length) appended in any order (the host sorts them), and
// stats[0] = number of such rows, stats[1] = their entries (u64 words, zeroed by the caller).
static __global__ void long_rows_kernel(const uint32_t* __restrict__ cnt_pos, uint64_t nq, uint32_t* __restrict__ long_pos,
                                        uint32_t* __restrict__ long_len, unsigned long long* __restrict__ stats) {
  const uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= nq) return;
  const uint32_t c = cnt_pos[i];
  if (c > (uint32_t)SHORT_MAX) {
    const unsigned long long slot = atomicAdd(&stats[0], 1ull);
    long_pos[slot] = (uint32_t)i;
    long_len[slot] = c;
    atomicAdd(&stats[1], (unsigned long long)c);
  }
}

__device__ __forceinline__ void emit_entry(uint64_t key, uint64_t o, int squared, int32_t* __restrict__ idx_out,
                                           float* __restrict__ dist_out) {
  idx_out[o] = key_idx(key);
  if (dist_out) dist_out[o] = squared ? key_d2(key) : __fsqrt_rn(key_d2(key));
}

// ---- short rows: one warp per row, bitonic sort of the row padded to a power of two in shared memory ------------------
static __global__ void __launch_bounds__(SORT_WARPS * 32) sort_rows_warp_kernel(
    const uint64_t* __restrict__ keys, const uint64_t* __restrict__ off_pos, const uint32_t* __restrict__ cnt_pos,
    const float4* __restrict__ queries, uint64_t nq, const uint64_t* __restrict__ off_row, int squared,
    int32_t* __restrict__ idx_out, float* __restrict__ dist_out) {
  __shared__ uint64_t s_keys[SORT_WARPS][SHORT_MAX];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const uint64_t pos = (uint64_t)blockIdx.x * SORT_WARPS + warp;
  if (pos >= nq) return;
  const uint32_t len = cnt_pos[pos];
  if (len == 0 || len > (uint32_t)SHORT_MAX) return;
  const uint64_t* src = keys + off_pos[pos];
  const uint64_t dst = off_row[(uint32_t)__float_as_int(queries[pos].w)];
  if (len == 1) {
    if (lane == 0) emit_entry(src[0], dst, squared, idx_out, dist_out);
    return;
  }
  uint64_t* s = s_keys[warp];
  const uint32_t p2 = 1u << (32 - __clz(len - 1));  // len rounded up to a power of two
  for (uint32_t i = lane; i < p2; i += 32) s[i] = i < len ? src[i] : ~0ull;  // padding sorts last
  __syncwarp();
  for (uint32_t k = 2; k <= p2; k <<= 1) {
    for (uint32_t j = k >> 1; j > 0; j >>= 1) {
      for (uint32_t i = lane; i < p2 / 2; i += 32) {
        const uint32_t lo = ((i & ~(j - 1)) << 1) | (i & (j - 1)), hi = lo + j;
        const uint64_t a = s[lo], b = s[hi];
        if ((a > b) == ((lo & k) == 0)) { s[lo] = b; s[hi] = a; }
      }
      __syncwarp();
    }
  }
  for (uint32_t i = lane; i < len; i += 32) emit_entry(s[i], dst + i, squared, idx_out, dist_out);
}

// ---- long rows: a batch of rows [first, first + rows) of the sorted long-row list, boff = their global prefix --------
// keys_a / slot_a / row_of[e] for batch entry e: the key, e itself, the row's rank in the batch.  One block per row.
static __global__ void __launch_bounds__(THREADS) long_gather_kernel(const uint64_t* __restrict__ keys,
                                                                     const uint64_t* __restrict__ off_pos,
                                                                     const uint32_t* __restrict__ long_pos,
                                                                     const uint64_t* __restrict__ boff, uint32_t first,
                                                                     uint64_t* __restrict__ keys_a, uint32_t* __restrict__ slot_a,
                                                                     uint32_t* __restrict__ row_of) {
  const uint32_t r = blockIdx.x;
  const uint32_t pos = long_pos[first + r];
  const uint64_t b0 = boff[first + r] - boff[first], len = boff[first + r + 1] - boff[first + r];
  const uint64_t* src = keys + off_pos[pos];
  for (uint64_t j = threadIdx.x; j < len; j += THREADS) {
    keys_a[b0 + j] = src[j];
    slot_a[b0 + j] = (uint32_t)(b0 + j);
    row_of[b0 + j] = r;
  }
}

// after the key sort: row rank of the entry in sorted place i as the next sort's key, i as its value
static __global__ void long_rowkey_kernel(const uint32_t* __restrict__ slot_sorted, const uint32_t* __restrict__ row_of,
                                          uint64_t e, uint64_t* __restrict__ rkey, uint32_t* __restrict__ rval) {
  const uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= e) return;
  rkey[i] = row_of[slot_sorted[i]];
  rval[i] = (uint32_t)i;
}

// after the stable row sort: entry i of the batch is key_sorted[rval[i]], in row rkey[i] at rank i - (its row's start)
static __global__ void long_emit_kernel(const uint64_t* __restrict__ key_sorted, const uint64_t* __restrict__ rkey,
                                        const uint32_t* __restrict__ rval, uint64_t e, const uint32_t* __restrict__ long_pos,
                                        const uint64_t* __restrict__ boff, uint32_t first, const float4* __restrict__ queries,
                                        const uint64_t* __restrict__ off_row, int squared, int32_t* __restrict__ idx_out,
                                        float* __restrict__ dist_out) {
  const uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= e) return;
  const uint32_t r = first + (uint32_t)rkey[i];
  const uint64_t rank = i - (boff[r] - boff[first]);
  const uint64_t dst = off_row[(uint32_t)__float_as_int(queries[long_pos[r]].w)] + rank;
  emit_entry(key_sorted[rval[i]], dst, squared, idx_out, dist_out);
}

}  // namespace radius
}  // namespace tknn
