// voxel.cuh — exact voxel-grid clustering and pooling over batches of clouds (tknn_voxel_grid, tknn_voxel_members,
// tknn_voxel_pool; torch_cluster's grid_cluster and PyG's voxel_grid / GridSampling, DESIGN.md §3.9).
//
// Raw ids (include/trueknn.h): c = sum_d (int64) fl(fl(p_d - start_d) / size_d) * m_d over the D coordinate columns and,
// for a batch, the cloud id column (size 1).  The host picks start / end, the multipliers m_d and a bound [lo, hi] of
// every raw id from the exact column box (box_kernel), and rejects inputs whose ids would leave int64 there, so the
// kernels never overflow.  Clustering: raw - lo is packed above the point index (or paired with it) and radix-sorted
// (rsort), heads of equal keys are flagged, the existing popc scan ranks them, and label_kernel scatters the dense ids,
// the CSR offsets, the lowest index of every voxel and its cloud.
//
// Pooling over members in ascending index: mean = chunked sum (chunks of 32 consecutive members, each summed from +0,
// then the chunk sums in chunk order from +0) / count; max = the first maximum in index order.  Every (voxel, column)
// is one thread of voxel_kernel, column fastest, so a warp reads consecutive columns of a row (whole sectors once
// f >= 8).  Voxels above LONG_VOXEL members first get their chunks reduced in parallel by chunk_kernel (one thread per
// (chunk, column)); fold_kernel (one warp per (long voxel, column)) then folds the chunk results in order.  Every mapping performs the contract's
// operations in the contract's order, so launch shapes cannot change a bit.
#pragma once
#include "common.cuh"

namespace tknn {
namespace voxel {

constexpr int THREADS = 256;
constexpr int CHUNK = 32;        // members per chunk of the mean's two-level sum (part of the contract)
constexpr uint32_t LONG_VOXEL = 256;  // voxels with more members reduce their chunks in parallel (chunk_kernel)
constexpr int IDX_BITS = 31;     // packed sort keys: (raw - lo) << 31 | point index

__device__ __forceinline__ uint32_t ordered(float v) {
  const uint32_t b = __float_as_uint(v);
  return (b & 0x80000000u) ? ~b : (b | 0x80000000u);
}

// Column min / max of the D coordinate columns as order-preserving words (box[d] = min, box[4 + d] = max; the caller
// sets the mins to ~0 and the maxes to 0) and the non-finite flag.
static __global__ void __launch_bounds__(THREADS) box_kernel(const float* __restrict__ p, uint64_t n, int dim, int stride,
                                                             uint32_t* __restrict__ box, uint32_t* __restrict__ bad) {
  uint32_t lo[3] = {~0u, ~0u, ~0u}, hi[3] = {0u, 0u, 0u};
  bool nf = false;
  for (uint64_t i = (uint64_t)blockIdx.x * THREADS + threadIdx.x; i < n; i += (uint64_t)gridDim.x * THREADS) {
#pragma unroll
    for (int d = 0; d < 3; ++d) {
      if (d < dim) {
        const float v = __ldg(p + i * (uint64_t)stride + d);
        if (!isfinite(v)) {
          nf = true;
        } else {
          const uint32_t o = ordered(v);
          lo[d] = min(lo[d], o);
          hi[d] = max(hi[d], o);
        }
      }
    }
  }
#pragma unroll
  for (int d = 0; d < 3; ++d) {
    lo[d] = __reduce_min_sync(FULL_MASK, lo[d]);
    hi[d] = __reduce_max_sync(FULL_MASK, hi[d]);
  }
  if ((threadIdx.x & 31) == 0) {
    for (int d = 0; d < dim; ++d) {
      if (lo[d] != ~0u) atomicMin(&box[d], lo[d]);
      if (hi[d] != 0u) atomicMax(&box[4 + d], hi[d]);
    }
  }
  if (__any_sync(FULL_MASK, nf) && (threadIdx.x & 31) == 0) *bad = 1u;
}

// last s with off[s] <= i, for off[0] = 0 <= i < off[m]
__device__ __forceinline__ uint32_t segment_of(const uint64_t* __restrict__ off, uint32_t m, uint64_t i) {
  uint32_t a = 0, b = m;  // off[a] <= i < off[b]
  while (b - a > 1) {
    const uint32_t h = (a + b) >> 1;
    if (__ldg(off + h) <= i) a = h; else b = h;
  }
  return a;
}

struct RawParams {
  const float* p;
  uint64_t n;
  int dim, stride;
  const uint64_t* seg_off;  // device offsets (n_seg + 1) of a batch, or NULL: no cloud id column
  uint32_t n_seg;
  float start[4], size[4];  // per column; column `dim` is the cloud id
  long long mult[4];
  long long lo;             // every raw id is >= lo (the host's bound)
  int packed;
  long long* raw;
  uint64_t* keys;
  uint32_t* vals;           // pair sort only
};

static __global__ void __launch_bounds__(THREADS) raw_kernel(const RawParams P) {
  const uint64_t i = (uint64_t)blockIdx.x * THREADS + threadIdx.x;
  if (i >= P.n) return;
  long long c = 0;
#pragma unroll
  for (int d = 0; d < 3; ++d)
    if (d < P.dim) {
      const float q = __fdiv_rn(__fsub_rn(__ldg(P.p + i * (uint64_t)P.stride + d), P.start[d]), P.size[d]);
      c += (long long)q * P.mult[d];  // truncation toward zero; |q| < 2^63 and no overflow (host bound)
    }
  if (P.seg_off) {
    const float s = (float)segment_of(P.seg_off, P.n_seg, i);  // < 2^24: exact
    const float q = __fdiv_rn(__fsub_rn(s, P.start[P.dim]), P.size[P.dim]);
    c += (long long)q * P.mult[P.dim];
  }
  P.raw[i] = c;
  const uint64_t u = (uint64_t)c - (uint64_t)P.lo;
  if (P.packed) {
    P.keys[i] = (u << IDX_BITS) | i;
  } else {
    P.keys[i] = u;
    P.vals[i] = (uint32_t)i;
  }
}

// words[w] bit l = sorted position 32 w + l starts a voxel (its key differs from its predecessor's)
static __global__ void __launch_bounds__(THREADS) heads_kernel(const uint64_t* __restrict__ keys, uint64_t n, int shift,
                                                               uint32_t* __restrict__ words) {
  const uint64_t i = (uint64_t)blockIdx.x * THREADS + threadIdx.x;
  bool head = false;
  if (i < n) head = i == 0 || (__ldg(keys + i) >> shift) != (__ldg(keys + i - 1) >> shift);
  const uint32_t b = __ballot_sync(FULL_MASK, head);
  if ((threadIdx.x & 31) == 0 && i < n) words[i >> 5] = b;
}

struct LabelParams {
  const uint64_t* keys;
  const uint32_t* vals;  // pair sort: the point index of every sorted position; NULL: packed keys
  uint64_t n;
  const uint32_t* words;
  const uint32_t* word_off;  // exclusive popc scan of words
  const uint64_t* seg_off;   // NULL: one cloud
  uint32_t n_seg;
  uint32_t* members;  // point index by sorted position
  int32_t* cluster;   // dense id by point index
  uint64_t* vox_off;  // nv + 1
  int32_t* first;     // lowest point index by voxel
  int32_t* vseg;      // cloud by voxel
};

static __global__ void __launch_bounds__(THREADS) label_kernel(const LabelParams P) {
  const uint64_t i = (uint64_t)blockIdx.x * THREADS + threadIdx.x;
  if (i >= P.n) return;
  const uint32_t idx = P.vals ? __ldg(P.vals + i) : (uint32_t)(__ldg(P.keys + i) & ((1ull << IDX_BITS) - 1));
  const uint32_t w = __ldg(P.words + (i >> 5)), lane = (uint32_t)(i & 31);
  const bool head = (w >> lane) & 1u;
  const uint32_t r = __ldg(P.word_off + (i >> 5)) + __popc(w & ((1u << lane) - 1u)) + (head ? 1u : 0u) - 1u;
  P.members[i] = idx;
  P.cluster[idx] = (int32_t)r;
  if (head) {
    P.vox_off[r] = i;
    P.first[r] = (int32_t)idx;
    P.vseg[r] = P.seg_off ? (int32_t)segment_of(P.seg_off, P.n_seg, idx) : 0;
  }
  if (i == P.n - 1) P.vox_off[r + 1] = P.n;
}

// chunks[v] = the 32-member chunks of voxel v when it has more than LONG_VOXEL members, else 0 (v < *nv; 0 past it);
// the long voxels are listed in longs[0 .. *n_long) in no particular order (each is pooled on its own)
static __global__ void __launch_bounds__(THREADS) long_chunks_kernel(const uint64_t* __restrict__ vox_off,
                                                                     const uint32_t* __restrict__ nv, uint64_t n,
                                                                     uint32_t* __restrict__ chunks,
                                                                     uint32_t* __restrict__ longs, uint32_t* n_long) {
  const uint64_t v = (uint64_t)blockIdx.x * THREADS + threadIdx.x;
  if (v >= n) return;
  uint32_t c = 0;
  if (v < *nv) {
    const uint64_t cnt = vox_off[v + 1] - vox_off[v];
    if (cnt > LONG_VOXEL) {
      c = (uint32_t)((cnt + CHUNK - 1) / CHUNK);
      longs[atomicAdd(n_long, 1u)] = (uint32_t)v;
    }
  }
  chunks[v] = c;
}

struct PoolParams {
  const float* x;
  int stride, f, c0, cb;       // columns [c0, c0 + cb) of this pass
  const uint32_t* members;
  const uint64_t* vox_off;
  const uint64_t* chunk_off;  // exclusive scan of long_chunks_kernel's counts (nv + 1)
  uint64_t nv, n_chunks;
  float* cs;                  // chunk results of this pass: cs[g * cb + (c - c0)]
  float* out;                 // nv x f
};

template <bool MAX>
__device__ __forceinline__ float reduce_run(const PoolParams& P, uint64_t j0, uint64_t j1, int c) {
  float a = MAX ? __ldg(P.x + (uint64_t)__ldg(P.members + j0) * P.stride + c) : 0.0f;
  for (uint64_t j = MAX ? j0 + 1 : j0; j < j1; ++j) {
    const float v = __ldg(P.x + (uint64_t)__ldg(P.members + j) * P.stride + c);
    if (MAX) a = v > a ? v : a;  // strict: the lowest index keeps a tie
    else a = __fadd_rn(a, v);
  }
  return a;
}

// one thread per (long-voxel chunk, column): the chunk's sum from +0 (or its first maximum)
template <bool MAX>
static __global__ void __launch_bounds__(THREADS) chunk_kernel(const PoolParams P) {
  const uint64_t total = P.n_chunks * (uint64_t)P.cb;
  for (uint64_t t = (uint64_t)blockIdx.x * THREADS + threadIdx.x; t < total; t += (uint64_t)gridDim.x * THREADS) {
    const uint64_t g = t / (uint64_t)P.cb;
    const int c = P.c0 + (int)(t - g * (uint64_t)P.cb);
    uint64_t a = 0, b = P.nv;  // last v with chunk_off[v] <= g
    while (b - a > 1) {
      const uint64_t h = (a + b) >> 1;
      if (__ldg(P.chunk_off + h) <= g) a = h; else b = h;
    }
    const uint64_t j0 = __ldg(P.vox_off + a) + (g - __ldg(P.chunk_off + a)) * CHUNK;
    const uint64_t j1 = min(j0 + CHUNK, __ldg(P.vox_off + a + 1));
    P.cs[t] = reduce_run<MAX>(P, j0, j1, c);
  }
}

// one thread per (short voxel, column): the members chunk by chunk (long voxels are left to fold_kernel)
template <bool MAX>
static __global__ void __launch_bounds__(THREADS) voxel_kernel(const PoolParams P) {
  const uint64_t total = P.nv * (uint64_t)P.cb;
  for (uint64_t t = (uint64_t)blockIdx.x * THREADS + threadIdx.x; t < total; t += (uint64_t)gridDim.x * THREADS) {
    const uint64_t v = t / (uint64_t)P.cb;
    const int cc = (int)(t - v * (uint64_t)P.cb), c = P.c0 + cc;
    const uint64_t j0 = __ldg(P.vox_off + v), j1 = __ldg(P.vox_off + v + 1);
    if (__ldg(P.chunk_off + v + 1) > __ldg(P.chunk_off + v)) continue;
    float a;
    if (MAX) {
      a = reduce_run<true>(P, j0, j1, c);
    } else {
      a = 0.0f;
      for (uint64_t k = j0; k < j1; k += CHUNK) a = __fadd_rn(a, reduce_run<false>(P, k, min(k + CHUNK, j1), c));
    }
    if (!MAX) a = __fdiv_rn(a, (float)(j1 - j0));
    P.out[v * (uint64_t)P.f + c] = a;
  }
}

// one warp per (long voxel, column): the chunk results in chunk order.  The lanes load 32 consecutive chunk results at a
// time and every lane folds them in order from the shuffles, so the serial chain is shuffles and adds, not loads.
template <bool MAX>
static __global__ void __launch_bounds__(THREADS) fold_kernel(const PoolParams P, const uint32_t* __restrict__ longs,
                                                              uint64_t n_long) {
  const int lane = threadIdx.x & 31;
  const uint64_t total = n_long * (uint64_t)P.cb, warps = (uint64_t)gridDim.x * (THREADS / 32);
  for (uint64_t w = ((uint64_t)blockIdx.x * THREADS + threadIdx.x) >> 5; w < total; w += warps) {
    const uint64_t li = w / (uint64_t)P.cb;
    const int cc = (int)(w - li * (uint64_t)P.cb);
    const uint32_t v = __ldg(longs + li);
    const uint64_t g0 = __ldg(P.chunk_off + v), g1 = __ldg(P.chunk_off + v + 1);
    float a = MAX ? P.cs[g0 * P.cb + cc] : 0.0f;
    for (uint64_t base = MAX ? g0 + 1 : g0; base < g1; base += 32) {
      const uint64_t g = base + lane;
      const float s = g < g1 ? P.cs[g * P.cb + cc] : 0.0f;
      const int m = g1 - base < 32 ? (int)(g1 - base) : 32;
#pragma unroll
      for (int j = 0; j < 32; ++j) {
        const float sj = __shfl_sync(FULL_MASK, s, j);
        if (j < m) {
          if (MAX) a = sj > a ? sj : a;
          else a = __fadd_rn(a, sj);
        }
      }
    }
    if (lane == 0) {
      if (!MAX) a = __fdiv_rn(a, (float)(__ldg(P.vox_off + v + 1) - __ldg(P.vox_off + v)));
      P.out[(uint64_t)v * P.f + P.c0 + cc] = a;
    }
  }
}

}  // namespace voxel
}  // namespace tknn
