// fps.cuh — exact farthest point sampling of the built cloud (tknn_fps), in two tiers chosen per segment by its size.
//
// D(p) is the smallest d2(c, p) over the samples c of p's segment so far (+inf before the first); sample i + 1 maximises
// the key (bits(D) << 32 | (0xFFFFFFFF - index)), i.e. the largest D with ties to the lowest index.  Both tiers compute
// the same D with the one distance formula and pick by the same key, so the result does not depend on the tier.
//
//   block tier  segments of at most BLOCK_CAP points: one CTA per segment stages it in shared memory, keeps D in
//               registers and runs all its iterations in one launch (warp argmax, then one __syncthreads per iteration
//               over double-buffered per-warp slots).
//   grid tier   larger segments: one cooperative kernel advances all of them in lockstep, one sample per iteration and
//               one grid barrier per iteration.  Per leaf it keeps the box and the key of its points; a leaf whose box is
//               no nearer to the new sample than its largest D is skipped (exact: RN monotonicity gives
//               box_dist2 <= d2(c, p) for every p in the box, and p changes only if d2 < D(p) <= the leaf's largest D).
#pragma once
#include <cooperative_groups.h>

#include "common.cuh"

namespace tknn {
namespace fps {

constexpr int BLOCK_CAP = 14336;      // 14 x 1024 points: 224 KB of float4, the most one CTA's shared memory holds
constexpr int MAX_PER_THREAD = 14;    // BLOCK_CAP / 1024: points (and D registers) per thread of the block tier
constexpr int BLOCK_TARGET_PER = 8;   // CTAs are sized for about 8 points per thread, so small clouds get small CTAs
constexpr int GRID_THREADS = 512;
constexpr int INIT_THREADS = 256;
constexpr uint32_t NO_SLOT = 0xFFFFFFFFu;

// one segment to sample: points at sorted positions [begin, begin + count), samples to out[0 .. m), start = global index
struct Seg {
  uint32_t begin, count, out, m;
  uint32_t start, pad0, pad1, pad2;
};

__device__ __forceinline__ uint64_t fps_key(float d2, uint32_t idx) {
  return ((uint64_t)__float_as_uint(d2) << 32) | (0xFFFFFFFFu - idx);
}
__device__ __forceinline__ uint32_t fps_key_idx(uint64_t key) { return 0xFFFFFFFFu - (uint32_t)key; }
__device__ __forceinline__ float fps_key_d2(uint64_t key) { return __uint_as_float((uint32_t)(key >> 32)); }

// largest key of the warp: the largest D bits, then the largest low word (= the lowest index) among the lanes at it
__device__ __forceinline__ uint64_t warp_max_key(uint64_t k) {
  const uint32_t hi = __reduce_max_sync(FULL_MASK, (uint32_t)(k >> 32));
  const uint32_t lo = __reduce_max_sync(FULL_MASK, (uint32_t)(k >> 32) == hi ? (uint32_t)k : 0u);
  return ((uint64_t)hi << 32) | lo;
}

__device__ __forceinline__ void write_sample(int32_t* __restrict__ idx_out, float* __restrict__ dist_out, uint32_t at,
                                             uint64_t key, int squared) {
  idx_out[at] = (int32_t)fps_key_idx(key);
  if (dist_out) {
    const float d2 = fps_key_d2(key);
    dist_out[at] = squared ? d2 : sqrtf(d2);
  }
}

// ---- block tier ----------------------------------------------------------------------------------------------------
// One CTA per segment.  Dynamic shared memory: the CTA's count rows of float4 (sized for the largest segment of the
// launch), then 2 x 32 u64 warp keys and 2 x 32 u32 warp positions (double-buffered by iteration parity, so a warp
// that runs ahead into iteration i + 1 never overwrites the slots another warp still reads for iteration i).
static __global__ void __launch_bounds__(1024) fps_block_kernel(const float4* __restrict__ pts, const Seg* __restrict__ segs,
                                                               uint32_t pts_cap, int32_t* __restrict__ idx_out,
                                                               float* __restrict__ dist_out, int squared) {
  extern __shared__ float4 s_pts[];
  __shared__ uint32_t s_start;
  uint64_t* s_key = reinterpret_cast<uint64_t*>(s_pts + pts_cap);
  uint32_t* s_pos = reinterpret_cast<uint32_t*>(s_key + 2 * WARP);
  const Seg sg = segs[blockIdx.x];
  const uint32_t T = blockDim.x, tid = threadIdx.x, lane = tid & 31u, warp = tid >> 5, nw = T >> 5;
  for (uint32_t i = tid; i < sg.count; i += T) {
    const float4 p = __ldg(&pts[sg.begin + i]);
    s_pts[i] = p;
    if (__float_as_uint(p.w) == sg.start) s_start = i;
  }
  if (tid == 0) {
    idx_out[sg.out] = (int32_t)sg.start;
    if (dist_out) dist_out[sg.out] = FLT_MAX;
  }
  float D[MAX_PER_THREAD];
#pragma unroll
  for (int k = 0; k < MAX_PER_THREAD; ++k) D[k] = INFINITY;
  __syncthreads();
  float4 c = s_pts[s_start];
  for (uint32_t i = 1; i < sg.m; ++i) {
    uint64_t best = 0;
    uint32_t bpos = 0;
#pragma unroll
    for (int k = 0; k < MAX_PER_THREAD; ++k) {
      const uint32_t j = tid + (uint32_t)k * T;
      if (j < sg.count) {
        const float4 p = s_pts[j];
        D[k] = fminf(D[k], dist2(c.x, c.y, c.z, p.x, p.y, p.z));
        const uint64_t key = fps_key(D[k], __float_as_uint(p.w));
        if (key > best) { best = key; bpos = j; }
      }
    }
    const uint64_t wk = warp_max_key(best);
    const uint32_t wpos = __shfl_sync(FULL_MASK, bpos, __ffs(__ballot_sync(FULL_MASK, best == wk)) - 1);
    const uint32_t buf = (i & 1u) * WARP;
    if (lane == 0) { s_key[buf + warp] = wk; s_pos[buf + warp] = wpos; }
    __syncthreads();
    const uint64_t k2 = lane < nw ? s_key[buf + lane] : 0ull;
    const uint64_t win = warp_max_key(k2);
    const uint32_t p2 = lane < nw ? s_pos[buf + lane] : 0u;
    c = s_pts[__shfl_sync(FULL_MASK, p2, __ffs(__ballot_sync(FULL_MASK, k2 == win)) - 1)];
    if (tid == 0) write_sample(idx_out, dist_out, sg.out + i, win, squared);
  }
}

// ---- grid tier: set-up ---------------------------------------------------------------------------------------------
// one bit per leaf of the BVH: the leaf belongs to a segment of the grid tier (slot_of_seg[segment] != NO_SLOT)
static __global__ void __launch_bounds__(INIT_THREADS) leaf_flag_kernel(const uint32_t* __restrict__ leaf_start, uint32_t n_leaves,
                                                                       const uint32_t* __restrict__ seg_of,
                                                                       const uint32_t* __restrict__ slot_of_seg,
                                                                       uint32_t* __restrict__ words) {
  const uint32_t leaf = blockIdx.x * INIT_THREADS + threadIdx.x;
  bool f = false;
  if (leaf < n_leaves) f = slot_of_seg[seg_of ? seg_of[leaf_start[leaf]] : 0u] != NO_SLOT;
  const uint32_t w = __ballot_sync(FULL_MASK, f);
  if ((threadIdx.x & 31u) == 0 && leaf < n_leaves) words[leaf >> 5] = w;
}

// One warp per flagged leaf: its compact record (box; lo.w = slot, hi.w = point count; first position), its key (+inf,
// lowest index), D = +inf for its points, and pos_of[index] = position for its points.
static __global__ void __launch_bounds__(INIT_THREADS) leaf_init_kernel(const float4* __restrict__ pts,
                                                                       const uint32_t* __restrict__ leaf_start, uint32_t n_leaves,
                                                                       const uint32_t* __restrict__ seg_of,
                                                                       const uint32_t* __restrict__ slot_of_seg,
                                                                       const uint32_t* __restrict__ words,
                                                                       const uint32_t* __restrict__ word_offsets,
                                                                       float4* __restrict__ leaf_lo, float4* __restrict__ leaf_hi,
                                                                       uint32_t* __restrict__ leaf_first, uint64_t* __restrict__ leaf_key,
                                                                       float* __restrict__ D, uint32_t* __restrict__ pos_of) {
  const uint32_t leaf = (uint32_t)(((uint64_t)blockIdx.x * INIT_THREADS + threadIdx.x) >> 5), lane = threadIdx.x & 31u;
  if (leaf >= n_leaves) return;
  const uint32_t w = words[leaf >> 5], bit = leaf & 31u;
  if (!((w >> bit) & 1u)) return;
  const uint32_t ci = word_offsets[leaf >> 5] + __popc(w & ((1u << bit) - 1u));
  const uint32_t b = leaf_start[leaf], cnt = leaf_start[leaf + 1] - b;
  float lx = INFINITY, ly = INFINITY, lz = INFINITY, hx = -INFINITY, hy = -INFINITY, hz = -INFINITY;
  uint32_t idx = 0xFFFFFFFFu;
  if (lane < cnt) {
    const float4 p = __ldg(&pts[b + lane]);
    lx = hx = p.x; ly = hy = p.y; lz = hz = p.z;
    idx = __float_as_uint(p.w);
    D[b + lane] = INFINITY;
    pos_of[idx] = b + lane;
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    lx = fminf(lx, __shfl_xor_sync(FULL_MASK, lx, o)); ly = fminf(ly, __shfl_xor_sync(FULL_MASK, ly, o));
    lz = fminf(lz, __shfl_xor_sync(FULL_MASK, lz, o)); hx = fmaxf(hx, __shfl_xor_sync(FULL_MASK, hx, o));
    hy = fmaxf(hy, __shfl_xor_sync(FULL_MASK, hy, o)); hz = fmaxf(hz, __shfl_xor_sync(FULL_MASK, hz, o));
  }
  const uint32_t min_idx = __reduce_min_sync(FULL_MASK, idx);
  if (lane == 0) {
    const uint32_t slot = slot_of_seg[seg_of ? seg_of[b] : 0u];
    leaf_lo[ci] = make_float4(lx, ly, lz, __uint_as_float(slot));
    leaf_hi[ci] = make_float4(hx, hy, hz, __uint_as_float(cnt));
    leaf_first[ci] = b;
    leaf_key[ci] = fps_key(INFINITY, min_idx);
  }
}

// per grid-tier segment: the three key slots (slot 0 holds sample 0 for the first iteration) and sample 0's output
static __global__ void __launch_bounds__(INIT_THREADS) slot_init_kernel(const Seg* __restrict__ segs, uint32_t n_slots,
                                                                       uint64_t* __restrict__ best, int32_t* __restrict__ idx_out,
                                                                       float* __restrict__ dist_out) {
  const uint32_t j = blockIdx.x * INIT_THREADS + threadIdx.x;
  if (j >= n_slots) return;
  const Seg sg = segs[j];
  best[j] = fps_key(0.0f, sg.start);
  best[n_slots + j] = 0;
  best[2 * (size_t)n_slots + j] = 0;
  idx_out[sg.out] = (int32_t)sg.start;
  if (dist_out) dist_out[sg.out] = FLT_MAX;
}

// ---- grid tier: the cooperative kernel -----------------------------------------------------------------------------
struct GridParams {
  const float4* pts;
  const float4* leaf_lo;
  const float4* leaf_hi;
  const uint32_t* leaf_first;
  uint64_t* leaf_key;
  float* D;
  const uint32_t* pos_of;
  const Seg* segs;          // per slot
  uint32_t n_slots;
  uint32_t max_m;           // largest sample count of the slots: iterations 1 .. max_m - 1
  const uint32_t* n_leaves; // device word: compact leaves (the popc scan's total)
  uint64_t* best;           // 3 x n_slots keys, rotated by iteration: written in it % 3, read in (it - 1) % 3, cleared
                            // in (it + 1) % 3 — that one was last read before the previous barrier, so one barrier suffices
  int32_t* idx_out;
  float* dist_out;
  int squared;
  unsigned long long* counters;  // COUNT: [0] leaf box tests, [1] point updates, [4] leaves updated
};

// Block b owns the compact leaves [nl * b / G, nl * (b + 1) / G) (leaves of a segment are contiguous, segments follow in
// slot order); its warps take 32-leaf chunks of that range in turn, one lane per leaf for the box test and the whole
// warp (one lane per point) for each leaf that needs an update.  Each chunk's leaf keys are reduced per segment into a
// running maximum that is flushed when the segment changes: into the block's shared slot for its first segment, or
// straight to the segment's global slot (atomicMax) for the others.
template <bool COUNT>
static __global__ void __launch_bounds__(GRID_THREADS) fps_grid_kernel(const GridParams P) {
  namespace cg = cooperative_groups;
  cg::grid_group grid = cg::this_grid();
  __shared__ unsigned long long s_best;
  const uint32_t lane = threadIdx.x & 31u, warp = threadIdx.x >> 5, nw = blockDim.x >> 5;
  const uint32_t nl = *P.n_leaves;
  const uint32_t bb = (uint32_t)((uint64_t)nl * blockIdx.x / gridDim.x), be = (uint32_t)((uint64_t)nl * (blockIdx.x + 1) / gridDim.x);
  const uint32_t first_slot = bb < be ? __float_as_uint(__ldg(&P.leaf_lo[bb]).w) : NO_SLOT;
  if (threadIdx.x == 0) s_best = 0;
  __syncthreads();
  unsigned long long n_box = 0, n_leaf = 0, n_pts = 0;
  for (uint32_t it = 1; it < P.max_m; ++it) {
    const uint64_t* rd = P.best + (size_t)((it - 1) % 3) * P.n_slots;
    unsigned long long* wr = reinterpret_cast<unsigned long long*>(P.best + (size_t)(it % 3) * P.n_slots);
    if (blockIdx.x == 0) {
      uint64_t* clr = P.best + (size_t)((it + 1) % 3) * P.n_slots;
      for (uint32_t j = threadIdx.x; j < P.n_slots; j += blockDim.x) {
        clr[j] = 0;
        const Seg sg = P.segs[j];
        if (it >= 2 && it - 1 < sg.m) write_sample(P.idx_out, P.dist_out, sg.out + it - 1, __ldcg(rd + j), P.squared);
      }
    }
    uint32_t run_slot = NO_SLOT;
    uint64_t run_key = 0;
    uint32_t c_slot = NO_SLOT;  // this lane's cached current sample: its slot, whether it is active, its coordinates
    bool c_act = false;
    float cx = 0.f, cy = 0.f, cz = 0.f;
    for (uint32_t base = bb + warp * WARP; base < be; base += nw * WARP) {
      const uint32_t l = base + lane;
      uint32_t slot = NO_SLOT, first = 0, cnt = 0;
      uint64_t lk = 0;
      bool need = false;
      if (l < be) {
        const float4 lo = __ldg(&P.leaf_lo[l]);
        const uint32_t s = __float_as_uint(lo.w);
        if (s != c_slot) {
          c_slot = s;
          c_act = it < P.segs[s].m;
          if (c_act) {
            const float4 q = __ldg(&P.pts[__ldg(&P.pos_of[fps_key_idx(__ldcg(rd + s))])]);
            cx = q.x; cy = q.y; cz = q.z;
          }
        }
        if (c_act) {
          slot = s;
          lk = __ldcg(&P.leaf_key[l]);
          const float4 hi = __ldg(&P.leaf_hi[l]);
          cnt = __float_as_uint(hi.w);
          if (COUNT) ++n_box;
          need = box_dist2(cx, cy, cz, lo, hi) < fps_key_d2(lk);
          if (need) first = __ldg(&P.leaf_first[l]);
        }
      }
      uint32_t todo = __ballot_sync(FULL_MASK, need);
      while (todo) {
        const int src = __ffs(todo) - 1;
        todo &= todo - 1;
        const uint32_t f = __shfl_sync(FULL_MASK, first, src), m = __shfl_sync(FULL_MASK, cnt, src);
        const float qx = __shfl_sync(FULL_MASK, cx, src), qy = __shfl_sync(FULL_MASK, cy, src),
                    qz = __shfl_sync(FULL_MASK, cz, src);
        uint64_t key = 0;
        if (lane < m) {
          const float4 p = __ldg(&P.pts[f + lane]);
          const float d = __ldcg(&P.D[f + lane]);
          const float nd = fminf(d, dist2(qx, qy, qz, p.x, p.y, p.z));
          if (nd < d) P.D[f + lane] = nd;
          key = fps_key(nd, __float_as_uint(p.w));
        }
        const uint64_t nk = warp_max_key(key);
        if (lane == (uint32_t)src) {
          lk = nk;
          P.leaf_key[l] = nk;
        }
        if (COUNT && lane == 0) { ++n_leaf; n_pts += m; }
      }
      uint32_t pending = __ballot_sync(FULL_MASK, slot != NO_SLOT);
      while (pending) {
        const uint32_t s = __shfl_sync(FULL_MASK, slot, __ffs(pending) - 1);
        const bool mine = slot == s;
        pending &= ~__ballot_sync(FULL_MASK, mine);
        const uint64_t k = warp_max_key(mine ? lk : 0ull);
        if (s != run_slot) {
          if (lane == 0 && run_slot != NO_SLOT) atomicMax(run_slot == first_slot ? &s_best : wr + run_slot, (unsigned long long)run_key);
          run_slot = s;
          run_key = k;
        } else if (k > run_key) {
          run_key = k;
        }
      }
    }
    if (lane == 0 && run_slot != NO_SLOT) atomicMax(run_slot == first_slot ? &s_best : wr + run_slot, (unsigned long long)run_key);
    __syncthreads();
    if (threadIdx.x == 0 && s_best != 0) {
      atomicMax(wr + first_slot, s_best);
      s_best = 0;
    }
    grid.sync();
  }
  if (blockIdx.x == 0 && P.max_m >= 2) {
    const uint64_t* rd = P.best + (size_t)((P.max_m - 1) % 3) * P.n_slots;
    for (uint32_t j = threadIdx.x; j < P.n_slots; j += blockDim.x) {
      const Seg sg = P.segs[j];
      if (P.max_m - 1 < sg.m) write_sample(P.idx_out, P.dist_out, sg.out + P.max_m - 1, __ldcg(rd + j), P.squared);
    }
  }
  if (COUNT) {
    if (n_box) atomicAdd(&P.counters[0], n_box);
    if (n_pts) atomicAdd(&P.counters[1], n_pts);
    if (n_leaf) atomicAdd(&P.counters[4], n_leaf);
  }
}

}  // namespace fps
}  // namespace tknn
