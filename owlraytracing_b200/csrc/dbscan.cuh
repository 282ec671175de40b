// dbscan.cuh — the small kernels of tknn_dbscan around the traversal passes of traverse.cuh.
//
// Pipeline (all on the device, positions = sorted positions of the BVH's points):
//   1. core test   traverse_kernel<MODE_DBSCAN_CORE>: one "is core" ballot word per 32 positions (the core bitset);
//                  split_queues_kernel turns it into the core queue and the non-core queue.
//   2. link        traverse_kernel<MODE_DBSCAN_LINK> over the core queue: every core point within eps of a core
//                  query is united with it in a lock-free union-find over positions (uf_unite).
//   3. labelling   flatten_kernel (every core point -> its root, atomicMin of the original index per root),
//                  mark_kernel (one bit per cluster at its smallest original index), popc scan of those bits
//                  (dense cluster ids in ascending order of the smallest core index, and C), label_core_kernel.
//   4. border      traverse_kernel<MODE_DBSCAN_BORDER> over the non-core queue: the lowest cluster id among the core
//                  points of the ball, or -1.
// Races in the union-find change only the shape of its trees, never the components, so the labels are deterministic.
#pragma once
#include "common.cuh"

namespace tknn {
namespace dbscan {

constexpr int THREADS = 256;

// ---- lock-free union-find over positions (ECL-CC style) ----------------------------------------
// Invariant: parent[x] <= x, so every chain strictly decreases and ends at a root (parent[r] == r).  Loads are volatile:
// other threads hook roots and halve paths while a find runs.  Path halving only ever writes an ancestor of x into
// parent[x], so concurrent halvings keep every chain valid.
__device__ __forceinline__ int uf_find(int* parent, int x) {
  volatile int* P = parent;
  int cur = P[x];
  if (cur != x) {
    int prev = x, next;
    while (cur > (next = P[cur])) {
      P[prev] = next;  // path halving
      prev = cur;
      cur = next;
    }
  }
  return cur;
}

// root of x without writes (the labelling pass: no concurrent unions any more)
__device__ __forceinline__ int uf_root(const int* parent, int x) {
  const volatile int* P = parent;
  int cur = P[x];
  while (cur != x) {
    x = cur;
    cur = P[x];
  }
  return cur;
}

// Hooks the larger root under the smaller one; a failed CAS means the root gained a parent meanwhile: retry from there.
// Returns 1 when this call performed the hook.
__device__ __forceinline__ int uf_unite(int* parent, int a, int b) {
  int ra = uf_find(parent, a), rb = uf_find(parent, b);
  while (ra != rb) {
    if (ra < rb) {
      const int old = atomicCAS(&parent[rb], rb, ra);
      if (old == rb) return 1;
      rb = old;
    } else {
      const int old = atomicCAS(&parent[ra], ra, rb);
      if (old == ra) return 1;
      ra = old;
    }
  }
  return 0;
}

// Bits pos0 .. pos0 + 31 of a bitset over positions: the core flags of one leaf (<= 32 consecutive positions) with at
// most two word loads.  Bits past the bitset's last word read as 0.
__device__ __forceinline__ uint32_t bits_at(const uint32_t* __restrict__ words, uint32_t n_words, uint32_t pos0) {
  const uint32_t w = pos0 >> 5, s = pos0 & 31u;
  const uint32_t lo = __ldg(&words[w]);
  const uint32_t hi = (s != 0u && w + 1 < n_words) ? __ldg(&words[w + 1]) : 0u;
  return __funnelshift_r(lo, hi, s);
}

// ---- 1. core / non-core queues, union-find and per-root minimum reset ---------------------------
// core_offsets = exclusive scan of popc(core_words).  Positions keep their order in both queues, so the groups of 32
// of either queue stay compact in space.  counts[0] = core points, counts[1] = the rest.
static __global__ void __launch_bounds__(THREADS) split_queues_kernel(const uint32_t* __restrict__ core_words,
                                                                      const uint32_t* __restrict__ core_offsets, uint64_t n,
                                                                      uint32_t* __restrict__ core_queue,
                                                                      uint32_t* __restrict__ noncore_queue,
                                                                      int* __restrict__ parent, int* __restrict__ min_idx,
                                                                      uint32_t* __restrict__ counts) {
  const uint64_t p = (uint64_t)blockIdx.x * THREADS + threadIdx.x;
  if (p >= n) return;
  const uint32_t g = (uint32_t)(p >> 5), lane = (uint32_t)(p & 31u);
  const uint32_t w = core_words[g];
  const uint32_t before = core_offsets[g] + __popc(w & ((1u << lane) - 1u));  // core points at positions < p
  if ((w >> lane) & 1u) core_queue[before] = (uint32_t)p;
  else noncore_queue[p - before] = (uint32_t)p;
  parent[p] = (int)p;
  min_idx[p] = 0x7fffffff;
  if (p == n - 1) {
    const uint32_t n_core = before + ((w >> lane) & 1u);
    counts[0] = n_core;
    counts[1] = (uint32_t)(n - n_core);
  }
}

// ---- 3. labelling -------------------------------------------------------------------------------
__device__ __forceinline__ bool is_core(const uint32_t* __restrict__ core_words, uint64_t p) {
  return (__ldg(&core_words[p >> 5]) >> (p & 31u)) & 1u;
}

// every core point points straight at its root; each root receives the smallest original index of its members
static __global__ void __launch_bounds__(THREADS) flatten_kernel(const uint32_t* __restrict__ core_words, const float4* __restrict__ pts,
                                                                 uint64_t n, int* parent, int* __restrict__ min_idx) {
  const uint64_t p = (uint64_t)blockIdx.x * THREADS + threadIdx.x;
  if (p >= n || !is_core(core_words, p)) return;
  const int r = uf_root(parent, (int)p);
  parent[p] = r;  // only this thread writes parent[p] here; readers see the old ancestor or the root
  atomicMin(&min_idx[r], __float_as_int(__ldg(&pts[p]).w));
}

// one bit per cluster, at its smallest original index (the cluster's rank among these bits is its id)
static __global__ void __launch_bounds__(THREADS) mark_kernel(const uint32_t* __restrict__ core_words, uint64_t n,
                                                              const int* __restrict__ parent, const int* __restrict__ min_idx,
                                                              uint32_t* __restrict__ cluster_bits) {
  const uint64_t p = (uint64_t)blockIdx.x * THREADS + threadIdx.x;
  if (p >= n || !is_core(core_words, p) || parent[p] != (int)p) return;
  const uint32_t m = (uint32_t)min_idx[p];
  atomicOr(&cluster_bits[m >> 5], 1u << (m & 31u));
}

// cluster id of every core point, to build order (label_out, core_out) and by position (pos_label, read by the border pass)
static __global__ void __launch_bounds__(THREADS) label_core_kernel(const uint32_t* __restrict__ core_words,
                                                                    const float4* __restrict__ pts, uint64_t n,
                                                                    const int* __restrict__ parent, const int* __restrict__ min_idx,
                                                                    const uint32_t* __restrict__ cluster_bits,
                                                                    const uint32_t* __restrict__ cluster_offsets,
                                                                    int32_t* __restrict__ pos_label, int32_t* __restrict__ label_out,
                                                                    uint8_t* __restrict__ core_out) {
  const uint64_t p = (uint64_t)blockIdx.x * THREADS + threadIdx.x;
  if (p >= n || !is_core(core_words, p)) return;
  const uint32_t m = (uint32_t)min_idx[parent[p]];
  const int32_t id = (int32_t)(cluster_offsets[m >> 5] + __popc(cluster_bits[m >> 5] & ((1u << (m & 31u)) - 1u)));
  pos_label[p] = id;
  const uint32_t row = __float_as_uint(__ldg(&pts[p]).w);
  label_out[row] = id;
  if (core_out) core_out[row] = 1;
}

}  // namespace dbscan
}  // namespace tknn
