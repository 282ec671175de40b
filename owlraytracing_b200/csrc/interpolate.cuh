// interpolate.cuh — exact, deterministic k-NN interpolation over kNN rows and its backward pass (tknn_interpolate,
// tknn_interpolate_backward; PyG's knn_interpolate, the feature propagation of PointNet++, DESIGN.md §3.10).
//
// Forward, per query row i and its slots s = 0 .. k-1 in slot order (idx = -1 slots skipped):
//   w[i,s] = fl(1 / max(d2[i,s], 1e-16)),  den[i] = sum_s w[i,s],  out[i,c] = fl(sum_s fl(x[idx[i,s], c] * w[i,s]) / den[i])
// every sum from +0 in slot order, every product rounded on its own (no FMA).  One group of G lanes per row
// (G = 32 for f > 16, else the next power of two >= f, at least 4; 32 / G rows per warp): the lanes load G slots at a
// time, share them by shuffle and walk the columns in blocks of G, each lane folding its column in slot order.
//
// Backward: grad_x[j,c] = sum over the edges e = i*k + s with idx[i,s] = j, in ascending e, from +0, of
// fl(fl(grad_out[i,c] / den[i]) * w[i,s]) (PyG's autograd chain evaluated in edge order).
//   1. edge_kernel:   key j and value e per edge (a -1 slot gets the key n, which sorts behind every data row), the
//                     number of edges of every j (integer atomics: exact in any order).
//   2. rsort::sort_pairs by j, ceil(bits(n) / 8) passes.  Stable, input in ascending e: each run comes out in ascending e.
//   3. the u64 scan of radius.cuh turns the counts into run offsets.
//   4. colsum_kernel: one group per (data row, column block) folds its run in edge order.  The lanes load G edges at a
//      time (value, weight, den) and G grad_out values each before the serial adds, so the chain waits on shuffles and
//      arithmetic, not on loads.  A data row that many queries reference is one long serial run: the order is the
//      contract.
// Every mapping performs the contract's operations in the contract's order, so launch shapes cannot change a bit.
#pragma once
#include "common.cuh"

namespace tknn {
namespace interp {

constexpr int THREADS = 256;
constexpr float MIN_D2 = 1e-16f;  // PyG's clamp(min=1e-16) of the squared distance

// lanes per row: f > 16 -> 32, else the next power of two >= f (at least 4)
inline int group_of(int f) { return f > 16 ? 32 : f > 8 ? 16 : f > 4 ? 8 : 4; }

__device__ __forceinline__ float weight_of(float d2) {
  return __fdiv_rn(1.0f, d2 < MIN_D2 ? MIN_D2 : d2);  // NaN passes the comparison untouched, as in torch.clamp
}

struct FwdParams {
  const int32_t* idx;  // nq x k
  const float* d2;     // nq x k
  const float* x;      // n rows, pitch x_stride
  uint64_t nq;
  uint32_t n;
  int k, f, x_stride;
  float* out;          // nq x f
  float* weight;       // nq x k or NULL
  float* den;          // nq or NULL
  uint32_t* bad;       // set when an idx entry lies outside {-1} u [0, n)
};

// (index, weight) of slot s of row i (slot-valid lanes only); a bad index is flagged and skipped like -1
__device__ __forceinline__ void load_slot(const FwdParams& P, uint64_t i, int s, bool live, int& j, float& w) {
  j = -1;
  w = 0.0f;
  if (live && s < P.k) {
    const uint64_t e = i * (uint64_t)P.k + s;
    j = __ldg(P.idx + e);
    if (j >= 0 && (uint32_t)j < P.n) {
      w = weight_of(__ldg(P.d2 + e));
    } else {
      if (j != -1) *P.bad = 1u;
      j = -1;
    }
  }
}

template <int G>
static __global__ void __launch_bounds__(THREADS) forward_kernel(const FwdParams P) {
  const int gl = threadIdx.x & (G - 1);
  const uint64_t groups = (uint64_t)gridDim.x * (THREADS / G);
  // every group of a warp runs the same trip counts (k and f are uniform), so the warp stays converged for the shuffles
  const uint64_t first = ((uint64_t)blockIdx.x * THREADS + threadIdx.x) / G;
  const uint64_t rounds = (P.nq + groups - 1) / groups;
  for (uint64_t r = 0; r < rounds; ++r) {
    const uint64_t i = first + r * groups;
    const bool live = i < P.nq;
    // slot chunk 0 stays in registers; den over all chunks in slot order
    int j0;
    float w0;
    load_slot(P, i, gl, live, j0, w0);
    if (live && P.weight && gl < P.k) P.weight[i * (uint64_t)P.k + gl] = w0;
    float den = 0.0f;
    for (int s0 = 0; s0 < P.k; s0 += G) {
      int js = j0;
      float ws = w0;
      if (s0) {
        load_slot(P, i, s0 + gl, live, js, ws);
        if (live && P.weight && s0 + gl < P.k) P.weight[i * (uint64_t)P.k + s0 + gl] = ws;
      }
      const int m = min(G, P.k - s0);
      for (int t = 0; t < m; ++t) {
        const int jt = __shfl_sync(FULL_MASK, js, t, G);
        const float wt = __shfl_sync(FULL_MASK, ws, t, G);
        if (jt >= 0) den = __fadd_rn(den, wt);
      }
    }
    if (live && P.den && gl == 0) P.den[i] = den;
    for (int c0 = 0; c0 < P.f; c0 += G) {
      const int c = c0 + gl;
      const bool col = live && c < P.f;
      float num = 0.0f;
      for (int s0 = 0; s0 < P.k; s0 += G) {
        int js = j0;
        float ws = w0;
        if (s0) load_slot(P, i, s0 + gl, live, js, ws);
        const int m = min(G, P.k - s0);
#pragma unroll 4
        for (int t = 0; t < m; ++t) {
          const int jt = __shfl_sync(FULL_MASK, js, t, G);
          const float wt = __shfl_sync(FULL_MASK, ws, t, G);
          if (col && jt >= 0) num = __fadd_rn(num, __fmul_rn(__ldg(P.x + (uint64_t)jt * P.x_stride + c), wt));
        }
      }
      if (col) P.out[i * (uint64_t)P.f + c] = __fdiv_rn(num, den);
    }
  }
}

// 1. keys (data row, or n for a skipped slot), values (edge number) and per-row edge counts
static __global__ void __launch_bounds__(THREADS) edge_kernel(const int32_t* __restrict__ idx, uint64_t edges, uint32_t n,
                                                              uint64_t* __restrict__ keys, uint32_t* __restrict__ vals,
                                                              uint32_t* __restrict__ counts, uint32_t* bad) {
  for (uint64_t e = (uint64_t)blockIdx.x * THREADS + threadIdx.x; e < edges; e += (uint64_t)gridDim.x * THREADS) {
    const int32_t j = __ldg(idx + e);
    uint32_t key = n;
    if (j >= 0 && (uint32_t)j < n) {
      key = (uint32_t)j;
      atomicAdd(counts + j, 1u);
    } else if (j != -1) {
      *bad = 1u;
    }
    keys[e] = key;
    vals[e] = (uint32_t)e;
  }
}

struct BwdParams {
  const uint32_t* vals;  // edge numbers, sorted by data row (runs in ascending e)
  const uint64_t* off;   // run offsets (n + 1)
  const float* weight;   // nq x k
  const float* den;      // nq
  const float* grad;     // nq rows, pitch g_stride
  uint32_t n;
  int k, f, g_stride, blocks;  // blocks: column blocks of G per data row
  float* grad_x;               // n x f
};

// 4. one group per (data row j, column block): its run folded in edge order
template <int G>
static __global__ void __launch_bounds__(THREADS) colsum_kernel(const BwdParams P) {
  const int gl = threadIdx.x & (G - 1);
  const uint64_t items = (uint64_t)P.n * P.blocks, groups = (uint64_t)gridDim.x * (THREADS / G);
  const uint64_t first = ((uint64_t)blockIdx.x * THREADS + threadIdx.x) / G;
  const uint64_t rounds = (items + groups - 1) / groups;
  for (uint64_t r = 0; r < rounds; ++r) {
    const uint64_t w = first + r * groups;
    const bool live = w < items;
    const uint64_t j = live ? w / P.blocks : 0;
    const int c = (live ? (int)(w - j * P.blocks) : 0) * G + gl;
    const bool col = live && c < P.f;
    const uint64_t p0 = live ? __ldg(P.off + j) : 0, p1 = live ? __ldg(P.off + j + 1) : 0;
    // runs differ between the groups of a warp: every lane walks the warp's longest run, past its own run idle
    const uint32_t chunks = __reduce_max_sync(FULL_MASK, (uint32_t)((p1 - p0 + G - 1) / G));
    float acc = 0.0f;
    for (uint32_t ch = 0; ch < chunks; ++ch) {
      const uint64_t p = p0 + (uint64_t)ch * G + gl;
      uint32_t my_i = 0;
      float my_w = 0.0f, my_d = 1.0f;
      if (p < p1) {
        const uint32_t e = __ldg(P.vals + p);
        my_i = e / (uint32_t)P.k;
        my_w = __ldg(P.weight + e);
        my_d = __ldg(P.den + my_i);
      }
      const uint64_t left = p0 + (uint64_t)ch * G < p1 ? p1 - (p0 + (uint64_t)ch * G) : 0;
      const int m = left < (uint64_t)G ? (int)left : G;
      float g[G];
#pragma unroll
      for (int t = 0; t < G; ++t) {
        const uint32_t it = __shfl_sync(FULL_MASK, my_i, t, G);
        g[t] = col && t < m ? __ldg(P.grad + (uint64_t)it * P.g_stride + c) : 0.0f;
      }
#pragma unroll
      for (int t = 0; t < G; ++t) g[t] = __fmul_rn(__fdiv_rn(g[t], __shfl_sync(FULL_MASK, my_d, t, G)),
                                                   __shfl_sync(FULL_MASK, my_w, t, G));
#pragma unroll
      for (int t = 0; t < G; ++t)
        if (t < m) acc = __fadd_rn(acc, g[t]);
    }
    if (col) P.grad_x[j * (uint64_t)P.f + c] = acc;
  }
}

}  // namespace interp
}  // namespace tknn
