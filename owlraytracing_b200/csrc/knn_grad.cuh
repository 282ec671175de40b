// knn_grad.cuh — gradient of kNN squared distances with respect to both point sets (tknn_knn_backward: PyTorch3D's
// knn_points backward, the backward pass of the Chamfer distance, DESIGN.md §3.11).
//
// For every edge e = i*k + s with j = idx[i,s] (idx = -1 slots skipped), t = fl(2 * grad_d2[i,s]) and per column c:
//   term_q[e,c] = fl(t * fl(q[i,c] - p[j,c])),   term_p[e,c] = fl(t * fl(p[j,c] - q[i,c]))
// grad_q[i] is the chunked sum of row i's terms in slot order and grad_p[j] the chunked sum of the terms of the edges
// with idx = j in ascending e (chunks of 32 consecutive terms, each summed from +0, then the chunk sums in order from +0:
// the voxel mean's rule without the division).  No FMA, no float atomics.
//   1. terms_kernel:   one thread per query row: grad_q, the E x dim array of term_p, the bad-index flag.
//   2. grad_p reuses the backward of interpolate.cuh and the pooling of voxel.cuh unchanged: interp::edge_kernel (keys
//      and per-row counts), rsort::sort_pairs (stable, so every run stays in ascending e), the u64 scan of radius.cuh
//      (run offsets), then the chunk / voxel / fold kernels of voxel.cuh in R_SUM mode over the sorted edge numbers.
//      A point that 2^20 edges reference is 32 768 chunks summed in parallel and one fold, not one serial chain.
// Every mapping performs the contract's operations in the contract's order, so launch shapes cannot change a bit.
#pragma once
#include "common.cuh"

namespace tknn {
namespace kgrad {

constexpr int THREADS = 256;
constexpr int CHUNK = 32;  // terms per chunk of the two-level sum (part of the contract; voxel::CHUNK)

struct Params {
  const float* q;      // nq rows, pitch q_stride
  const float* p;      // n rows, pitch p_stride
  const int32_t* idx;  // nq x k
  const float* g;      // nq x k: grad_d2
  uint64_t nq;
  uint32_t n;
  int k, q_stride, p_stride;
  float* grad_q;  // nq x D or NULL
  float* term_p;  // nq * k x D or NULL (entries of skipped slots are not written)
  uint32_t* bad;  // set when an idx entry lies outside {-1} u [0, n)
};

template <int D>
static __global__ void __launch_bounds__(THREADS) terms_kernel(const Params P) {
  for (uint64_t i = (uint64_t)blockIdx.x * THREADS + threadIdx.x; i < P.nq; i += (uint64_t)gridDim.x * THREADS) {
    float qi[D], acc[D], part[D];
#pragma unroll
    for (int c = 0; c < D; ++c) {
      qi[c] = __ldg(P.q + i * (uint64_t)P.q_stride + c);
      acc[c] = part[c] = 0.0f;
    }
    int m = 0;  // terms in the current chunk
    for (int s = 0; s < P.k; ++s) {
      const uint64_t e = i * (uint64_t)P.k + s;
      const int32_t j = __ldg(P.idx + e);
      if (j < 0 || (uint32_t)j >= P.n) {
        if (j != -1) *P.bad = 1u;
        continue;
      }
      const float t = __fmul_rn(2.0f, __ldg(P.g + e));
#pragma unroll
      for (int c = 0; c < D; ++c) {
        const float pj = __ldg(P.p + (uint64_t)j * P.p_stride + c);
        part[c] = __fadd_rn(part[c], __fmul_rn(t, __fsub_rn(qi[c], pj)));
        if (P.term_p) P.term_p[e * D + c] = __fmul_rn(t, __fsub_rn(pj, qi[c]));
      }
      if (++m == CHUNK) {
#pragma unroll
        for (int c = 0; c < D; ++c) {
          acc[c] = __fadd_rn(acc[c], part[c]);
          part[c] = 0.0f;
        }
        m = 0;
      }
    }
    if (P.grad_q) {
#pragma unroll
      for (int c = 0; c < D; ++c) P.grad_q[i * D + c] = m ? __fadd_rn(acc[c], part[c]) : acc[c];
    }
  }
}

}  // namespace kgrad
}  // namespace tknn
