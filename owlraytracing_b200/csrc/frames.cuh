// frames.cuh — surface normals and local frames from the covariance of neighbourhoods (tknn_local_frames; PyTorch3D's
// estimate_pointcloud_local_coord_frames, DESIGN.md §3.12).
//
// One thread per row, in the order of the contract (include/trueknn.h):
//   pass 1  gathers the row's points for the chunked sums of the centroid, keeps the anchor (the first valid slot) and
//           flags an idx outside {-1} u [0, n);
//   pass 2  gathers them again for the six chunked covariance sums;
//           then cyclic Jacobi on the 3 x 3 matrix in registers and the three compare-exchanges;
//   pass 3  (disambiguate only) gathers them a third time to count the positive projections onto columns 0 and 2.
// A row of up to 512 slots does not fit in registers, so the passes re-read it; the second and third reads of a row
// mostly hit L1 / L2.  Every pass loads G slots before it folds them in slot order, so G gathers per thread are in flight.
// No atomics except the error flag, and every row is one fixed sequence of operations: launch shapes cannot change a bit.
#pragma once
#include "common.cuh"

namespace tknn {
namespace frames {

constexpr int THREADS = 256;
constexpr int CHUNK = 32;  // terms per chunk of the two-level sums (part of the contract; kgrad::CHUNK)
constexpr int SWEEPS = 8;  // the Jacobi sweep cap (part of the contract)
constexpr int G = 4;       // slots a pass loads before it folds them

struct Params {
  const float* p;      // n rows, pitch stride
  const int32_t* idx;  // m x k
  uint64_t m;
  uint32_t n;
  int k, stride, disambiguate;
  float* eig;          // m x 3 or NULL
  float* frames;       // m x 9 (row-major 3 x 3, eigenvectors in columns) or NULL
  uint32_t* bad;       // set when an idx entry lies outside {-1} u [0, n)
};

// Calls f(x, y, z) for the valid slots of row i in slot order.  FLAG: report entries outside {-1} u [0, n).
template <bool FLAG, class F>
__device__ __forceinline__ void each_point(const Params& P, uint64_t i, F&& f) {
  const int32_t* row = P.idx + i * (uint64_t)P.k;
  for (int s0 = 0; s0 < P.k; s0 += G) {
    bool ok[G];
    float x[G], y[G], z[G];
#pragma unroll
    for (int u = 0; u < G; ++u) {
      const int32_t j = s0 + u < P.k ? __ldg(row + s0 + u) : -1;
      ok[u] = j >= 0 && (uint32_t)j < P.n;
      if (FLAG && !ok[u] && j != -1) *P.bad = 1u;
      x[u] = y[u] = z[u] = 0.0f;
      if (ok[u]) {
        const float* q = P.p + (uint64_t)j * P.stride;
        x[u] = __ldg(q);
        y[u] = __ldg(q + 1);
        z[u] = __ldg(q + 2);
      }
    }
#pragma unroll
    for (int u = 0; u < G; ++u)
      if (ok[u]) f(x[u], y[u], z[u]);
  }
}

// R running chunked sums that share one chunk counter
template <int R>
struct Chunked {
  float acc[R], part[R];
  int in_chunk = 0;
  __device__ __forceinline__ Chunked() {
#pragma unroll
    for (int r = 0; r < R; ++r) acc[r] = part[r] = 0.0f;
  }
  __device__ __forceinline__ void add(const float (&v)[R]) {
#pragma unroll
    for (int r = 0; r < R; ++r) part[r] = __fadd_rn(part[r], v[r]);
    if (++in_chunk == CHUNK) {
#pragma unroll
      for (int r = 0; r < R; ++r) {
        acc[r] = __fadd_rn(acc[r], part[r]);
        part[r] = 0.0f;
      }
      in_chunk = 0;
    }
  }
  __device__ __forceinline__ float result(int r) const { return in_chunk ? __fadd_rn(acc[r], part[r]) : acc[r]; }
};

// One Jacobi rotation of the pair (p, q): Numerical Recipes' t, the plain (c, s) update of the third row and of V.
template <int p, int q>
__device__ __forceinline__ void rotate(float (&A)[3][3], float (&V)[3][3]) {
  constexpr int r = 3 - p - q;
  const float apq = A[p][q];
  if (apq == 0.0f) return;
  const float tau = __fdiv_rn(__fsub_rn(A[q][q], A[p][p]), __fmul_rn(2.0f, apq));
  const float tt = __fmul_rn(tau, tau);
  const float t = isinf(tt) ? __fdiv_rn(0.5f, tau)
                            : __fdiv_rn(tau < 0.0f ? -1.0f : 1.0f, __fadd_rn(fabsf(tau), __fsqrt_rn(__fadd_rn(1.0f, tt))));
  const float c = __fdiv_rn(1.0f, __fsqrt_rn(__fadd_rn(1.0f, __fmul_rn(t, t))));
  const float s = __fmul_rn(t, c);
  const float ta = __fmul_rn(t, apq);
  A[p][p] = __fsub_rn(A[p][p], ta);
  A[q][q] = __fadd_rn(A[q][q], ta);
  A[p][q] = A[q][p] = 0.0f;
  const float arp = A[r][p], arq = A[r][q];
  A[r][p] = A[p][r] = __fsub_rn(__fmul_rn(c, arp), __fmul_rn(s, arq));
  A[r][q] = A[q][r] = __fadd_rn(__fmul_rn(s, arp), __fmul_rn(c, arq));
#pragma unroll
  for (int u = 0; u < 3; ++u) {
    const float vp = V[u][p], vq = V[u][q];
    V[u][p] = __fsub_rn(__fmul_rn(c, vp), __fmul_rn(s, vq));
    V[u][q] = __fadd_rn(__fmul_rn(s, vp), __fmul_rn(c, vq));
  }
}

template <int a, int b>
__device__ __forceinline__ void compare_exchange(float (&w)[3], float (&V)[3][3]) {
  if (w[a] > w[b]) {
    const float t = w[a];
    w[a] = w[b];
    w[b] = t;
#pragma unroll
    for (int u = 0; u < 3; ++u) {
      const float v = V[u][a];
      V[u][a] = V[u][b];
      V[u][b] = v;
    }
  }
}

// #{slots s : fl(fl(fl(v0 f0) + fl(v1 f1)) + fl(v2 f2)) > 0}, f = fl(p_s - anchor)
__device__ __forceinline__ bool projects_positive(float v0, float v1, float v2, float f0, float f1, float f2) {
  return __fadd_rn(__fadd_rn(__fmul_rn(v0, f0), __fmul_rn(v1, f1)), __fmul_rn(v2, f2)) > 0.0f;
}

static __global__ void __launch_bounds__(THREADS) frames_kernel(const Params P) {
  for (uint64_t i = (uint64_t)blockIdx.x * THREADS + threadIdx.x; i < P.m; i += (uint64_t)gridDim.x * THREADS) {
    // 1. centroid and anchor
    Chunked<3> sum;
    int c = 0;
    float a0 = 0.0f, a1 = 0.0f, a2 = 0.0f;
    each_point<true>(P, i, [&](float x, float y, float z) {
      if (c == 0) {
        a0 = x;
        a1 = y;
        a2 = z;
      }
      ++c;
      sum.add({x, y, z});
    });
    float w[3], V[3][3];
    if (c == 0) {  // no neighbour: NaN everywhere
      const float nan = __int_as_float(0x7fc00000);
#pragma unroll
      for (int u = 0; u < 3; ++u) {
        w[u] = nan;
#pragma unroll
        for (int j = 0; j < 3; ++j) V[u][j] = nan;
      }
    } else {
      const float fc = (float)c;
      const float m0 = __fdiv_rn(sum.result(0), fc), m1 = __fdiv_rn(sum.result(1), fc), m2 = __fdiv_rn(sum.result(2), fc);
      // 2. covariance (mean over the neighbourhood)
      Chunked<6> cov;
      each_point<false>(P, i, [&](float x, float y, float z) {
        const float e0 = __fsub_rn(x, m0), e1 = __fsub_rn(y, m1), e2 = __fsub_rn(z, m2);
        cov.add({__fmul_rn(e0, e0), __fmul_rn(e0, e1), __fmul_rn(e0, e2), __fmul_rn(e1, e1), __fmul_rn(e1, e2),
                 __fmul_rn(e2, e2)});
      });
      float A[3][3];
      A[0][0] = __fdiv_rn(cov.result(0), fc);
      A[0][1] = A[1][0] = __fdiv_rn(cov.result(1), fc);
      A[0][2] = A[2][0] = __fdiv_rn(cov.result(2), fc);
      A[1][1] = __fdiv_rn(cov.result(3), fc);
      A[1][2] = A[2][1] = __fdiv_rn(cov.result(4), fc);
      A[2][2] = __fdiv_rn(cov.result(5), fc);
      // cyclic Jacobi from V = I
#pragma unroll
      for (int u = 0; u < 3; ++u)
#pragma unroll
        for (int j = 0; j < 3; ++j) V[u][j] = u == j ? 1.0f : 0.0f;
      for (int sweep = 0; sweep < SWEEPS; ++sweep) {
        if (A[0][1] == 0.0f && A[0][2] == 0.0f && A[1][2] == 0.0f) break;
        rotate<0, 1>(A, V);
        rotate<0, 2>(A, V);
        rotate<1, 2>(A, V);
      }
      w[0] = A[0][0];
      w[1] = A[1][1];
      w[2] = A[2][2];
      compare_exchange<0, 1>(w, V);
      compare_exchange<1, 2>(w, V);
      compare_exchange<0, 1>(w, V);
      if (P.disambiguate) {
        // 3. signs of the normal (column 0) and of the main curvature direction (column 2), then y = n x z
        int pos0 = 0, pos2 = 0;
        each_point<false>(P, i, [&](float x, float y, float z) {
          const float f0 = __fsub_rn(x, a0), f1 = __fsub_rn(y, a1), f2 = __fsub_rn(z, a2);
          pos0 += projects_positive(V[0][0], V[1][0], V[2][0], f0, f1, f2);
          pos2 += projects_positive(V[0][2], V[1][2], V[2][2], f0, f1, f2);
        });
        if (2 * pos0 < c) {
#pragma unroll
          for (int u = 0; u < 3; ++u) V[u][0] = -V[u][0];
        }
        if (2 * pos2 < c) {
#pragma unroll
          for (int u = 0; u < 3; ++u) V[u][2] = -V[u][2];
        }
        V[0][1] = __fsub_rn(__fmul_rn(V[1][0], V[2][2]), __fmul_rn(V[2][0], V[1][2]));
        V[1][1] = __fsub_rn(__fmul_rn(V[2][0], V[0][2]), __fmul_rn(V[0][0], V[2][2]));
        V[2][1] = __fsub_rn(__fmul_rn(V[0][0], V[1][2]), __fmul_rn(V[1][0], V[0][2]));
      }
    }
    if (P.eig) {
#pragma unroll
      for (int j = 0; j < 3; ++j) P.eig[i * 3 + j] = w[j];
    }
    if (P.frames) {
#pragma unroll
      for (int u = 0; u < 3; ++u)
#pragma unroll
        for (int j = 0; j < 3; ++j) P.frames[i * 9 + u * 3 + j] = V[u][j];
    }
  }
}

}  // namespace frames
}  // namespace tknn
