// features.cuh — exact segmented k-nearest neighbours in feature space (tknn_feature_knn): a tiled brute force on the
// CUDA cores over row-major rows of f columns, for inputs the LBVH cannot serve (f = 64 or 128 in DGCNN's dynamic
// graphs, where boxes prune nothing).
//
// Distance rule (include/trueknn.h): d_j = fl(y_j - x_j), d2 = d_0 * d_0, then d2 = fmaf(d_j, d_j, d2) for j = 1 .. f - 1
// in that order.  The kernel starts every accumulator at +0 (fmaf(d, d, +0) has the bits of d * d) and walks the
// columns in order, so each pair sees exactly that sequence of roundings whatever the tile shape.  The data tile is
// staged NEGATED, so one packed __fadd2_rn gives two fl(y - x) (an IEEE subtraction is the addition of the negation)
// and one __ffma2_rn two accumulations; each component is the scalar op, bit for bit.  Columns past f are staged as
// zeros on both sides: fl(0 + -0) = 0 and fmaf(0, 0, a) = a, so padding never changes a sum.
//
// Work: one CTA per item (segment, tile of QT query rows, contiguous split of the segment's data rows).  Per data tile
// of PT rows, the query and data chunks of DC columns are staged transposed in shared memory (a warp reads 4 rows x 8
// columns: 32-byte sectors, and the padded row pitch makes the transposing stores conflict-free); each thread keeps
// 4 queries x 8 data rows of accumulators.  When a data tile is finished, every pair is compared with its query's
// current k-th distance (conservative: d2 <= bound lets ties through), survivors are marked in a per-query bit mask,
// and thread t then pushes query t's survivors into its key heap (trav::heap_push / heap_sift_root, the (d2, index)
// order of make_key).  So the k-list holds the smallest keys of all rows seen, which is the exact answer.
#pragma once
#include "common.cuh"
#include "traverse.cuh"

namespace tknn {
namespace feat {

constexpr int PT = 128;     // data rows per tile (16 threads x 8 rows)
constexpr int DC = 32;      // columns per staged chunk
constexpr int XS = PT + 4;  // row pitch of the transposed data chunk and of the d2 tile (floats)

// One CTA's work: query rows [q0, q0 + nq) against data rows [x0, x1) (one split of the query rows' segment).
struct Item {
  uint32_t q0, nq, x0, x1, split, pad0, pad1, pad2;
};

struct Params {
  const float* x;       // data rows (device), pitch x_stride floats
  const float* y;       // query rows (device), pitch y_stride floats
  const int32_t* sid;   // per query row: the data index to exclude, or NULL
  const Item* items;
  int f, x_stride, y_stride, k, squared;
  uint32_t nq;          // all query rows (layout of the partial lists)
  int32_t* idx_out;     // final rows (one split), device
  float* dist_out;      // final rows, device, may be NULL
  uint64_t* partial;    // several splits: partial[(split * nq + q) * k + i], ascending keys, ~0 = empty
};

// query tile for a k: QT queries keep QT * k keys in shared memory
__host__ __device__ constexpr int query_tile(int k) { return k <= 64 ? 64 : 32; }

template <int QT>
__host__ __device__ constexpr size_t smem_bytes(int k) {
  return (size_t)QT * k * sizeof(uint64_t) + sizeof(float) * ((size_t)DC * (QT + 4) + (size_t)DC * XS + (size_t)QT * XS) +
         sizeof(uint32_t) * QT * (PT / 32) + sizeof(float) * QT + sizeof(int32_t) * QT;
}

// Stages rows [row0, row0 + rows) x columns [c0, c0 + DC) of `src` transposed into dst[c * pitch + r] (R rows in the
// tile; rows past `rows` and columns past f become 0).  A warp covers 4 rows x 8 columns per instruction.
template <int R, int THREADS, bool NEG>
__device__ __forceinline__ void stage_chunk(float* __restrict__ dst, int pitch, const float* __restrict__ src, int stride,
                                            uint32_t row0, int rows, int c0, int f) {
  static_assert((R * DC) % THREADS == 0, "a chunk is a whole number of passes");
#pragma unroll 8
  for (int pass = 0; pass < R * DC / THREADS; ++pass) {
    const int e = pass * THREADS + (int)threadIdx.x;
    const int lane = e & 31, slot = e >> 5;
    const int r = (slot % (R / 4)) * 4 + (lane >> 3);
    const int c = (slot / (R / 4)) * 8 + (lane & 7);
    float v = 0.0f;
    if (r < rows && c0 + c < f) v = __ldg(src + (uint64_t)(row0 + r) * (uint64_t)stride + (uint64_t)(c0 + c));
    dst[c * pitch + r] = NEG ? -v : v;
  }
}

template <int QT>
__global__ void __launch_bounds__(QT * 4) feature_knn_kernel(const Params P) {
  constexpr int THREADS = QT * 4, QS = QT + 4, MW = PT / 32;
  extern __shared__ __align__(16) unsigned char smem[];
  const int k = P.k;
  uint64_t* heap = reinterpret_cast<uint64_t*>(smem);
  float* sQ = reinterpret_cast<float*>(heap + (size_t)QT * k);  // [DC][QS]
  float* sX = sQ + DC * QS;                                      // [DC][XS], negated
  float* sD = sX + DC * XS;                                      // [QT][XS]
  uint32_t* sMask = reinterpret_cast<uint32_t*>(sD + QT * XS);   // [QT][MW]
  float* sBound = reinterpret_cast<float*>(sMask + QT * MW);
  int32_t* sSelf = reinterpret_cast<int32_t*>(sBound + QT);

  const Item it = P.items[blockIdx.x];
  const int tid = threadIdx.x, tx = tid & 15, ty = tid >> 4;
  const int nqt = (int)it.nq;
  if (tid < QT) {
    sBound[tid] = tid < nqt ? INFINITY : -1.0f;  // -1: a padding query accepts nothing
    sSelf[tid] = (tid < nqt && P.sid) ? P.sid[it.q0 + tid] : -1;
#pragma unroll
    for (int w = 0; w < MW; ++w) sMask[tid * MW + w] = 0u;
  }
  uint64_t* H = heap + (size_t)(tid >> 5) * 32 * k + (tid & 31);  // query tid's heap (stride 32, trav's layout)
  int cnt = 0;

  for (uint32_t xb = it.x0; xb < it.x1; xb += PT) {
    const int rows = (int)min((uint32_t)PT, it.x1 - xb);
    float2 acc[4][4];
#pragma unroll
    for (int i = 0; i < 4; ++i)
#pragma unroll
      for (int j = 0; j < 4; ++j) acc[i][j] = make_float2(0.0f, 0.0f);
    for (int c0 = 0; c0 < P.f; c0 += DC) {
      __syncthreads();  // the previous chunk's reads (and the previous tile's inserts) are done
      stage_chunk<QT, THREADS, false>(sQ, QS, P.y, P.y_stride, it.q0, nqt, c0, P.f);
      stage_chunk<PT, THREADS, true>(sX, XS, P.x, P.x_stride, xb, rows, c0, P.f);
      __syncthreads();
      const int dc = (min(DC, P.f - c0) + 3) & ~3;  // columns past f are zeros on both sides
      const float* q = sQ + 4 * ty;
      const float* xn = sX + 8 * tx;
#pragma unroll 4
      for (int c = 0; c < dc; ++c) {
        const float4 qv = *reinterpret_cast<const float4*>(q + c * QS);
        const float4 xa = *reinterpret_cast<const float4*>(xn + c * XS);
        const float4 xc = *reinterpret_cast<const float4*>(xn + c * XS + 4);
        const float2 x2[4] = {make_float2(xa.x, xa.y), make_float2(xa.z, xa.w), make_float2(xc.x, xc.y),
                              make_float2(xc.z, xc.w)};
        const float qs[4] = {qv.x, qv.y, qv.z, qv.w};
#pragma unroll
        for (int i = 0; i < 4; ++i) {
          const float2 q2 = make_float2(qs[i], qs[i]);
#pragma unroll
          for (int j = 0; j < 4; ++j) {
            const float2 d = __fadd2_rn(q2, x2[j]);
            acc[i][j] = __ffma2_rn(d, d, acc[i][j]);
          }
        }
      }
    }
    // filter: pairs with d2 <= the query's k-th distance (stale bounds are larger, so still conservative)
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      const int qi = 4 * ty + i;
      const float bound = sBound[qi];
      const int self = sSelf[qi];
      const float v[8] = {acc[i][0].x, acc[i][0].y, acc[i][1].x, acc[i][1].y,
                          acc[i][2].x, acc[i][2].y, acc[i][3].x, acc[i][3].y};
      uint32_t bits = 0;
#pragma unroll
      for (int j = 0; j < 8; ++j) {
        const int p = 8 * tx + j;
        bits |= (p < rows && v[j] <= bound && (int)(xb + p) != self ? 1u : 0u) << j;
      }
      float* drow = sD + qi * XS + 8 * tx;
      *reinterpret_cast<float4*>(drow) = make_float4(v[0], v[1], v[2], v[3]);
      *reinterpret_cast<float4*>(drow + 4) = make_float4(v[4], v[5], v[6], v[7]);
      if (bits) atomicOr(&sMask[qi * MW + (tx >> 2)], bits << (8 * (tx & 3)));
    }
    __syncthreads();
    // insert: thread t owns query t's heap
    if (tid < nqt) {
#pragma unroll
      for (int w = 0; w < MW; ++w) {
        uint32_t m = sMask[tid * MW + w];
        sMask[tid * MW + w] = 0u;
        while (m) {
          const int p = w * 32 + __ffs(m) - 1;
          m &= m - 1u;
          const uint64_t key = make_key(sD[tid * XS + p], (int)(xb + p));
          if (cnt < k) trav::heap_push(H, cnt, key);
          else if (key < H[0]) trav::heap_sift_root(H, k, key);
        }
      }
      if (cnt == k) sBound[tid] = key_d2(H[0]);
    }
  }

  if (tid >= nqt) return;
  const uint64_t row = (uint64_t)it.q0 + tid;
  if (P.partial) {
    uint64_t* out = P.partial + ((uint64_t)it.split * P.nq + row) * (uint64_t)k;
    for (int i = k - 1; i >= cnt; --i) out[i] = ~0ull;
    for (int i = cnt - 1; i >= 0; --i) {
      out[i] = H[0];
      if (i > 0) trav::heap_sift_root(H, i, H[i * 32]);
    }
    return;
  }
  int32_t* io = P.idx_out + row * (uint64_t)k;
  float* dd = P.dist_out ? P.dist_out + row * (uint64_t)k : nullptr;
  for (int i = k - 1; i >= cnt; --i) {
    io[i] = -1;
    if (dd) dd[i] = FLT_MAX;
  }
  for (int i = cnt - 1; i >= 0; --i) {
    const uint64_t top = H[0];
    io[i] = key_idx(top);
    if (dd) dd[i] = P.squared ? key_d2(top) : __fsqrt_rn(key_d2(top));
    if (i > 0) trav::heap_sift_root(H, i, H[i * 32]);
  }
}

// Sets *flag when one of the first f columns of `rows` rows is not finite.
static __global__ void __launch_bounds__(256) finite_kernel(const float* __restrict__ a, uint64_t rows, int f, int stride,
                                                            uint32_t* __restrict__ flag) {
  const uint64_t total = rows * (uint64_t)f;
  for (uint64_t i = (uint64_t)blockIdx.x * 256 + threadIdx.x; i < total; i += (uint64_t)gridDim.x * 256) {
    const uint64_t r = i / (uint64_t)f, c = i - r * (uint64_t)f;
    if (!isfinite(__ldg(a + r * (uint64_t)stride + c))) *flag = 1u;
  }
}

}  // namespace feat
}  // namespace tknn
