// brute.cuh — exact tiled brute-force kNN (no BVH), the k-way list merge, the synthetic generator
// and the bandwidth probe.
//
// The brute-force kernel is the GPU-side second oracle for sampled queries at sizes no CPU oracle
// reaches (SURVEY.md §7 M0 / §8c).  It shares the distance formula, key order and heap with the
// traversal kernel but none of its culling logic, so a culling bug cannot hide in both.
#pragma once
#include "common.cuh"
#include "traverse.cuh"

namespace tknn {
namespace brute {

// Finds the sorted position of each requested original index: ids_sorted ascending, nq entries.
// qpts[rank] = (x, y, z, original index bits).
static __global__ void __launch_bounds__(256) lookup_queries_kernel(const float4* __restrict__ pts, uint64_t n,
                                                             const int32_t* __restrict__ ids_sorted, uint32_t nq,
                                                             float4* __restrict__ qpts) {
  const uint64_t i = (uint64_t)blockIdx.x * 256 + threadIdx.x;
  if (i >= n) return;
  const float4 p = __ldg(&pts[i]);
  const int id = __float_as_int(p.w);
  uint32_t lo = 0, hi = nq;
  while (lo < hi) {
    const uint32_t mid = (lo + hi) >> 1;
    if (ids_sorted[mid] < id) lo = mid + 1; else hi = mid;
  }
  if (lo < nq && ids_sorted[lo] == id) qpts[lo] = p;
}

// One warp per (group of 32 queries, split of the point range).  partial[(split * nq + q) * k + i]
// receives the ascending key list (~0 = empty slot).
static __global__ void __launch_bounds__(32) brute_kernel(const float4* __restrict__ pts, uint64_t n,
                                                   const float4* __restrict__ qpts, uint32_t nq, int k, int splits,
                                                   uint64_t* __restrict__ partial) {
  extern __shared__ __align__(16) unsigned char smem[];
  float4* stage = reinterpret_cast<float4*>(smem);
  const int lane = threadIdx.x;
  uint64_t* H = reinterpret_cast<uint64_t*>(smem + 32 * sizeof(float4)) + lane;
  const uint32_t group = blockIdx.x;
  const int split = blockIdx.y;
  const uint32_t qi = group * 32 + lane;
  const bool valid = qi < nq;
  float4 q = make_float4(0.f, 0.f, 0.f, 0.f);
  if (valid) q = qpts[qi];
  const int self = __float_as_int(q.w);
  const uint64_t chunk = (((n + splits - 1) / splits) + 31) / 32 * 32;
  const uint64_t begin = (uint64_t)split * chunk;
  const uint64_t end = begin + chunk < n ? begin + chunk : n;
  int cnt = 0;
  float bound = valid ? INFINITY : -1.0f;
  for (uint64_t base = begin; base < end; base += 32) {
    const int m = (int)((end - base) < 32 ? (end - base) : 32);
    if (lane < m) stage[lane] = __ldg(&pts[base + lane]);
    __syncwarp();
    uint32_t mask = 0;
    for (int j = 0; j < m; ++j) {
      const float4 p = stage[j];
      const float d = dist2(q.x, q.y, q.z, p.x, p.y, p.z);
      mask |= (d <= bound ? 1u : 0u) << j;
    }
    while (mask) {
      const int j = __ffs(mask) - 1;
      mask &= mask - 1u;
      const float4 p = stage[j];
      const float d = dist2(q.x, q.y, q.z, p.x, p.y, p.z);
      const int pid = __float_as_int(p.w);
      if (pid == self) continue;
      const uint64_t key = make_key(d, pid);
      if (cnt < k) {
        trav::heap_push(H, cnt, key);
        if (cnt == k) bound = key_d2(H[0]);
      } else if (key < H[0]) {
        trav::heap_sift_root(H, k, key);
        bound = key_d2(H[0]);
      }
    }
    __syncwarp();
  }
  if (valid) {
    uint64_t* out = partial + ((uint64_t)split * nq + qi) * (uint64_t)k;
    for (int i = k - 1; i >= cnt; --i) out[i] = ~0ull;
    for (int i = cnt - 1; i >= 0; --i) {
      out[i] = H[0];
      if (i > 0) trav::heap_sift_root(H, i, H[i * 32]);
    }
  }
}

// Merge `parts` ascending key lists per query into one; writes (idx, sqrt(d2)) rows.
// row_of[q] (optional) redirects the output row.
static __global__ void __launch_bounds__(32) merge_keys_kernel(const uint64_t* __restrict__ partial, int parts, uint32_t nq, int k,
                                                        const uint32_t* __restrict__ row_of, int squared,
                                                        int32_t* __restrict__ idx_out, float* __restrict__ dist_out) {
  extern __shared__ __align__(16) unsigned char smem[];
  const int lane = threadIdx.x;
  uint64_t* H = reinterpret_cast<uint64_t*>(smem) + lane;
  const uint32_t qi = blockIdx.x * 32 + lane;
  if (qi >= nq) return;
  int cnt = 0;
  for (int s = 0; s < parts; ++s) {
    const uint64_t* in = partial + ((uint64_t)s * nq + qi) * (uint64_t)k;
    for (int i = 0; i < k; ++i) {
      const uint64_t key = in[i];
      if (key == ~0ull) break;
      if (cnt < k) trav::heap_push(H, cnt, key);
      else if (key < H[0]) trav::heap_sift_root(H, k, key);
      else break;  // lists ascend: nothing smaller follows
    }
  }
  const uint64_t row = row_of ? row_of[qi] : qi;
  int32_t* io = idx_out + row * (uint64_t)k;
  float* dd = dist_out + row * (uint64_t)k;
  for (int i = k - 1; i >= cnt; --i) { io[i] = -1; dd[i] = FLT_MAX; }
  for (int i = cnt - 1; i >= 0; --i) {
    const uint64_t top = H[0];
    io[i] = key_idx(top);
    dd[i] = squared ? key_d2(top) : __fsqrt_rn(key_d2(top));
    if (i > 0) trav::heap_sift_root(H, i, H[i * 32]);
  }
}

// Merge of (idx, d2) partial lists (point-partitioned driver, SURVEY.md §8e).  The partial lists
// carry SQUARED distances (contexts run with TKNN_OPT_SQUARED_DIST = 1): sqrtf maps two adjacent
// d2 values to one float about half of the time, so ordering on the reported distance would not
// be the (d2, index) order.  Duplicates by index are dropped; the output distance is sqrtf(d2).
static __global__ void __launch_bounds__(32) merge_lists_kernel(const int32_t* __restrict__ idx_parts,
                                                         const float* __restrict__ dist_parts, int parts, uint32_t nq, int k,
                                                         int squared, int32_t* __restrict__ idx_out,
                                                         float* __restrict__ dist_out) {
  extern __shared__ __align__(16) unsigned char smem[];
  const int lane = threadIdx.x;
  uint64_t* H = reinterpret_cast<uint64_t*>(smem) + lane;
  const uint32_t qi = blockIdx.x * 32 + lane;
  if (qi >= nq) return;
  int cnt = 0;
  for (int s = 0; s < parts; ++s) {
    const uint64_t off = ((uint64_t)s * nq + qi) * (uint64_t)k;
    for (int i = 0; i < k; ++i) {
      const int id = idx_parts[off + i];
      if (id < 0) break;
      const uint64_t key = make_key(dist_parts[off + i], id);
      bool dup = false;
      for (int h = 0; h < cnt; ++h)
        if (key_idx(H[h * 32]) == id) { dup = true; break; }
      if (dup) continue;
      if (cnt < k) trav::heap_push(H, cnt, key);
      else if (key < H[0]) trav::heap_sift_root(H, k, key);
    }
  }
  int32_t* io = idx_out + (uint64_t)qi * k;
  float* dd = dist_out + (uint64_t)qi * k;
  for (int i = k - 1; i >= cnt; --i) { io[i] = -1; dd[i] = FLT_MAX; }
  for (int i = cnt - 1; i >= 0; --i) {
    const uint64_t top = H[0];
    io[i] = key_idx(top);
    dd[i] = squared ? key_d2(top) : __fsqrt_rn(key_d2(top));
    if (i > 0) trav::heap_sift_root(H, i, H[i * 32]);
  }
}

// small gathers used by tknn_query to follow the Morton order of the queries
static __global__ void __launch_bounds__(256) gather_i32_kernel(const int32_t* __restrict__ in, const uint32_t* __restrict__ order,
                                                         uint64_t n, int32_t* __restrict__ out) {
  const uint64_t i = (uint64_t)blockIdx.x * 256 + threadIdx.x;
  if (i < n) out[i] = in[order[i]];
}
static __global__ void __launch_bounds__(256) gather_r2_kernel(const float* __restrict__ radius2, const uint32_t* __restrict__ order,
                                                        uint64_t n, float* __restrict__ r2_out) {
  const uint64_t i = (uint64_t)blockIdx.x * 256 + threadIdx.x;
  if (i < n) {
    const float r2 = radius2[order[i]];
    r2_out[i] = r2 >= 0.0f ? r2 : INFINITY;  // negative = no cap
  }
}

// Point-partitioned driver: which remote ranks can the closed ball (q, sqrt(reach2)) reach?  Every rank
// publishes the tight box of its points inside each top-level Morton cell (2^bits cells per axis on the
// global cubic grid, cell id = the top 3*bits bits of the Morton code).  A ball only touches the cells
// between the cells of its two extreme corners — computed with the builder's own monotone quantiser, so
// no point of the ball can lie in a cell outside that range — usually 1..8 of them.  mask bit s = rank s.
//
// The ball is the fp32 rule, not the real one: a point p must be reached when dist2(q, p) <= r2.  The fma chain only
// adds non-negative terms, so RN(da * da) <= r2 on every axis; that rounding errs by 2^-24 relative, or by up to 2^-150
// absolute where da * da is subnormal or underflows to 0, so da^2 <= r2 (1 + 2^-23) + 2^-150 and, since
// sqrt(r2 + 2^-148) <= sqrt(r2) + 2^-74, |q - p| <= rho = fma(sqrt_ru(r2), 1.000001, 2^-74) per axis with room for the
// rounding of the fma.  q -/+ rho rounds outward and the quantiser is monotone, so p's cell lies in [c0, c1].  Without
// the absolute term a subnormal or zero r2 (a cloud at 1e-21 scale) misses remote points whose d2 underflows to it.
// lim needs no such change: a box holding p is no farther from q than p on any axis, so the box's sum is the point's
// chain up to reassociation, and its 1e-5 relative and 1e-30 absolute slack exceed that rounding, subnormal included.
__device__ __forceinline__ uint32_t reach_mask_of(float qx, float qy, float qz, float r2, const float* __restrict__ box6,
                                                  const float* __restrict__ summ, int n_ranks, int bits, int self_rank) {
  const float lx = box6[0], ly = box6[1], lz = box6[2];
  const float ext = fmaxf(fmaxf(box6[3] - lx, box6[4] - ly), fmaxf(box6[5] - lz, FLT_MIN));
  const float scale = 2097152.0f / ext;  // identical to morton_kernel
  const int cells = 1 << bits, shift = 21 - bits;
  int c0[3] = {0, 0, 0}, c1[3] = {cells - 1, cells - 1, cells - 1};
  const float rho = __fmaf_rn(__fsqrt_ru(r2), 1.000001f, 0x1p-74f);
  if (rho < 1e30f) {
    const float q[3] = {qx, qy, qz}, l[3] = {lx, ly, lz};
#pragma unroll
    for (int a = 0; a < 3; ++a) {
      c0[a] = (int)((uint32_t)fminf(fmaxf((__fsub_rd(q[a], rho) - l[a]) * scale, 0.0f), 2097151.0f) >> shift);
      c1[a] = (int)((uint32_t)fminf(fmaxf((__fadd_ru(q[a], rho) - l[a]) * scale, 0.0f), 2097151.0f) >> shift);
    }
  }
  const float lim = __fmaf_rn(r2, 1e-5f, r2) + 1e-30f;  // the boxes are tested in plain fp32: widen a little
  uint32_t mask = 0;
  for (int cz = c0[2]; cz <= c1[2]; ++cz)
    for (int cy = c0[1]; cy <= c1[1]; ++cy)
      for (int cx = c0[0]; cx <= c1[0]; ++cx) {
        uint32_t cell = 0;  // Morton interleave of the cell coordinates: x bit highest, then y, then z
        for (int b = 0; b < bits; ++b)
          cell |= (((uint32_t)cx >> b) & 1u) << (3 * b + 2) | (((uint32_t)cy >> b) & 1u) << (3 * b + 1) | (((uint32_t)cz >> b) & 1u) << (3 * b);
        for (int s = 0; s < n_ranks; ++s) {
          if (s == self_rank || ((mask >> s) & 1u)) continue;
          const float* bx = summ + ((size_t)s * ((size_t)1 << (3 * bits)) + cell) * 6;
          const float dx = fmaxf(fmaxf(bx[0] - qx, qx - bx[3]), 0.0f);
          const float dy = fmaxf(fmaxf(bx[1] - qy, qy - bx[4]), 0.0f);
          const float dz = fmaxf(fmaxf(bx[2] - qz, qz - bx[5]), 0.0f);
          if (dx * dx + dy * dy + dz * dz <= lim) mask |= 1u << s;  // an empty (inverted) box gives +inf
        }
      }
  return mask;
}

static __global__ void __launch_bounds__(256) reach_mask_kernel(const float* __restrict__ xyz, uint64_t n, int stride,
                                                         const float* __restrict__ reach2, const float* __restrict__ box6,
                                                         const float* __restrict__ summ, int n_ranks, int bits, int self_rank,
                                                         uint32_t* __restrict__ mask_out) {
  const uint64_t i = (uint64_t)blockIdx.x * 256 + threadIdx.x;
  if (i >= n) return;
  const float* p = xyz + i * (uint64_t)stride;
  mask_out[i] = reach_mask_of(p[0], p[1], p[2], reach2[i], box6, summ, n_ranks, bits, self_rank);
}

// u(i, a) = (mix64(seed ^ ((3 i + a) * phi64)) >> 40) * 2^-24  in [0, 1)   (SURVEY.md §8d)
static __global__ void __launch_bounds__(256) generate_uniform_kernel(uint64_t seed, uint64_t first, uint64_t n,
                                                               float* __restrict__ xyz) {
  const uint64_t t = (uint64_t)blockIdx.x * 256 + threadIdx.x;
  if (t >= 3 * n) return;
  const uint64_t c = 3 * first + t;  // = 3 i + a
  const uint64_t h = mix64(seed ^ (c * 0x9E3779B97F4A7C15ull));
  xyz[t] = (float)(h >> 40) * 5.9604644775390625e-08f;
}

// read-bandwidth probe: sums `words` uint4 per pass, `passes` passes
static __global__ void __launch_bounds__(256) read_probe_kernel(const uint4* __restrict__ buf, uint64_t words, int passes,
                                                         uint32_t* __restrict__ sink) {
  uint32_t acc = 0;
  const uint64_t step = (uint64_t)gridDim.x * 256;
  for (int p = 0; p < passes; ++p)
    for (uint64_t i = (uint64_t)blockIdx.x * 256 + threadIdx.x; i < words; i += step) {
      const uint4 v = __ldcg(&buf[i]);
      acc += v.x ^ v.y ^ v.z ^ v.w;
    }
  if (acc == 0x12345678u) *sink = acc;
}

// Shared-memory bandwidth probe: every thread issues `iters` x 8 independent LDS.128.  broadcast = 0: the lanes of a
// warp read 32 consecutive float4 (conflict-free, 512 B per instruction = 4 wavefronts of 128 B); broadcast = 1: all
// lanes of a warp read ONE float4 (the access pattern of the traversal kernel's leaf filter: one wavefront per
// instruction).  Bytes DELIVERED to lanes = threads x iters x 8 x 16 in both cases.
static __global__ void __launch_bounds__(256) smem_probe_kernel(int iters, int broadcast, int stride, uint32_t* __restrict__ sink) {
  __shared__ float4 s[1024];
  for (int i = threadIdx.x; i < 1024; i += 256) s[i] = make_float4((float)i, 1.0f, 2.0f, 3.0f);
  __syncthreads();
  uint32_t ax = 0, ay = 0, az = 0, aw = 0;
  const int base = broadcast ? (int)(threadIdx.x >> 5) * 37 : (int)threadIdx.x;
  const uint32_t s0 = (uint32_t)__cvta_generic_to_shared(s);
  for (int it = 0; it < iters; ++it) {
#pragma unroll
    for (int u = 0; u < 8; ++u) {
      // asm volatile: every load is issued (the compiler may neither hoist nor merge them); `stride` is a run-time value
      const uint32_t addr = s0 + 16u * (uint32_t)((base + it * stride + u * 32) & 1023);
      uint32_t x, y, z, w;
      asm volatile("ld.shared.v4.u32 {%0, %1, %2, %3}, [%4];" : "=r"(x), "=r"(y), "=r"(z), "=r"(w) : "r"(addr));
      ax ^= x; ay ^= y; az ^= z; aw ^= w;
    }
  }
  if ((ax ^ ay ^ az ^ aw) == 0x12345678u) *sink = ax;
}

}  // namespace brute
}  // namespace tknn
