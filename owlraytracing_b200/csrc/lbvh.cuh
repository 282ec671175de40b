// lbvh.cuh — LBVH builder kernels: scene bounds, Morton codes, leaf cut, Karras hierarchy, refit.
//
// Stands in for UserGeomGroup::buildAccel (owl/UserGeomGroup.cpp:39-241: bounds program +
// optixAccelBuild) and the 1-instance IAS on top of it (owl/InstanceGroup.cpp:110-280).  Unlike
// the reference's bounds program (samples/s01-trueknn/deviceCode.cu:38-48) the boxes here bound
// the POINTS, not radius-inflated spheres: the search radius is a kernel argument of the
// traversal, so nothing is rebuilt or refitted between rounds (hostCode.cpp:326-327 disappears).
#pragma once
#include "common.cuh"

namespace tknn {
namespace lbvh {

constexpr int THREADS = 256;

// ------------------------------------------------------------------------------------------------
// scene AABB: warp-shuffle + block reduce, one atomicMin/Max per block on order-preserving uints.
// Also flags non-finite coordinates (bad != 0 => tknn_build returns TKNN_EINVAL).
// bounds[0..2] = ordered(min xyz), bounds[3..5] = ordered(max xyz), bounds[6] = bad flag.
// ------------------------------------------------------------------------------------------------
static __global__ void __launch_bounds__(THREADS) bounds_kernel(const float* __restrict__ xyz, uint64_t n, int dim, int stride,
                                                         uint32_t* __restrict__ bounds) {
  float lo[3] = {INFINITY, INFINITY, INFINITY}, hi[3] = {-INFINITY, -INFINITY, -INFINITY};
  int bad = 0;
  const uint64_t step = (uint64_t)gridDim.x * THREADS;
  for (uint64_t i = (uint64_t)blockIdx.x * THREADS + threadIdx.x; i < n; i += step) {
    const float* p = xyz + i * (uint64_t)stride;
#pragma unroll
    for (int a = 0; a < 3; ++a) {
      const float v = (a < dim) ? p[a] : 0.0f;
      if (!isfinite(v)) bad = 1;
      lo[a] = fminf(lo[a], v);
      hi[a] = fmaxf(hi[a], v);
    }
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
#pragma unroll
    for (int a = 0; a < 3; ++a) {
      lo[a] = fminf(lo[a], __shfl_xor_sync(FULL_MASK, lo[a], o));
      hi[a] = fmaxf(hi[a], __shfl_xor_sync(FULL_MASK, hi[a], o));
    }
    bad |= __shfl_xor_sync(FULL_MASK, bad, o);
  }
  __shared__ float s_lo[THREADS / 32][3], s_hi[THREADS / 32][3];
  __shared__ int s_bad[THREADS / 32];
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  if (lane == 0) {
    for (int a = 0; a < 3; ++a) { s_lo[warp][a] = lo[a]; s_hi[warp][a] = hi[a]; }
    s_bad[warp] = bad;
  }
  __syncthreads();
  if (threadIdx.x < 3) {
    const int a = threadIdx.x;
    float l = s_lo[0][a], h = s_hi[0][a];
    for (int w = 1; w < THREADS / 32; ++w) { l = fminf(l, s_lo[w][a]); h = fmaxf(h, s_hi[w][a]); }
    atomicMin(&bounds[a], float_to_ordered(l));
    atomicMax(&bounds[3 + a], float_to_ordered(h));
  }
  if (threadIdx.x == 3) {
    int b = 0;
    for (int w = 0; w < THREADS / 32; ++w) b |= s_bad[w];
    if (b) atomicOr(&bounds[6], 1u);
  }
}

// ------------------------------------------------------------------------------------------------
// Morton code with `bits` bits per axis (<= 21, i.e. <= 63 bits) on a CUBIC grid spanning the longest
// scene extent, so cells are cubes whatever the aspect ratio of the cloud.  vals[i] = i (the sort
// payload).  The builder picks bits = ceil(log2(n) / 3) + 8: cells 256x finer per axis than the mean
// point spacing, which keeps the radix-sort pass count at ceil(3 * bits / 8) (6 instead of 8 at 10 M
// points).  Points that still share a cell are ordered by index — tree quality, never exactness.
// ------------------------------------------------------------------------------------------------
__device__ __forceinline__ uint64_t spread21(uint32_t v) {
  uint64_t x = v & 0x1fffffu;
  x = (x | (x << 32)) & 0x001f00000000ffffull;
  x = (x | (x << 16)) & 0x001f0000ff0000ffull;
  x = (x | (x << 8)) & 0x100f00f00f00f00full;
  x = (x | (x << 4)) & 0x10c30c30c30c30c3ull;
  x = (x | (x << 2)) & 0x1249249249249249ull;
  return x;
}

// Hilbert index of a cell of the 2^bits cubic grid in "transposed" form (Skilling 2004, AxesToTranspose): afterwards the
// three words hold the index's bits interleaved exactly like a Morton code holds the coordinates' bits, so the same
// spread21 interleave yields the key.  A Hilbert key has the Morton key's prefix property — the first 3 m bits name the
// same octree cell at level m, only the order of the eight children differs — so the leaf cut and the Karras hierarchy
// see the same cells and build the same tree up to child order.  What changes is the ORDER of the points: consecutive
// points on the Hilbert curve are always neighbours in space, while the Z-curve jumps at every octant seam.  The
// traversal's work unit is 32 consecutive sorted points whose balls are searched TOGETHER: on 2 M uniform points the
// bounding box of such a group, inflated by the k-th-neighbour radius, holds 245 points on average along the Hilbert
// curve and 427 along the Z-curve (p90: 306 vs 642).
__device__ __forceinline__ void hilbert_transpose(uint32_t& x0, uint32_t& x1, uint32_t& x2, int bits) {
  for (uint32_t q = 1u << (bits - 1); q > 1u; q >>= 1) {
    const uint32_t p = q - 1u;
    if (x0 & q) x0 ^= p;  // axis 0: invert (the exchange with itself is the identity)
    if (x1 & q) x0 ^= p; else { const uint32_t t = (x0 ^ x1) & p; x0 ^= t; x1 ^= t; }
    if (x2 & q) x0 ^= p; else { const uint32_t t = (x0 ^ x2) & p; x0 ^= t; x2 ^= t; }
  }
  x1 ^= x0;  // Gray encode
  x2 ^= x1;
  uint32_t t = x2 >> 1;  // t bit j = xor of the bits of x2 above j
  t ^= t >> 1; t ^= t >> 2; t ^= t >> 4; t ^= t >> 8; t ^= t >> 16;
  x0 ^= t; x1 ^= t; x2 ^= t;
}

// The key's quantisation: the cubic frame over the scene bounds (origin = the box's low corner, 2^21 cells along the
// longest axis) and a coordinate's 21-bit cell.  The grid table (grid.cuh) reuses both, so a point's level-L cell there is
// exactly the one the top 3 L bits of its sort key name.  Every step is monotone in v (RN subtract and multiply, clamps,
// truncation), which grid.cuh relies on too.
struct KeyFrame {
  float lx, ly, lz, scale;
};
__device__ __forceinline__ KeyFrame key_frame(const uint32_t* __restrict__ bounds) {
  KeyFrame f;
  f.lx = ordered_to_float(bounds[0]); f.ly = ordered_to_float(bounds[1]); f.lz = ordered_to_float(bounds[2]);
  const float ex = ordered_to_float(bounds[3]) - f.lx, ey = ordered_to_float(bounds[4]) - f.ly,
              ez = ordered_to_float(bounds[5]) - f.lz;
  const float ext = fmaxf(fmaxf(ex, ey), fmaxf(ez, FLT_MIN));
  f.scale = 2097152.0f / ext;  // 2^21 cells along the longest axis
  return f;
}
__device__ __forceinline__ uint32_t quantise21(float v, float lo, float scale) {
  return (uint32_t)fminf(fmaxf(__fmul_rn(__fsub_rn(v, lo), scale), 0.0f), 2097151.0f);
}

// curve: 0 = Morton (Z-order); h > 0 = Hilbert order on the top h bits per axis, Morton order below.  The curve only
// has to keep consecutive points together down to the level where a cell holds about one point (log2(n) / 3 bits per
// axis); the builder asks for two levels more.  Below that the digits stay plain Morton digits — each still names one
// octant of its cell, so the key keeps its prefix property — and the transform loop is 40 % shorter (10 of 16 levels
// at 10 M points: 0.22 -> 0.15 ms).
static __global__ void __launch_bounds__(THREADS) morton_kernel(const float* __restrict__ xyz, uint64_t n, int dim, int stride,
                                                         const uint32_t* __restrict__ bounds, int bits, int curve,
                                                         int idx_bits, uint64_t* __restrict__ keys,
                                                         uint32_t* __restrict__ vals) {
  const uint64_t i = (uint64_t)blockIdx.x * THREADS + threadIdx.x;
  if (i >= n) return;
  const KeyFrame f = key_frame(bounds);
  const float* p = xyz + i * (uint64_t)stride;
  const float x = p[0], y = p[1], z = dim > 2 ? p[2] : 0.0f;
  const int drop = 21 - bits;  // keep the top `bits` bits of each 21-bit coordinate
  uint32_t cx = quantise21(x, f.lx, f.scale) >> drop;
  uint32_t cy = quantise21(y, f.ly, f.scale) >> drop;
  uint32_t cz = quantise21(z, f.lz, f.scale) >> drop;
  if (curve > 0) {
    const int h = curve < bits ? curve : bits, low = bits - h;
    uint32_t hx = cx >> low, hy = cy >> low, hz = cz >> low;
    hilbert_transpose(hx, hy, hz, h);
    const uint32_t lm = (1u << low) - 1u;
    cx = (hx << low) | (cx & lm);
    cy = (hy << low) | (cy & lm);
    cz = (hz << low) | (cz & lm);
  }
  const uint64_t code = (spread21(cx) << 2) | (spread21(cy) << 1) | spread21(cz);
  if (idx_bits > 0) {
    // packed key: the code above the point's index (3 * bits + idx_bits <= 64).  The sort runs on the code bits only
    // and moves 8 instead of 12 bytes per point and pass; keys are distinct, ties of the code are in index order.
    keys[i] = (code << idx_bits) | i;
  } else {
    keys[i] = code;
    vals[i] = (uint32_t)i;
  }
}

// sorted float4 points: (x, y, z, id bits).  The id is the row number of the point in the caller's array, or —
// ids_in_w (point-partitioned driver) — the bits of the row's 4th float, so that a rank's BVH carries GLOBAL ids
// and its (d2, id) tie-breaks are the global ones.  bad_flag (optional): set when a coordinate is not finite.
// The source row of sorted position i is order[i], or — order == nullptr — the low idx_bits bits of packed[i].
static __global__ void __launch_bounds__(THREADS) gather_points_kernel(const float* __restrict__ xyz, int dim, int stride,
                                                                const uint32_t* __restrict__ order,
                                                                const uint64_t* __restrict__ packed, int idx_bits, uint64_t n,
                                                                int ids_in_w, float4* __restrict__ pts,
                                                                uint32_t* __restrict__ bad_flag = nullptr) {
  const uint64_t i = (uint64_t)blockIdx.x * THREADS + threadIdx.x;
  if (i >= n) return;
  const uint32_t src = order ? order[i] : (uint32_t)(packed[i] & ((1ull << idx_bits) - 1ull));
  const float* p = xyz + (uint64_t)src * (uint64_t)stride;
  const float x = p[0], y = p[1], z = dim > 2 ? p[2] : 0.0f;
  if (bad_flag && !(isfinite(x) && isfinite(y) && isfinite(z))) *bad_flag = 1u;
  pts[i] = make_float4(x, y, z, ids_in_w ? p[3] : __uint_as_float(src));
}

// ------------------------------------------------------------------------------------------------
// Leaf cut.  Policy 0 (default): the leaves are the maximal subtrees of the point-level radix tree
// holding <= leaf_max points ("treelet collapse"), found WITHOUT building that tree: the internal
// node that splits at boundary b spans the points between the nearest strictly stronger boundaries
// on each side, and b is a leaf boundary iff that span exceeds leaf_max — a +-leaf_max window scan.
// Policy 1: fixed chunks of leaf_max consecutive points.
// delta[b] = length of the common prefix of the augmented keys (code, position) at sorted positions b-1 and b
// (Karras 2012); smaller = stronger split; delta[0] = 0.  It is computed from the keys while staging.
// Output: one ballot word per 32 boundaries.
// ------------------------------------------------------------------------------------------------
static __global__ void __launch_bounds__(THREADS) leaf_flag_kernel(const uint64_t* __restrict__ keys, uint64_t n, int leaf_max,
                                                            int policy, uint64_t force_split,
                                                            uint32_t* __restrict__ ballots) {
  // The block's boundaries plus a halo of MAX_LEAF on both sides, staged once in shared memory.  Positions
  // outside [0, n) hold 0 = "stronger than anything" (delta[0] is 0 too), which makes the array ends behave
  // like the boundaries at 0 and n without special cases.
  __shared__ __align__(4) uint8_t s_delta[THREADS + 2 * MAX_LEAF];
  const int64_t block0 = (int64_t)blockIdx.x * THREADS;
  const int64_t in = (int64_t)n;
  for (int i = threadIdx.x; i < THREADS + 2 * MAX_LEAF; i += THREADS) {
    const int64_t g = block0 - MAX_LEAF + i;
    uint8_t dv = 0;
    if (g > 0 && g < in) {
      const uint64_t x = __ldg(&keys[g - 1]) ^ __ldg(&keys[g]);
      dv = (uint8_t)(x ? __clzll((long long)x) : 64 + __clz((uint32_t)(g - 1) ^ (uint32_t)g));
    }
    s_delta[i] = dv;
  }
  __syncthreads();
  const int64_t ib = block0 + threadIdx.x;
  bool cut = false;
  if (ib < in) {
    if (ib == 0 || (force_split && (uint64_t)ib == force_split)) cut = true;
    else if (policy == 1) cut = (ib % leaf_max) == 0;
    else {
      // nearest strictly stronger boundary within leaf_max - 1 positions on each side, four bytes per step
      const uint32_t* w32 = reinterpret_cast<const uint32_t*>(s_delta);
      const int m = MAX_LEAF + (int)threadIdx.x;  // my position in the window
      const uint32_t sb = (uint32_t)s_delta[m] * 0x01010101u;
      const int none = 4 * MAX_LEAF;
      int dl = none, dr = none;
      {  // left: highest position p in [m - (leaf_max - 1), m - 1] with s_delta[p] < s
        const int lo_lim = m - (leaf_max - 1);
        int wi = (m - 1) >> 2;
        uint32_t lt = __vcmpltu4(w32[wi], sb) & (0xFFFFFFFFu >> (8 * (3 - ((m - 1) & 3))));
        for (;;) {
          if (lt) {
            const int pos = wi * 4 + ((31 - __clz(lt)) >> 3);
            if (pos >= lo_lim) dl = m - pos;
            break;
          }
          if (wi * 4 <= lo_lim) break;
          --wi;
          lt = __vcmpltu4(w32[wi], sb);
        }
      }
      {  // right: lowest position p in [m + 1, m + (leaf_max - 1)] with s_delta[p] < s
        const int hi_lim = m + (leaf_max - 1);
        int wi = (m + 1) >> 2;
        uint32_t lt = __vcmpltu4(w32[wi], sb) & (0xFFFFFFFFu << (8 * ((m + 1) & 3)));
        for (;;) {
          if (lt) {
            const int pos = wi * 4 + ((__ffs(lt) - 1) >> 3);
            if (pos <= hi_lim) dr = pos - m;
            break;
          }
          if (wi * 4 + 3 >= hi_lim) break;
          ++wi;
          lt = __vcmpltu4(w32[wi], sb);
        }
      }
      cut = dl + dr > leaf_max;  // the node that splits here spans more than leaf_max points
    }
  }
  const uint32_t word = __ballot_sync(FULL_MASK, cut);
  if ((threadIdx.x & 31) == 0 && ib < in) ballots[ib >> 5] = word;
}

// ------------------------------------------------------------------------------------------------
// Exclusive scan of popc(ballots[i]) (three-phase reduce / scan-of-sums / apply).
// ------------------------------------------------------------------------------------------------
constexpr int SCAN_ITEMS = 8;
constexpr int SCAN_CHUNK = THREADS * SCAN_ITEMS;

__device__ __forceinline__ uint32_t block_exclusive_scan(uint32_t v, uint32_t* s_warp, uint32_t* total) {
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  uint32_t inc = v;
#pragma unroll
  for (int o = 1; o < 32; o <<= 1) {
    const uint32_t t = __shfl_up_sync(FULL_MASK, inc, o);
    if (lane >= o) inc += t;
  }
  if (lane == 31) s_warp[warp] = inc;
  __syncthreads();
  uint32_t off = 0, tot = 0;
  for (int w = 0; w < THREADS / 32; ++w) {
    const uint32_t x = s_warp[w];
    if (w < warp) off += x;
    tot += x;
  }
  __syncthreads();
  if (total) *total = tot;
  return off + inc - v;
}

static __global__ void __launch_bounds__(THREADS) popc_reduce_kernel(const uint32_t* __restrict__ words, uint64_t nw,
                                                              uint32_t* __restrict__ block_sums) {
  __shared__ uint32_t s_warp[THREADS / 32];
  const uint64_t base = (uint64_t)blockIdx.x * SCAN_CHUNK + (uint64_t)threadIdx.x * SCAN_ITEMS;
  uint32_t v = 0;
#pragma unroll
  for (int i = 0; i < SCAN_ITEMS; ++i)
    if (base + i < nw) v += __popc(words[base + i]);
  uint32_t total;
  block_exclusive_scan(v, s_warp, &total);
  if (threadIdx.x == 0) block_sums[blockIdx.x] = total;
}

// single block: exclusive scan of block_sums in place, grand total -> *total_out
static __global__ void __launch_bounds__(THREADS) scan_sums_kernel(uint32_t* __restrict__ block_sums, uint32_t nb,
                                                            uint32_t* __restrict__ total_out) {
  __shared__ uint32_t s_warp[THREADS / 32];
  uint32_t carry = 0;
  for (uint32_t base = 0; base < nb; base += THREADS) {
    const uint32_t i = base + threadIdx.x;
    const uint32_t v = i < nb ? block_sums[i] : 0u;
    uint32_t total;
    const uint32_t ex = block_exclusive_scan(v, s_warp, &total);
    if (i < nb) block_sums[i] = carry + ex;
    carry += total;
  }
  if (threadIdx.x == 0) *total_out = carry;
}

static __global__ void __launch_bounds__(THREADS) popc_apply_kernel(const uint32_t* __restrict__ words, uint64_t nw,
                                                             const uint32_t* __restrict__ block_sums,
                                                             uint32_t* __restrict__ offsets) {
  __shared__ uint32_t s_warp[THREADS / 32];
  const uint64_t base = (uint64_t)blockIdx.x * SCAN_CHUNK + (uint64_t)threadIdx.x * SCAN_ITEMS;
  uint32_t c[SCAN_ITEMS];
  uint32_t v = 0;
#pragma unroll
  for (int i = 0; i < SCAN_ITEMS; ++i) {
    c[i] = (base + i < nw) ? __popc(words[base + i]) : 0u;
    v += c[i];
  }
  uint32_t ex = block_exclusive_scan(v, s_warp, nullptr) + block_sums[blockIdx.x];
#pragma unroll
  for (int i = 0; i < SCAN_ITEMS; ++i) {
    if (base + i < nw) offsets[base + i] = ex;
    ex += c[i];
  }
}

// leaf_start[offsets[w] + rank-in-word] = b for every flagged boundary; leaf_key = its Morton code
static __global__ void __launch_bounds__(THREADS) leaf_emit_kernel(const uint32_t* __restrict__ ballots,
                                                            const uint32_t* __restrict__ offsets,
                                                            const uint64_t* __restrict__ keys, uint64_t n,
                                                            uint32_t n_leaves, uint32_t* __restrict__ leaf_start,
                                                            uint64_t* __restrict__ leaf_key) {
  const uint64_t b = (uint64_t)blockIdx.x * THREADS + threadIdx.x;
  if (b == 0) leaf_start[n_leaves] = (uint32_t)n;
  if (b >= n) return;
  const uint32_t w = ballots[b >> 5];
  const int bit = (int)(b & 31);
  if ((w >> bit) & 1u) {
    const uint32_t pos = offsets[b >> 5] + __popc(w & ((1u << bit) - 1u));
    leaf_start[pos] = (uint32_t)b;
    leaf_key[pos] = keys[b];
  }
}

// ------------------------------------------------------------------------------------------------
// Karras radix-tree hierarchy over the M leaves (keys = first Morton code of each leaf, ties broken
// by leaf index).  One thread per internal node.  child_info[node] = (ref0, cnt0, ref1, cnt1):
// cnt == 0 => internal child (ref = node index) else leaf child (ref = first sorted point).
// parent_*[] = (parent node << 1) | child slot;  node 0 is the root.
// ------------------------------------------------------------------------------------------------
__device__ __forceinline__ int karras_delta(const uint64_t* __restrict__ key, int64_t m, int64_t i, int64_t j) {
  if (j < 0 || j >= m) return -1;
  const uint64_t x = key[i] ^ key[j];
  return x ? __clzll((long long)x) : 64 + __clz((uint32_t)i ^ (uint32_t)j);
}

// the leaf range [lo, hi] of internal node i and its split: child 0 covers leaves lo .. gamma, child 1 gamma + 1 .. hi
__device__ __forceinline__ void karras_range(const uint64_t* __restrict__ leaf_key, int64_t m, int64_t i, int64_t& lo,
                                             int64_t& hi, int64_t& gamma) {
  const int d = (karras_delta(leaf_key, m, i, i + 1) - karras_delta(leaf_key, m, i, i - 1)) >= 0 ? 1 : -1;
  const int dmin = karras_delta(leaf_key, m, i, i - d);
  int64_t lmax = 2;
  while (karras_delta(leaf_key, m, i, i + lmax * d) > dmin) lmax <<= 1;
  int64_t l = 0;
  for (int64_t t = lmax >> 1; t >= 1; t >>= 1)
    if (karras_delta(leaf_key, m, i, i + (l + t) * d) > dmin) l += t;
  const int64_t j = i + l * d;
  const int dnode = karras_delta(leaf_key, m, i, j);
  int64_t s = 0, t = l;
  do {
    t = (t + 1) >> 1;
    if (karras_delta(leaf_key, m, i, i + (s + t) * d) > dnode) s += t;
  } while (t > 1);
  gamma = i + s * d + (d < 0 ? -1 : 0);
  lo = i < j ? i : j;
  hi = i < j ? j : i;
}

static __global__ void __launch_bounds__(THREADS) karras_kernel(const uint64_t* __restrict__ leaf_key,
                                                         const uint32_t* __restrict__ leaf_start, uint32_t n_leaves,
                                                         int4* __restrict__ child_info, int32_t* __restrict__ parent_leaf,
                                                         int32_t* __restrict__ parent_node) {
  const int64_t i = (int64_t)blockIdx.x * THREADS + threadIdx.x;
  const int64_t m = n_leaves;
  if (i >= m - 1) return;
  int64_t lo, hi, gamma;
  karras_range(leaf_key, m, i, lo, hi, gamma);
  int4 info;
  if (lo == gamma) {
    info.x = (int)leaf_start[gamma];
    info.y = (int)(leaf_start[gamma + 1] - leaf_start[gamma]);
    parent_leaf[gamma] = (int)((i << 1) | 0);
  } else {
    info.x = (int)gamma;
    info.y = 0;
    parent_node[gamma] = (int)((i << 1) | 0);
  }
  if (hi == gamma + 1) {
    info.z = (int)leaf_start[gamma + 1];
    info.w = (int)(leaf_start[gamma + 2] - leaf_start[gamma + 1]);
    parent_leaf[gamma + 1] = (int)((i << 1) | 1);
  } else {
    info.z = (int)(gamma + 1);
    info.w = 0;
    parent_node[gamma + 1] = (int)((i << 1) | 1);
  }
  child_info[i] = info;
  if (i == 0) parent_node[0] = -1;
}

// ------------------------------------------------------------------------------------------------
// Segmented builds (tknn_build_segments).  Segment s is the points with indices in [off[s], off[s + 1]).  Its id sits in
// the top bits of the sort key, above the curve code, so the sort keeps the segments contiguous and in order: the sorted
// positions of segment s are [off[s], off[s + 1]) as well, and seg_of serves both numberings.
// ------------------------------------------------------------------------------------------------
// seg_of[i] = the segment of index i (the last s with off[s] <= i: an empty segment never wins); keys[i] |= seg << shift
static __global__ void __launch_bounds__(THREADS) segment_key_kernel(const uint64_t* __restrict__ off, uint64_t n_segments,
                                                                     uint64_t n, int shift, uint64_t* __restrict__ keys,
                                                                     uint32_t* __restrict__ seg_of) {
  const uint64_t i = (uint64_t)blockIdx.x * THREADS + threadIdx.x;
  if (i >= n) return;
  uint64_t lo = 0, hi = n_segments;  // off[lo] <= i < off[hi]
  while (hi - lo > 1) {
    const uint64_t mid = (lo + hi) >> 1;
    if (__ldg(&off[mid]) <= i) lo = mid; else hi = mid;
  }
  seg_of[i] = (uint32_t)lo;
  keys[i] |= lo << shift;
}

// a leaf boundary at the start of every non-empty segment: no leaf holds points of two segments
static __global__ void __launch_bounds__(THREADS) segment_cut_kernel(const uint64_t* __restrict__ off, uint64_t n_segments,
                                                                     uint64_t n, uint32_t* __restrict__ ballots) {
  const uint64_t s = (uint64_t)blockIdx.x * THREADS + threadIdx.x;
  if (s >= n_segments) return;
  const uint64_t b = off[s];
  if (b < n && b < off[s + 1]) atomicOr(&ballots[b >> 5], 1u << (b & 31));
}

// node_seg[i] = the segment ranges of node i's children: (first, last segment under child 0, the same for child 1).  With
// the segment prefix and the cut above, a node lies inside one segment or is a union of whole segments.
static __global__ void __launch_bounds__(THREADS) node_segments_kernel(const uint64_t* __restrict__ leaf_key,
                                                                       const uint32_t* __restrict__ leaf_start, uint32_t n_leaves,
                                                                       const uint32_t* __restrict__ seg_of,
                                                                       int4* __restrict__ node_seg) {
  const int64_t i = (int64_t)blockIdx.x * THREADS + threadIdx.x;
  const int64_t m = n_leaves;
  if (i >= m - 1) return;
  int64_t lo, hi, gamma;
  karras_range(leaf_key, m, i, lo, hi, gamma);
  const uint32_t p0 = leaf_start[lo], p1 = leaf_start[gamma + 1], p2 = leaf_start[hi + 1];
  node_seg[i] = make_int4((int)seg_of[p0], (int)seg_of[p1 - 1], (int)seg_of[p1], (int)seg_of[p2 - 1]);
}

// ------------------------------------------------------------------------------------------------
// Bottom-up refit: one thread per leaf computes the leaf box and climbs; at every internal node the
// first arriver parks its child's record (box + ref + count, two 16-byte stores) in its half of the node
// and stops; the second one reads it back, writes the whole node in its final interleaved layout
// (common.cuh: Node) with four 16-byte stores, merges and continues.
// ------------------------------------------------------------------------------------------------
static __global__ void __launch_bounds__(THREADS) refit_kernel(const float4* __restrict__ pts,
                                                        const uint32_t* __restrict__ leaf_start, uint32_t n_leaves,
                                                        const int4* __restrict__ child_info,
                                                        const int32_t* __restrict__ parent_leaf,
                                                        const int32_t* __restrict__ parent_node,
                                                        uint32_t* __restrict__ arrive, Node* nodes,
                                                        int* node_min_idx, uint32_t* __restrict__ dup_leaf_flag,
                                                        uint32_t dup_min, float* __restrict__ scene_box) {
  const uint32_t leaf = blockIdx.x * THREADS + threadIdx.x;
  if (leaf >= n_leaves) return;
  const uint32_t b = leaf_start[leaf], e = leaf_start[leaf + 1];
  float3 lo = make_float3(INFINITY, INFINITY, INFINITY), hi = make_float3(-INFINITY, -INFINITY, -INFINITY);
  int mn = 0x7fffffff;  // smallest original index in the subtree (index-aware pruning of exact distance ties)
  for (uint32_t i = b; i < e; ++i) {
    const float4 p = __ldg(&pts[i]);
    lo.x = fminf(lo.x, p.x); lo.y = fminf(lo.y, p.y); lo.z = fminf(lo.z, p.z);
    hi.x = fmaxf(hi.x, p.x); hi.y = fmaxf(hi.y, p.y); hi.z = fmaxf(hi.z, p.z);
    mn = min(mn, __float_as_int(p.w));
  }
  // A leaf of >= dup_min coincident points: the cloud has duplicate CLUSTERS; searches enable tie pruning.  Tie pruning
  // pays when a cluster fills many leaves (all at box distance == bound: D / 32 leaf visits per group without it); a few
  // doubled points do not, and the pruning variant of the kernel costs 4.5 % on such a cloud (cfg3: 10 000 doubled points
  // in 10 M, 46.3 ms with it, 44.2 ms without, the same node and test counts: profiles/r2_ab_ties_cfg3.jsonl).
  if (e - b >= dup_min && lo.x == hi.x && lo.y == hi.y && lo.z == hi.z) *dup_leaf_flag = 1u;
  int32_t link = parent_leaf[leaf];
  for (;;) {
    const int node = link >> 1, slot = link & 1;
    const int4 info = child_info[node];
    const int ref = slot ? info.z : info.x, cnt = slot ? info.w : info.y;
    float4* rec = reinterpret_cast<float4*>(nodes + node) + 2 * slot;
    __stcg(rec, make_float4(lo.x, lo.y, lo.z, __int_as_float(ref)));
    __stcg(rec + 1, make_float4(hi.x, hi.y, hi.z, __int_as_float(cnt)));
    __stcg(&node_min_idx[2 * node + slot], mn);
    __threadfence();
    if (atomicAdd(&arrive[node], 1u) == 0u) return;
    __threadfence();  // acquire side: the sibling's record was written before its arrival
    const float4* sib = reinterpret_cast<const float4*>(nodes + node) + 2 * (1 - slot);
    const float4 slo = __ldcg(sib), shi = __ldcg(sib + 1);
    mn = min(mn, __ldcg(&node_min_idx[2 * node + (1 - slot)]));
    {  // both children are known: the node in its final layout (child 0 low, child 1 high in every pair)
      const float4 mlo = make_float4(lo.x, lo.y, lo.z, __int_as_float(ref)), mhi = make_float4(hi.x, hi.y, hi.z, __int_as_float(cnt));
      const float4 l0 = slot ? slo : mlo, h0 = slot ? shi : mhi, l1 = slot ? mlo : slo, h1 = slot ? mhi : shi;
      float4* out = reinterpret_cast<float4*>(nodes + node);
      __stcg(out, make_float4(l0.x, l1.x, l0.y, l1.y));
      __stcg(out + 1, make_float4(l0.z, l1.z, h0.x, h1.x));
      __stcg(out + 2, make_float4(h0.y, h1.y, h0.z, h1.z));
      __stcg(out + 3, make_float4(l0.w, l1.w, h0.w, h1.w));
    }
    lo.x = fminf(lo.x, slo.x); lo.y = fminf(lo.y, slo.y); lo.z = fminf(lo.z, slo.z);
    hi.x = fmaxf(hi.x, shi.x); hi.y = fmaxf(hi.y, shi.y); hi.z = fmaxf(hi.z, shi.z);
    if (node == 0) {
      scene_box[0] = lo.x; scene_box[1] = lo.y; scene_box[2] = lo.z;
      scene_box[3] = hi.x; scene_box[4] = hi.y; scene_box[5] = hi.z;
      return;
    }
    link = parent_node[node];
  }
}

}  // namespace lbvh
}  // namespace tknn
