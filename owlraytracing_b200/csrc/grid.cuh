// grid.cuh — a uniform cell grid over the sorted points, and the dense kNN round kernel that walks it.
//
// The build sorts the points by a key whose top 3 L bits name the level-L octree cell (Morton and Hilbert digits alike,
// lbvh.cuh), so every level-L cell is one contiguous run of sorted positions.  A table of runs per cell, indexed by the
// linear (x, y, z) cell, turns the sorted points into a grid with no extra copy of them.  On a uniform cloud a 32-query
// group then lists the cells that meet its lanes' balls directly: a cell holds a few points instead of a leaf's ~21, and
// there is no tree walk (DESIGN.md §3.2).
//
// Exactness.  Cell c along an axis holds exactly the points whose coordinate v has quantise21(v) >> (21 - L) == c
// (lbvh.cuh: the key's own arithmetic, monotone in v).  The table stores per axis B[c] = the smallest float in the scene's
// range whose cell is >= c (found by bisection over the float bit patterns with that same arithmetic; B[0] and B[2^L] are
// the scene's own bounds), so every point of cell c lies in [B[c], B[c + 1]] with no rounding margin at all, and the
// point-to-box distance of that box (box_dist2's chain) never exceeds the point's dist2 (the argument of common.cuh).
// The cull is therefore conservative, the filter and the (d2, index) keys are the LBVH kernel's, and the k-lists end
// bit-identical.
#pragma once
#include "common.cuh"
#include "lbvh.cuh"
#include "traverse.cuh"

namespace tknn {
namespace grid {

constexpr int MAX_LEVEL = 8;   // 2^24 cells (134 MB of runs) at most
constexpr int MAX_SPAN = 31;   // cells per axis a group may span (its 32 boundaries fill one warp-wide load)
#ifndef TKNN_GRID_CAP
#define TKNN_GRID_CAP 1024     // cells a group may test; a larger range is left unresolved to the LBVH rounds
#endif
#ifndef TKNN_GRID_FLUSH
#define TKNN_GRID_FLUSH 64     // staged points that trigger the filter + insert pass (<= 64: the staging area)
#endif
// Selection: the grid serves a build only while its fullest cell holds at most this many points.  Uniform clouds stay far
// below it (10 M points at level 7: 4.8 per cell on average, 23 at most); clustered clouds (LiDAR-like scans, duplicate
// clusters) exceed it by orders of magnitude, and there cells as large as the leaves' boxes would gain nothing.
constexpr uint32_t SELECT_MAX_CELL = 64;

// Frame of the table: the key's cubic frame (lbvh::KeyFrame), the highest occupied cell per axis, then the boundaries.
// Words: [0..3] lx, ly, lz, scale; [4..6] highest cell per axis (u32); [7] unused; [8 ..] B_x[0 .. 2^L], B_y, B_z.
constexpr int FRAME_WORDS = 8;
__host__ __device__ inline size_t frame_words(int level) { return FRAME_WORDS + 3 * (((size_t)1 << level) + 1); }

__device__ __forceinline__ uint32_t cell_of(float v, float lo, float scale, int shift) {
  return lbvh::quantise21(v, lo, scale) >> shift;
}

// one thread per sorted position: the run boundaries of its cell.  A run start takes the cell's `start` slot with an
// exchange: finding it taken means the cell's points are not one contiguous run (`split` counts such starts; the table
// is then not used).  Empty cells keep 0xffffffff in both words: end - start = 0.
static __global__ void __launch_bounds__(256) fill_kernel(const float4* __restrict__ pts, uint64_t n,
                                                          const uint32_t* __restrict__ bounds, int level,
                                                          uint2* __restrict__ cells, uint32_t* __restrict__ split) {
  const uint64_t i = (uint64_t)blockIdx.x * 256 + threadIdx.x;
  if (i >= n) return;
  const lbvh::KeyFrame f = lbvh::key_frame(bounds);
  const int sh = 21 - level;
  auto lin = [&](const float4 p) -> uint64_t {
    return ((uint64_t)cell_of(p.x, f.lx, f.scale, sh) << (2 * level)) | ((uint64_t)cell_of(p.y, f.ly, f.scale, sh) << level) |
           cell_of(p.z, f.lz, f.scale, sh);
  };
  const uint64_t c = lin(__ldg(&pts[i]));
  if (i == 0 || lin(__ldg(&pts[i - 1])) != c) {
    if (atomicExch(&cells[c].x, (uint32_t)i) != 0xffffffffu) atomicAdd(split, 1u);
  }
  if (i + 1 == n || lin(__ldg(&pts[i + 1])) != c) cells[c].y = (uint32_t)(i + 1);
}

// The frame words: one thread per boundary (3 x (2^L + 1)), bisection over the ordered bit patterns of [lo, hi].
static __global__ void __launch_bounds__(256) frame_kernel(const uint32_t* __restrict__ bounds, int level,
                                                           float* __restrict__ frame) {
  const int per = (1 << level) + 1;
  const int t = blockIdx.x * 256 + threadIdx.x;
  if (t >= 3 * per) return;
  const int a = t / per, c = t - a * per;
  const lbvh::KeyFrame f = lbvh::key_frame(bounds);
  const float lo = ordered_to_float(bounds[a]), hi = ordered_to_float(bounds[3 + a]);
  const float org = a == 0 ? f.lx : (a == 1 ? f.ly : f.lz);
  const int sh = 21 - level;
  if (t == 0) {
    frame[0] = f.lx; frame[1] = f.ly; frame[2] = f.lz; frame[3] = f.scale;
  }
  if (c == 0) reinterpret_cast<uint32_t*>(frame)[4 + a] = cell_of(hi, org, f.scale, sh);
  float b;
  if (c == 0) {
    b = lo;
  } else if (c == per - 1 || cell_of(hi, org, f.scale, sh) < (uint32_t)c) {
    b = hi;  // no coordinate reaches cell c: the cells from c up are empty
  } else {   // smallest float v in [lo, hi] with cell(v) >= c: cell(hi) >= c > cell(lo) = 0
    uint32_t olo = float_to_ordered(lo), ohi = float_to_ordered(hi);  // pred(olo) false, pred(ohi) true
    while (ohi - olo > 1) {
      const uint32_t mid = olo + (ohi - olo) / 2;
      if (cell_of(ordered_to_float(mid), org, f.scale, sh) >= (uint32_t)c) ohi = mid; else olo = mid;
    }
    b = ordered_to_float(ohi);
  }
  frame[FRAME_WORDS + t] = b;
}

// out[0] = max(out[0], the largest run of a cell)
static __global__ void __launch_bounds__(256) occupancy_kernel(const uint2* __restrict__ cells, uint64_t n_cells,
                                                               uint32_t* __restrict__ out) {
  uint32_t m = 0;
  for (uint64_t i = (uint64_t)blockIdx.x * 256 + threadIdx.x; i < n_cells; i += (uint64_t)gridDim.x * 256) {
    const uint2 r = __ldg(&cells[i]);
    m = max(m, r.y - r.x);
  }
  m = __reduce_max_sync(FULL_MASK, m);
  if ((threadIdx.x & 31) == 0) atomicMax(out, m);
}

struct GridParams {
  const uint2* cells;   // per linear cell (x << 2L | y << L | z): sorted positions [x, y) of its points
  const float* frame;   // frame_kernel's words
  int level;
};

// per warp: the LBVH list kernel's layout (staging 64 points, stack area = the group's 3 x 32 cell boundaries, k-list,
// SoA coordinates) + the visit order of the group's cells per axis (3 x 32 bytes) + its low cell and width per axis
// (kept in shared memory: registers stay free for the loop nest)
__host__ __device__ inline size_t smem_per_warp(int k) { return trav::smem_per_warp(k) + 128; }

// Visit order along one axis of w cells, outward from cell c: c, c + 1, c - 1, c + 2, ... and, once one side is used up,
// the rest of the other side.  Near cells first, so the bounds tighten early.
__device__ __forceinline__ int zigzag(int j, int w, int c) {
  const int below = c, above = w - 1 - c, m = min(below, above);
  if (j <= 2 * m) return (j & 1) ? c + ((j + 1) >> 1) : c - (j >> 1);
  return above > below ? c + (j - m) : c - (j - m);
}

// 1-D term of box_dist2 (common.cuh), the same operations in the same order
__device__ __forceinline__ float axis_gap(float q, float lo, float hi) {
  return fmaxf(fmaxf(__fsub_rn(lo, q), __fsub_rn(q, hi)), 0.0f);
}

// Dense MODE_KNN round with k <= 24 on the grid: the persistent grid, 32-query groups, Params, emit and unresolved ballots of
// trav::traverse_kernel (ascending lists, exact filter).  Never a final round: a group whose cell range is too large (a huge or
// infinite radius: r2_dev may hold the estimator's +inf fallback) tests nothing and leaves its lanes unresolved, and the LBVH
// rounds after it finish them exactly.
// Per group: the integer cell range of the union of the lanes' boxes [q - s, q + s] (s >= sqrt(bound), see below), visited
// x-slab, y-row, z-cell, each axis outward from the middle; a slab, row or cell is entered when ANY lane's box distance to it
// is within that lane's current bound (warp vote).  The box term of each axis enters the chain in dist2's order (x first), so
// the slab and row terms are partial sums of the cell's distance and cull as conservatively.  Wanted cells' runs are staged
// into the 64-point area (NaN-padded), filtered into two masks by filter4 and inserted in one loop (the sibling-pair path of
// the LBVH kernel) whenever TKNN_GRID_FLUSH points are staged.
// Counting build: counters[0] = cell tests x active lanes (the nodes_visited field), [1] = staged points x active lanes,
// [2] = inserts, [3] = cell tests per warp, [4] = cells staged per warp, [5] = points staged per warp, [7] = groups left
// unresolved by the cap.
template <bool COUNT>
static __global__ void __launch_bounds__(256, COUNT ? 1 : 5) grid_knn_kernel(const trav::Params P, const GridParams G) {
  extern __shared__ __align__(16) unsigned char smem[];
  constexpr int NS = trav::stage_pts(false);  // 64
  constexpr int S = trav::KLS;
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int k = P.k;
  unsigned char* wbase = smem + (size_t)warp * smem_per_warp(k);
  float4* stage = reinterpret_cast<float4*>(wbase);
  float* gb = reinterpret_cast<float*>(wbase + NS * sizeof(float4));  // boundaries: x at [0, 32), y at [32, 64), z at [64, 96)
  uint64_t* H = reinterpret_cast<uint64_t*>(wbase + NS * sizeof(float4) + STACK_DEPTH * sizeof(int)) + lane;
  float* soa = reinterpret_cast<float*>(wbase + NS * sizeof(float4) + STACK_DEPTH * sizeof(int) + trav::klist_bytes(k));
  uint8_t* ord = reinterpret_cast<uint8_t*>(soa + 3 * NS);  // visit order: x at [0, 32), y at [32, 64), z at [64, 96)
  uint32_t* rng = reinterpret_cast<uint32_t*>(ord + 96);    // low cell per axis [0, 3), width per axis [3, 6)
  const int level = G.level, sh = 21 - level;
  const int per = (1 << level) + 1;

  unsigned long long c_cells = 0, c_tests = 0, c_ins = 0, c_wcells = 0, c_wstaged = 0, c_wpts = 0, c_defer = 0;
  const float round_r2 = P.r2_dev ? __ldg(P.r2_dev) : P.r2;
  const uint64_t n_active = P.n_active_dev ? min((uint64_t)__ldg(P.n_active_dev), P.n_active) : P.n_active;
  const uint32_t n_groups = (uint32_t)((n_active + 31) / 32);

  for (;;) {
    uint32_t group = 0;
    if (lane == 0) group = atomicAdd(P.group_counter, 1u);
    group = __shfl_sync(FULL_MASK, group, 0);
    if (group >= n_groups) break;

    const uint64_t gi = (uint64_t)group * 32 + lane;
    const bool valid = gi < n_active;
    uint64_t qpos = 0;
    if (valid) qpos = P.queue ? (uint64_t)P.queue[gi] : P.q_begin + gi;
    float4 q = make_float4(0.f, 0.f, 0.f, 0.f);
    if (valid) q = __ldg(&P.queries[qpos]);
    const int row_id = __float_as_int(q.w);
    int self = -1;
    if (valid) self = P.self_ids ? P.self_ids[qpos] : (P.self_is_row ? row_id : -1);
    float r2 = round_r2;
    if (valid && P.query_r2) r2 = fminf(r2, P.query_r2[qpos]);
    float bound = valid ? r2 : -1.0f;  // d2 >= 0 > -1: an idle lane never wants anything
    int cnt = 0;
    H[0] = 0;  // sentinel of this lane's k-list

    // ---- the group's cell range ----
    // A point p with dist2(q, p) <= bound has RN(dx * dx) <= bound (the fma chain only adds non-negative terms).  Rounding
    // errs by at most u = 2^-24 relative, or by 2^-150 absolute where dx * dx is subnormal, so dx^2 <= bound (1 + 2u) + 2^-150
    // and |q - p| <= sqrt(bound) (1 + 2u) + 2^-75 per axis.  s = fma(sqrtf(bound), 1.0001, fma(|q|, 2^-18, 2^-74)) exceeds
    // that by more than the rounding of q -/+ s (<= u (|q| + s)), so p lies in [RN(q - s), RN(q + s)], and the monotone cell
    // function maps it into the range.  Without the 2^-74 term a bound that is subnormal or 0 (a tiny cloud, a tiny start
    // radius) would miss points whose d2 underflows to it.  bound = +inf gives the whole grid (and the cap below).
    bool defer = false;
    {
      const float sb = valid ? sqrtf(bound) : 0.0f;
      const float scale = __ldg(&G.frame[3]);
      uint32_t vol = 1;
#pragma unroll
      for (int a = 0; a < 3; ++a) {
        const float qa = a == 0 ? q.x : (a == 1 ? q.y : q.z);
        const float org = __ldg(&G.frame[a]);
        const uint32_t top = __ldg(reinterpret_cast<const uint32_t*>(G.frame) + 4 + a);
        const float s = __fmaf_rn(sb, 1.0001f, __fmaf_rn(fabsf(qa), 0x1p-18f, 0x1p-74f));
        const uint32_t l = cell_of(__fsub_rn(qa, s), org, scale, sh);
        const uint32_t h = min(cell_of(__fadd_rn(qa, s), org, scale, sh), top);
        const uint32_t glo = __reduce_min_sync(FULL_MASK, valid ? l : 0xffffffffu);
        const uint32_t w = __reduce_max_sync(FULL_MASK, valid ? h : 0u) - glo + 1;
        if (w > (uint32_t)MAX_SPAN) defer = true;
        vol *= min(w, 32u);
        // the range's boundaries and the visit order along this axis
        if (w <= (uint32_t)MAX_SPAN) {
          if (lane <= (int)w) gb[32 * a + lane] = __ldg(&G.frame[FRAME_WORDS + a * per + glo + lane]);
          if (lane < (int)w) ord[32 * a + lane] = (uint8_t)zigzag(lane, (int)w, ((int)w - 1) >> 1);
        }
        if (lane == 0) { rng[a] = glo; rng[3 + a] = w; }
      }
      if (vol > (uint32_t)TKNN_GRID_CAP) defer = true;
    }
    __syncwarp();

    if (!defer) {

      int fill = 0;  // points staged
      // filter the staged points against the bounds as they are now, then insert the survivors (one divergent loop)
      auto flush = [&]() {
        if (lane < 8 && fill + lane < NS) soa[fill + lane] = __int_as_float(0x7fc00000);  // NaN x: the padded tail never passes
        __syncwarp();
        if (COUNT) { c_tests += valid ? fill : 0; c_wpts += fill; }
        const float2 qx2 = make_float2(q.x, q.x), qy2 = make_float2(q.y, q.y), qz2 = make_float2(q.z, q.z);
        uint32_t mask_a = 0, mask_b = 0;  // survivors among staged points 0..31 / 32..63
        const int na = min(fill, MAX_LEAF);
#pragma unroll 1
        for (int j0 = 0; j0 < na; j0 += 8)
          mask_a |= (trav::filter4<NS>(soa, j0, qx2, qy2, qz2, bound) | (trav::filter4<NS>(soa, j0 + 4, qx2, qy2, qz2, bound) << 4)) << j0;
#pragma unroll 1
        for (int j0 = MAX_LEAF; j0 < fill; j0 += 8)
          mask_b |= (trav::filter4<NS>(soa, j0, qx2, qy2, qz2, bound) | (trav::filter4<NS>(soa, j0 + 4, qx2, qy2, qz2, bound) << 4))
                    << (j0 - MAX_LEAF);
        while (mask_a | mask_b) {
          int j;
          if (mask_a) { j = __ffs(mask_a) - 1; mask_a &= mask_a - 1u; }
          else { j = MAX_LEAF + __ffs(mask_b) - 1; mask_b &= mask_b - 1u; }
          const float4 p = stage[j];
          const float d = dist2(q.x, q.y, q.z, p.x, p.y, p.z);
          const int pid = __float_as_int(p.w);
          if (pid != self && d <= bound) trav::list_take<S, COUNT>(H, cnt, k, bound, d, pid, c_ins);
        }
        __syncwarp();
        fill = 0;
      };

#pragma unroll 1
      for (int ix = 0; ix < (int)rng[3]; ++ix) {
        const int ox = ord[ix];
        const float tx = axis_gap(q.x, gb[ox], gb[ox + 1]);
        const float ax2 = __fmul_rn(tx, tx);
        if (!__any_sync(FULL_MASK, ax2 <= bound)) continue;
#pragma unroll 1
        for (int iy = 0; iy < (int)rng[4]; ++iy) {
          const int oy = ord[32 + iy];
          const float ty = axis_gap(q.y, gb[32 + oy], gb[33 + oy]);
          const float ay2 = __fmaf_rn(ty, ty, ax2);
          if (!__any_sync(FULL_MASK, ay2 <= bound)) continue;
          // the row's runs, lane j: cell (x, y, lo_z + j); one load for the whole row
          const int wz = (int)rng[5];
          uint2 run = make_uint2(0u, 0u);
          if (lane < wz)
            run = __ldg(&G.cells[((uint64_t)(rng[0] + ox) << (2 * level)) | ((uint64_t)(rng[1] + oy) << level) | (rng[2] + lane)]);
          const uint32_t full = __ballot_sync(FULL_MASK, run.y != run.x);
#pragma unroll 1
          for (int iz = 0; iz < wz; ++iz) {
            const int oz = ord[64 + iz];
            if (!((full >> oz) & 1u)) continue;
            const float tz = axis_gap(q.z, gb[64 + oz], gb[65 + oz]);
            const float d = __fmaf_rn(tz, tz, ay2);
            if (COUNT) { c_cells += valid ? 1 : 0; c_wcells += 1; }
            if (!__any_sync(FULL_MASK, d <= bound)) continue;
            uint32_t src = __shfl_sync(FULL_MASK, run.x, oz);
            int rem = (int)(__shfl_sync(FULL_MASK, run.y, oz) - src);
            if (COUNT) c_wstaged += 1;
            while (rem > 0) {  // a run longer than the free space continues after a flush
              const int take = min(rem, NS - fill);
#pragma unroll
              for (int h = 0; h < NS; h += 32) {
                if (lane + h < take) {
                  const float4 p = __ldg(&P.pts[(uint64_t)src + lane + h]);
                  const int j = fill + lane + h;
                  stage[j] = p;
                  soa[j] = p.x; soa[NS + j] = p.y; soa[2 * NS + j] = p.z;
                }
              }
              fill += take;
              src += take;
              rem -= take;
              if (fill == NS) flush();
            }
            if (fill >= TKNN_GRID_FLUSH) flush();
          }
        }
      }
      if (fill > 0) flush();
    } else if (COUNT && lane == 0) {
      c_defer += 1;
    }

    // ---- emit (non-final round: resolved lanes only) ----
    const bool resolved = valid && cnt == k;
    const unsigned un = __ballot_sync(FULL_MASK, valid && !resolved);
    if (lane == 0 && P.unresolved) P.unresolved[group] = un;
    if (resolved) {
      const uint64_t row = P.row_mode == 0 ? (uint64_t)(uint32_t)row_id : (P.row_mode == 1 ? qpos - P.q_begin : gi);
      if (P.row_mode && P.qid_out) P.qid_out[row] = row_id;
      trav::kl_emit<true, S>(H, cnt, k, false, P.squared != 0, P.idx_out + row * (uint64_t)k, P.dist_out + row * (uint64_t)k);
    }
    __syncwarp();
  }

  if (COUNT && P.counters) {
    atomicAdd(&P.counters[0], c_cells);
    atomicAdd(&P.counters[1], c_tests);
    atomicAdd(&P.counters[2], c_ins);
    if (lane == 0) {
      atomicAdd(&P.counters[3], c_wcells);
      atomicAdd(&P.counters[4], c_wstaged);
      atomicAdd(&P.counters[5], c_wpts);
      if (c_defer) atomicAdd(&P.counters[7], c_defer);
    }
  }
}

}  // namespace grid
}  // namespace tknn
