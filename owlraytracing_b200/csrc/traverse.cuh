// traverse.cuh — the persistent, warp-cooperative LBVH traversal kernel.
//
// Replaces, in one kernel, the reference's raygen program (samples/s01-trueknn/deviceCode.cu:140-152),
// the RT-core traversal behind optixTrace (owl/include/owl/owl_device.h:150-174) and the
// intersection program with its global-memory sorted k-list (deviceCode.cu:62-138).
//
// Work unit = a GROUP of 32 consecutive queries in Morton order, one query per lane.  The warp
// walks ONE stack for the group; a node is entered when ANY lane's exact point-to-box distance is
// within that lane's own bound min(r^2, k-th best d2) (warp vote), so culling is per query, never
// per group box.  A wanted leaf (<= 32 points, one coalesced 512 B float4 load) is staged in shared
// memory and broadcast to all lanes: 32 queries x 32 points of distance tests per 512 B fetched.
// Each lane owns a bounded k-list of (d2, index) keys (ascending list for k <= 24, padded 4-ary max-heap
// above); candidates are filtered against the bound into a bit mask first — two points per issue slot
// with Blackwell's packed fp32x2 instructions — and inserted afterwards, so the divergent part only
// runs for real hits.
//
// Three kernels share the rules and produce identical results: traverse_kernel (above; dense rounds),
// traverse_sparse_kernel (one thread per query; rounds whose survivors are spatially incoherent) and
// traverse_warp_kernel (one warp per query; tiny rounds and the start-radius sample).
//
// Exactness: box distances use the same fmaf chain as point distances (monotone under RN), pruning
// is strict (`>`), ties are resolved on the full (d2, index) key, self is excluded by index.
#pragma once
#include "common.cuh"
#include "dbscan.cuh"

namespace tknn {
namespace trav {

// MODE_DBSCAN_*: the three traversal passes of tknn_dbscan (dbscan.cuh has the pipeline around them).  All three use the
// closed eps-ball of MODE_RANGE_COUNT, the query's own point included.
//   CORE    every position; a lane stops wanting nodes (bound = -1) once its ball holds min_pts (= P.k) points; one
//           "is core" ballot word per group of 32 positions (P.unresolved, the core bitset).
//   LINK    the core queue; every core point of the ball is united with the query in the union-find (P.uf_parent).
//   BORDER  the non-core queue; the lowest cluster id (P.pos_label) among the core points of the ball, or -1.
// MODE_RANGE_LIST_*: the two traversal passes of tknn_radius_search / tknn_radius_query (radius.cuh has the pipeline).
// Both take the exact closed ball and drop the excluded point by POSITION (P.self_pos, or the query's own position when
// self_is_row): one bit of the leaf mask, which is "index != self" because positions and indices are a bijection.
//   COUNT   every query position; the ball's size minus self, written by position (P.count_out) and by row (P.count_row).
//   FILL    every query position; each member as the key make_key(d2, index) at the lane's cursor, which starts at
//           P.list_off[position] in P.list_keys (unsorted; the order pass sorts every row).
enum Mode { MODE_KNN = 0, MODE_RANGE_COUNT = 1, MODE_DBSCAN_CORE = 2, MODE_DBSCAN_LINK = 3, MODE_DBSCAN_BORDER = 4,
            MODE_RANGE_LIST_COUNT = 5, MODE_RANGE_LIST = 6 };

struct Params {
  const Node* nodes;
  const int2* node_min_idx;  // per node: smallest original index under child 0 / child 1 (tie pruning)
  const float4* pts;         // sorted data points (x, y, z, original index bits)
  const float4* queries;     // query points (x, y, z, row-id bits); == pts when all points are queries
  const uint32_t* queue;     // optional list of query positions (rounds >= 2); nullptr = identity
  const int32_t* self_ids;   // optional data index to exclude per query position; nullptr => see self_is_row
  const float* query_r2;     // optional per-query-position squared radius cap
  uint64_t n_active;         // queries in this launch
  uint64_t q_begin;          // first query position when queue == nullptr
  uint32_t n_groups;         // ceil(n_active / 32)
  float r2;                  // squared search radius of this round (may be +inf)
  int k;
  int self_is_row;           // 1: exclude the data point whose index equals the query's row id
  int row_mode;              // 0: output row = row id (scatter to build order); 1: row = position - q_begin;
                             // 2: row = index inside this launch
  int final_round;           // 1: emit every query, resolved or not (sentinels fill the rest)
  int squared;               // 1: dist_out receives d2 instead of sqrtf(d2)
  uint32_t* error;           // bit 0: traversal stack overflow (cannot happen for depth <= 95)
  int32_t* idx_out;
  float* dist_out;
  int32_t* qid_out;          // row_mode 1: row id of each compact row (may be nullptr)
  uint32_t* count_out;       // MODE_RANGE_COUNT
  uint32_t* unresolved;      // one ballot word per group
  uint32_t* group_counter;   // persistent-grid work counter
  const float* r2_dev;           // optional: the squared radius of this round, read from device memory (the start-radius
                                 // estimate stays on the device: no host round trip before round 1); overrides r2
  const uint32_t* n_active_dev;  // optional: min(*n_active_dev, n_active) queries are active (a round launched before the
                                 // host knows how many queries the previous round left unresolved)
  unsigned long long* counters;  // [0] node visits x active lanes, [1] point tests x active lanes, [2] inserts,
                                 // [3] warp node loads, [4] warp leaf loads, [5] warp point loads,
                                 // [6] pre-filter violations (must stay 0)
  // MODE_DBSCAN_LINK / _BORDER
  const uint32_t* core_words;    // the core bitset over positions, n_core_words words
  uint32_t n_core_words;
  int* uf_parent;                // LINK: union-find parents over positions
  const int32_t* pos_label;      // BORDER: cluster id of every core position
  int32_t* label_out;            // BORDER: label per original index (-1 = noise)
  uint8_t* core_out;             // BORDER: 0 per original index (may be nullptr)
  // MODE_RANGE_LIST_COUNT / _LIST
  const int32_t* self_pos;       // per query position: the data position to exclude or -1; nullptr => see self_is_row
  uint32_t* count_row;           // LIST_COUNT: ball size per output row (count_out: per query position)
  const uint64_t* list_off;      // LIST: first key slot of every query position
  uint64_t* list_keys;           // LIST: the unsorted rows, in position order
  // segmented builds (the SEG kernels)
  const uint32_t* seg_of;        // segment of every query position (built positions, or a staged query set's sorted rows)
  const uint64_t* seg_off;       // data segment offsets, n_segments + 1
  const int4* node_seg;          // per node: first / last segment under child 0, the same under child 1
};

// ---- segmented builds -----------------------------------------------------------------------------
// A lane searches only its query's segment.  At every node visit a child whose segment range does not hold the lane's
// segment gets box distance NaN for that lane: NaN fails every `<=`, `<` and `==` the walk makes, so the lane never wants
// it, even in an unbounded round (+inf would pass `<= +inf`).  Leaves never straddle segments, so a leaf staged for other
// lanes is foreign to this lane as a whole and its filter mask is cleared.  A row whose data segment has too few eligible
// points is resolved once it holds all of them (need = segment size minus the query's self id when that lies inside the
// segment), so it does not wait for the radius to pass the scene diagonal.  SegLane is empty in the other kernels.
template <bool SEG> struct SegLane {};
template <> struct SegLane<true> {
  int seg = -1;  // the lane's segment
};

__device__ __forceinline__ void seg_lane_init(SegLane<true>& sl, const Params& P, uint64_t qpos) { sl.seg = (int)__ldg(&P.seg_of[qpos]); }

// MODE_KNN: min(k, size - [self in the segment]) entries resolve the row (read at emit: nothing more stays live during
// the walk).  A built point is always in its own segment (size - 1); an empty data segment needs 0.
__device__ __forceinline__ int seg_need(const Params& P, int seg, int k, int self) {
  const uint64_t lo = __ldg(&P.seg_off[seg]), size = __ldg(&P.seg_off[seg + 1]) - lo;
  const uint64_t eligible = size - (self >= 0 && (uint64_t)self - lo < size ? 1 : 0);
  return (uint64_t)k < eligible ? k : (int)eligible;
}

__device__ __forceinline__ void seg_cull(const Params& P, int node, int seg, float& d0, float& d1) {
  const int4 r = __ldg(&P.node_seg[node]);
  const float qnan = __int_as_float(0x7fc00000);
  if (seg < r.x || seg > r.y) d0 = qnan;
  if (seg < r.z || seg > r.w) d1 = qnan;
}

// per-lane state of the MODE_RANGE_LIST_* passes (an empty object in the other modes)
template <bool LIST> struct ListLane {};
template <> struct ListLane<true> {
  int64_t spos = -1;    // position of the excluded data point (-1: none)
  uint64_t cursor = 0;  // MODE_RANGE_LIST: next key slot of the lane's row
};

// ---- bounded 4-ary max-heap of u64 keys in shared memory, slot s of lane l at H[s * 32 + l] ----
// Four children per node: k = 64 is three levels deep instead of six, and the four child loads of a level
// are independent, so an insert costs three shared-memory latencies instead of six (the binary heap left
// the k = 64 kernel latency bound: issue slots 42 % busy at 12 resident warps per SM).
__device__ __forceinline__ void heap_push(uint64_t* H, int& cnt, uint64_t key) {
  int i = cnt++;
  while (i > 0) {
    const int par = (i - 1) >> 2;
    const uint64_t pk = H[par * 32];
    if (pk >= key) break;
    H[i * 32] = pk;
    i = par;
  }
  H[i * 32] = key;
}

// place `key` at the root of a heap of `size` entries and sift it down
__device__ __forceinline__ void heap_sift_root(uint64_t* H, int size, uint64_t key) {
  int i = 0;
  for (;;) {
    const int c = 4 * i + 1;
    if (c >= size) break;
    const uint64_t k0 = H[c * 32];
    const uint64_t k1 = (c + 1 < size) ? H[(c + 1) * 32] : 0ull;  // 0 never beats a real child
    const uint64_t k2 = (c + 2 < size) ? H[(c + 2) * 32] : 0ull;
    const uint64_t k3 = (c + 3 < size) ? H[(c + 3) * 32] : 0ull;
    int m = c;
    uint64_t mk = k0;
    if (k1 > mk) { mk = k1; m = c + 1; }
    if (k2 > mk) { mk = k2; m = c + 2; }
    if (k3 > mk) { mk = k3; m = c + 3; }
    if (mk <= key) break;
    H[i * 32] = mk;
    i = m;
  }
  H[i * 32] = key;
}

// ---- padded D-ary max-heap of the cooperative kernel ---------------------------------------------
// Every slot a sift can read past the heap's last entry holds 0 (<= every key), so the D child loads of a
// level need no bounds tests, and the maximum is found by a tournament (independent compares first) instead
// of a chain: 32 instead of 48 SASS instructions per level of the 4-ary heap.  heap_pads(k) zero slots follow
// the k entries; kl_emit zeroes the slots it vacates so the invariant also holds while the heap shrinks.
// Arity 8 (k = 64 two levels deep: two dependent shared-memory round trips per replacement instead of three)
// was measured SLOWER on cfg3 (round 1: 55.5 vs 51.0 ms): seven compare-selects per level cost more issue
// slots than the saved round trip returns.
#ifndef TKNN_HEAP_ARITY
#define TKNN_HEAP_ARITY 4
#endif
constexpr int PAD_D = TKNN_HEAP_ARITY;  // 4 or 8
static_assert(PAD_D == 4 || PAD_D == 8, "padded heap arity");

// zero slots needed behind a heap of k entries: the last internal node's children end at PAD_D * ((k - 2) / PAD_D) + PAD_D
__host__ __device__ inline int heap_pads(int k) { return k >= 2 ? PAD_D * ((k - 2) / PAD_D) + PAD_D - (k - 1) : 1; }

__device__ __forceinline__ void pheap_push(uint64_t* A, int& cnt, uint64_t key) {
  int i = cnt++;
  while (i > 0) {
    const int par = (i - 1) / PAD_D;
    const uint64_t pk = A[par * 32];
    if (pk >= key) break;
    A[i * 32] = pk;
    i = par;
  }
  A[i * 32] = key;
}

// larger of two (key, slot) pairs, the slot selected with the key so that the predicate dies here
#define TKNN_MAX2(ka, ia, kb, ib, ko, io)      \
  const bool b_##ko = (kb) > (ka);               \
  const uint64_t ko = b_##ko ? (kb) : (ka);      \
  const int io = b_##ko ? (ib) : (ia);

__device__ __forceinline__ void pheap_sift_root(uint64_t* A, int size, uint64_t key) {
  int i = 0;
  for (;;) {
    const int c = PAD_D * i + 1;
    if (c >= size) break;
    const uint64_t* p = A + c * 32;
    const uint64_t k0 = p[0], k1 = p[32], k2 = p[64], k3 = p[96];
    TKNN_MAX2(k0, c, k1, c + 1, m01, i01)
    TKNN_MAX2(k2, c + 2, k3, c + 3, m23, i23)
    TKNN_MAX2(m01, i01, m23, i23, m03, i03)
    uint64_t mk = m03;
    int im = i03;
    if (PAD_D == 8) {
      const uint64_t k4 = p[128], k5 = p[160], k6 = p[192], k7 = p[224];
      TKNN_MAX2(k4, c + 4, k5, c + 5, m45, i45)
      TKNN_MAX2(k6, c + 6, k7, c + 7, m67, i67)
      TKNN_MAX2(m45, i45, m67, i67, m47, i47)
      TKNN_MAX2(m03, i03, m47, i47, m07, i07)
      mk = m07;
      im = i07;
    }
    if (mk <= key) break;
    A[i * 32] = mk;
    i = im;
  }
  A[i * 32] = key;
}
#undef TKNN_MAX2

// A warp-COOPERATIVE insert (lane i owns rank i of one query's list, rows padded to 33 keys) for iterations with few
// lanes holding a candidate was measured and rejected in round 2 (profiles/r2_ab_coop_cfg2.jsonl, cfg2 round 1: off 7.48 ms,
// <= 2 lanes 7.98, <= 3 lanes 8.36, <= 5 lanes 9.25, <= 8 lanes 10.57 ms): a chain of dependent warp-wide steps per candidate
// with no overlap between candidates, while the private path lets every lane walk its own list at once.  The code was
// removed when the leaf section was unified (git history: 5fc7c56).

// ---- bounded ASCENDING list of u64 keys in shared memory (slot s of lane l at L[s * S + l]) ----
// Candidates arrive roughly nearest-first, so a new key usually lands near the tail: the backward
// shift is short, and the list needs no heap-sort at emit time.  Precondition: cnt < k or key < L[k-1].
// L points at a SENTINEL slot holding 0 (<= every key); entries live in slots 1..k.  The sentinel ends
// the backward walk without a bounds test, so the loop unrolls to 5 instructions per step.
// S = slot stride in keys: 32 (one 256-byte row per slot; the 32 lanes of a warp touch 32 consecutive keys: conflict-free).
constexpr int KLS = 32;

// Returns the key left in the slot that was filled, i.e. the list's new LAST entry — the new worst once the list is
// full — so the caller keeps the bound and the worst index in registers instead of re-reading them.
template <int S = 32>
__device__ __forceinline__ uint64_t list_insert(uint64_t* L, int& cnt, int k, uint64_t key) {
  uint64_t* p = L + (cnt < k ? cnt + 1 : k) * S;  // the slot being filled
  if (cnt < k) ++cnt;
  uint64_t tail;
  {
    // four independent loads in flight: one shared-memory latency per four steps.  Slots below the
    // sentinel (at most three) are never used: the walk stops at the sentinel; they lie inside this
    // warp's own staging area, so the reads are in bounds.
    const uint64_t a = *(p - S), b = *(p - 2 * S), c = *(p - 3 * S), d = *(p - 4 * S);
    if (a <= key) { *p = key; return key; }
    *p = a;
    tail = a;
    if (b <= key) { *(p - S) = key; return tail; }
    *(p - S) = b;
    if (c <= key) { *(p - 2 * S) = key; return tail; }
    *(p - 2 * S) = c;
    if (d <= key) { *(p - 3 * S) = key; return tail; }
    *(p - 3 * S) = d;
    p -= 4 * S;
  }
  for (;;) {
    const uint64_t a = *(p - S), b = *(p - 2 * S), c = *(p - 3 * S), d = *(p - 4 * S);
    if (a <= key) { *p = key; return tail; }
    *p = a;
    if (b <= key) { *(p - S) = key; return tail; }
    *(p - S) = b;
    if (c <= key) { *(p - 2 * S) = key; return tail; }
    *(p - 2 * S) = c;
    if (d <= key) { *(p - 3 * S) = key; return tail; }
    *(p - 3 * S) = d;
    p -= 4 * S;
  }
}

// k-list policy: ascending list for small k (short shifts, no sort at emit), 4-ary max-heap above
// (O(log4 k) per insert; heap-sorted at emit).  Warp-uniform choice.
constexpr int LIST_MAX_K = 24;

// H = sentinel slot of the lane's region; the heap (large k) uses slots 1..k as its 0-based array (stride 32 always)
template <int S = 32>
__device__ __forceinline__ uint64_t kl_worst(const uint64_t* H, int k, bool heap) { return heap ? H[32] : H[k * S]; }

// PADDED: the padded D-ary heap of the cooperative kernel (pheap_*)
template <bool PADDED = false, int S = 32>
__device__ __forceinline__ void kl_insert(uint64_t* H, int& cnt, int k, uint64_t key, bool heap) {
  if (heap) {
    if (PADDED) {
      if (cnt < k) pheap_push(H + 32, cnt, key);
      else pheap_sift_root(H + 32, k, key);
    } else {
      if (cnt < k) heap_push(H + 32, cnt, key);
      else heap_sift_root(H + 32, k, key);
    }
  } else {
    list_insert<S>(H, cnt, k, key);
  }
}

// writes the k-list ascending to (io, dd); destroys the heap (PADDED: leaves it all zero)
template <bool PADDED = false, int S = 32>
__device__ __forceinline__ void kl_emit(uint64_t* H, int cnt, int k, bool heap, bool squared, int32_t* io, float* dd) {
  for (int i = k - 1; i >= cnt; --i) { io[i] = -1; dd[i] = FLT_MAX; }
  if (heap) {
    uint64_t* A = H + 32;
    if (PADDED && cnt < k) {  // a short heap (capped final round): slots past it may hold an earlier group's keys
      const int last_slot = k - 1 + heap_pads(k);
      for (int j = cnt; j < cnt + PAD_D - 1 && j <= last_slot; ++j) A[j * 32] = 0;
    }
    for (int i = cnt - 1; i >= 0; --i) {
      const uint64_t top = A[0];
      io[i] = key_idx(top);
      dd[i] = squared ? key_d2(top) : __fsqrt_rn(key_d2(top));
      if (PADDED) {
        const uint64_t last = A[i * 32];
        A[i * 32] = 0;  // the vacated slot joins the zero padding
        if (i > 0) pheap_sift_root(A, i, last);
      } else if (i > 0) {
        heap_sift_root(A, i, A[i * 32]);
      }
    }
  } else {
    for (int i = 0; i < cnt; ++i) {
      const uint64_t e = H[(i + 1) * S];
      io[i] = key_idx(e);
      dd[i] = squared ? key_d2(e) : __fsqrt_rn(key_d2(e));
    }
  }
}

// k-list slots per lane in the cooperative kernel: sentinel + k entries, + heap_pads(k) zero slots behind a heap
__host__ __device__ inline int klist_slots(int k) { return k > LIST_MAX_K ? k + 1 + heap_pads(k) : k + 1; }

// bytes of the 32 k-lists of a warp: rows of KLS keys for the ascending lists, of 32 keys for the heaps; a multiple of 16
__host__ __device__ inline size_t klist_bytes(int k) {
  const size_t b = (size_t)klist_slots(k) * (k > LIST_MAX_K ? 32 : KLS) * sizeof(uint64_t);
  return (b + 15) / 16 * 16;
}

// Sibling leaves together (TKNN_PAIR_LEAVES): when BOTH children of a node are leaves and the group wants both, the two
// leaves are staged side by side, filtered into two masks and inserted in ONE divergent loop.  The insert loop runs
// max-over-lanes(survivors) iterations of ~90 warp instructions at ~5 active lanes — 41 % of the dense kernel's
// instructions — and the lanes that find survivors in two sibling leaves are mostly different lanes, so one loop over both
// is shorter than two loops; the price is that the second leaf is filtered against the bound as it was before the first
// one tightened it (its stale survivors fail the re-test at insert time).  1: ascending-list kernel only (k <= 24);
// 2: heap kernel too (+768 B of staging per warp: one resident warp fewer at k = 64).
#ifndef TKNN_PAIR_LEAVES
#define TKNN_PAIR_LEAVES 1
#endif
// Measured (profiles/r2_ab_pair.jsonl, r2_ab_pairfilter.jsonl; round 1 of cfg2 / cfg4): off 6.70 / 67.6 ms, on 6.50 / 65.2 ms,
// on with the pair's filter in chunks of 8 (compile-time bit positions) 6.49 / 65.1 ms (default); chunks of 4 only in the
// single-leaf filter as well: 6.70 / 67.2 ms — the unrolled chunks of 8 are worth 3 %.  Heap kernel (cfg3): 46.0 ms off, 49.2 on.
#ifndef TKNN_PAIR_FILTER8
#define TKNN_PAIR_FILTER8 1
#endif
__host__ __device__ constexpr bool pair_leaves(bool heap) { return TKNN_PAIR_LEAVES >= 2 || (TKNN_PAIR_LEAVES == 1 && !heap); }
// points staged per warp = axis stride of the SoA staging area
__host__ __device__ constexpr int stage_pts(bool heap) { return pair_leaves(heap) ? 2 * MAX_LEAF : MAX_LEAF; }

__host__ __device__ inline size_t smem_per_warp(int k) {
  const int ns = stage_pts(k > LIST_MAX_K);
  return klist_bytes(k) + (size_t)ns * sizeof(float4) + (ns > MAX_LEAF ? 3 * ns * sizeof(float) : MAX_LEAF * sizeof(float4)) +
         STACK_DEPTH * sizeof(int);
}

// ---- index-aware pruning of exact ties ----------------------------------------------------------
// A child whose box distance EQUALS a lane's bound can only matter to that lane through a point at
// exactly the k-th distance with a LOWER index than the current k-th neighbour.  So when no lane is
// strictly inside (d < bound), the child is entered only if its smallest original index could win such
// a tie for some lane.  Without this, a cluster of D coincident points (bound = 0, every cluster box at
// distance 0) costs D/32 leaf visits per group — 272 ms for 400 K duplicates in a 2 M cloud; with it the
// walk reaches the lowest-index leaf of the cluster first (child 0 first among equals) and prunes the rest
// Queries NEAR such a cluster tie at a non-zero distance (their k nearest are k of the duplicates), so the
// test applies to every exact tie, not only to bound == 0.  It lives in its own kernel variant (VARIANT 2),
// selected only when the build saw a leaf of coincident points: compiled into the default variant it cost
// 9 % on tie-free data (8.45 -> 9.2 ms on cfg2).
template <int MODE, int S>
__device__ __forceinline__ bool child_wanted(float dc, float bound, int cnt, int k, const uint64_t* H, bool heap,
                                             int child_min_idx) {
  if (!__any_sync(FULL_MASK, dc <= bound)) return false;
  if (MODE != MODE_KNN) return true;
  if (__any_sync(FULL_MASK, dc < bound)) return true;
  const bool tie_can_win = (dc == bound) && (cnt < k || child_min_idx < key_idx(kl_worst<S>(H, k, heap)));
  return __any_sync(FULL_MASK, tie_can_win);
}

// ---- conservative pre-filter -------------------------------------------------------------------
// The exact test costs 6 FP instructions per (query, point).  With coordinates taken relative to a
// group-local origin c (lane 0's query), qr = q - c and pr = p - c are small, and
//     t = fma(-2qr.x, pr.x, fma(-2qr.y, pr.y, fma(-2qr.z, pr.z, |pr|^2)))  ~  |q - p|^2 - |qr|^2
// costs 3.  A point passes the pre-filter iff t <= tau with tau = bound - |qr|^2 + margin; survivors
// are re-tested with the exact fmaf chain in the insert loop, so false positives cost time, never
// correctness.  No false negatives: writing u = 2^-23 and R = |qr| + |pr|, the roundings of qr, pr
// (<= u R per vector), of |pr|^2 and |qr|^2 (3 ops each) and of the three fmas (each <= u R^2) put the
// computed t + |qr|^2 within 19 u R^2 of the exact chain's d2 (whose own relative error is <= 6u), and
// any point with d2 <= bound has |pr| <= |qr| + 1.01 sqrt(bound), i.e. R^2 <= 8|qr|^2 + 2.1 bound.  So
// margin = 19u (8|qr|^2 + 2.1 bound) ~ 1.8e-5 |qr|^2 + 4.8e-6 bound suffices; the kernel uses
// 1e-4 |qr|^2 + 2e-5 bound (5x slack).  Non-finite or huge operands fall back to tau = +inf (all pass).
// The counting build (TKNN_OPT_COUNTERS) also evaluates the exact test for every pair and counts
// violations (tknn_stats.filter_violations, asserted zero by the tests).
// Measured on cfg2: 8.45 ms vs 8.54 ms for the exact filter (-1 %): the 3 FFMA per pair saturate the FMA
// pipe (one warp instruction per two cycles) where the exact form splits 3 FADD (ALU pipe) / 3 FMUL+FFMA.
// It is therefore OFF by default (TKNN_OPT_APPROX_FILTER) — kept as a measured, audited option.
__device__ __forceinline__ float prefilter_tau(float bound, float qq) {
  const float tau = __fadd_rn(__fsub_rn(bound, qq), __fmaf_rn(1e-4f, qq, __fmul_rn(2e-5f, bound)));
  return (qq < 1e30f && bound < 1e30f) ? tau : INFINITY;
}

// ---- packed exact filter (sm_100a FADD2 / FMUL2 / FFMA2) -----------------------------------------
// The traversal is instruction-issue bound (DESIGN.md 3.2), and Blackwell's packed fp32x2 instructions
// evaluate the distance chain of TWO points per issue slot with the same IEEE round-to-nearest result
// per component as the scalar __fsub_rn/__fmul_rn/__fmaf_rn chain of dist2().  The leaf is therefore
// also staged as three coordinate arrays (sx, sy, sz), so one LDS.128 per axis yields two aligned
// operand pairs: 4 points cost 3 LDS.128 + 12 packed FP + 4 FSETP/SEL instead of 4 LDS.128 + 24 FP + 8.
// Lanes past the leaf's last point stage NaN in sx: a NaN distance never satisfies d <= bound, so the
// padded tail of the last chunk of 4 drops out without a bounds test.
__device__ __forceinline__ float2 dist2_x2(float2 qx, float2 qy, float2 qz, float2 px, float2 py, float2 pz) {
  const float2 dx = __fadd2_rn(qx, make_float2(-px.x, -px.y));
  const float2 dy = __fadd2_rn(qy, make_float2(-py.x, -py.y));
  const float2 dz = __fadd2_rn(qz, make_float2(-pz.x, -pz.y));
  return __ffma2_rn(dz, dz, __ffma2_rn(dy, dy, __fmul2_rn(dx, dx)));
}

// bit i of the result: point j0 + i of the staged leaf is within `bound` of the lane's query
template <int NS = MAX_LEAF>  // NS = axis stride of the staging area (stage_pts)
__device__ __forceinline__ uint32_t filter4(const float* sx, int j0, float2 qx, float2 qy, float2 qz, float bound) {
  const float4 X = *reinterpret_cast<const float4*>(sx + j0);
  const float4 Y = *reinterpret_cast<const float4*>(sx + NS + j0);
  const float4 Z = *reinterpret_cast<const float4*>(sx + 2 * NS + j0);
  const float2 a = dist2_x2(qx, qy, qz, make_float2(X.x, X.y), make_float2(Y.x, Y.y), make_float2(Z.x, Z.y));
  const float2 b = dist2_x2(qx, qy, qz, make_float2(X.z, X.w), make_float2(Y.z, Y.w), make_float2(Z.z, Z.w));
  uint32_t m = 0;
  if (a.x <= bound) m |= 1u;
  if (a.y <= bound) m |= 2u;
  if (b.x <= bound) m |= 4u;
  if (b.y <= bound) m |= 8u;
  return m;
}

// Insert loop of the dense kernel: every lane walks its own survivors and the warp reconverges once behind the loop.
// Round 1's warp-voted loop (one candidate per lane per iteration) cost ~10 of the ~100 warp instructions of an iteration in
// the vote, its divergence check and the reconvergence points (profiles/r2_ab_insert.jsonl: cfg2 7.53 -> 7.35 ms, cfg3
// 48.95 -> 45.79 ms); it was removed with the unification of the leaf section.
// Worst entry of a full ascending list: 2 (default) = list_insert hands back the new tail, so the bound is updated from
// registers, and the stored worst key is re-read only when a candidate TIES the bound (its index then decides);
// 0 = re-read the tail slot before and after every insert (round 1); 1 = also keep the worst index in a register
// (55 registers instead of 47: 36 instead of 40 resident warps).  cfg2 (profiles/r2_ab_insert.jsonl, r2_ab_wreg2.jsonl):
// 0: 7.33 ms, 1: 7.65 ms, 2: 7.30 ms.
// 1: the two internal-child votes as one REDUX.OR and the near-first majority as one REDUX.SUM.  Measured neutral (cfg2 round 1
// 6.630 vs 6.632 ms, cfg3 44.43 vs 44.44 ms, profiles/r2_ab_team.jsonl): off.
#ifndef TKNN_REDUX_VOTES
#define TKNN_REDUX_VOTES 0
#endif
#ifndef TKNN_WORST_REG
#define TKNN_WORST_REG 2
#endif

// The insert rule of the ascending list with TKNN_WORST_REG 2, for a candidate that passed `d <= bound` and is not self:
// the key beats the worst entry unless the list is full and it TIES the bound's distance with a higher index.  The bound
// becomes the new tail's distance once the list is full.  (The LBVH kernel and the grid kernel, grid.cuh.)
template <int S, bool COUNT>
__device__ __forceinline__ void list_take(uint64_t* H, int& cnt, int k, float& bound, float d, int pid, unsigned long long& c_ins) {
  if (cnt < k || d < bound || pid < key_idx(kl_worst<S>(H, k, false))) {
    const uint64_t tail = list_insert<S>(H, cnt, k, make_key(d, pid));
    if (cnt == k) bound = key_d2(tail);
    if (COUNT) c_ins += 1;
  }
}
// MODE_DBSCAN_LINK: 1 = a core query unites only the core points of its ball at LOWER positions (every edge joins two core
// queries, so each is still united once); 0 = every core point of the ball (each edge twice).
#ifndef TKNN_DBSCAN_HALF_EDGES
#define TKNN_DBSCAN_HALF_EDGES 1
#endif

// VARIANT: 0 = exact filter, 1 = conservative pre-filter (audited option), 2 = exact filter + index-aware
// tie pruning (chosen by the host when the build found leaves of coincident points).
// HEAP: k > LIST_MAX_K (compile-time, so the small-k kernel does not carry the heap code).
// Launch bounds: the list kernels are capped at 48 registers (5 blocks of 8 warps = 40 resident warps; uncapped, the
// unified leaf section compiles to 64 and loses a fifth of them); the heap kernels (12 resident warps: shared memory)
// and the counting variants (diagnostics) take what they need.
// SEG: segmented build (MODE_KNN, MODE_RANGE_COUNT, MODE_RANGE_LIST_*): the per-lane segment cull above.
template <int MODE, bool COUNT, int VARIANT, bool HEAP, bool SEG = false>
static __global__ void __launch_bounds__(256, (HEAP || COUNT) ? 1 : 5) traverse_kernel(const Params P) {
  constexpr bool APPROX = VARIANT == 1;
  constexpr bool TIES = VARIANT == 2 && MODE == MODE_KNN;
  extern __shared__ __align__(16) unsigned char smem[];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int k = P.k;
  constexpr bool heap = HEAP;
  unsigned char* wbase = smem + (size_t)warp * smem_per_warp(MODE == MODE_KNN ? k : 0);
  constexpr int NS = stage_pts(HEAP);  // staged points = SoA axis stride (64 with sibling-leaf pairs)
  constexpr bool PAIR = pair_leaves(HEAP) && MODE == MODE_KNN && VARIANT != 1;
  float4* stage = reinterpret_cast<float4*>(wbase);
  int* stack = reinterpret_cast<int*>(wbase + NS * sizeof(float4));
  constexpr int S = HEAP ? 32 : KLS;  // slot stride of the k-lists (keys)
  uint64_t* H = reinterpret_cast<uint64_t*>(wbase + NS * sizeof(float4) + STACK_DEPTH * sizeof(int)) + lane;
  // second staging array (relative coordinates + squared norm) for the pre-filter, behind the k-list
  float4* stage2 = reinterpret_cast<float4*>(wbase + NS * sizeof(float4) + STACK_DEPTH * sizeof(int) +
                                             klist_bytes(MODE == MODE_KNN ? k : 0));
  float* soa = reinterpret_cast<float*>(stage2);  // exact filter: the leaf's x[32] | y[32] | z[32] (same region)

  unsigned long long c_nodes = 0, c_tests = 0, c_ins = 0, c_wnodes = 0, c_wleaves = 0, c_wpts = 0, c_viol = 0;
  if (HEAP && MODE == MODE_KNN) {  // zero padding behind the heap (never written again)
    for (int j = 0; j < heap_pads(k); ++j) H[(k + 1 + j) * 32] = 0;
  }
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
    int cnt = 0;                       // MODE_DBSCAN_BORDER: 1 + the lowest cluster id of a core point in the ball so far, 0: none
    int widx = 0x7fffffff;             // index of the list's worst entry once it is full (TKNN_WORST_REG)
    if (MODE == MODE_KNN) H[0] = 0;    // sentinel of this lane's k-list
    ListLane<MODE == MODE_RANGE_LIST_COUNT || MODE == MODE_RANGE_LIST> rl;  // empty in every other mode
    if constexpr (MODE == MODE_RANGE_LIST_COUNT || MODE == MODE_RANGE_LIST) {
      if (valid) rl.spos = P.self_pos ? (int64_t)P.self_pos[qpos] : (P.self_is_row ? (int64_t)qpos : -1);
      if (MODE == MODE_RANGE_LIST && valid) rl.cursor = P.list_off[qpos];
    }
    SegLane<SEG> sl;
    if constexpr (SEG) {
      if (valid) seg_lane_init(sl, P, qpos);
    }
    // group-local origin and this lane's pre-filter constants
    float ax, ay, az, qq;
    {
      const float cx = __shfl_sync(FULL_MASK, q.x, 0), cy = __shfl_sync(FULL_MASK, q.y, 0), cz = __shfl_sync(FULL_MASK, q.z, 0);
      const float qrx = __fsub_rn(q.x, cx), qry = __fsub_rn(q.y, cy), qrz = __fsub_rn(q.z, cz);
      ax = -2.0f * qrx; ay = -2.0f * qry; az = -2.0f * qrz;
      qq = __fmaf_rn(qrz, qrz, __fmaf_rn(qry, qry, __fmul_rn(qrx, qrx)));
    }

    // one candidate of the staged leaf (or leaf pair): exact distance, self test, bound test, insert; the bound tightens
    auto try_insert = [&](int j) {
      const float4 p = stage[j];
      const float d = dist2(q.x, q.y, q.z, p.x, p.y, p.z);
      const int pid = __float_as_int(p.w);
      if (pid != self && d <= bound) {
        const uint64_t key = make_key(d, pid);
        if (!HEAP && TKNN_WORST_REG == 2) {
          list_take<S, COUNT>(H, cnt, k, bound, d, pid, c_ins);
        } else if (!HEAP && TKNN_WORST_REG) {
          // (d, pid) < (bound, widx): the worst entry's key lives in registers (bound = its d2)
          if (cnt < k || d < bound || pid < widx) {
            const uint64_t tail = list_insert<S>(H, cnt, k, key);
            if (cnt == k) { bound = key_d2(tail); widx = key_idx(tail); }
            if (COUNT) c_ins += 1;
          }
        } else if (cnt < k || key < kl_worst<S>(H, k, heap)) {
          kl_insert<true, S>(H, cnt, k, key, heap);
          if (cnt == k) bound = key_d2(kl_worst<S>(H, k, heap));
          if (COUNT) c_ins += 1;
        }
      }
    };

    int sp = 0;
    int node = 0;
    for (;;) {
      const float4* np = reinterpret_cast<const float4*>(P.nodes + node);
      const float4 na = __ldg(np), nb = __ldg(np + 1), nc = __ldg(np + 2), nd = __ldg(np + 3);
      const float2 d01 = box_dist2_x2(q.x, q.y, q.z, na, nb, nc);
      float d0 = d01.x, d1 = d01.y;
      if constexpr (SEG) seg_cull(P, node, sl.seg, d0, d1);
      if (COUNT) { c_nodes += valid ? 1 : 0; c_wnodes += 1; }
      const int ref0 = __float_as_int(nd.x), cnt0 = __float_as_int(nd.z);
      const int ref1 = __float_as_int(nd.y), cnt1 = __float_as_int(nd.w);

      // ---- leaf children first (they tighten the bounds before anything is pushed) ----
      if ((cnt0 | cnt1) != 0) {
        // near-first among two leaves, by majority of lanes
        bool swap = false;
        if (cnt0 > 0 && cnt1 > 0)
          swap = __popc(__ballot_sync(FULL_MASK, d1 < d0)) > __popc(__ballot_sync(FULL_MASK, d0 < d1));
        // does the group want leaf child 0 / 1 (second)?  Evaluated against the bounds as they are NOW.
        auto leaf_wanted = [&](bool second) -> bool {
          if ((second ? cnt1 : cnt0) <= 0) return false;
          const float dc = second ? d1 : d0;
          if (!__any_sync(FULL_MASK, dc <= bound)) return false;
          if (TIES && !__any_sync(FULL_MASK, dc < bound)) {  // only exact ties: can any of them win?
            const int2 mi = __ldg(&P.node_min_idx[node]);
            return child_wanted<MODE, S>(dc, bound, cnt, k, H, heap, second ? mi.y : mi.x);
          }
          return true;
        };
        // sibling leaves both wanted: one staging, two masks, ONE insert loop (TKNN_PAIR_LEAVES)
        const bool pair = PAIR && cnt0 > 0 && cnt1 > 0 && leaf_wanted(false) && leaf_wanted(true);
#pragma unroll 1
        for (int c = 0; c < 2; ++c) {
          uint32_t mask_a = 0, mask_b = 0;  // survivors among staged points 0..31 / 32..63
          if (pair) {
            if (c == 1) break;
            const float qnan = __int_as_float(0x7fc00000);
            float4 pa = make_float4(qnan, 0.f, 0.f, 0.f), pb = pa;  // NaN x: a padded slot never passes the filter
            if (lane < cnt0) pa = __ldg(&P.pts[(uint64_t)(uint32_t)ref0 + lane]);
            if (lane < cnt1) pb = __ldg(&P.pts[(uint64_t)(uint32_t)ref1 + lane]);
            stage[lane] = pa;
            stage[MAX_LEAF + lane] = pb;
            soa[lane] = pa.x; soa[NS + lane] = pa.y; soa[2 * NS + lane] = pa.z;
            soa[MAX_LEAF + lane] = pb.x; soa[NS + MAX_LEAF + lane] = pb.y; soa[2 * NS + MAX_LEAF + lane] = pb.z;
            __syncwarp();
            if (COUNT) { c_tests += valid ? cnt0 + cnt1 : 0; c_wleaves += 2; c_wpts += cnt0 + cnt1; }
            const float2 qx2 = make_float2(q.x, q.x), qy2 = make_float2(q.y, q.y), qz2 = make_float2(q.z, q.z);
#if TKNN_PAIR_FILTER8
            {
              int j0 = 0;
              for (; j0 + 8 <= cnt0; j0 += 8)
                mask_a |= (filter4<NS>(soa, j0, qx2, qy2, qz2, bound) | (filter4<NS>(soa, j0 + 4, qx2, qy2, qz2, bound) << 4)) << j0;
#pragma unroll 1
              for (; j0 < cnt0; j0 += 4) mask_a |= filter4<NS>(soa, j0, qx2, qy2, qz2, bound) << j0;
              j0 = 0;
              for (; j0 + 8 <= cnt1; j0 += 8)
                mask_b |= (filter4<NS>(soa + MAX_LEAF, j0, qx2, qy2, qz2, bound) |
                           (filter4<NS>(soa + MAX_LEAF, j0 + 4, qx2, qy2, qz2, bound) << 4)) << j0;
#pragma unroll 1
              for (; j0 < cnt1; j0 += 4) mask_b |= filter4<NS>(soa + MAX_LEAF, j0, qx2, qy2, qz2, bound) << j0;
            }
#else
#pragma unroll 1
            for (int j0 = 0; j0 < cnt0; j0 += 4) mask_a |= filter4<NS>(soa, j0, qx2, qy2, qz2, bound) << j0;
#pragma unroll 1
            for (int j0 = 0; j0 < cnt1; j0 += 4) mask_b |= filter4<NS>(soa + MAX_LEAF, j0, qx2, qy2, qz2, bound) << j0;
#endif
            if constexpr (SEG) {  // a leaf of another segment: nothing in it is this lane's
              if (isnan(d0)) mask_a = 0;
              if (isnan(d1)) mask_b = 0;
            }
          } else {
            const bool second = (c == 1) != swap;  // false: child 0, true: child 1
            if (!leaf_wanted(second)) continue;
            const int lcount = second ? cnt1 : cnt0;
            const int start = second ? ref1 : ref0;
            const bool own = !SEG || !isnan(second ? d1 : d0);  // SEG: the leaf holds this lane's segment
            float cx = 0.f, cy = 0.f, cz = 0.f;
            if (APPROX && MODE == MODE_KNN) {  // the group origin = lane 0's query (re-broadcast: saves 3 registers)
              cx = __shfl_sync(FULL_MASK, q.x, 0); cy = __shfl_sync(FULL_MASK, q.y, 0); cz = __shfl_sync(FULL_MASK, q.z, 0);
            }
            if (lane < lcount) {
              const float4 pl = __ldg(&P.pts[(uint64_t)(uint32_t)start + lane]);
              stage[lane] = pl;
              if (APPROX && MODE == MODE_KNN) {
                const float rx = __fsub_rn(pl.x, cx), ry = __fsub_rn(pl.y, cy), rz = __fsub_rn(pl.z, cz);
                stage2[lane] = make_float4(rx, ry, rz, __fmaf_rn(rz, rz, __fmaf_rn(ry, ry, __fmul_rn(rx, rx))));
              } else {
                soa[lane] = pl.x; soa[NS + lane] = pl.y; soa[2 * NS + lane] = pl.z;
              }
            } else if (!(APPROX && MODE == MODE_KNN)) {
              soa[lane] = __int_as_float(0x7fc00000);  // NaN: the padded tail of the last chunk never passes
            }
            __syncwarp();
            if (COUNT) { c_tests += valid ? lcount : 0; c_wleaves += 1; c_wpts += lcount; }
            if (MODE == MODE_RANGE_COUNT || MODE == MODE_DBSCAN_CORE) {
              // every point within the radius, the query's own point included: it lies at distance 0 in the one
              // leaf that holds it and is taken off again at emit time
              const float2 qx2 = make_float2(q.x, q.x), qy2 = make_float2(q.y, q.y), qz2 = make_float2(q.z, q.z);
              if (own) {
#pragma unroll 1
                for (int j0 = 0; j0 < lcount; j0 += 4) cnt += __popc(filter4<NS>(soa, j0, qx2, qy2, qz2, bound));
              }
              // decided: a core point wants nothing more, and the group's walk ends once every lane is decided
              if (MODE == MODE_DBSCAN_CORE && cnt >= k) bound = -1.0f;
            } else {
              // filter: full chunks of 8 with compile-time bit positions, then the remainder in chunks of 4
              int j0 = 0;
              if (APPROX) {
                const float tau = valid ? prefilter_tau(bound, qq) : -INFINITY;
                for (; j0 + 8 <= lcount; j0 += 8) {
                  uint32_t m8 = 0;
#pragma unroll
                  for (int jj = 0; jj < 8; ++jj) {
                    const float4 p = stage2[j0 + jj];
                    const float t = __fmaf_rn(ax, p.x, __fmaf_rn(ay, p.y, __fmaf_rn(az, p.z, p.w)));
                    if (t <= tau) m8 |= (1u << jj);
                  }
                  mask_a |= m8 << j0;
                }
                for (; j0 < lcount; ++j0) {
                  const float4 p = stage2[j0];
                  const float t = __fmaf_rn(ax, p.x, __fmaf_rn(ay, p.y, __fmaf_rn(az, p.z, p.w)));
                  if (t <= tau) mask_a |= (1u << j0);
                }
                if (COUNT) {  // audit: an exactly-passing pair the pre-filter rejected would be a wrong result
                  for (int j = 0; j < lcount; ++j) {
                    const float4 p = stage[j];
                    const float d = dist2(q.x, q.y, q.z, p.x, p.y, p.z);
                    if (valid && d <= bound && !((mask_a >> j) & 1u)) c_viol += 1;
                  }
                }
              } else {
                const float2 qx2 = make_float2(q.x, q.x), qy2 = make_float2(q.y, q.y), qz2 = make_float2(q.z, q.z);
                for (; j0 + 8 <= lcount; j0 += 8) {
                  const uint32_t m8 = filter4<NS>(soa, j0, qx2, qy2, qz2, bound) | (filter4<NS>(soa, j0 + 4, qx2, qy2, qz2, bound) << 4);
                  mask_a |= m8 << j0;
                }
#pragma unroll 1
                for (; j0 < lcount; j0 += 4)  // tail in chunks of 4, NaN-padded past the last point
                  mask_a |= filter4<NS>(soa, j0, qx2, qy2, qz2, bound) << j0;
              }
              if (!own) mask_a = 0;
            }
            if constexpr (MODE == MODE_RANGE_LIST_COUNT || MODE == MODE_RANGE_LIST) {
              // the excluded point is one slot of this leaf at most
              const int64_t rel = rl.spos - (int64_t)(uint32_t)start;
              uint32_t m = mask_a & ((rel >= 0 && rel < 32) ? ~(1u << rel) : FULL_MASK);
              if (MODE == MODE_RANGE_LIST_COUNT) {
                cnt += __popc(m);
              } else {
                while (m) {  // the distance of the filter, recomputed with the chain of try_insert (bit-identical)
                  const int j = __ffs(m) - 1;
                  m &= m - 1u;
                  const float4 p = stage[j];
                  P.list_keys[rl.cursor++] = make_key(dist2(q.x, q.y, q.z, p.x, p.y, p.z), __float_as_int(p.w));
                  if (COUNT) c_ins += 1;
                }
              }
            }
            if (MODE == MODE_DBSCAN_LINK || MODE == MODE_DBSCAN_BORDER) {
              // the survivors that are core points: the leaf's core bits come with one bitset load (<= 32 consecutive positions)
              uint32_t m = mask_a & dbscan::bits_at(P.core_words, P.n_core_words, (uint32_t)start);
              if (MODE == MODE_DBSCAN_LINK) {
#if TKNN_DBSCAN_HALF_EDGES
                // both ends of an edge are core queries: only the end at the higher position unites it
                const int64_t below = (int64_t)qpos - (int64_t)(uint32_t)start;  // leaf slots at positions < qpos
                m &= below >= 32 ? FULL_MASK : (below <= 0 ? 0u : (1u << below) - 1u);
#endif
                while (m) {
                  const int j = __ffs(m) - 1;
                  m &= m - 1u;
                  const int hooked = dbscan::uf_unite(P.uf_parent, (int)qpos, start + j);
                  if (COUNT) c_ins += hooked;
                }
              } else {
                while (m) {
                  const int j = __ffs(m) - 1;
                  m &= m - 1u;
                  const int id1 = __ldg(&P.pos_label[(uint32_t)start + j]) + 1;
                  cnt = (cnt == 0 || id1 < cnt) ? id1 : cnt;
                  if (COUNT) c_ins += 1;
                }
              }
            }
          }
          if (MODE == MODE_KNN) {
            // insert: only lanes with survivors do work; the bound tightens as they go.  Every lane walks its own survivors
            // (a pair: those of its nearer leaf first) and the warp reconverges once, behind the loop.
            int off_a = 0;
            if (PAIR && d1 < d0) { const uint32_t t = mask_a; mask_a = mask_b; mask_b = t; off_a = MAX_LEAF; }
            while (mask_a | mask_b) {
              int j;
              if (!PAIR || mask_a) { j = off_a + __ffs(mask_a) - 1; mask_a &= mask_a - 1u; }
              else { j = (MAX_LEAF - off_a) + __ffs(mask_b) - 1; mask_b &= mask_b - 1u; }
              try_insert(j);
            }
          }
          __syncwarp();
        }
      }

      // ---- internal children, voted against the (tightened) bounds ----
#if TKNN_REDUX_VOTES
      // one warp reduction for both children (REDUX.OR) instead of two votes, one (REDUX.SUM) for the near-first majority
      const unsigned want = __reduce_or_sync(FULL_MASK, (d0 <= bound ? 1u : 0u) | (d1 <= bound ? 2u : 0u));
      bool w0 = (cnt0 == 0) && (want & 1u);
      bool w1 = (cnt1 == 0) && (want & 2u);
#else
      bool w0 = (cnt0 == 0) && __any_sync(FULL_MASK, d0 <= bound);
      bool w1 = (cnt1 == 0) && __any_sync(FULL_MASK, d1 <= bound);
#endif
      if (TIES && (w0 || w1)) {
        const int2 mi = __ldg(&P.node_min_idx[node]);
        if (w0) w0 = child_wanted<MODE, S>(d0, bound, cnt, k, H, heap, mi.x);
        if (w1) w1 = child_wanted<MODE, S>(d1, bound, cnt, k, H, heap, mi.y);
      }
      if (w0 && w1) {
#if TKNN_REDUX_VOTES
        const bool far0 = __reduce_add_sync(FULL_MASK, (d1 < d0 ? 1 : 0) - (d0 < d1 ? 1 : 0)) > 0;
#else
        const bool far0 = __popc(__ballot_sync(FULL_MASK, d1 < d0)) > __popc(__ballot_sync(FULL_MASK, d0 < d1));
#endif
        const int nearc = far0 ? ref1 : ref0, farc = far0 ? ref0 : ref1;
        if (sp < STACK_DEPTH) {
          if (lane == 0) stack[sp] = farc;
          ++sp;
        } else if (lane == 0) {
          atomicOr(P.error, 1u);
        }
        node = nearc;
      } else if (w0) {
        node = ref0;
      } else if (w1) {
        node = ref1;
      } else {
        if (sp == 0) break;
        --sp;
        __syncwarp();
        node = stack[sp];
      }
    }

    // ---- emit ----
    if (MODE == MODE_RANGE_COUNT) {
      if (valid) P.count_out[row_id] = (uint32_t)(cnt - (self >= 0 ? 1 : 0));
    } else if (MODE == MODE_DBSCAN_CORE) {
      const unsigned core = __ballot_sync(FULL_MASK, valid && cnt >= k);
      if (lane == 0) P.unresolved[group] = core;  // groups are positions 32 g .. 32 g + 31 (no queue)
    } else if (MODE == MODE_RANGE_LIST_COUNT) {
      if (valid) {
        P.count_out[qpos] = (uint32_t)cnt;
        P.count_row[row_id] = (uint32_t)cnt;
      }
    } else if (MODE == MODE_RANGE_LIST) {
      // nothing to emit: the keys are written
    } else if (MODE == MODE_DBSCAN_LINK) {
      // nothing to emit: the unions are the result
    } else if (MODE == MODE_DBSCAN_BORDER) {
      if (valid) {
        P.label_out[row_id] = cnt - 1;  // -1: noise
        if (P.core_out) P.core_out[row_id] = 0;
      }
    } else {
      int need = k;
      if constexpr (SEG) {
        if (valid && cnt < k) need = seg_need(P, sl.seg, k, self);
      }
      const bool resolved = valid && cnt == need;
      const bool emit = valid && (resolved || P.final_round);
      const unsigned un = __ballot_sync(FULL_MASK, valid && !resolved);
      if (lane == 0 && P.unresolved) P.unresolved[group] = un;
      if (emit) {
        const uint64_t row = P.row_mode == 0 ? (uint64_t)(uint32_t)row_id : (P.row_mode == 1 ? qpos - P.q_begin : gi);
        int32_t* io = P.idx_out + row * (uint64_t)k;
        float* dd = P.dist_out + row * (uint64_t)k;
        if (P.row_mode && P.qid_out) P.qid_out[row] = row_id;
        kl_emit<true, S>(H, cnt, k, heap, P.squared != 0, io, dd);
      }
    }
    __syncwarp();
  }

  if (COUNT && P.counters) {
    atomicAdd(&P.counters[0], c_nodes);
    atomicAdd(&P.counters[1], c_tests);
    atomicAdd(&P.counters[2], c_ins);
    if (c_viol) atomicAdd(&P.counters[6], c_viol);
    if (lane == 0) {
      atomicAdd(&P.counters[3], c_wnodes);
      atomicAdd(&P.counters[4], c_wleaves);
      atomicAdd(&P.counters[5], c_wpts);
    }
  }
}

// ------------------------------------------------------------------------------------------------
// Sparse rounds: when only a small fraction of the queries is still unresolved, 32 consecutive queue
// entries are no longer neighbours in space, and a shared stack would walk the union of 32 unrelated
// traversals on one warp (measured: 1.2 ms for 2 743 queries).  This variant gives every query its
// own thread, stack and k-list; it is divergent but embarrassingly parallel.  Same distance formula,
// same strict pruning, same (d2, index) keys => same results.
// ------------------------------------------------------------------------------------------------
constexpr int SPARSE_THREADS = 128;
// Measured (profiles/r2_ab_chunk.jsonl): 8 per step 0.414 vs 0.447 ms on cfg2's 97 478 leftovers but 1.98 vs 1.66 ms on cfg4's
// 568 002; 16 and 32 per step 1.0 / 1.8 ms (registers, wasted tail loads).  4 stays.
#ifndef TKNN_SPARSE_CHUNK
#define TKNN_SPARSE_CHUNK 4
#endif
constexpr int SPARSE_CHUNK = TKNN_SPARSE_CHUNK;  // leaf points fetched per step of the thread-per-query kernel

// + 3 slots of padding in front: list_insert prefetches up to three slots below the sentinel
__host__ __device__ inline size_t sparse_smem(int k) { return ((size_t)(k + 1) * SPARSE_THREADS + 3 * 32) * sizeof(uint64_t); }

template <bool COUNT, bool SEG = false>
static __global__ void __launch_bounds__(SPARSE_THREADS) traverse_sparse_kernel(const Params P) {
  extern __shared__ __align__(16) unsigned char smem[];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int k = P.k;
  uint64_t* H = reinterpret_cast<uint64_t*>(smem) + 3 * 32 + (size_t)warp * (k + 1) * 32 + lane;
  H[0] = 0;  // sentinel
  const bool heap = k > LIST_MAX_K;
  int stack[STACK_DEPTH];
  unsigned long long c_nodes = 0, c_tests = 0, c_ins = 0;

  const uint64_t gi = (uint64_t)blockIdx.x * SPARSE_THREADS + threadIdx.x;
  const uint64_t n_active = P.n_active_dev ? min((uint64_t)__ldg(P.n_active_dev), P.n_active) : P.n_active;
  const bool valid = gi < n_active;
  uint64_t qpos = 0;
  if (valid) qpos = P.queue ? (uint64_t)P.queue[gi] : P.q_begin + gi;
  float4 q = make_float4(0.f, 0.f, 0.f, 0.f);
  if (valid) q = __ldg(&P.queries[qpos]);
  const int row_id = __float_as_int(q.w);
  int self = -1;
  if (valid) self = P.self_ids ? P.self_ids[qpos] : (P.self_is_row ? row_id : -1);
  float r2 = P.r2_dev ? __ldg(P.r2_dev) : P.r2;
  if (valid && P.query_r2) r2 = fminf(r2, P.query_r2[qpos]);
  float bound = r2;
  int cnt = 0;
  SegLane<SEG> sl;
  if constexpr (SEG) {
    if (valid) seg_lane_init(sl, P, qpos);
  }

  if (valid) {
    int sp = 0;
    int node = 0;
    for (;;) {
      const float4* np = reinterpret_cast<const float4*>(P.nodes + node);
      const float4 na = __ldg(np), nb = __ldg(np + 1), nc = __ldg(np + 2), nd = __ldg(np + 3);
      const float2 d01 = box_dist2_x2(q.x, q.y, q.z, na, nb, nc);
      float d0 = d01.x, d1 = d01.y;
      if constexpr (SEG) seg_cull(P, node, sl.seg, d0, d1);
      if (COUNT) c_nodes += 1;
      const int ref0 = __float_as_int(nd.x), cnt0 = __float_as_int(nd.z);
      const int ref1 = __float_as_int(nd.y), cnt1 = __float_as_int(nd.w);
      const bool swap = d1 < d0;
#pragma unroll 1
      for (int c = 0; c < 2; ++c) {
        const bool second = (c == 1) != swap;
        const int lcount = second ? cnt1 : cnt0;
        if (lcount <= 0) continue;
        const float dcs = second ? d1 : d0;
        if (!(dcs <= bound)) continue;
        if (dcs == bound && cnt == k) {  // exact tie: only a lower index can still win
          const int2 mi = __ldg(&P.node_min_idx[node]);
          if ((second ? mi.y : mi.x) >= key_idx(kl_worst(H, k, heap))) continue;
        }
        const float4* lp = P.pts + (uint64_t)(uint32_t)(second ? ref1 : ref0);
        if (COUNT) c_tests += lcount;
        // SPARSE_CHUNK independent loads in flight per step (the tail re-reads the last point; masked off)
        for (int j = 0; j < lcount; j += SPARSE_CHUNK) {
          float4 p[SPARSE_CHUNK];
#pragma unroll
          for (int u = 0; u < SPARSE_CHUNK; ++u) p[u] = __ldg(lp + min(j + u, lcount - 1));
#pragma unroll
          for (int u = 0; u < SPARSE_CHUNK; ++u) {
            const float d = dist2(q.x, q.y, q.z, p[u].x, p[u].y, p[u].z);
            const int pid = __float_as_int(p[u].w);
            if (j + u < lcount && d <= bound && pid != self) {
              const uint64_t key = make_key(d, pid);
              if (cnt < k || key < kl_worst(H, k, heap)) {
                kl_insert(H, cnt, k, key, heap);
                if (cnt == k) bound = key_d2(kl_worst(H, k, heap));
                if (COUNT) c_ins += 1;
              }
            }
          }
        }
      }
      bool w0 = (cnt0 == 0) && (d0 <= bound);
      bool w1 = (cnt1 == 0) && (d1 <= bound);
      if (cnt == k && ((w0 && d0 == bound) || (w1 && d1 == bound))) {
        const int2 mi = __ldg(&P.node_min_idx[node]);
        const int wi = key_idx(kl_worst(H, k, heap));
        if (w0 && d0 == bound && mi.x >= wi) w0 = false;
        if (w1 && d1 == bound && mi.y >= wi) w1 = false;
      }
      if (w0 && w1) {
        if (sp < STACK_DEPTH) stack[sp++] = swap ? ref0 : ref1;
        else atomicOr(P.error, 1u);
        node = swap ? ref1 : ref0;
      } else if (w0) {
        node = ref0;
      } else if (w1) {
        node = ref1;
      } else {
        if (sp == 0) break;
        node = stack[--sp];
      }
    }
  }

  int need = k;
  if constexpr (SEG) {
    if (valid && cnt < k) need = seg_need(P, sl.seg, k, self);
  }
  const bool resolved = valid && cnt == need;
  const unsigned un = __ballot_sync(FULL_MASK, valid && !resolved);
  if (lane == 0 && P.unresolved && (gi >> 5) < P.n_groups) P.unresolved[gi >> 5] = un;  // P.n_groups: the launch's capacity
  if (valid && (resolved || P.final_round)) {
    const uint64_t row = P.row_mode == 0 ? (uint64_t)(uint32_t)row_id : (P.row_mode == 1 ? qpos - P.q_begin : gi);
    int32_t* io = P.idx_out + row * (uint64_t)k;
    float* dd = P.dist_out + row * (uint64_t)k;
    if (P.row_mode && P.qid_out) P.qid_out[row] = row_id;
    kl_emit(H, cnt, k, heap, P.squared != 0, io, dd);
  }
  if (COUNT && P.counters) {
    atomicAdd(&P.counters[0], c_nodes);
    atomicAdd(&P.counters[1], c_tests);
    atomicAdd(&P.counters[2], c_ins);
    // every load is private to its thread here: the per-warp figures equal the per-query ones
    atomicAdd(&P.counters[3], c_nodes);
    atomicAdd(&P.counters[5], c_tests);
  }
}

// ------------------------------------------------------------------------------------------------
// Tiny rounds: one WARP per query.  A thread-per-query walk is a chain of ~100 dependent global loads plus
// ~670 serial distance tests and takes ~0.3 ms however few queries there are (the start-radius sample of
// 4 096 queries, a third round of a few hundred stragglers).  Here the 32 lanes test the <= 32 points of a
// leaf at once (one coalesced load, one ballot) and keep the k-list as one ascending array in shared
// memory that they shift cooperatively, so the chain shrinks to the node and leaf round trips.  Node
// decisions are scalar (one query), same strict pruning, same (d2, index) keys => same results.
// Unresolved queries set their bit in P.unresolved with atomicOr: the host zeroes the words first.
// ------------------------------------------------------------------------------------------------
constexpr int WQ_WARPS = 4;  // warps per block

// T = lanes per query: 32 (one warp per query: tiny rounds) or a TEAM of 4 / 8 / 16 lanes, 32 / T queries per warp
// (TKNN_OPT_SPARSE_TEAM, for sparse rounds).  A team loads its node and its leaf chunk coalesced, tests T points per step,
// and its k-list is one ascending array in shared memory shifted cooperatively; teams of one warp follow different paths,
// so every warp-level primitive below is masked to the team (independent thread scheduling), nothing is block-wide.
// MEASURED (profiles/r2_ab_team.jsonl): for sparse rounds the teams LOSE to the thread-per-query kernel — cfg2's 97 478
// leftover queries: 0.447 ms with threads, 0.78 / 0.65 / 0.63 ms with teams of 4 / 8 / 16; cfg4's 568 002: 1.64 vs 3.71 ms —
// the teams of a warp serialise on their diverging paths and each repeats the node test on all its lanes, while 32
// private walks keep 32 loads in flight per warp.  So T = 32 serves the tiny rounds and the teams stay an option.
__host__ __device__ inline size_t warpq_smem(int k, int T = 32) {
  return (size_t)WQ_WARPS * (32 / T) * ((size_t)k * sizeof(uint64_t) + STACK_DEPTH * sizeof(int));
}

// inserts `key` into the ascending list L[0, cnt) of capacity k (the largest entry falls off a full list);
// precondition: cnt < k or key < L[k - 1]; keys are distinct.  All T lanes of the team call it together
// (tl = lane within the team, tmask = the team's lanes, tshift = its first lane).
template <int T>
__device__ __forceinline__ void team_list_insert(uint64_t* L, int& cnt, int k, uint64_t key, int tl, unsigned tmask) {
  int pos = 0;  // entries smaller than key
  for (int c0 = 0; c0 < cnt; c0 += T) {
    const int i = c0 + tl;
    const uint64_t e = i < cnt ? L[i] : ~0ull;
    pos += __popc(__ballot_sync(tmask, e < key));
  }
  const int n_new = cnt < k ? cnt + 1 : k;
  // shift [pos, n_new - 1) one slot up, T entries at a time from the top: a chunk reads its old values
  // (and the last entry of the still untouched chunk below) before it writes
  for (int c0 = ((n_new - 1) / T) * T; c0 >= (pos / T) * T; c0 -= T) {
    const int i = c0 + tl;
    const bool moved = i > pos && i < n_new;
    uint64_t prev = 0;
    if (moved) prev = L[i - 1];
    __syncwarp(tmask);
    if (moved) L[i] = prev;
    else if (i == pos) L[i] = key;
    __syncwarp(tmask);
  }
  cnt = n_new;
}

template <bool COUNT, int T, bool SEG = false>
static __global__ void __launch_bounds__(WQ_WARPS * 32) traverse_warp_kernel(const Params P) {
  extern __shared__ __align__(16) unsigned char smem[];
  constexpr int TEAMS = 32 / T;                 // queries per warp
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int team = lane / T, tl = lane % T, tshift = team * T;
  const unsigned tmask = T == 32 ? FULL_MASK : (((1u << (T & 31)) - 1u) << tshift);
  const int k = P.k;
  const int slot = warp * TEAMS + team;         // this query's list and stack inside the block
  uint64_t* L = reinterpret_cast<uint64_t*>(smem) + (size_t)slot * k;
  int* stack = reinterpret_cast<int*>(smem + (size_t)WQ_WARPS * TEAMS * k * sizeof(uint64_t)) + slot * STACK_DEPTH;
  const uint64_t gi = ((uint64_t)blockIdx.x * WQ_WARPS + warp) * TEAMS + team;
  const uint64_t n_active = P.n_active_dev ? min((uint64_t)__ldg(P.n_active_dev), P.n_active) : P.n_active;
  if (gi >= n_active) return;  // the whole team leaves; the kernel has no block-wide barrier
  const uint64_t qpos = P.queue ? (uint64_t)P.queue[gi] : P.q_begin + gi;
  const float4 q = __ldg(&P.queries[qpos]);
  const int row_id = __float_as_int(q.w);
  const int self = P.self_ids ? P.self_ids[qpos] : (P.self_is_row ? row_id : -1);
  float bound = P.r2_dev ? __ldg(P.r2_dev) : P.r2;
  if (P.query_r2) bound = fminf(bound, P.query_r2[qpos]);
  int cnt = 0;
  uint64_t worst = ~0ull;  // L[k - 1] once the list is full
  unsigned long long c_nodes = 0, c_tests = 0, c_ins = 0;
  SegLane<SEG> sl;
  if constexpr (SEG) seg_lane_init(sl, P, qpos);

  int sp = 0;
  int node = 0;
  for (;;) {
    const float4* np = reinterpret_cast<const float4*>(P.nodes + node);
    const float4 na = __ldg(np), nb = __ldg(np + 1), nc = __ldg(np + 2), nd = __ldg(np + 3);
    const float2 d01 = box_dist2_x2(q.x, q.y, q.z, na, nb, nc);
    float d0 = d01.x, d1 = d01.y;
    if constexpr (SEG) seg_cull(P, node, sl.seg, d0, d1);
    if (COUNT) c_nodes += 1;
    const int ref0 = __float_as_int(nd.x), cnt0 = __float_as_int(nd.z);
    const int ref1 = __float_as_int(nd.y), cnt1 = __float_as_int(nd.w);
    const bool swap = d1 < d0;
#pragma unroll 1
    for (int c = 0; c < 2; ++c) {
      const bool second = (c == 1) != swap;
      const int lcount = second ? cnt1 : cnt0;
      if (lcount <= 0) continue;
      const float dcs = second ? d1 : d0;
      if (!(dcs <= bound)) continue;
      if (dcs == bound && cnt == k) {  // exact tie: only a lower index can still win
        const int2 mi = __ldg(&P.node_min_idx[node]);
        if ((second ? mi.y : mi.x) >= key_idx(worst)) continue;
      }
      if (COUNT) c_tests += lcount;
      const float4* lp = P.pts + (uint64_t)(uint32_t)(second ? ref1 : ref0);
#pragma unroll 1
      for (int j0 = 0; j0 < lcount; j0 += T) {  // T points per step; the bound tightens between steps
        bool pass = false;
        uint64_t key = 0;
        if (j0 + tl < lcount) {
          const float4 p = __ldg(lp + j0 + tl);
          const float d = dist2(q.x, q.y, q.z, p.x, p.y, p.z);
          const int pid = __float_as_int(p.w);
          pass = d <= bound && pid != self;
          key = make_key(d, pid);
        }
        unsigned m = __ballot_sync(tmask, pass) >> tshift;
        while (m) {
          const int src = __ffs(m) - 1;
          m &= m - 1u;
          const uint64_t kk = __shfl_sync(tmask, key, tshift + src);
          if (cnt == k && kk >= worst) continue;
          team_list_insert<T>(L, cnt, k, kk, tl, tmask);
          if (COUNT) c_ins += 1;
          if (cnt == k) {
            worst = L[k - 1];
            bound = key_d2(worst);
          }
        }
      }
    }
    bool w0 = (cnt0 == 0) && (d0 <= bound);
    bool w1 = (cnt1 == 0) && (d1 <= bound);
    if (cnt == k && ((w0 && d0 == bound) || (w1 && d1 == bound))) {
      const int2 mi = __ldg(&P.node_min_idx[node]);
      const int wi = key_idx(worst);
      if (w0 && d0 == bound && mi.x >= wi) w0 = false;
      if (w1 && d1 == bound && mi.y >= wi) w1 = false;
    }
    if (w0 && w1) {
      if (sp < STACK_DEPTH) {
        if (tl == 0) stack[sp] = swap ? ref0 : ref1;
        ++sp;
      } else if (tl == 0) {
        atomicOr(P.error, 1u);
      }
      node = swap ? ref1 : ref0;
    } else if (w0) {
      node = ref0;
    } else if (w1) {
      node = ref1;
    } else {
      if (sp == 0) break;
      --sp;
      __syncwarp(tmask);
      node = stack[sp];
    }
  }

  int need = k;
  if constexpr (SEG) {
    if (cnt < k) need = seg_need(P, sl.seg, k, self);
  }
  const bool resolved = cnt == need;
  if (!resolved && P.unresolved && tl == 0) atomicOr(&P.unresolved[gi >> 5], 1u << (unsigned)(gi & 31));
  if (resolved || P.final_round) {
    const uint64_t row = P.row_mode == 0 ? (uint64_t)(uint32_t)row_id : (P.row_mode == 1 ? qpos - P.q_begin : gi);
    int32_t* io = P.idx_out + row * (uint64_t)k;
    float* dd = P.dist_out + row * (uint64_t)k;
    if (P.row_mode && P.qid_out && tl == 0) P.qid_out[row] = row_id;
    __syncwarp(tmask);
    for (int i = tl; i < k; i += T) {
      if (i < cnt) {
        const uint64_t e = L[i];
        io[i] = key_idx(e);
        dd[i] = P.squared ? key_d2(e) : __fsqrt_rn(key_d2(e));
      } else {
        io[i] = -1;
        dd[i] = FLT_MAX;
      }
    }
  }
  if (COUNT && P.counters && tl == 0) {
    atomicAdd(&P.counters[0], c_nodes);
    atomicAdd(&P.counters[1], c_tests);
    atomicAdd(&P.counters[2], c_ins);
    atomicAdd(&P.counters[3], c_nodes);
    atomicAdd(&P.counters[5], c_tests);
  }
}

// Start-radius estimator, device side.  The sample = `sg` runs of 32 consecutive sorted positions spread evenly over
// the `groups` groups of the query range (only the last group of the range can be short, and it is the last run).
static __global__ void __launch_bounds__(256) sample_queue_kernel(uint64_t groups, uint32_t sg, uint64_t q_begin, uint64_t nq,
                                                                  uint32_t* __restrict__ queue) {
  const uint32_t t = blockIdx.x * 256 + threadIdx.x;
  if (t >= sg * 32u) return;
  const uint64_t g = groups * (uint64_t)(t >> 5) / sg;
  const uint64_t pos = g * 32 + (t & 31u);
  if (pos < nq) queue[t] = (uint32_t)(q_begin + pos);
}

// out[0] = the `pos`-th smallest (0-based) of the m sampled k-th-neighbour distances dist[i * k + k - 1], out[1] = its
// square (the round's r2, the same fp32 product the host forms).  Radix select over the bit patterns (non-negative
// floats order like unsigned ints): four 8-bit passes of one block.  A degenerate sample (the quantile is 0: duplicate
// clusters) falls back to the largest finite positive value, or +inf (one unbounded round) when there is none.
// quantile_pm >= 0 (segmented builds): rows that came back unfilled (k-th distance FLT_MAX: their segment has at most k
// points) are left out, and the position is quantile_pm per mille of the filled rows; +inf when no row is filled.
static __global__ void __launch_bounds__(1024) radius_quantile_kernel(const float* __restrict__ dist, uint32_t m, int k, uint32_t pos,
                                                                      float* __restrict__ out, int quantile_pm = -1) {
  __shared__ uint32_t s_hist[256];
  __shared__ uint32_t s_prefix, s_want, s_maxpos, s_filled;
  constexpr uint32_t UNFILLED = 0x7f7fffffu;  // FLT_MAX
  const bool skip = quantile_pm >= 0;
  if (skip) {
    if (threadIdx.x == 0) s_filled = 0;
    __syncthreads();
    uint32_t f = 0;
    for (uint32_t i = threadIdx.x; i < m; i += 1024) f += __float_as_uint(dist[(uint64_t)i * k + (k - 1)]) != UNFILLED;
    atomicAdd(&s_filled, f);
    __syncthreads();
    if (s_filled == 0) {
      if (threadIdx.x == 0) { out[0] = INFINITY; out[1] = INFINITY; }
      return;
    }
    pos = (uint32_t)((double)(s_filled - 1) * quantile_pm / 1000.0);
  }
  uint32_t prefix = 0, mask = 0, want = pos;
  if (threadIdx.x == 0) s_maxpos = 0;
  for (int shift = 24; shift >= 0; shift -= 8) {
    if (threadIdx.x < 256) s_hist[threadIdx.x] = 0;
    __syncthreads();
    for (uint32_t i = threadIdx.x; i < m; i += 1024) {
      const uint32_t u = __float_as_uint(dist[(uint64_t)i * k + (k - 1)]);
      if (skip && u == UNFILLED) continue;
      if ((u & mask) == prefix) atomicAdd(&s_hist[(u >> shift) & 255u], 1u);
      if (shift == 24 && u > 0u && u < 0x7f800000u) atomicMax(&s_maxpos, u);
    }
    __syncthreads();
    if (threadIdx.x < 32) {  // warp 0: lane l owns bins 8 l .. 8 l + 7; the bin whose cumulative count passes `want`
      uint32_t mine = 0;
#pragma unroll
      for (int j = 0; j < 8; ++j) mine += s_hist[threadIdx.x * 8 + j];
      uint32_t inc = mine;
#pragma unroll
      for (int o = 1; o < 32; o <<= 1) {
        const uint32_t t = __shfl_up_sync(FULL_MASK, inc, o);
        if ((int)threadIdx.x >= o) inc += t;
      }
      const uint32_t before = inc - mine;
      const int owner = __ffs(__ballot_sync(FULL_MASK, inc > want)) - 1;  // first lane whose inclusive sum passes it
      if ((int)threadIdx.x == (owner < 0 ? 31 : owner)) {
        uint32_t acc = before;
        int b = threadIdx.x * 8;
        for (; b < (int)threadIdx.x * 8 + 7; ++b) {
          if (acc + s_hist[b] > want) break;
          acc += s_hist[b];
        }
        s_prefix = prefix | ((uint32_t)b << shift);
        s_want = want - acc;
      }
    }
    __syncthreads();
    prefix = s_prefix;
    want = s_want;
    mask |= 0xffu << shift;
  }
  if (threadIdx.x == 0) {
    float r = __uint_as_float(prefix);
    if (!(r > 0.0f) || !isfinite(r)) r = s_maxpos ? __uint_as_float(s_maxpos) : INFINITY;
    out[0] = r;
    out[1] = __fmul_rn(r, r);
  }
}

// Ballot words of "the point at sorted position p has an original index in [lo, hi)": the first step of
// cutting the query list into FILE-order slices whose output rows are contiguous (pipelined host output).
static __global__ void __launch_bounds__(256) index_range_flag_kernel(const float4* __restrict__ pts, uint64_t n, uint32_t lo,
                                                               uint32_t hi, uint32_t* __restrict__ words) {
  const uint64_t p = (uint64_t)blockIdx.x * 256 + threadIdx.x;
  bool in = false;
  if (p < n) {
    const uint32_t id = __float_as_uint(__ldg(&pts[p]).w);
    in = id >= lo && id < hi;
  }
  const uint32_t w = __ballot_sync(FULL_MASK, in);
  if ((threadIdx.x & 31) == 0 && p < n) words[p >> 5] = w;
}

// ------------------------------------------------------------------------------------------------
// Round compaction: unresolved ballot words -> the next round's queue, order preserved (so the
// next round's groups are still Morton-coherent).  offsets[] = exclusive scan of popc(words).
// ------------------------------------------------------------------------------------------------
static __global__ void __launch_bounds__(256) compact_queue_kernel(const uint32_t* __restrict__ words,
                                                            const uint32_t* __restrict__ offsets, uint32_t n_groups,
                                                            const uint32_t* __restrict__ queue_in, uint64_t q_begin,
                                                            uint32_t* __restrict__ queue_out) {
  const uint64_t t = (uint64_t)blockIdx.x * 256 + threadIdx.x;
  const uint32_t g = (uint32_t)(t >> 5);
  if (g >= n_groups) return;
  const int lane = (int)(t & 31);
  const uint32_t w = words[g];
  if ((w >> lane) & 1u) {
    const uint32_t pos = offsets[g] + __popc(w & ((1u << lane) - 1u));
    const uint64_t gi = (uint64_t)g * 32 + lane;
    queue_out[pos] = queue_in ? queue_in[gi] : (uint32_t)(q_begin + gi);
  }
}

}  // namespace trav
}  // namespace tknn
