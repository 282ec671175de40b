/*
 * trueknn.h — C ABI of libtrueknn: the B200-native (sm_100a) replacement for the hot path of
 * vani-nag/OWLRayTracing's samples/s01-trueknn (TrueKNN): accel build -> traverse / intersect /
 * k-list -> radius-doubling rounds.  Citations are relative to the reference repository root.
 *
 * The reference has no kNN library interface: its sample drives ~25 OWL C-API calls
 * (owl/include/owl/owl_host.h:336-1240, call sites samples/s01-trueknn/hostCode.cpp:141-362).
 * Each entry point below names the slice of that sequence it replaces.
 *
 * Conventions (all functions): plain pointers and sizes, no C++ types; returns TKNN_OK (0) or a
 * TKNN_E* code and never throws or exits (the reference throws std::runtime_error through
 * extern "C" — owl/helper/cuda.h:22-31 — and exit(2)s on OptiX errors — owl/helper/optix.h:34-42);
 * the message of the last failure is available from tknn_last_error().  A context is bound to one
 * CUDA device and is not thread-safe; distinct contexts are independent.  Input/output arrays may
 * be HOST or DEVICE pointers (detected with cudaPointerGetAttributes); host buffers are staged
 * through device memory inside the call.  Calls are synchronous on return, like owlLaunch2D
 * (owl/impl.cpp:168-176).  There is no CPU fallback: without a CUDA device tknn_create fails.
 *
 * Result semantics (north star): for query q the k data points p != q BY INDEX minimising
 * (d2(q,p), index(p)) lexicographically, d2 = fmaf(dz,dz,fmaf(dy,dy,dx*dx)) in fp32;
 * idx_out[q*k+i] ascending, dist_out[q*k+i] = sqrtf(d2); unfilled slots are -1 / FLT_MAX
 * (hostCode.cpp:129).  Indices refer to the order of the points passed to tknn_build
 * (= file order in the sample, hostCode.cpp:115-124).
 */
#ifndef TRUEKNN_H
#define TRUEKNN_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#if defined(_WIN32)
#define TKNN_API
#else
#define TKNN_API __attribute__((visibility("default")))
#endif

#define TKNN_VERSION 100

enum {
  TKNN_OK = 0,
  TKNN_EINVAL = 1, /* bad argument (k >= n, dim not 2|3, non-finite coordinate, ...) */
  TKNN_ENOMEM = 2, /* host or device allocation failed */
  TKNN_ECUDA = 3,  /* CUDA runtime error (text in tknn_last_error) */
  TKNN_ENCCL = 4,  /* NCCL error, or libnccl.so.2 could not be loaded (multi-GPU calls only) */
  TKNN_ESTATE = 5  /* call order (search before build, ...) */
};

#define TKNN_MAX_K 512
#define TKNN_MAX_ROUNDS 48

/* option keys for tknn_set_option */
enum {
  TKNN_OPT_LEAF_SIZE = 1,   /* max points per BVH leaf, 4..32 (default 32)                         */
  TKNN_OPT_COUNTERS = 2,    /* 1: run the counting variant of the traversal kernel (V/T of §8d)   */
  TKNN_OPT_LEAF_POLICY = 3, /* 0: Morton-aligned maximal subtrees (default); 1: fixed chunks       */
  TKNN_OPT_SAMPLE_GROUPS = 4, /* groups of 32 queries sampled by the start-radius estimator (128) */
  TKNN_OPT_BLOCKS_PER_SM = 5, /* persistent-grid size of the traversal kernel, 0 = auto            */
  TKNN_OPT_SQUARED_DIST = 6,  /* 1: dist_out receives d2 instead of sqrtf(d2)                      */
  TKNN_OPT_RADIUS_QUANTILE = 7 /* start-radius estimator: per-mille quantile of the sampled k-th
                                  neighbour distance (default 990)                                */
  ,TKNN_OPT_KEEP_SCRATCH = 8   /* 1 (default): keep the build scratch buffers for the next tknn_build    */
  ,TKNN_OPT_APPROX_FILTER = 10 /* 1: conservative 3-FMA pre-filter before the exact distance test
                                  (DESIGN.md §3.2; audited, -1 % time); 0 (default): exact test on every pair */
  ,TKNN_OPT_OUTPUT_CHUNKS = 11 /* tknn_search_shard with HOST outputs: number of Morton slices whose
                                  device->host copies overlap the search of the next slice (default 4; 1 = off) */
  ,TKNN_OPT_FILE_ORDER_CHUNKS = 12 /* tknn_search with HOST outputs: slices by original index (rows of a slice are
                                  contiguous and final), copies overlapped like above (default 0 = auto: 5, or 2 when
                                  dist_out is NULL; for k > 24: 2 and 1; 1 = off)   */
  ,TKNN_OPT_MORTON_BITS = 13   /* curve-code bits per axis for the next build: 0 = auto (see TKNN_OPT_SORT_MODE), else 4..21 */
  ,TKNN_OPT_TIE_PRUNING = 14   /* index-aware pruning of exact distance ties: 0 = auto (kernel variant used when the
                                  build found a leaf of >= 8 coincident points, i.e. a duplicate cluster), 1 = always,
                                  2 = never           */
  ,TKNN_OPT_WARP_ROUND_MAX = 15 /* rounds with at most this many active queries (the start-radius sample, late rounds of a
                                  few stragglers, small query sets) run one WARP per query (default 49152; 0 = never) */
  ,TKNN_OPT_CURVE = 16          /* space-filling curve the next build sorts the points by: 0 = Hilbert (default; consecutive
                                  points are always neighbours in space, so a 32-query group is compact), 1 = Morton */
  ,TKNN_OPT_SPECULATIVE_MAX = 17 /* searches of at most this many queries run without a host decision between their launches:
                                  round 2 is launched as the final round before the host knows how many queries round 1 left
                                  (default 2^20; 0 = always wait for the count) */
  ,TKNN_OPT_SPARSE_TEAM = 18    /* sparse rounds (more than WARP_ROUND_MAX leftover queries, fewer than n / SPARSE_DIVISOR): 0 (default)
                                  = one thread per query; 4, 8, 16 = a team of that many lanes shares one traversal (measured
                                  slower: cfg2's 97 478 leftovers 0.45 ms with threads, 0.78 / 0.65 / 0.63 ms with teams) */
  ,TKNN_OPT_SORT_MODE = 19      /* build sort: 0 (default) = packed keys when they fit — (curve code << index bits | point index) in one
                                  u64, as many code bits per axis as fit beside the index (at most 13: five 8-bit passes), sorted
                                  keys-only at 16 B per point and pass; falls back to 1 when fewer than log2(n)/3 + 3 bits per axis
                                  would fit (n > 2^28) or TKNN_OPT_MORTON_BITS asks for more than fit; 1 = (u64 code, u32 index)
                                  pairs, log2(n)/3 + 8 bits per axis, 24 B per point and pass (round 1's sort) */
  ,TKNN_OPT_SPARSE_DIVISOR = 9 /* rounds >= 2 with fewer than n/divisor active queries run the
                                  thread-per-query kernel (default 8; 0 = never)                  */
  ,TKNN_OPT_GRID = 20           /* cell grid over the sorted points for round 1 of a dense kNN search with k <= 24 (same results):
                                  0 (default) = auto: a plain build without coincident-point leaves makes the table, and uses it
                                  when no cell holds more than 64 points (uniform clouds); 1 = off (the LBVH only); 2 = whenever
                                  the table is valid, whatever its occupancy (tests, A/B)  */
  ,TKNN_OPT_GRID_LEVEL = 21     /* cells per axis of the grid = 2^level: 0 (default) = floor(log2(n) / 3), else 1..8 (at most the
                                  key's code bits per axis) */
};

typedef struct tknn_ctx tknn_ctx;

typedef struct tknn_stats {
  /* build (replaces "Build time", hostCode.cpp:201-212) */
  uint64_t n_points;
  uint32_t n_leaves;
  uint32_t n_nodes;
  float build_ms;     /* points on device -> BVH ready (sum of the phases below) */
  float bounds_ms;    /* scene AABB reduce                                        */
  float morton_ms;    /* Morton codes                                             */
  float sort_ms;      /* onesweep radix sort (8 passes)                           */
  float leaves_ms;    /* leaf cut + point gather                                  */
  float hierarchy_ms; /* Karras hierarchy                                         */
  float refit_ms;     /* bottom-up AABB refit                                     */
  float h2d_ms;       /* host->device staging of the points (0 for device input)  */
  /* last search (replaces "True KNN time", hostCode.cpp:279-347) */
  uint64_t n_queries;
  int32_t k;
  int32_t rounds;
  float start_radius; /* the radius round 1 ran with (after auto-estimation)      */
  float final_radius;
  float estimate_ms;  /* start-radius estimator (0 when the caller gave a radius) */
  float search_ms;    /* first launch -> last result written on device, all rounds, incl. estimate */
  float d2h_ms;       /* device->host copy of results (0 for device output)       */
  float round_ms[TKNN_MAX_ROUNDS];  /* round incl. compaction + the host termination check */
  float kernel_ms[TKNN_MAX_ROUNDS]; /* the traversal kernel alone, CUDA events on the launching stream */
  uint64_t round_queries[TKNN_MAX_ROUNDS]; /* queries active in each round */
  uint32_t kernel_launches; /* kernels launched by the last search */
  uint32_t build_launches;  /* kernels launched by the last build  */
  /* counters (TKNN_OPT_COUNTERS=1), summed over all rounds; per-query, i.e. a 32-query group
   * visiting a node counts once per active query (SURVEY.md §8d: V(q), T(q)) */
  uint64_t nodes_visited;   /* sum_q V(q): 64-byte node records a query's warp read           */
  uint64_t points_tested;   /* sum_q T(q): float4 points distance-tested per query            */
  uint64_t heap_inserts;    /* accepted candidates                                            */
  uint64_t warp_node_visits;/* node records actually loaded (once per warp)                   */
  uint64_t warp_leaf_visits;/* leaves actually loaded (once per warp)                         */
  uint64_t warp_point_loads;/* float4 points actually loaded (once per warp)                  */
  uint64_t filter_violations;/* counting build: pairs the pre-filter rejected but the exact test accepts; must be 0 */
  uint64_t h2d_bytes, d2h_bytes; /* staging traffic of the last build / search */
  /* cell grid (TKNN_OPT_GRID) of the last build; with it, nodes_visited / warp_node_visits count the non-empty cells a
   * round-1 group tested and warp_leaf_visits the cells it staged */
  int32_t grid_level;        /* 2^grid_level cells per axis; 0: no table was made                         */
  int32_t grid_selected;     /* 1: round 1 of dense kNN searches (k <= 24) walks the grid                  */
  uint32_t grid_max_cell;    /* points in the fullest cell                                                */
  uint32_t grid_split_cells; /* cells whose points were not one contiguous run of the sort (always 0)     */
  float grid_ms;             /* table build, included in build_ms                                         */
  uint32_t grid_reserved;
  uint64_t grid_deferred;    /* counting build: round-1 groups whose cell range exceeded the cap, left to the LBVH rounds */
} tknn_stats;

/* Replaces owlContextCreate + module/program/pipeline/SBT setup (hostCode.cpp:141-159,267-269).
 * device = CUDA ordinal.  Fails with TKNN_ECUDA when no usable device exists. */
TKNN_API int tknn_create(int device, tknn_ctx** out);

/* Replaces owlContextDestroy (hostCode.cpp:362): frees every device allocation of the context. */
TKNN_API int tknn_destroy(tknn_ctx* ctx);

/* Run all work of this context on `cuda_stream` (a cudaStream_t; NULL = the context's own
 * non-blocking stream; pass cudaStreamLegacy / cudaStreamPerThread for the default streams).  Inputs
 * produced on another stream must be complete before a call: the library only orders its work on the
 * stream it was given.  The reference uses one stream per LaunchParams (owl/LaunchParams.cpp:46). */
TKNN_API int tknn_set_stream(tknn_ctx* ctx, void* cuda_stream);

TKNN_API int tknn_set_option(tknn_ctx* ctx, int key, int64_t value);

/* Replaces owlDeviceBufferCreate(points) + owlUserGeomGroupCreate + owlGroupBuildAccel(GAS) +
 * owlInstanceGroupCreate + owlGroupBuildAccel(IAS) (hostCode.cpp:165-175,199-212), i.e.
 * UserGeomGroup::buildAccel (owl/UserGeomGroup.cpp:39-241) and the bounds program
 * (deviceCode.cu:38-56): builds an LBVH over the n points.
 * xyz: n rows of `stride_floats` floats (>= dim); dim 2 => z = 0 (hostCode.cpp:114-118), dim 3. */
TKNN_API int tknn_build(tknn_ctx* ctx, const float* xyz, uint64_t n, int dim, int stride_floats);

/* Segmented build: a batch of independent point clouds in one BVH (torch_cluster's `batch`).  Segment s is the points
 * with indices in [seg_offsets[s], seg_offsets[s + 1]); seg_offsets holds n_segments + 1 entries, host or device, that
 * start at 0, never decrease and end at n (empty segments are legal); anything else, or n_segments outside
 * [1, 2^31 - 1]: TKNN_EINVAL.  n_segments = 1 is tknn_build, bit for bit.  A later tknn_build clears the segments.
 * After a segmented build:
 *   tknn_search / tknn_estimate_start_radius: row q holds the k points p of q's segment with index(p) != q and the
 *     smallest (d2, index), i.e. tknn_search run on q's segment alone with indices shifted by seg_offsets[s].  A row
 *     whose segment has at most k points ends in -1 / FLT_MAX.  k <= min(n - 1, TKNN_MAX_K) stays the global check.
 *   tknn_range_count / tknn_radius_search: only points of q's own segment are in its ball; nothing else changes.
 *   tknn_query / tknn_radius_query: TKNN_ESTATE; a separate query set takes tknn_query_segments /
 *     tknn_radius_query_segments, which give each query segment the data segment of the same number.
 *   tknn_fps: samples every segment on its own (sample_offsets give each segment its count).
 *   tknn_search_shard, tknn_dbscan, tknn_brute_force, tknn_partition_search and tknn_partition_verify: TKNN_ESTATE
 *     (segmented builds do not support them yet). */
TKNN_API int tknn_build_segments(tknn_ctx* ctx, const float* xyz, uint64_t n, int dim, int stride_floats,
                                 const uint64_t* seg_offsets, uint64_t n_segments);

/* Replaces the whole round loop (hostCode.cpp:285-340: owlLaunch2D + host termination scan +
 * radius *= 2 + 2x owlGroupRefitAccel) and the raygen / intersection programs
 * (deviceCode.cu:62-152).  All n points are the queries (samples/s01-trueknn/README.md:2).
 * start_radius > 0: round 1 searches the closed ball of that radius, unresolved queries double it
 * (hostCode.cpp:323); start_radius <= 0: estimated from a sample (Util/random_sample.py's role);
 * start_radius = +inf: one unbounded round.  idx_out/dist_out: n*k each, rows in build order.
 * dist_out may be NULL (tknn_search and tknn_search_shard): indices only — with host outputs that halves the
 * device->host copy, which bounds the end-to-end time of a large search (DESIGN.md §5).
 * k must satisfy 1 <= k <= min(n-1, TKNN_MAX_K) (the reference never terminates for k > n-1). */
TKNN_API int tknn_search(tknn_ctx* ctx, int k, float start_radius, int32_t* idx_out, float* dist_out);

/* Query-sharded variant (SURVEY.md §8e, cfg4): this context answers shard `shard` of `n_shards`
 * contiguous Morton slices of the queries over its (replicated) BVH.  Rows are written compactly:
 * row r holds the neighbours of query qid_out[r]; *n_out rows are produced.  Capacity of each
 * output array must be at least tknn_shard_capacity(n, n_shards) rows. */
TKNN_API int tknn_search_shard(tknn_ctx* ctx, int k, float start_radius, int shard, int n_shards, int32_t* qid_out,
                               int32_t* idx_out, float* dist_out, uint64_t* n_out);
TKNN_API uint64_t tknn_shard_capacity(uint64_t n, int n_shards);

/* Separate query set on the built BVH (SURVEY.md §8f rank 3).  queries: nq rows; self_ids (may be
 * NULL) names the data index to exclude per query (-1: none); init_radius2 (may be NULL): per-query
 * cap on the SQUARED distance, closed (d2 <= cap; negative = no cap) — squared so that the
 * point-partitioned driver can pass a k-th-neighbour d2 bit-exactly for its boundary queries.
 * Output rows follow the query order; rows with fewer than k neighbours end in -1 / FLT_MAX. */
TKNN_API int tknn_query(tknn_ctx* ctx, const float* queries, uint64_t nq, int dim, int stride_floats,
                        const int32_t* self_ids, const float* init_radius2, int k, float start_radius,
                        int32_t* idx_out, float* dist_out);

/* Fixed-radius neighbour count per point (closed ball, self excluded) on the same traversal
 * (SURVEY.md §8f rank 4: the DBSCAN core-point test; tknn_dbscan below clusters with it).  count_out: n entries,
 * build order. */
TKNN_API int tknn_range_count(tknn_ctx* ctx, float radius, uint32_t* count_out);

/* Exact DBSCAN over the built cloud (SURVEY.md §8f rank 4; the reference README's RT-DBSCAN).  p is in q's eps-ball iff
 * d2(q, p) <= fl(eps * eps) with the d2 rule above (closed ball, as tknn_range_count); q is a CORE point iff its ball
 * holds at least min_pts points, q itself and coincident duplicates included (scikit-learn's min_samples, i.e.
 * range_count(eps)[q] >= min_pts - 1).  Clusters are the connected components of the core points under "within eps",
 * numbered 0 .. C-1 in ascending order of their smallest core index; a non-core point with a core point in its ball
 * takes the lowest cluster id among those core points (border); every other point is noise (-1).  The result is
 * deterministic and equals sklearn.cluster.DBSCAN(eps, min_samples=min_pts) wherever no pair distance lies within
 * rounding of eps.  eps = +inf and min_pts > n are legal; eps NaN or < 0, min_pts < 1 or a NULL label_out: TKNN_EINVAL;
 * before a build or on a point-partitioned context: TKNN_ESTATE.
 * label_out: n entries, build order, cluster id or -1 (noise); core_out (may be NULL): n bytes, 1 = core point;
 * *n_clusters_out (may be NULL): number of clusters.  Host or device arrays.
 * Statistics: rounds = 4 phases (core test, link, labelling, border) in round_ms / round_queries, the traversal kernel of
 * each in kernel_ms (0 for the labelling), search_ms = the whole call on the device, k = min_pts, radii = eps. */
TKNN_API int tknn_dbscan(tknn_ctx* ctx, float eps, int min_pts, int32_t* label_out, uint8_t* core_out,
                         uint64_t* n_clusters_out);

/* Exact fixed-radius neighbour lists (scipy's cKDTree.query_ball_point, scikit-learn's radius_neighbors).  The row of
 * query q holds every data point p with index(p) != self(q) and d2(q, p) <= fl(radius * radius), the d2 rule and closed
 * ball of tknn_range_count, sorted ascending by (d2, index): coincident duplicates are neighbours at distance 0, ties
 * are ordered by index.  So in the all-points form row q has range_count(radius)[q] entries, and a row of length >= k
 * starts with row q of tknn_search(k), bit for bit.
 * Output, CSR: offsets_out[0 .. nq] (u64, offsets_out[0] = 0); idx_out[offsets[q] .. offsets[q + 1]) = data indices;
 * dist_out the same entries' sqrtf(d2), or d2 while TKNN_OPT_SQUARED_DIST is set (may be NULL: indices only).
 * Sizing: idx_out == NULL asks for the size (offsets_out and *total_out are filled, TKNN_OK); capacity < total fills
 * offsets_out and *total_out, writes no entries and returns TKNN_EINVAL; otherwise all rows are written.
 * tknn_radius_search: every built point is a query, rows in build order, self = the point itself.
 * tknn_radius_query: nq query rows (dim, stride and self_ids as tknn_query; self_ids may be NULL, -1 = no exclusion),
 * rows in query order.  Host or device arrays.  radius = +inf is legal; radius NaN or < 0 or a NULL offsets_out:
 * TKNN_EINVAL; before a build or on a point-partitioned context: TKNN_ESTATE.
 * Statistics: rounds = 3 phases (count + scans, fill, order) in round_ms, their traversal kernels in kernel_ms (the
 * order phase: all of its kernels), round_queries = {queries, queries filled, rows sorted by the long-row radix sort},
 * search_ms = the whole call on the device. */
TKNN_API int tknn_radius_search(tknn_ctx* ctx, float radius, uint64_t* offsets_out, int32_t* idx_out, float* dist_out,
                                uint64_t capacity, uint64_t* total_out);
TKNN_API int tknn_radius_query(tknn_ctx* ctx, const float* queries, uint64_t nq, int dim, int stride_floats,
                               const int32_t* self_ids, float radius, uint64_t* offsets_out, int32_t* idx_out,
                               float* dist_out, uint64_t capacity, uint64_t* total_out);

/* Segmented query sets (torch_cluster's knn(x, y, k, batch_x, batch_y) and radius(x, y, r, batch_x, batch_y)): query
 * segment s is rows [q_seg_offsets[s], q_seg_offsets[s + 1]) and searches data segment s of the last build only.
 * q_seg_offsets: n_segments + 1 entries, host or device, that start at 0, never decrease and end at nq (empty query
 * segments are legal); n_segments must equal the segment count of the last build (1 after tknn_build).  NULL, a count
 * mismatch or malformed offsets: TKNN_EINVAL.  Before a build or on a point-partitioned context: TKNN_ESTATE.
 *   tknn_query_segments: row j of segment s holds the k points p with index(p) in [off[s], off[s + 1]),
 *     index(p) != self_ids[j] and d2 <= init_radius2[j] (when given) with the smallest (d2, index), i.e. tknn_query run
 *     on data segment s alone with indices shifted by off[s].  A self id of -1 or outside data segment s excludes
 *     nothing.  A row with fewer eligible points (an empty data segment included) ends in -1 / FLT_MAX.  The argument
 *     checks are those of tknn_query (1 <= k <= min(n, TKNN_MAX_K) globally).
 *   tknn_radius_query_segments: row j of segment s holds every p of data segment s with index(p) != self_ids[j] and
 *     d2 <= fl(radius * radius), sorted by (d2, index); output, sizing, capacity, statistics and errors as
 *     tknn_radius_query.
 * After a segmented build with the built points as queries, self_ids = 0 .. n - 1 and the build's offsets, the two
 * calls equal tknn_search and tknn_radius_search bit for bit; on a plain build with n_segments = 1 they are tknn_query
 * and tknn_radius_query. */
TKNN_API int tknn_query_segments(tknn_ctx* ctx, const float* queries, uint64_t nq, int dim, int stride_floats,
                                 const uint64_t* q_seg_offsets, uint64_t n_segments, const int32_t* self_ids,
                                 const float* init_radius2, int k, float start_radius, int32_t* idx_out, float* dist_out);
TKNN_API int tknn_radius_query_segments(tknn_ctx* ctx, const float* queries, uint64_t nq, int dim, int stride_floats,
                                        const uint64_t* q_seg_offsets, uint64_t n_segments, const int32_t* self_ids,
                                        float radius, uint64_t* offsets_out, int32_t* idx_out, float* dist_out,
                                        uint64_t capacity, uint64_t* total_out);

/* Exact farthest point sampling of the last build (torch_cluster's fps), plain (one segment) or segmented; segment s is
 * the points with indices [off[s], off[s + 1]).  Per segment, with a sample count m_s and a start index start_s in it:
 * D(p) is the minimum over the samples selected so far in p's segment of d2(c, p) (the d2 rule above; +inf before the
 * first sample).  Sample 0 is start_s; sample i + 1 is the point of the segment that maximises D(p), ties to the LOWEST
 * index (torch.argmax's first occurrence), i.e. the largest u64 key (bits(D) << 32) | (0xFFFFFFFF - index), which orders
 * +inf correctly too.  When every point of a segment has D = 0 (duplicates, m_s above its distinct locations) the rule
 * picks the segment's lowest index again, so samples may repeat; for distinct points and m_s = n_s they are a
 * permutation of the segment.  The result depends only on the points, the offsets, the counts and the starts (not on
 * leaf size, curve, sort mode, grid option or stream) and is identical from call to call.
 * sample_offsets: n_segments + 1 u64 entries, host or device, starting at 0, non-decreasing, with m_s =
 * sample_offsets[s+1] - sample_offsets[s] <= the segment's point count; n_segments must equal the build's segment count
 * (1 after tknn_build).  start_ids (may be NULL: the first point of every segment, off[s]): n_segments global indices,
 * each inside its segment wherever m_s > 0.  idx_out: sample_offsets[n_segments] entries, idx_out[soff[s] + i] = the
 * i-th sample of segment s as a global index; dist_out (may be NULL): sqrtf(D(sample i)) when it was selected (the
 * coverage radius after i samples, non-increasing in i), d2 while TKNN_OPT_SQUARED_DIST is set, FLT_MAX for sample 0.
 * Host or device arrays.  Errors: malformed offsets, a count above its segment, a start outside its segment, a NULL
 * idx_out or n > 2^31 - 1: TKNN_EINVAL; before a build, on a point-partitioned context or a BVH with caller-chosen ids:
 * TKNN_ESTATE; a device without cooperative launch when a segment is above the block tier's capacity: TKNN_ECUDA.
 * Statistics: rounds = 2 tiers (segments of at most 14 336 points: one CTA each; larger ones: one cooperative kernel,
 * leaf-culled) in round_ms / kernel_ms, round_queries = the samples of each tier, n_queries = all samples, search_ms =
 * the whole call on the device.  TKNN_OPT_COUNTERS: nodes_visited = leaf box tests of the grid tier, warp_leaf_visits
 * = leaves whose points were updated, points_tested = point distance updates. */
TKNN_API int tknn_fps(tknn_ctx* ctx, const uint64_t* sample_offsets, uint64_t n_segments, const int32_t* start_ids,
                      int32_t* idx_out, float* dist_out);

/* Exact k-nearest neighbours in feature space over a batch of clouds (torch_cluster's knn / knn_graph on features, as
 * DGCNN's dynamic graphs use them).  x: n data rows, y: nq query rows, both row-major with their own pitch (stride >= f
 * floats); only the first f columns are read.  y may alias x (the all-points form passes the same pointer twice).
 * Distance rule, with d_j = fl(y_j - x_j): d2 = d_0 * d_0, then d2 = fmaf(d_j, d_j, d2) for j = 1 .. f - 1 in that
 * order, in fp32.  For f = 3 this is the d2 rule above; for f = 2 it equals the 2-D path (z = 0).  fmaf(d, d, +0) has
 * the bits of d * d, so the sum may start at +0.
 * Segments: query segment s (rows [y_off[s], y_off[s + 1])) searches data segment s (rows [x_off[s], x_off[s + 1]))
 * only.  Each offset array holds n_segments + 1 entries, host or device, that start at 0, never decrease and end at n
 * (nq for y_off); empty segments are legal.  Both NULL: one segment, and n_segments must be 1; one NULL: TKNN_EINVAL.
 * Row j holds the k points p of its data segment with index(p) != self_ids[j] and the smallest (d2, index), ordered
 * ascending by that key (the key of make_key: +inf distances from overflow are ordered by index).  self_ids (may be
 * NULL: nothing excluded): nq global data indices; -1 or an index outside the data segment excludes nothing.  Rows
 * with fewer eligible points end in -1 / FLT_MAX.  dist_out (may be NULL: indices only) receives sqrtf(d2), or d2
 * while TKNN_OPT_SQUARED_DIST is set.  idx_out / dist_out: nq * k entries.  Host or device arrays.
 * The call needs no build and touches none: it works before tknn_build, and a search after it returns what it
 * returned before.  No option selects its path: a tiled brute force on the CUDA cores (DESIGN.md §3.8), split over the
 * data rows when the query tiles alone would leave the GPU idle, with a k-way merge of the splits.
 * Errors (TKNN_EINVAL): f outside [1, 1024], a stride below f, k outside [1, min(n, TKNN_MAX_K)], n or nq >= 2^31, a
 * non-finite value in the first f columns of x or y, malformed offsets, a NULL x, y or idx_out.  nq = 0 is a no-op.
 * Statistics: n_queries, k, search_ms; rounds = 1 (the tile kernel) or 2 (tile kernel, then the merge of the splits),
 * with round_ms / kernel_ms / round_queries per round; points_tested = the pair distances evaluated, sum_s nq_s * n_s. */
TKNN_API int tknn_feature_knn(tknn_ctx* ctx, const float* x, uint64_t n, int f, int x_stride_floats,
                              const uint64_t* x_seg_offsets, const float* y, uint64_t nq, int y_stride_floats,
                              const uint64_t* y_seg_offsets, uint64_t n_segments, const int32_t* self_ids, int k,
                              int32_t* idx_out, float* dist_out);

/* Exact voxel-grid clustering over a batch of clouds (torch_cluster's grid_cluster, PyG's voxel_grid; DESIGN.md §3.9).
 * points: n rows of `stride_floats` floats (host or device), the first dim (2 or 3) columns are the position.  size,
 * start, end: HOST arrays of dim floats; start / end may be NULL (the column min / max).  Raw voxel id of a point, in
 * fp32 with IEEE rounding and int64 arithmetic, over its columns d = 0 .. D - 1:
 *   c = 0; m = 1;  for each d:  c += (int64) fl(fl(p_d - start_d) / size_d) * m;  m *= (int64) fl(fl(end_d - start_d) / size_d) + 1
 * with truncation toward zero, so a point up to one voxel below start lands in cell 0, one further below gives a
 * negative term, and one beyond end aliases into the next row: all as torch_cluster computes them.
 * Batches (seg_offsets, n_segments + 1 entries, host or device, validated as for tknn_build_segments; NULL: one cloud,
 * n_segments must be 1): the rule runs over [position | cloud id] (D = dim + 1) with size 1 for the id column, which
 * starts at 0 when start is given and at the first non-empty cloud's id otherwise, and ends at the last non-empty
 * cloud's id (PyG's voxel_grid).  A single cloud gives the ids of the position columns alone.
 * Consecutive ids: the rank of the raw id among the distinct raw ids, ascending as int64 (torch.unique(sorted=True,
 * return_inverse=True)).  raw_out (int64, may be NULL) and cluster_out (int32, may be NULL): n entries by point, host
 * or device.  *n_voxels_out: the number of distinct ids (0 for n = 0).  The clustering stays in the context for
 * tknn_voxel_members / tknn_voxel_pool until the next tknn_voxel_grid or tknn_destroy; builds and searches neither
 * need it nor touch it, and it touches no build state.
 * Errors (TKNN_EINVAL): dim not 2 or 3, a stride below dim, n > 2^30 - 1 (the sort's limit), n_segments >= 2^24 (ids
 * exact in fp32), malformed offsets, a NULL points, size or n_voxels_out, a non-finite coordinate, size, start or end,
 * a size <= 0, a per-axis cell count or a product of counts outside int64, and a raw id outside int64 at a corner of the
 * points' bounding box (points far outside a given [start, end]; every raw id lies between those of the corners). */
TKNN_API int tknn_voxel_grid(tknn_ctx* ctx, const float* points, uint64_t n, int dim, int stride_floats,
                             const uint64_t* seg_offsets, uint64_t n_segments, const float* size, const float* start,
                             const float* end, int64_t* raw_out, int32_t* cluster_out, uint64_t* n_voxels_out);

/* Members of the last tknn_voxel_grid's voxels, each output may be NULL, host or device: offsets_out (n_voxels + 1)
 * CSR offsets into members_out (n point indices, voxel by voxel, ascending index inside a voxel), first_out (n_voxels)
 * the lowest point index of each voxel (PyG's consecutive_cluster picks an arbitrary one), seg_out (n_voxels) the cloud
 * of each voxel.  Before any tknn_voxel_grid: TKNN_ESTATE. */
TKNN_API int tknn_voxel_members(tknn_ctx* ctx, uint64_t* offsets_out, int32_t* members_out, int32_t* first_out,
                                int32_t* seg_out);

#define TKNN_REDUCE_MEAN 0
#define TKNN_REDUCE_MAX 1
/* Pools the rows x (n x f, pitch stride_floats >= f, 1 <= f <= 1024, host or device) over the last clustering into
 * out (n_voxels x f, host or device).  n must be the clustering's point count.  Members are taken in ascending index.
 * TKNN_REDUCE_MEAN: the members are split into chunks of 32 consecutive members, each chunk summed in order from +0.0f,
 * the chunk sums summed in chunk order from +0.0f, and mean = sum / (float)count, all round-to-nearest (a voxel of at
 * most 32 points is the plain sequential sum).  TKNN_REDUCE_MAX: the largest value as a float, the lowest index among
 * equal ones (so +0 / -0 ties keep the first), and a non-finite value anywhere in x's first f columns is TKNN_EINVAL.
 * The result depends on the inputs only.  Any number of calls per clustering.  Before any tknn_voxel_grid: TKNN_ESTATE;
 * another n, f or stride out of range, an unknown reduce or a NULL x or out (with n_voxels > 0): TKNN_EINVAL. */
TKNN_API int tknn_voxel_pool(tknn_ctx* ctx, const float* x, uint64_t n, int f, int stride_floats, int reduce, float* out);

/* Exact k-NN interpolation (PyG's knn_interpolate: the feature propagation, or upsampling, of PointNet++; DESIGN.md
 * §3.10).  idx / d2: the nq x k rows of tknn_query / tknn_query_segments with TKNN_OPT_SQUARED_DIST = 1 (squared
 * distances); x: n feature rows of f columns with pitch x_stride_floats >= f.  For row i and its slots s = 0 .. k-1 in
 * slot order, a slot with idx = -1 is skipped wherever it lies; for every other slot, in fp32 with round-to-nearest:
 *   w[i,s]   = fl(1 / max(d2[i,s], (float)1e-16))            (a NaN d2 stays NaN, d2 = +inf gives w = 0)
 *   den[i]   = sum_s w[i,s]                                   (from +0, in slot order)
 *   num[i,c] = sum_s fl(x[idx[i,s], c] * w[i,s])              (each product rounded on its own, no FMA; from +0, in slot order)
 *   out[i,c] = fl(num[i,c] / den[i])
 * Since the slot order is PyG's edge order (rows ascending by (d2, index)), this is PyG's arithmetic on the same d2.
 * A row without a filled slot gives 0 / 0 = NaN in every column, as in PyG; NaN in d2 or x propagates (which NaN, its
 * sign and payload, is not part of the contract).
 * out: nq x f, dense; weight_out (may be NULL): nq x k, w of every slot and +0 for skipped slots; den_out (may be NULL):
 * nq entries.  These are what tknn_interpolate_backward takes.  Host or device arrays.
 * The call needs no build and touches none: it works before tknn_build, and a search after it returns what it returned
 * before.
 * Errors (TKNN_EINVAL): k outside [1, TKNN_MAX_K], f < 1, a stride below f, n or nq >= 2^31, an idx entry outside {-1}
 * and [0, n) (found on the device and reported after the call, whose outputs are then undefined), and a NULL idx, d2 or
 * out, or a NULL x with n > 0, when nq > 0.  nq = 0 is a no-op.
 * Statistics: n_queries, k, search_ms, d2h_ms; rounds = 1 with its round_ms / kernel_ms / round_queries (nq). */
TKNN_API int tknn_interpolate(tknn_ctx* ctx, const int32_t* idx, const float* d2, uint64_t nq, int k, const float* x,
                              uint64_t n, int f, int x_stride_floats, float* out, float* weight_out, float* den_out);

/* Backward pass of tknn_interpolate with respect to x (PyG computes the weights without gradient, so there is none for
 * the positions).  idx, weight and den: what tknn_interpolate took and returned for nq rows of k slots; grad_out: nq
 * rows of f columns with pitch g_stride_floats >= f; grad_x: n x f, dense.  For data row j and column c:
 *   grad_x[j,c] = sum over the edges e = i*k + s with idx[i,s] = j, in ascending e, from +0, of
 *                 fl( fl(grad_out[i,c] / den[i]) * weight[i,s] )
 * i.e. PyG's autograd chain (DivBackward, the gather of the scatter sum, MulBackward, index_add_ into zeros) evaluated
 * sequentially in edge order.  A data row no edge references gets +0.  No float atomics: the result depends only on
 * the inputs and is identical from call to call, on any stream and launch shape.  A data row that many queries
 * reference is summed as one serial run (DESIGN.md §3.10 gives its cost).  Host or device arrays.
 * Errors (TKNN_EINVAL): those of tknn_interpolate (with g_stride_floats for the stride), nq * k above 2^30 - 1 edges
 * (the limit of the edge sort: 357 913 941 queries at k = 3), an idx entry outside {-1} and [0, n) (reported after the
 * call), and a NULL idx, weight, den or grad_out, or a NULL grad_x with n > 0, when nq > 0.  nq = 0 fills grad_x with +0.
 * Statistics: n_queries, k, search_ms, d2h_ms; rounds = 3 phases in round_ms: edge keys and counts, the sort, then the
 * run offsets and the column sums; kernel_ms: the edge kernel, the whole sort, the column-sum kernel; round_queries =
 * {nq, nq * k, n}. */
TKNN_API int tknn_interpolate_backward(tknn_ctx* ctx, const int32_t* idx, const float* weight, const float* den, uint64_t nq,
                                       int k, const float* grad_out, int g_stride_floats, uint64_t n, int f, float* grad_x);

/* Start-radius estimator alone (replaces samples/s01-trueknn/Util/random_sample.py:5-32). */
TKNN_API int tknn_estimate_start_radius(tknn_ctx* ctx, int k, float* radius_out);

/* Exact brute-force kNN of selected data points on the GPU (tiled, no BVH): the second oracle for
 * sampled queries at sizes no CPU oracle reaches (SURVEY.md §7 M0, §8c).  query_ids: nq data
 * indices (host or device).  Output rows follow query_ids. */
TKNN_API int tknn_brute_force(tknn_ctx* ctx, const int32_t* query_ids, uint64_t nq, int k, int32_t* idx_out,
                              float* dist_out);

/* k-way merge of partial neighbour lists on (d2, index): for each of nq rows, merge `parts` lists
 * of k (idx, d2) pairs (layout [parts][nq][k], a list ends at its first -1 index, duplicates by
 * index removed) into one list of k.  d2_parts holds SQUARED distances (produced with
 * TKNN_OPT_SQUARED_DIST = 1: sqrtf is not injective, so only d2 gives the exact order); dist_out
 * receives sqrtf(d2), or d2 again while TKNN_OPT_SQUARED_DIST is set (chained merges).  Used by the
 * point-partitioned driver (SURVEY.md §8e). */
TKNN_API int tknn_merge_topk(tknn_ctx* ctx, const int32_t* idx_parts, const float* d2_parts, int parts, uint64_t nq,
                             int k, int32_t* idx_out, float* dist_out);

TKNN_API int tknn_get_stats(const tknn_ctx* ctx, tknn_stats* out);
TKNN_API const char* tknn_last_error(const tknn_ctx* ctx);
TKNN_API int tknn_version(void);

/* ================================ multi-GPU (SURVEY.md §8b row 2, §8e) ================================
 * The reference's multi-GPU model is "replicate every object on every device and split the launch"
 * (owl/RayGen.cpp:150-200, owl/Context.cpp:75-120), created from a device list (owlContextCreate(ids, n),
 * owl/include/owl/owl_host.h:360) and unused by its sample (hostCode.cpp:141 passes one device).  Both
 * variants below live INSIDE the library, over NCCL (NVLink 5 / NVSwitch):
 *
 *   TKNN_SHARD_QUERIES    the BVH is replicated on every GPU, GPU g answers the g-th contiguous Morton slice of
 *                         the queries; no collective on the search path (one all-gather of the points at build).
 *   TKNN_PARTITION_POINTS every GPU owns one Morton range of the points (clouds that should not be replicated):
 *                         redistribution by Morton range, local LBVH, local search, boundary-query exchange,
 *                         remote bounded search, partial top-k merge on (d2, GLOBAL index).
 *
 * Two ways in: (a) ONE PROCESS drives all devices — tknn_create_multi (ncclCommInitAll inside) + tknn_multi_build
 * + tknn_multi_search, host arrays in, host arrays in FILE order out: the drop-in for the sample; (b) ONE RANK
 * PER PROCESS (torchrun, MPI): every rank creates its own tknn_ctx, rank 0 makes a unique id, everyone calls
 * tknn_comm_init, then the per-rank calls below; results stay sharded on the ranks.
 * Collective calls must be made by every rank in the same order.  NCCL failures return TKNN_ENCCL. */

enum { TKNN_SHARD_QUERIES = 1, TKNN_PARTITION_POINTS = 2 };

#define TKNN_UNIQUE_ID_BYTES 128

typedef struct tknn_dist_stats {
  int32_t n_ranks, rank;
  uint64_t n_global, n_owned;
  /* build, ms between CUDA events on this rank's stream (time spent waiting for peers inside a collective included) */
  float h2d_ms;          /* staging of this rank's slice (0 for device input)                              */
  float allgather_ms;    /* replicated build: the one all-gather of the points                             */
  float box_ms;          /* partitioned build: global box (local reduce + all-reduce)                      */
  float codes_ms;        /* Morton codes on the global grid + cell histogram + its all-reduce              */
  float splitters_ms;    /* histogram read-back and the host's splitter choice                             */
  float bucket_ms;       /* destination ranks, one onesweep pass on them, row packing                      */
  float exchange_ms;     /* all-to-all of (x, y, z, global id) rows                                        */
  float lbvh_ms;         /* the local (or replicated) LBVH build                                           */
  float summaries_ms;    /* per-cell boxes + all-gather                                                    */
  float build_total_ms;
  /* partitioned search */
  float local_search_ms, reach_ms, exchange_out_ms, remote_search_ms, exchange_back_ms, merge_ms, finish_ms, d2h_ms;
  float search_total_ms; /* first launch -> last result written on the device                              */
  uint64_t boundary_sent, boundary_received;
  uint64_t bytes_sent_build, bytes_sent_search; /* bytes this rank handed to NCCL (self copies excluded)   */
} tknn_dist_stats;

/* (b) one rank per process.  tknn_comm_unique_id: rank 0 fills 128 bytes (ncclGetUniqueId) and ships them to the
 * other ranks by any means; tknn_comm_init: ncclCommInitRank on the context's device. */
TKNN_API int tknn_comm_unique_id(void* id128_out);
TKNN_API int tknn_comm_init(tknn_ctx* ctx, int n_ranks, int rank, const void* id128);
TKNN_API int tknn_get_dist_stats(const tknn_ctx* ctx, tknn_dist_stats* out);

/* TKNN_SHARD_QUERIES build: this rank holds rows [first, first + n_local) of the n_total-point cloud (host or
 * device); slices must tile the cloud in rank order.  Uploads the slice, assembles the cloud on every GPU with one
 * ncclAllGather, builds the replicated LBVH.  Search with tknn_search_shard(ctx, k, r, rank, n_ranks, ...). */
TKNN_API int tknn_build_replicated(tknn_ctx* ctx, const float* xyz_local, uint64_t n_local, uint64_t first,
                                   uint64_t n_total, int dim, int stride_floats);

/* TKNN_PARTITION_POINTS build: this rank STARTS with rows of global indices [first_index, first_index + n_local)
 * (host or device) and ENDS owning one Morton range of the global cloud (tknn_partition_owned rows).  Global
 * indices must stay below 2^31. */
TKNN_API int tknn_partition_build(tknn_ctx* ctx, const float* xyz_local, uint64_t n_local, uint64_t first_index, int dim,
                                  int stride_floats);
TKNN_API uint64_t tknn_partition_owned(const tknn_ctx* ctx);

/* Exact kNN of the owned points against the GLOBAL cloud.  Row r: gid_out[r] = global index of the query,
 * idx_out[r*k..] = global neighbour indices, dist_out[r*k..] = distances (d2 while TKNN_OPT_SQUARED_DIST is set).
 * Arrays (host or device) hold `capacity` >= tknn_partition_owned rows; *n_out rows are written. */
TKNN_API int tknn_partition_search(tknn_ctx* ctx, int k, float start_radius, int32_t* gid_out, int32_t* idx_out,
                                   float* dist_out, uint64_t capacity, uint64_t* n_out);

/* Proof at sizes no replica fits (2 B points): every rank samples `samples` of its result rows, all ranks brute-force
 * ALL sampled queries against their OWN points (exact tiled kernel, no BVH), the partial lists are all-gathered and
 * merged on (d2, global index), and each rank compares its rows bit for bit.  gid/idx/dist: the arrays
 * tknn_partition_search filled (n_rows rows).  *n_checked / *n_bad: GLOBAL sums (identical on every rank). */
TKNN_API int tknn_partition_verify(tknn_ctx* ctx, int k, int samples, const int32_t* gid, const int32_t* idx, const float* dist,
                                   uint64_t n_rows, uint64_t* n_checked, uint64_t* n_bad);

/* (a) one process, all devices.  device_ids: CUDA ordinals (owlContextCreate's device list); distinct devices talk
 * over NCCL (ncclCommInitAll); a list that NAMES ONE DEVICE SEVERAL TIMES runs that many ranks on it over an
 * in-process transport (device-to-device copies) — NCCL refuses two ranks on one GPU — which is how the single-GPU
 * test suite exercises the multi-rank paths.  mode: TKNN_SHARD_QUERIES | TKNN_PARTITION_POINTS. */
typedef struct tknn_multi tknn_multi;
TKNN_API int tknn_create_multi(const int* device_ids, int n_devices, int mode, tknn_multi** out);
TKNN_API int tknn_multi_destroy(tknn_multi* m);
TKNN_API int tknn_multi_set_option(tknn_multi* m, int key, int64_t value); /* applied to every rank's context */
/* xyz: n host rows; replaces the same calls as tknn_build on every device */
TKNN_API int tknn_multi_build(tknn_multi* m, const float* xyz, uint64_t n, int dim, int stride_floats);
/* idx_out / dist_out: HOST arrays, n*k each, rows in build (file) order — the layout of tknn_search.  Every rank
 * writes its result rows straight into the owner GPU's slice of the file-order array through peer pointers (P2P
 * stores over NVLink), then each GPU copies its contiguous slice to the host. */
TKNN_API int tknn_multi_search(tknn_multi* m, int k, float start_radius, int32_t* idx_out, float* dist_out);
TKNN_API int tknn_multi_ranks(const tknn_multi* m);
TKNN_API tknn_ctx* tknn_multi_ctx(tknn_multi* m, int rank); /* per-rank context: stats, options (owned by m) */
TKNN_API const char* tknn_multi_last_error(const tknn_multi* m);
/* wall-clock phases of the last tknn_multi_build / tknn_multi_search (ms): [0] build, [1] search (all ranks done),
 * [2] row exchange to the owners, [3] device->host copies */
TKNN_API int tknn_multi_get_times(const tknn_multi* m, float* ms4);

/* ---- introspection used by the tests and the bench (not part of the drop-in surface) ---- */

/* The sort-key layout tknn_build would choose for n points under TKNN_OPT_MORTON_BITS = morton_bits (0 = auto) and
 * TKNN_OPT_SORT_MODE = sort_mode: curve-code bits per axis, index bits packed below the code (0 = pair sort) and the
 * number of 8-bit onesweep passes.  Pure host arithmetic: needs no context and no device. */
TKNN_API int tknn_key_layout(uint64_t n, int morton_bits, int sort_mode, int* code_bits_per_axis, int* index_bits,
                             int* sort_passes);

/* Stand-alone onesweep radix sort of (u64 key, u32 value) pairs, stable, in place; device or host
 * pointers.  values == NULL: keys only (the kernel variant behind the builder's packed keys). */
TKNN_API int tknn_sort_pairs(tknn_ctx* ctx, uint64_t* keys, uint32_t* values, uint64_t n);

/* Copies of the built BVH: nodes (n_nodes x 16 words, see DESIGN.md), sorted points
 * (n x float4: x, y, z, original index bits), leaf starts (n_leaves + 1).  NULL pointers skipped. */
TKNN_API int tknn_get_bvh(const tknn_ctx* ctx, void* nodes_out, void* points_out, uint32_t* leaf_start_out);

/* 63-bit Morton codes of n points on the cubic grid spanning box = {lo.xyz, hi.xyz} (the same code
 * the builder sorts by); the point-partitioned driver uses it with the GLOBAL box to assign Morton
 * ranges to ranks.  Device or host arrays. */
TKNN_API int tknn_morton_codes(tknn_ctx* ctx, const float* xyz, uint64_t n, int dim, int stride_floats,
                               const float* box6, uint64_t* codes_out);

/* Point-partitioned driver (SURVEY.md §8e): for each of n points with squared reach reach2[i], the set of
 * REMOTE ranks whose published per-cell boxes the closed ball (p, sqrt(reach2)) touches, as a bit mask
 * (bit s = rank s, n_ranks <= 32).  summaries: [n_ranks][8^cell_bits][6] floats (lo.xyz, hi.xyz; an
 * untouched cell holds an inverted box); box6: the global box the Morton grid spans.  Device arrays. */
TKNN_API int tknn_reach_mask(tknn_ctx* ctx, const float* xyz, uint64_t n, int stride_floats, const float* reach2,
                             const float* box6, const float* summaries, int n_ranks, int cell_bits, int self_rank,
                             uint32_t* mask_out);

/* Synthetic clouds generated on the device by the stateless hash of SURVEY.md §8d:
 * u(i,a) = (mix64(seed ^ ((3i+a) * 0x9E3779B97F4A7C15)) >> 40) * 2^-24.  Writes n rows of xyz
 * for indices [first, first+n) to a DEVICE or HOST array. */
TKNN_API int tknn_generate_uniform(tknn_ctx* ctx, uint64_t seed, uint64_t first, uint64_t n, float* xyz_out);

/* Point-file ingest and neighbour writer (SURVEY.md §8f rank 2; host only, no CUDA).
 * tknn_read_points: the sample's file grammar (hostCode.cpp:83-124), mmap + parallel parse; names
 * ending in ".f32" are raw little-endian float32 rows of `dim`.  xyz_out: n_cap rows of 3 floats; when the rows do
 * not fit (the grammar consumes the last line whole, so more than n rows can come back) the call returns
 * TKNN_EINVAL with *n_out = the capacity needed.
 * tknn_write_neighbours: `query,neighbourIndex,distance` lines (the dump commented out at
 * hostCode.cpp:312-319), or raw arrays (path + ".idx.i32" / ".dist.f32") when binary != 0. */
TKNN_API int tknn_read_points(const char* path, uint64_t n, int dim, float* xyz_out, uint64_t n_cap, uint64_t* n_out);
TKNN_API int tknn_write_neighbours(const char* path, const int32_t* idx, const float* dist, uint64_t n, int k, int binary);
/* tknn_write_neighbour_lists: the CSR rows of tknn_radius_search / _query (host arrays; dist may be NULL).  Text: one
 * `query,neighbourIndex,distance` line per entry (no distance column without dist); binary: path.off.u64 (nq + 1
 * offsets), path.idx.i32 and path.dist.f32 (raw little-endian arrays). */
TKNN_API int tknn_write_neighbour_lists(const char* path, const uint64_t* offsets, const int32_t* idx, const float* dist,
                                        uint64_t nq, int binary);

/* Device properties the roofline needs: SM count, L2 bytes, and a measured L2 / HBM read
 * bandwidth (GB/s) from a short read loop over an L2-resident / HBM-sized buffer. */
TKNN_API int tknn_measure_bandwidth(tknn_ctx* ctx, double* l2_gbs, double* hbm_gbs, int* sm_count, uint64_t* l2_bytes);

/* Measured aggregate shared-memory bandwidth (GB/s of bytes delivered to lanes): conflict-free LDS.128 — the
 * 128 B/clk/SM crossbar — and warp-broadcast LDS.128, the access pattern of the traversal kernel's leaf filter.
 * The traversal kernel is bound by this data path (and by issue slots), not by HBM: bench.py's roofline uses it. */
TKNN_API int tknn_measure_smem_bandwidth(tknn_ctx* ctx, double* conflict_free_gbs, double* broadcast_gbs);

#ifdef __cplusplus
}
#endif
#endif /* TRUEKNN_H */
