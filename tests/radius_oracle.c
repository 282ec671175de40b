/*
 * radius_oracle.c — CPU reference of tknn_radius_search / tknn_radius_query (test infrastructure only; never loaded by
 * the library).
 *
 * The contract (include/trueknn.h): the row of query q holds every data point p with index(p) != self(q) and
 * d2(q, p) <= fl(r * r), with the project's one distance rule d2 = fmaf(dz, dz, fmaf(dy, dy, dx * dx)) in fp32, sorted
 * ascending by the key (d2 bits << 32 | index) — the tko_key order of oracle/knn_oracle.c.
 *
 * Balls come from closed-ball walks of a kd-tree (the tree of dbscan_oracle.c), pruned with the same fp32 chain on the
 * clamped per-axis gaps, which never exceeds the chain of any point inside the box, so no member is ever pruned.  Two
 * passes over the queries (OpenMP): count, then fill each row at its offset and sort it.  It runs at 10 M points.
 * Build: gcc -O2 -std=gnu11 -fPIC -fopenmp -ffp-contract=off -shared -o libradius_oracle.so radius_oracle.c -lm
 */
#include <math.h>
#include <stdint.h>
#include <stdlib.h>
#include <string.h>
#ifdef _OPENMP
#include <omp.h>
#endif

#define LEAF 16

typedef struct {
  float lo[3], hi[3];
  int64_t begin, end; /* ids[begin, end) */
  int32_t left, right; /* children; -1 for a leaf */
} node_t;

typedef struct {
  const float* xyz;
  int32_t* ids;
  node_t* nodes;
  int64_t n_nodes;
} tree_t;

static inline float dist2(const float* q, const float* p) {
  const float dx = q[0] - p[0], dy = q[1] - p[1], dz = q[2] - p[2];
  return fmaf(dz, dz, fmaf(dy, dy, dx * dx));
}

static inline float box_dist2(const float* q, const node_t* b) {
  float d[3];
  for (int a = 0; a < 3; ++a) d[a] = fmaxf(fmaxf(b->lo[a] - q[a], q[a] - b->hi[a]), 0.0f);
  return fmaf(d[2], d[2], fmaf(d[1], d[1], d[0] * d[0]));
}

/* total order on (coordinate a, index): distinct keys, so the selection below needs no special case for ties */
static inline int less(const float* xyz, int a, int32_t i, int32_t j) {
  const float u = xyz[3 * (int64_t)i + a], v = xyz[3 * (int64_t)j + a];
  return u < v || (u == v && i < j);
}

#define SWAP(i, j) do { const int32_t t_ = ids[i]; ids[i] = ids[j]; ids[j] = t_; } while (0)

/* quickselect: ids[nth] gets the element of rank nth in [lo, hi), smaller ones before it, larger ones after */
static void select_nth(const float* xyz, int32_t* ids, int64_t lo, int64_t hi, int64_t nth, int a) {
  while (hi - lo > 2) {
    const int64_t m = lo + (hi - lo) / 2, r = hi - 1;
    if (less(xyz, a, ids[m], ids[lo])) SWAP(m, lo);
    if (less(xyz, a, ids[r], ids[lo])) SWAP(r, lo);
    if (less(xyz, a, ids[r], ids[m])) SWAP(r, m);
    SWAP(m, r); /* median of three as the pivot, at r */
    const int32_t piv = ids[r];
    int64_t s = lo;
    for (int64_t i = lo; i < r; ++i)
      if (less(xyz, a, ids[i], piv)) { SWAP(i, s); ++s; }
    SWAP(s, r);
    if (nth == s) return;
    if (nth < s) hi = s; else lo = s + 1;
  }
  if (hi - lo == 2 && less(xyz, a, ids[lo + 1], ids[lo])) SWAP(lo, lo + 1);
}

static int32_t build_rec(tree_t* t, int64_t begin, int64_t end) {
  const int32_t me = (int32_t)t->n_nodes++;
  node_t* nd = &t->nodes[me];
  for (int a = 0; a < 3; ++a) { nd->lo[a] = INFINITY; nd->hi[a] = -INFINITY; }
  for (int64_t i = begin; i < end; ++i) {
    const float* p = t->xyz + 3 * (int64_t)t->ids[i];
    for (int a = 0; a < 3; ++a) { nd->lo[a] = fminf(nd->lo[a], p[a]); nd->hi[a] = fmaxf(nd->hi[a], p[a]); }
  }
  nd->begin = begin;
  nd->end = end;
  nd->left = nd->right = -1;
  if (end - begin <= LEAF) return me;
  int axis = 0;
  for (int a = 1; a < 3; ++a)
    if (nd->hi[a] - nd->lo[a] > nd->hi[axis] - nd->lo[axis]) axis = a;
  const int64_t mid = begin + (end - begin) / 2;
  select_nth(t->xyz, t->ids, begin, end, mid, axis);
  const int32_t l = build_rec(t, begin, mid);
  const int32_t r = build_rec(t, mid, end);
  t->nodes[me].left = l; /* t->nodes is preallocated: nd stays valid, but say it plainly */
  t->nodes[me].right = r;
  return me;
}


/* One closed-ball walk around q: the number of members other than self, written as keys to out when out != NULL. */
static int64_t walk(const tree_t* t, const float* q, int32_t self, float r2, uint64_t* out) {
  int32_t stack[256];
  int sp = 0;
  int64_t cnt = 0;
  stack[sp++] = 0;
  while (sp) {
    const node_t* nd = &t->nodes[stack[--sp]];
    if (!(box_dist2(q, nd) <= r2)) continue;
    if (nd->left >= 0) {
      stack[sp++] = nd->left;
      stack[sp++] = nd->right;
      continue;
    }
    for (int64_t i = nd->begin; i < nd->end; ++i) {
      const int32_t j = t->ids[i];
      if (j == self) continue;
      const float d = dist2(q, t->xyz + 3 * (int64_t)j);
      if (!(d <= r2)) continue;
      if (out) {
        uint32_t bits;
        memcpy(&bits, &d, sizeof(bits));
        out[cnt] = ((uint64_t)bits << 32) | (uint32_t)j;
      }
      ++cnt;
    }
  }
  return cnt;
}

static int cmp_u64(const void* a, const void* b) {
  const uint64_t x = *(const uint64_t*)a, y = *(const uint64_t*)b;
  return x < y ? -1 : x > y;
}

static void sort_row(uint64_t* a, int64_t m) {
  if (m > 32) { qsort(a, (size_t)m, sizeof(uint64_t), cmp_u64); return; }
  for (int64_t i = 1; i < m; ++i) { /* insertion sort: most rows are short */
    const uint64_t v = a[i];
    int64_t j = i - 1;
    while (j >= 0 && a[j] > v) { a[j + 1] = a[j]; --j; }
    a[j + 1] = v;
  }
}

__attribute__((visibility("default"))) int tkr_num_threads(void) {
#ifdef _OPENMP
  return omp_get_max_threads();
#else
  return 1;
#endif
}

/* Data xyz [n][3]; queries q [nq][3] (NULL: the data points themselves, self = own index); self_ids [nq] (NULL: none,
 * -1: none).  offsets_out [nq + 1]; *keys_out: a malloc'd array of offsets_out[nq] row-sorted keys (free with tkr_free).
 * Returns 0, or -1 on bad arguments / no memory. */
__attribute__((visibility("default"))) int tkr_radius_lists(const float* xyz, int64_t n, const float* q, int64_t nq,
                                                            const int32_t* self_ids, float r, int64_t* offsets_out,
                                                            uint64_t** keys_out) {
  if (n < 1 || n > INT32_MAX || nq < 0 || !(r >= 0.0f) || !offsets_out || !keys_out) return -1;
  const float r2 = r * r;
  const int all = q == NULL;
  if (all) nq = n;
  tree_t t;
  t.xyz = xyz;
  t.ids = (int32_t*)malloc(sizeof(int32_t) * (size_t)n);
  t.nodes = (node_t*)malloc(sizeof(node_t) * (size_t)(2 * (n / (LEAF / 2) + 2)));
  t.n_nodes = 0;
  if (!t.ids || !t.nodes) { free(t.ids); free(t.nodes); return -1; }
  for (int64_t i = 0; i < n; ++i) t.ids[i] = (int32_t)i;
  build_rec(&t, 0, n);

#pragma omp parallel for schedule(dynamic, 1024)
  for (int64_t i = 0; i < nq; ++i) {
    const int32_t self = all ? (int32_t)i : (self_ids ? self_ids[i] : -1);
    offsets_out[i + 1] = walk(&t, all ? xyz + 3 * i : q + 3 * i, self, r2, NULL);
  }
  offsets_out[0] = 0;
  for (int64_t i = 0; i < nq; ++i) offsets_out[i + 1] += offsets_out[i];
  uint64_t* keys = (uint64_t*)malloc(sizeof(uint64_t) * (size_t)(offsets_out[nq] > 0 ? offsets_out[nq] : 1));
  if (!keys) { free(t.ids); free(t.nodes); return -1; }
#pragma omp parallel for schedule(dynamic, 1024)
  for (int64_t i = 0; i < nq; ++i) {
    const int32_t self = all ? (int32_t)i : (self_ids ? self_ids[i] : -1);
    uint64_t* row = keys + offsets_out[i];
    walk(&t, all ? xyz + 3 * i : q + 3 * i, self, r2, row);
    sort_row(row, offsets_out[i + 1] - offsets_out[i]);
  }
  *keys_out = keys;
  free(t.ids); free(t.nodes);
  return 0;
}

__attribute__((visibility("default"))) void tkr_free(void* p) { free(p); }
