/*
 * dbscan_oracle.c — CPU reference of tknn_dbscan (test infrastructure only; never loaded by the library).
 *
 * The contract (include/trueknn.h): p is in q's eps-ball iff d2(q, p) <= fl(eps * eps) with the project's one
 * distance rule d2 = fmaf(dz, dz, fmaf(dy, dy, dx * dx)) in fp32; q is a core point iff its ball holds at least
 * min_pts points, q itself and coincident duplicates included; clusters are the connected components of the core
 * points under "within eps", numbered in ascending order of their smallest core index; a non-core point with a core
 * point in its ball takes the lowest cluster id among those core points; every other point is noise (-1).
 *
 * Neighbourhoods come from closed-ball walks of a kd-tree (no neighbour lists are stored: at 10 M points they would
 * take gigabytes).  Boxes are pruned with the same fp32 chain on the clamped per-axis gaps, which under
 * round-to-nearest never exceeds the chain of any point inside the box, so no ball member is ever pruned.
 *   1. core flags: one walk per point (OpenMP), stopped as soon as min_pts members are found;
 *   2. components: one walk per core point (OpenMP) uniting it with every core member of lower index in a
 *      union-find whose roots are hooked with compare-and-swap (the larger root under the smaller one);
 *   3. cluster ids: one sequential pass in index order — the first core point of a component names it;
 *   4. border labels: one walk per non-core point (OpenMP), the minimum cluster id of its core members.
 * Build: gcc -O2 -std=gnu11 -fPIC -fopenmp -ffp-contract=off -shared -o libdbscan_oracle.so dbscan_oracle.c -lm
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

enum { WALK_COUNT = 0, WALK_UNITE = 1, WALK_BORDER = 2 };

static int32_t uf_find(int32_t* par, int32_t x) {
  for (;;) {
    const int32_t p = __atomic_load_n(&par[x], __ATOMIC_RELAXED);
    if (p == x) return x;
    const int32_t gp = __atomic_load_n(&par[p], __ATOMIC_RELAXED);
    if (gp != p) __atomic_store_n(&par[x], gp, __ATOMIC_RELAXED); /* path halving: gp is an ancestor of x */
    x = gp;
  }
}

static void uf_unite(int32_t* par, int32_t a, int32_t b) {
  int32_t ra = uf_find(par, a), rb = uf_find(par, b);
  while (ra != rb) {
    int32_t* slot = ra < rb ? &par[rb] : &par[ra];
    int32_t expect = ra < rb ? rb : ra;
    const int32_t want = ra < rb ? ra : rb;
    if (__atomic_compare_exchange_n(slot, &expect, want, 0, __ATOMIC_RELAXED, __ATOMIC_RELAXED)) return;
    ra = uf_find(par, ra);
    rb = uf_find(par, rb);
  }
}

/* One closed-ball walk around point qi.  WALK_COUNT: returns min(|ball|, limit).  WALK_UNITE: unites qi with every core
 * member of lower index, returns 0.  WALK_BORDER: returns the minimum label of the core members, or INT32_MAX. */
static int64_t walk(const tree_t* t, int32_t qi, float eps2, int mode, int64_t limit, const uint8_t* core, int32_t* par,
                    const int32_t* label) {
  const float* q = t->xyz + 3 * (int64_t)qi;
  int32_t stack[256];
  int sp = 0;
  int64_t acc = mode == WALK_BORDER ? INT32_MAX : 0;
  stack[sp++] = 0;
  while (sp) {
    const node_t* nd = &t->nodes[stack[--sp]];
    if (!(box_dist2(q, nd) <= eps2)) continue;
    if (nd->left >= 0) {
      stack[sp++] = nd->left;
      stack[sp++] = nd->right;
      continue;
    }
    for (int64_t i = nd->begin; i < nd->end; ++i) {
      const int32_t j = t->ids[i];
      if (!(dist2(q, t->xyz + 3 * (int64_t)j) <= eps2)) continue;
      if (mode == WALK_COUNT) {
        if (++acc >= limit) return acc;
      } else if (mode == WALK_UNITE) {
        if (j < qi && core[j]) uf_unite(par, qi, j);
      } else if (core[j] && label[j] < acc) {
        acc = label[j];
      }
    }
  }
  return acc;
}

__attribute__((visibility("default"))) int tkd_num_threads(void) {
#ifdef _OPENMP
  return omp_get_max_threads();
#else
  return 1;
#endif
}

/* label_out: n cluster ids or -1; core_out: n flags; *n_clusters_out: C.  Returns 0, or -1 on bad arguments / no memory. */
__attribute__((visibility("default"))) int tkd_dbscan(const float* xyz, int64_t n, float eps, int min_pts, int32_t* label_out,
                                                      uint8_t* core_out, int64_t* n_clusters_out) {
  if (n < 1 || n > INT32_MAX || !(eps >= 0.0f) || min_pts < 1 || !label_out || !core_out) return -1;
  const float eps2 = eps * eps;
  tree_t t;
  t.xyz = xyz;
  t.ids = (int32_t*)malloc(sizeof(int32_t) * (size_t)n);
  t.nodes = (node_t*)malloc(sizeof(node_t) * (size_t)(2 * (n / (LEAF / 2) + 2)));
  t.n_nodes = 0;
  int32_t* par = (int32_t*)malloc(sizeof(int32_t) * (size_t)n);
  int32_t* cid = (int32_t*)malloc(sizeof(int32_t) * (size_t)n);
  if (!t.ids || !t.nodes || !par || !cid) { free(t.ids); free(t.nodes); free(par); free(cid); return -1; }
  for (int64_t i = 0; i < n; ++i) t.ids[i] = (int32_t)i;
  build_rec(&t, 0, n);

#pragma omp parallel for schedule(dynamic, 1024)
  for (int64_t i = 0; i < n; ++i) core_out[i] = walk(&t, (int32_t)i, eps2, WALK_COUNT, min_pts, NULL, NULL, NULL) >= min_pts;

  for (int64_t i = 0; i < n; ++i) par[i] = (int32_t)i;
#pragma omp parallel for schedule(dynamic, 256)
  for (int64_t i = 0; i < n; ++i)
    if (core_out[i]) walk(&t, (int32_t)i, eps2, WALK_UNITE, 0, core_out, par, NULL);

  int64_t n_clusters = 0;
  for (int64_t i = 0; i < n; ++i) cid[i] = -1;
  for (int64_t i = 0; i < n; ++i) {
    label_out[i] = -1;
    if (!core_out[i]) continue;
    const int32_t r = uf_find(par, (int32_t)i);
    if (cid[r] < 0) cid[r] = (int32_t)n_clusters++;
    label_out[i] = cid[r];
  }

#pragma omp parallel for schedule(dynamic, 1024)
  for (int64_t i = 0; i < n; ++i) {
    if (core_out[i]) continue;
    const int64_t m = walk(&t, (int32_t)i, eps2, WALK_BORDER, 0, core_out, NULL, label_out);
    label_out[i] = m == INT32_MAX ? -1 : (int32_t)m;
  }
  if (n_clusters_out) *n_clusters_out = n_clusters;
  free(t.ids); free(t.nodes); free(par); free(cid);
  return 0;
}
