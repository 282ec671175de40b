/*
 * voxel_oracle.c — CPU reference of tknn_voxel_grid / tknn_voxel_members / tknn_voxel_pool (test infrastructure only;
 * never loaded by the library).
 *
 * The contract (include/trueknn.h), literally: per point, over the columns [position | cloud id],
 *   c += (int64_t)((p_d - start_d) / size_d) * m;  m *= (int64_t)((end_d - start_d) / size_d) + 1
 * in fp32 (-ffp-contract=off, so every operation rounds on its own), start / end defaulting to the column min / max.
 * Dense ids: ranks of the distinct raw ids ascending; members ascending by index inside a voxel.  Pooling: the mean as
 * chunks of 32 consecutive members summed from +0, then the chunk sums in order from +0, divided by (float)count; the
 * max as the first maximum in index order.
 * Build: gcc -O2 -std=gnu11 -fPIC -ffp-contract=off -shared -o libvoxel_oracle.so voxel_oracle.c
 */
#include <stdint.h>
#include <stdlib.h>

typedef struct {
  int64_t raw;
  int64_t idx;
} pair_t;

static int cmp_pair(const void* a, const void* b) {
  const pair_t *x = (const pair_t*)a, *y = (const pair_t*)b;
  if (x->raw != y->raw) return x->raw < y->raw ? -1 : 1;
  return x->idx < y->idx ? -1 : x->idx > y->idx;
}

/* points: n rows of `stride` floats, dim position columns; off: n_seg + 1 cloud offsets or NULL; size[dim]; start /
 * end: dim floats or NULL.  Outputs: raw[n], cluster[n], vox_off[n + 1], members[n], first[n], seg[n]; returns the
 * number of voxels, or -1 when n == 0 is mishandled (never). */
__attribute__((visibility("default"))) int64_t tkv_grid(const float* points, int64_t n, int dim, int stride,
                                                       const uint64_t* off, int64_t n_seg, const float* size,
                                                       const float* start, const float* end, int64_t* raw,
                                                       int32_t* cluster, uint64_t* vox_off, int32_t* members,
                                                       int32_t* first, int32_t* seg) {
  if (n == 0) {
    vox_off[0] = 0;
    return 0;
  }
  const int cols = dim + (off ? 1 : 0);
  float s0[4], e0[4], sz[4];
  int32_t* cloud = (int32_t*)malloc(sizeof(int32_t) * (size_t)n);
  for (int64_t s = 0; s < (off ? n_seg : 1); ++s)
    for (uint64_t i = off ? off[s] : 0; i < (off ? off[s + 1] : (uint64_t)n); ++i) cloud[i] = (int32_t)s;
  for (int d = 0; d < cols; ++d) {
    float mn, mx;
    if (d < dim) {
      mn = mx = points[d];
      for (int64_t i = 1; i < n; ++i) {
        const float v = points[i * stride + d];
        if (v < mn) mn = v;
        if (v > mx) mx = v;
      }
    } else {
      mn = (float)cloud[0];
      mx = (float)cloud[n - 1];
    }
    if (d < dim) {
      s0[d] = start ? start[d] : mn;
      e0[d] = end ? end[d] : mx;
      sz[d] = size[d];
    } else {
      s0[d] = start ? 0.0f : mn;
      e0[d] = mx;
      sz[d] = 1.0f;
    }
  }
  for (int64_t i = 0; i < n; ++i) {
    int64_t c = 0, m = 1;
    for (int d = 0; d < cols; ++d) {
      const float p = d < dim ? points[i * stride + d] : (float)cloud[i];
      const float q = (p - s0[d]) / sz[d];
      c += (int64_t)q * m;
      const float span = (e0[d] - s0[d]) / sz[d];
      m *= (int64_t)span + 1;
    }
    raw[i] = c;
  }
  pair_t* p = (pair_t*)malloc(sizeof(pair_t) * (size_t)n);
  for (int64_t i = 0; i < n; ++i) {
    p[i].raw = raw[i];
    p[i].idx = i;
  }
  qsort(p, (size_t)n, sizeof(pair_t), cmp_pair);
  int64_t nv = 0;
  for (int64_t j = 0; j < n; ++j) {
    if (j == 0 || p[j].raw != p[j - 1].raw) {
      vox_off[nv] = (uint64_t)j;
      first[nv] = (int32_t)p[j].idx;
      seg[nv] = cloud[p[j].idx];
      ++nv;
    }
    members[j] = (int32_t)p[j].idx;
    cluster[p[j].idx] = (int32_t)(nv - 1);
  }
  vox_off[nv] = (uint64_t)n;
  free(p);
  free(cloud);
  return nv;
}

/* out[v * f + c] for every voxel of (vox_off, members); reduce 0 = mean, 1 = max */
__attribute__((visibility("default"))) void tkv_pool(const float* x, int f, int stride, const uint64_t* vox_off,
                                                     const int32_t* members, int64_t nv, int reduce, float* out) {
  for (int64_t v = 0; v < nv; ++v)
    for (int c = 0; c < f; ++c) {
      const uint64_t j0 = vox_off[v], j1 = vox_off[v + 1];
      float a;
      if (reduce == 1) {
        a = x[(int64_t)members[j0] * stride + c];
        for (uint64_t j = j0 + 1; j < j1; ++j) {
          const float t = x[(int64_t)members[j] * stride + c];
          if (t > a) a = t;
        }
      } else {
        a = 0.0f;
        for (uint64_t k = j0; k < j1; k += 32) {
          float s = 0.0f;
          for (uint64_t j = k; j < j1 && j < k + 32; ++j) s = s + x[(int64_t)members[j] * stride + c];
          a = a + s;
        }
        a = a / (float)(int64_t)(j1 - j0);
      }
      out[v * f + c] = a;
    }
}
