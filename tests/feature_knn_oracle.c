/*
 * feature_knn_oracle.c — CPU reference of tknn_feature_knn (test infrastructure only; never loaded by the library).
 *
 * The contract (include/trueknn.h), literally: query row j of segment s is compared with every row p of data segment s
 * (p != self_ids[j]); d_c = y_c - x_c in fp32, d2 = d_0 * d_0, then d2 = fmaf(d_c, d_c, d2) for c = 1 .. f - 1 in that
 * order; the k smallest u64 keys (bits(d2) << 32) | index are kept (a max-heap of k keys) and emitted ascending.
 * Rows with fewer eligible points end in -1 / FLT_MAX.  OpenMP over query rows; `rows` (may be NULL) limits the work to
 * the query rows with rows[j] != 0 (the others are left untouched).
 * Build: gcc -O2 -std=gnu11 -fPIC -fopenmp -ffp-contract=off -shared -o libfeature_knn_oracle.so feature_knn_oracle.c -lm
 */
#include <float.h>
#include <math.h>
#include <stdint.h>
#include <stdlib.h>
#include <string.h>

static inline float dist2(const float* y, const float* x, int f) {
  const float d0 = y[0] - x[0];
  float d2 = d0 * d0;
  for (int c = 1; c < f; ++c) {
    const float d = y[c] - x[c];
    d2 = fmaf(d, d, d2);
  }
  return d2;
}

static inline uint64_t key_of(float d2, int64_t idx) {
  uint32_t b;
  memcpy(&b, &d2, 4);
  return ((uint64_t)b << 32) | (uint32_t)idx;
}

static void sift_down(uint64_t* h, int size, int i) {
  for (;;) {
    int m = i;
    const int l = 2 * i + 1, r = l + 1;
    if (l < size && h[l] > h[m]) m = l;
    if (r < size && h[r] > h[m]) m = r;
    if (m == i) return;
    const uint64_t t = h[i];
    h[i] = h[m];
    h[m] = t;
    i = m;
  }
}

static void sift_up(uint64_t* h, int i) {
  while (i > 0) {
    const int p = (i - 1) / 2;
    if (h[p] >= h[i]) return;
    const uint64_t t = h[i];
    h[i] = h[p];
    h[p] = t;
    i = p;
  }
}

static int cmp_u64(const void* a, const void* b) {
  const uint64_t x = *(const uint64_t*)a, y = *(const uint64_t*)b;
  return x < y ? -1 : x > y;
}

__attribute__((visibility("default"))) int tkfk_knn(const float* x, int64_t n, int f, int64_t xs, const uint64_t* xoff,
                                                    const float* y, int64_t nq, int64_t ys, const uint64_t* yoff,
                                                    int64_t n_segments, const int32_t* self_ids, int k,
                                                    const uint8_t* rows, int32_t* idx_out, float* d2_out) {
  if (f < 1 || k < 1 || n < 0 || nq < 0) return 1;
  for (int64_t s = 0; s < n_segments; ++s) {
    const int64_t a = (int64_t)xoff[s], b = (int64_t)xoff[s + 1], c = (int64_t)yoff[s], d = (int64_t)yoff[s + 1];
    int failed = 0;
#pragma omp parallel
    {
      uint64_t* h = (uint64_t*)malloc(sizeof(uint64_t) * (size_t)k);
      if (!h) {
#pragma omp atomic write
        failed = 1;
      }
#pragma omp for schedule(dynamic, 16)
      for (int64_t j = c; j < d; ++j) {
        if (!h || (rows && !rows[j])) continue;
        const int64_t self = self_ids ? self_ids[j] : -1;
        const float* q = y + j * ys;
        int cnt = 0;
        for (int64_t p = a; p < b; ++p) {
          if (p == self) continue;
          const uint64_t key = key_of(dist2(q, x + p * xs, f), p);
          if (cnt < k) {
            h[cnt] = key;
            sift_up(h, cnt++);
          } else if (key < h[0]) {
            h[0] = key;
            sift_down(h, k, 0);
          }
        }
        qsort(h, (size_t)cnt, sizeof(uint64_t), cmp_u64);
        for (int i = 0; i < k; ++i) {
          if (i < cnt) {
            const uint32_t bits = (uint32_t)(h[i] >> 32);
            float v;
            memcpy(&v, &bits, 4);
            idx_out[j * k + i] = (int32_t)(uint32_t)h[i];
            d2_out[j * k + i] = v;
          } else {
            idx_out[j * k + i] = -1;
            d2_out[j * k + i] = FLT_MAX;
          }
        }
      }
      free(h);
    }
    if (failed) return 2;
  }
  (void)n;
  (void)nq;
  return 0;
}
