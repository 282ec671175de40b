/*
 * chamfer_oracle.c — CPU reference of tknn_knn_backward / tknn_segment_reduce (test infrastructure only; never loaded by
 * the library).
 *
 * The contract (include/trueknn.h), literally, in fp32 (-ffp-contract=off, so every operation rounds on its own):
 *   per edge e = i * k + s with j = idx[e] != -1: t = 2 * g[e], term_q = t * (q_i - p_j), term_p = t * (p_j - q_i);
 *   grad_q[i] = chunked sum of row i's term_q in slot order, grad_p[j] = chunked sum of the term_p of the edges with
 *   idx = j in ascending e.  Chunked sum: chunks of 32 consecutive terms, each summed from +0, then the chunk sums in
 *   order from +0.  segment_reduce: the chunked sum of each segment's rows, divided by (float)count for the mean, +0 for
 *   an empty segment.
 * Build: gcc -O2 -std=gnu11 -fPIC -ffp-contract=off -shared -o libchamfer_oracle.so chamfer_oracle.c
 */
#include <stdint.h>
#include <stdlib.h>
#include <string.h>

/* One running chunked sum: acc (chunk sums so far), part (the open chunk), m (its terms). */
typedef struct {
  float acc, part;
  int m;
} chunked_t;

static void chunked_add(chunked_t* s, float v) {
  s->part = s->part + v;
  if (++s->m == 32) {
    s->acc = s->acc + s->part;
    s->part = 0.0f;
    s->m = 0;
  }
}

static float chunked_result(const chunked_t* s) { return s->m ? s->acc + s->part : s->acc; }

/* q: nq rows of pitch qs; p: n rows of pitch ps; idx, g: nq x k; gq: nq x dim or NULL; gp: n x dim or NULL */
__attribute__((visibility("default"))) void tkc_knn_backward(const float* q, int64_t nq, int qs, const float* p, int64_t n,
                                                            int ps, int dim, const int32_t* idx, int k, const float* g,
                                                            float* gq, float* gp) {
  chunked_t* sp = (chunked_t*)calloc((size_t)(n > 0 ? n : 1) * (size_t)dim, sizeof(chunked_t));
  for (int64_t i = 0; i < nq; ++i) {
    chunked_t sq[3];
    memset(sq, 0, sizeof(sq));
    for (int s = 0; s < k; ++s) {
      const int64_t e = i * k + s;
      const int32_t j = idx[e];
      if (j < 0) continue;
      const float t = 2.0f * g[e];
      for (int c = 0; c < dim; ++c) {
        const float qc = q[i * qs + c], pc = p[(int64_t)j * ps + c];
        const float dq = qc - pc, dp = pc - qc;
        chunked_add(&sq[c], t * dq);
        chunked_add(&sp[(int64_t)j * dim + c], t * dp);
      }
    }
    if (gq)
      for (int c = 0; c < dim; ++c) gq[i * dim + c] = chunked_result(&sq[c]);
  }
  if (gp)
    for (int64_t r = 0; r < n * dim; ++r) gp[r] = chunked_result(&sp[r]);
  free(sp);
}

/* x: n rows of pitch stride, f columns; off: n_seg + 1 offsets; reduce 0 = mean, 2 = sum; out: n_seg x f */
__attribute__((visibility("default"))) void tkc_segment_reduce(const float* x, int f, int stride, const uint64_t* off,
                                                              int64_t n_seg, int reduce, float* out) {
  for (int64_t s = 0; s < n_seg; ++s)
    for (int c = 0; c < f; ++c) {
      chunked_t a;
      memset(&a, 0, sizeof(a));
      for (uint64_t r = off[s]; r < off[s + 1]; ++r) chunked_add(&a, x[(int64_t)r * stride + c]);
      float v = chunked_result(&a);
      const uint64_t cnt = off[s + 1] - off[s];
      if (reduce == 0 && cnt) v = v / (float)(int64_t)cnt;
      out[s * f + c] = v;
    }
}
