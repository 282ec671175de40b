/*
 * frames_oracle.c — CPU reference of tknn_local_frames (test infrastructure only; never loaded by the library).
 *
 * The contract (include/trueknn.h), literally, in fp32 (-ffp-contract=off, so every operation rounds on its own): per
 * row, the chunked-sum centroid and covariance over the valid slots, cyclic Jacobi (pairs (0,1), (0,2), (1,2), at most
 * 8 sweeps, stop before a sweep whose off-diagonal entries are all zero), three compare-exchanges on the eigenvalues,
 * and optionally the sign rule anchored at the first valid slot with column 1 = n x z.  c = 0 rows are NaN.
 * Also returns the covariance (a00 a01 a02 a11 a12 a22) and the number of sweeps run, for the accuracy tests.
 * Build: gcc -O2 -std=gnu11 -fPIC -ffp-contract=off -shared -o libframes_oracle.so frames_oracle.c
 */
#include <math.h>
#include <stdint.h>
#include <string.h>

/* R running chunked sums: chunks of 32 terms from +0, then the chunk sums in order from +0 */
typedef struct {
  float acc[6], part[6];
  int m;
} chunked_t;

static void chunked_add(chunked_t* s, const float* v, int r) {
  for (int i = 0; i < r; ++i) s->part[i] = s->part[i] + v[i];
  if (++s->m == 32) {
    for (int i = 0; i < r; ++i) {
      s->acc[i] = s->acc[i] + s->part[i];
      s->part[i] = 0.0f;
    }
    s->m = 0;
  }
}

static float chunked_result(const chunked_t* s, int i) { return s->m ? s->acc[i] + s->part[i] : s->acc[i]; }

static void rotate(float A[3][3], float V[3][3], int p, int q) {
  const int r = 3 - p - q;
  const float apq = A[p][q];
  if (apq == 0.0f) return;
  const float tau = (A[q][q] - A[p][p]) / (2.0f * apq);
  const float tt = tau * tau;
  float t;
  if (isinf(tt)) {
    t = 0.5f / tau;
  } else {
    const float sg = tau < 0.0f ? -1.0f : 1.0f;
    const float root = sqrtf(1.0f + tt);
    t = sg / (fabsf(tau) + root);
  }
  const float cs = 1.0f / sqrtf(1.0f + t * t);
  const float sn = t * cs;
  const float ta = t * apq;
  const float app = A[p][p] - ta, aqq = A[q][q] + ta;
  const float arp = A[r][p], arq = A[r][q];
  const float nrp = cs * arp - sn * arq, nrq = sn * arp + cs * arq;
  A[p][p] = app;
  A[q][q] = aqq;
  A[p][q] = A[q][p] = 0.0f;
  A[r][p] = A[p][r] = nrp;
  A[r][q] = A[q][r] = nrq;
  for (int u = 0; u < 3; ++u) {
    const float vp = V[u][p], vq = V[u][q];
    V[u][p] = cs * vp - sn * vq;
    V[u][q] = sn * vp + cs * vq;
  }
}

static void compare_exchange(float w[3], float V[3][3], int a, int b) {
  if (!(w[a] > w[b])) return;
  float t = w[a];
  w[a] = w[b];
  w[b] = t;
  for (int u = 0; u < 3; ++u) {
    t = V[u][a];
    V[u][a] = V[u][b];
    V[u][b] = t;
  }
}

/* points: n rows of pitch stride; idx: m x k; eig: m x 3, frames: m x 9, cov: m x 6, sweeps: m (each may be NULL) */
__attribute__((visibility("default"))) void tlf_local_frames(const float* points, int stride, const int32_t* idx,
                                                            int64_t m, int k, int disambiguate, float* eig,
                                                            float* frames, float* cov, int32_t* sweeps) {
  for (int64_t i = 0; i < m; ++i) {
    const int32_t* row = idx + i * k;
    int c = 0, first = -1;
    chunked_t s1;
    memset(&s1, 0, sizeof(s1));
    for (int s = 0; s < k; ++s) {
      if (row[s] < 0) continue;
      const float* p = points + (int64_t)row[s] * stride;
      if (first < 0) first = row[s];
      ++c;
      chunked_add(&s1, p, 3);
    }
    float w[3], V[3][3], C6[6];
    int used = 0;
    if (c == 0) {
      for (int u = 0; u < 3; ++u) {
        w[u] = NAN;
        for (int j = 0; j < 3; ++j) V[u][j] = NAN;
      }
      for (int e = 0; e < 6; ++e) C6[e] = NAN;
    } else {
      const float fc = (float)c;
      float mean[3];
      for (int d = 0; d < 3; ++d) mean[d] = chunked_result(&s1, d) / fc;
      chunked_t s2;
      memset(&s2, 0, sizeof(s2));
      for (int s = 0; s < k; ++s) {
        if (row[s] < 0) continue;
        const float* p = points + (int64_t)row[s] * stride;
        float e[3], t[6];
        for (int d = 0; d < 3; ++d) e[d] = p[d] - mean[d];
        t[0] = e[0] * e[0];
        t[1] = e[0] * e[1];
        t[2] = e[0] * e[2];
        t[3] = e[1] * e[1];
        t[4] = e[1] * e[2];
        t[5] = e[2] * e[2];
        chunked_add(&s2, t, 6);
      }
      for (int e = 0; e < 6; ++e) C6[e] = chunked_result(&s2, e) / fc;
      float A[3][3] = {{C6[0], C6[1], C6[2]}, {C6[1], C6[3], C6[4]}, {C6[2], C6[4], C6[5]}};
      for (int u = 0; u < 3; ++u)
        for (int j = 0; j < 3; ++j) V[u][j] = u == j ? 1.0f : 0.0f;
      while (used < 8 && !(A[0][1] == 0.0f && A[0][2] == 0.0f && A[1][2] == 0.0f)) {
        rotate(A, V, 0, 1);
        rotate(A, V, 0, 2);
        rotate(A, V, 1, 2);
        ++used;
      }
      for (int u = 0; u < 3; ++u) w[u] = A[u][u];
      compare_exchange(w, V, 0, 1);
      compare_exchange(w, V, 1, 2);
      compare_exchange(w, V, 0, 1);
      if (disambiguate) {
        const float* a = points + (int64_t)first * stride;
        for (int col = 0; col <= 2; col += 2) {
          int pos = 0;
          for (int s = 0; s < k; ++s) {
            if (row[s] < 0) continue;
            const float* p = points + (int64_t)row[s] * stride;
            const float f0 = p[0] - a[0], f1 = p[1] - a[1], f2 = p[2] - a[2];
            const float dot = (V[0][col] * f0 + V[1][col] * f1) + V[2][col] * f2;
            if (dot > 0.0f) ++pos;
          }
          if (2 * pos < c)
            for (int u = 0; u < 3; ++u) V[u][col] = -V[u][col];
        }
        const float n0 = V[0][0], n1 = V[1][0], n2 = V[2][0], z0 = V[0][2], z1 = V[1][2], z2 = V[2][2];
        V[0][1] = n1 * z2 - n2 * z1;
        V[1][1] = n2 * z0 - n0 * z2;
        V[2][1] = n0 * z1 - n1 * z0;
      }
    }
    if (eig)
      for (int j = 0; j < 3; ++j) eig[i * 3 + j] = w[j];
    if (frames)
      for (int u = 0; u < 3; ++u)
        for (int j = 0; j < 3; ++j) frames[i * 9 + u * 3 + j] = V[u][j];
    if (cov)
      for (int e = 0; e < 6; ++e) cov[i * 6 + e] = C6[e];
    if (sweeps) sweeps[i] = used;
  }
}
