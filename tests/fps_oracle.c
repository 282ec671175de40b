/*
 * fps_oracle.c — CPU reference of tknn_fps (test infrastructure only; never loaded by the library).
 *
 * The contract (include/trueknn.h), literally, per segment: D(p) = +inf; sample 0 = start; after each sample c every
 * point of the segment takes D(p) = min(D(p), d2(c, p)) with the project's one distance rule
 * d2 = fmaf(dz, dz, fmaf(dy, dy, dx * dx)) in fp32 (dx = c - p); the next sample maximises the u64 key
 * (bits(D) << 32) | (0xFFFFFFFF - index), i.e. the largest D with ties to the lowest index.
 *
 * Segments of at most SERIAL_MAX points run one per thread; larger ones run one at a time with the update and the
 * argmax parallel over points.  `limit` (>= 0) stops every segment after that many samples: the sequence for m samples
 * is the prefix of the sequence for more, so large clouds can be checked on their first samples.
 * Build: gcc -O2 -std=gnu11 -fPIC -fopenmp -ffp-contract=off -shared -o libfps_oracle.so fps_oracle.c -lm
 */
#include <math.h>
#include <stdint.h>
#include <stdlib.h>
#include <string.h>
#ifdef _OPENMP
#include <omp.h>
#endif

#define SERIAL_MAX 65536

static inline float dist2(const float* c, const float* p) {
  const float dx = c[0] - p[0], dy = c[1] - p[1], dz = c[2] - p[2];
  return fmaf(dz, dz, fmaf(dy, dy, dx * dx));
}

static inline uint64_t key_of(float d, int64_t idx) {
  uint32_t b;
  memcpy(&b, &d, 4);
  return ((uint64_t)b << 32) | (uint64_t)(0xFFFFFFFFu - (uint32_t)idx);
}

/* one segment: points [b, e) of xyz, m samples (m >= 1) into idx[0 .. m), d2[0 .. m) (d2[0] = +inf: no sample before) */
static void fps_segment(const float* xyz, int64_t b, int64_t e, int64_t m, int32_t start, float* D, int32_t* idx, float* d2,
                        int parallel) {
  const int64_t n = e - b;
  for (int64_t i = 0; i < n; ++i) D[i] = INFINITY;
  int64_t cur = start;
  idx[0] = start;
  d2[0] = INFINITY;
  for (int64_t s = 1; s < m; ++s) {
    const float* c = xyz + 3 * cur;
    uint64_t best = 0;
    if (parallel) {
#pragma omp parallel
      {
        uint64_t mine = 0;
#pragma omp for schedule(static)
        for (int64_t i = 0; i < n; ++i) {
          const float d = dist2(c, xyz + 3 * (b + i));
          if (d < D[i]) D[i] = d;
          const uint64_t k = key_of(D[i], b + i);
          if (k > mine) mine = k;
        }
#pragma omp critical
        if (mine > best) best = mine;
      }
    } else {
      for (int64_t i = 0; i < n; ++i) {
        const float d = dist2(c, xyz + 3 * (b + i));
        if (d < D[i]) D[i] = d;
        const uint64_t k = key_of(D[i], b + i);
        if (k > best) best = k;
      }
    }
    cur = (int64_t)(0xFFFFFFFFu - (uint32_t)best);
    const uint32_t hb = (uint32_t)(best >> 32);
    idx[s] = (int32_t)cur;
    memcpy(&d2[s], &hb, 4);
  }
}

__attribute__((visibility("default"))) int tkf_num_threads(void) {
#ifdef _OPENMP
  return omp_get_max_threads();
#else
  return 1;
#endif
}

/* xyz: n x 3; off: n_seg + 1 segment offsets; soff: n_seg + 1 sample offsets; starts: n_seg global indices; limit < 0:
 * all samples, else at most limit per segment.  idx_out / d2_out: soff[n_seg] entries (the skipped tail untouched). */
__attribute__((visibility("default"))) int tkf_fps(const float* xyz, int64_t n, const uint64_t* off, const uint64_t* soff,
                                                   int64_t n_seg, const int32_t* starts, int64_t limit, int32_t* idx_out,
                                                   float* d2_out) {
  if (n < 0 || n_seg < 1 || off[0] != 0 || (int64_t)off[n_seg] != n || soff[0] != 0) return 1;
  int64_t max_small = 0;
  for (int64_t s = 0; s < n_seg; ++s) {
    const int64_t ns = (int64_t)(off[s + 1] - off[s]), m = (int64_t)(soff[s + 1] - soff[s]);
    if (off[s + 1] < off[s] || soff[s + 1] < soff[s] || m > ns) return 1;
    if (m > 0 && (starts[s] < (int64_t)off[s] || starts[s] >= (int64_t)off[s + 1])) return 1;
    if (ns <= SERIAL_MAX && ns > max_small) max_small = ns;
  }
  int bad = 0;
#pragma omp parallel
  {
    float* D = malloc(sizeof(float) * (size_t)(max_small > 0 ? max_small : 1));
    if (!D) {
#pragma omp atomic write
      bad = 1;
    }
#pragma omp for schedule(dynamic, 1)
    for (int64_t s = 0; s < n_seg; ++s) {
      const int64_t ns = (int64_t)(off[s + 1] - off[s]);
      int64_t m = (int64_t)(soff[s + 1] - soff[s]);
      if (limit >= 0 && m > limit) m = limit;
      if (D && m > 0 && ns <= SERIAL_MAX)
        fps_segment(xyz, (int64_t)off[s], (int64_t)off[s + 1], m, starts[s], D, idx_out + soff[s], d2_out + soff[s], 0);
    }
    free(D);
  }
  if (bad) return 2;
  for (int64_t s = 0; s < n_seg; ++s) {
    const int64_t ns = (int64_t)(off[s + 1] - off[s]);
    int64_t m = (int64_t)(soff[s + 1] - soff[s]);
    if (limit >= 0 && m > limit) m = limit;
    if (m == 0 || ns <= SERIAL_MAX) continue;
    float* D = malloc(sizeof(float) * (size_t)ns);
    if (!D) return 2;
    fps_segment(xyz, (int64_t)off[s], (int64_t)off[s + 1], m, starts[s], D, idx_out + soff[s], d2_out + soff[s], 1);
    free(D);
  }
  return 0;
}
