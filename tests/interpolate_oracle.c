/*
 * interpolate_oracle.c — CPU reference of tknn_interpolate / tknn_interpolate_backward (test infrastructure only;
 * never loaded by the library).
 *
 * The contract (include/trueknn.h), literally, in fp32 (-ffp-contract=off, so every operation rounds on its own):
 *   w = 1 / max(d2, 1e-16) per filled slot (+0 for idx = -1), den = sum of w in slot order from +0,
 *   out = (sum in slot order from +0 of x[idx] * w) / den;
 *   grad_x[j] = sum over the edges e = i * k + s with idx[i, s] = j in ascending e, from +0, of (grad_out[i] / den[i]) * w[e].
 * Build: gcc -O2 -std=gnu11 -fPIC -ffp-contract=off -shared -o libinterpolate_oracle.so interpolate_oracle.c
 */
#include <stdint.h>
#include <string.h>

/* x: n rows of pitch xs; out: nq x f; w: nq x k; den: nq */
__attribute__((visibility("default"))) void tki_forward(const int32_t* idx, const float* d2, int64_t nq, int k,
                                                       const float* x, int f, int xs, float* out, float* w, float* den) {
  for (int64_t i = 0; i < nq; ++i) {
    float dsum = 0.0f;
    for (int s = 0; s < k; ++s) {
      const int64_t e = i * k + s;
      float ws = 0.0f;
      if (idx[e] >= 0) {
        const float d = d2[e] < 1e-16f ? 1e-16f : d2[e]; /* NaN stays NaN, as torch.clamp */
        ws = 1.0f / d;
        dsum = dsum + ws;
      }
      w[e] = ws;
    }
    den[i] = dsum;
    for (int c = 0; c < f; ++c) {
      float num = 0.0f;
      for (int s = 0; s < k; ++s) {
        const int64_t e = i * k + s;
        if (idx[e] >= 0) {
          const float p = x[(int64_t)idx[e] * xs + c] * w[e];
          num = num + p;
        }
      }
      out[i * f + c] = num / dsum;
    }
  }
}

/* grad: nq rows of pitch gs; gx: n x f */
__attribute__((visibility("default"))) void tki_backward(const int32_t* idx, const float* w, const float* den, int64_t nq,
                                                        int k, const float* grad, int gs, int64_t n, int f, float* gx) {
  memset(gx, 0, sizeof(float) * (size_t)n * (size_t)f);
  for (int64_t e = 0; e < nq * k; ++e) {
    const int32_t j = idx[e];
    if (j < 0) continue;
    const int64_t i = e / k;
    for (int c = 0; c < f; ++c) {
      const float q = grad[i * gs + c] / den[i];
      const float p = q * w[e];
      gx[(int64_t)j * f + c] = gx[(int64_t)j * f + c] + p;
    }
  }
}
