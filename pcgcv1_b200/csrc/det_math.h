// Bit-reproducible float32 math shared by the CUDA kernels (entropy.cu, gpu_coder.cu) and the host half of the library
// (coder.cpp): every operation is a single correctly rounded IEEE-754 binary32 add / sub / mul / div, rintf or an integer
// bit manipulation -- no FMA contraction, no libm / libdevice transcendental -- so the SAME inputs give the SAME bits on
// sm_100a and on any x86-64 / aarch64 host.  This is what makes a stream written with GPU-built CDF tables decodable on a
// CPU (and the other way round): models/conditional_entropy_model.py:95-124 and models/entropy_model.py:183-221 build the
// integer CDFs from float likelihoods, so one differing ulp in exp() can move a 16-bit table entry.
//
// Accuracy (vs the correctly rounded function): det_expf <= 2 ulp for x <= 0, det_tanhf <= 4e-7 relative, both far inside the
// 1e-3 relative tolerance north_star sets for likelihoods; the operation ORDER of the likelihood formulas is the reference's.
#pragma once
#include <math.h>
#include <stdint.h>
#include <string.h>

#if defined(__CUDACC__)
#define PCGC_DET __host__ __device__ __forceinline__
#else
#define PCGC_DET inline
#endif

namespace pcgc {

// ---- single IEEE operations that no compiler pass may fuse ------------------------------------------------------------
#if defined(__CUDA_ARCH__)
PCGC_DET float d_add(float a, float b) { return __fadd_rn(a, b); }
PCGC_DET float d_sub(float a, float b) { return __fadd_rn(a, -b); }
PCGC_DET float d_mul(float a, float b) { return __fmul_rn(a, b); }
PCGC_DET float d_div(float a, float b) { return __fdiv_rn(a, b); }
#else
// host: volatile keeps the optimiser from contracting a*b+c into an FMA on targets that have one (-march=native builds)
PCGC_DET float d_add(float a, float b) { volatile float r = a + b; return r; }
PCGC_DET float d_sub(float a, float b) { volatile float r = a - b; return r; }
PCGC_DET float d_mul(float a, float b) { volatile float r = a * b; return r; }
PCGC_DET float d_div(float a, float b) { volatile float r = a / b; return r; }
#endif

PCGC_DET float d_bits(uint32_t u) {
#if defined(__CUDA_ARCH__)
  return __uint_as_float(u);
#else
  float f; memcpy(&f, &u, 4); return f;
#endif
}

// exp(x), any x (the entropy models only call it with x <= 0 or |x| small).  x = k ln2 + r, |r| <= ln2/2 (Cody-Waite with
// a 16-bit ln2_hi so k*ln2_hi is exact), degree-7 Taylor polynomial in plain mul/add, scaled by 2^k through the exponent
// field; results below FLT_MIN are produced by ONE final rounding multiply, so denormals agree bit for bit as well.
PCGC_DET float det_expf(float x) {
  if (x != x) return x;
  if (x > 88.72f) return d_bits(0x7F800000u);        // +inf
  if (x < -104.0f) return 0.0f;
  const float kf = rintf(d_mul(x, 1.44269504088896341f));
  float r = d_sub(x, d_mul(kf, 0.693145751953125f));             // exact product (kf has <= 8 bits, ln2_hi 16)
  r = d_sub(r, d_mul(kf, 1.42860682030941723212e-6f));
  float p = 1.0f / 5040.0f;
  p = d_add(d_mul(p, r), 1.0f / 720.0f);
  p = d_add(d_mul(p, r), 1.0f / 120.0f);
  p = d_add(d_mul(p, r), 1.0f / 24.0f);
  p = d_add(d_mul(p, r), 1.0f / 6.0f);
  p = d_add(d_mul(p, r), 0.5f);
  p = d_add(d_mul(p, r), 1.0f);
  p = d_add(d_mul(p, r), 1.0f);
  int k = (int)kf;
  if (k > 127) { p = d_mul(p, 2.0f); k -= 1; }                    // x in (88.03, 88.72]: 2^128 is not a float
  if (k >= -126) return d_mul(p, d_bits((uint32_t)(k + 127) << 23));
  // k in [-151, -127]: p * 2^(k+100) is exact (normal), the last multiply rounds once into the denormal range
  return d_mul(d_mul(p, d_bits((uint32_t)(k + 100 + 127) << 23)), d_bits((uint32_t)(127 - 100) << 23));
}

// tanh(t): odd polynomial near 0, 1 - 2/(e^{2|t|}+1) elsewhere.
PCGC_DET float det_tanhf(float t) {
  if (t != t) return t;
  const float a = fabsf(t);
  if (a < 0.25f) {
    const float s = d_mul(t, t);
    float p = 62.0f / 2835.0f;
    p = d_add(d_mul(p, s), -17.0f / 315.0f);
    p = d_add(d_mul(p, s), 2.0f / 15.0f);
    p = d_add(d_mul(p, s), -1.0f / 3.0f);
    p = d_add(d_mul(p, s), 1.0f);
    return d_mul(t, p);
  }
  if (a > 12.0f) return t > 0.f ? 1.0f : -1.0f;
  const float e = det_expf(d_mul(2.0f, a));
  const float v = d_sub(1.0f, d_div(2.0f, d_add(e, 1.0f)));
  return t > 0.f ? v : -v;
}

PCGC_DET float det_sigmoidf(float x) { return d_div(1.0f, d_add(1.0f, det_expf(-x))); }
PCGC_DET float det_signf(float x) { return (x > 0.f) ? 1.f : ((x < 0.f) ? -1.f : 0.f); }

// ---- SymmetricConditional (models/conditional_entropy_model.py:21-56): LAPLACE cdf / likelihood, operation for operation ----
PCGC_DET float det_laplace_cdf(float t, float loc, float scale) {
  const float e = det_expf(d_div(-fabsf(d_sub(t, loc)), scale));
  const float c_l = d_mul(0.5f, e);
  const float c_r = d_sub(1.0f, c_l);
  return (t <= loc) ? c_l : ((t > loc) ? c_r : 0.f);          // NaN: both masks false -> 0 like the reference
}
PCGC_DET float det_laplace_likelihood(float x, float loc, float scale) {
  float upper = d_add(x, 0.5f), lower = d_sub(x, 0.5f);
  const float sgn = det_signf(d_sub(d_add(upper, lower), loc));   // sign(2x - loc): the reference's quirk (:47)
  upper = d_add(d_mul(-sgn, d_sub(upper, loc)), loc);
  lower = d_add(d_mul(-sgn, d_sub(lower, loc)), loc);
  return fabsf(d_sub(det_laplace_cdf(upper, loc, scale), det_laplace_cdf(lower, loc, scale)));
}

// The likelihoods of the CONSECUTIVE integers min_v .. min_v + n - 1 (SymmetricConditional._get_cdf, :95-124), each floored at
// `bound`: out[k] == max(det_laplace_likelihood(min_v + k, loc, scale), bound) bit for bit, with about half the exp() calls.
// Symbol k's upper edge and symbol k+1's lower edge are the same float (k + 1/2 is exact), and the reflected argument
// -s (t - loc) + loc only depends on the edge and on s = sign(2x - loc); s changes at most twice along the row, so the cdf at
// the upper edge of one symbol is re-used as the cdf at the lower edge of the next whenever their signs agree.
PCGC_DET void det_laplace_pmf_row(int min_v, int n, float loc, float scale, float bound, float* out, int st = 1) {
  float s_prev = 2.0f, c_prev = 0.0f;                          // no sign equals 2: the first symbol evaluates both edges
  for (int k = 0; k < n; ++k) {
    const float x = (float)(min_v + k);
    const float upper = d_add(x, 0.5f), lower = d_sub(x, 0.5f);
    const float sgn = det_signf(d_sub(d_add(upper, lower), loc));
    const float c_lo = (sgn == s_prev) ? c_prev : det_laplace_cdf(d_add(d_mul(-sgn, d_sub(lower, loc)), loc), loc, scale);
    const float c_up = det_laplace_cdf(d_add(d_mul(-sgn, d_sub(upper, loc)), loc), loc, scale);
    const float p = fabsf(d_sub(c_up, c_lo));
    out[k * st] = p > bound ? p : bound;                         // fmaxf(p, bound), NaN -> bound like fmaxf
    s_prev = sgn; c_prev = c_up;
  }
}

// ---- EntropyBottleneck (models/entropy_model.py:72-151) for filters (3,3,3) ------------------------------------------------
// p: 44 floats per channel as packed by pcgc_load_bottleneck: softplus(matrix), bias, tanh(factor) per layer.
PCGC_DET float det_bn_logits(float x, const float* p) {
  float h[3], g[3];
  for (int j = 0; j < 3; ++j) {               // layer 0: [3,1]
    const float t = d_add(d_mul(p[j], x), p[3 + j]);
    h[j] = d_add(t, d_mul(p[6 + j], det_tanhf(t)));
  }
  const float* q = p + 9;
  for (int l = 0; l < 2; ++l) {               // layers 1,2: [3,3]
    for (int j = 0; j < 3; ++j) {
      float t = d_mul(q[3 * j], h[0]);
      t = d_add(t, d_mul(q[3 * j + 1], h[1]));
      t = d_add(t, d_mul(q[3 * j + 2], h[2]));
      t = d_add(t, q[9 + j]);
      g[j] = d_add(t, d_mul(q[12 + j], det_tanhf(t)));
    }
    h[0] = g[0]; h[1] = g[1]; h[2] = g[2];
    q += 15;
  }
  float t = d_mul(q[0], h[0]);                // layer 3: [1,3]
  t = d_add(t, d_mul(q[1], h[1]));
  t = d_add(t, d_mul(q[2], h[2]));
  t = d_add(t, q[3]);
  return d_add(t, d_mul(q[4], det_tanhf(t)));
}
// _likelihood (entropy_model.py:131-139) at an already quantised value.
PCGC_DET float det_bn_likelihood(float xq, const float* p) {
  const float lower = det_bn_logits(d_sub(xq, 0.5f), p);
  const float upper = det_bn_logits(d_add(xq, 0.5f), p);
  const float sgn = -det_signf(d_add(lower, upper));
  return fabsf(d_sub(det_sigmoidf(d_mul(sgn, upper)), det_sigmoidf(d_mul(sgn, lower))));
}

}  // namespace pcgc
