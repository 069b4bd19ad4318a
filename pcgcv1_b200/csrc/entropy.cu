// Fused, HBM-bound entropy-model kernels (sm_100a).
//   factorized:  models/entropy_model.py:72-181  (quantise + per-channel 1-3-3-3-1 density + bits + min/max)
//   conditional: models/conditional_entropy_model.py:21-124 (quantise + LAPLACE likelihood + bits +
//                per-cube min/max; per-element quantised CDF rows / symbol intervals for the coder)
// The arithmetic follows the reference's operation order in FP32 with the bit-reproducible exp / tanh of det_math.h (shared
// with the host half of the library; this file must NOT be compiled with --use_fast_math).  Reductions are two-stage with a fixed order
// (block partials -> one finalising block), min/max use integer atomics: results are reproducible.
#include <float.h>
#include <limits.h>
#include <stdlib.h>

#include "cdf_norm.h"
#include "common.cuh"
#include "det_math.h"
#include "philox.cuh"

namespace pcgc {

constexpr int BN_PARAMS = 44;   // per channel: see api.cu pack_bottleneck()

// The likelihood formulas live in det_math.h (bit-reproducible on host and device): _logits_cumulative / _likelihood of
// entropy_model.py:72-151 and the Laplace cdf / likelihood of conditional_entropy_model.py:21-56.
__device__ __forceinline__ float bn_likelihood(float xq, const float* __restrict__ p) { return det_bn_likelihood(xq, p); }
__device__ __forceinline__ float laplace_likelihood(float x, float loc, float scale) { return det_laplace_likelihood(x, loc, scale); }

// ---------------------------------------------------------------------------------------------
__global__ void init_minmax_kernel(int32_t* mm, int n_pairs) {
  int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n_pairs) { mm[2 * i] = INT_MAX; mm[2 * i + 1] = INT_MIN; }
}

// Per-cube symbol ranges made codable and storable: the range gets 0 inside it (the .strings_head byte packs max*16 - min with
// min <= 0 <= max, inout_bitstream.py:95-96) and at least two symbols (pmf_to_quantized_cdf rejects a one-symbol alphabet,
// entropy_model.py:192-193).  The decoder builds its tables from the header's (min, max) alone, so the stream stays readable.
__global__ void widen_minmax_kernel(int32_t* mm, int n_pairs) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n_pairs) return;
  int lo = min(mm[2 * i], 0), hi = max(mm[2 * i + 1], 0);
  if (lo == hi) hi = 1;
  mm[2 * i] = lo; mm[2 * i + 1] = hi;
}

cudaError_t launch_widen_minmax(int32_t* minmax, int n_pairs, cudaStream_t s, int64_t* launches) {
  if (n_pairs <= 0) return cudaSuccess;
  widen_minmax_kernel<<<(n_pairs + 127) / 128, 128, 0, s>>>(minmax, n_pairs);
  if (launches) ++*launches;
  return cudaGetLastError();
}

struct BlockStats { double bits; int mn, mx; };

template <int THREADS>
__device__ __forceinline__ BlockStats block_reduce(double bits, int mn, int mx) {
  __shared__ double s_b[THREADS / 32];
  __shared__ int s_mn[THREADS / 32], s_mx[THREADS / 32];
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    bits += __shfl_down_sync(0xffffffffu, bits, o);
    mn = min(mn, __shfl_down_sync(0xffffffffu, mn, o));
    mx = max(mx, __shfl_down_sync(0xffffffffu, mx, o));
  }
  const int w = threadIdx.x >> 5, l = threadIdx.x & 31;
  if (l == 0) { s_b[w] = bits; s_mn[w] = mn; s_mx[w] = mx; }
  __syncthreads();
  BlockStats r{0.0, INT_MAX, INT_MIN};
  if (threadIdx.x == 0) {
    for (int i = 0; i < THREADS / 32; ++i) { r.bits += s_b[i]; r.mn = min(r.mn, s_mn[i]); r.mx = max(r.mx, s_mx[i]); }
  }
  return r;
}

// Final, fixed-order sum of per-block partials: out[g] = sum_j partial[g*per + j].
__global__ void finalize_bits_kernel(const double* __restrict__ partial, int per, double* __restrict__ out) {
  const int g = blockIdx.x;
  if (threadIdx.x == 0) {
    double s = 0.0;
    for (int j = 0; j < per; ++j) s += partial[(size_t)g * per + j];
    out[g] = s;
  }
}

constexpr int ENT_THREADS = 256;
constexpr int ENT_VEC = 4;

// ---- factorized: one thread = 4 consecutive elements (C % 4 == 0 => 4 consecutive channels) ----
__global__ void __launch_bounds__(ENT_THREADS)
factorized_kernel(const float* __restrict__ x, int64_t n, int C, const float* __restrict__ params, float bound,
                  float* __restrict__ x_hat, float* __restrict__ p_out, double* __restrict__ partial,
                  int32_t* __restrict__ minmax, int noise, uint64_t seed) {
  extern __shared__ float s_par[];
  for (int i = threadIdx.x; i < C * BN_PARAMS; i += ENT_THREADS) s_par[i] = params[i];
  __syncthreads();
  double bits = 0.0;
  int mn = INT_MAX, mx = INT_MIN;
  const int64_t nvec = n / ENT_VEC;
  for (int64_t v = (int64_t)blockIdx.x * ENT_THREADS + threadIdx.x; v < nvec; v += (int64_t)gridDim.x * ENT_THREADS) {
    const float4 xv = __ldg(reinterpret_cast<const float4*>(x) + v);
    float xs[4] = {xv.x, xv.y, xv.z, xv.w}, q[4], pr[4];
    const int c0 = (int)((v * ENT_VEC) % C);
    float u[4] = {0.f, 0.f, 0.f, 0.f};
    if (noise) noise4(seed, (uint64_t)v, u);
#pragma unroll
    for (int k = 0; k < 4; ++k) {
      q[k] = noise ? xs[k] + u[k] : rintf(xs[k]);                 // "noise" (:105-107) | tf.math.round: half to even
      pr[k] = fmaxf(bn_likelihood(q[k], s_par + (c0 + k) * BN_PARAMS), bound);
      bits -= (double)log2f(pr[k]);
      const int qi = (int)q[k];
      mn = min(mn, qi); mx = max(mx, qi);
    }
    if (x_hat) reinterpret_cast<float4*>(x_hat)[v] = make_float4(q[0], q[1], q[2], q[3]);
    if (p_out) reinterpret_cast<float4*>(p_out)[v] = make_float4(pr[0], pr[1], pr[2], pr[3]);
  }
  const BlockStats r = block_reduce<ENT_THREADS>(bits, mn, mx);
  if (threadIdx.x == 0) {
    if (partial) partial[blockIdx.x] = r.bits;
    if (minmax && r.mn <= r.mx) { atomicMin(minmax, r.mn); atomicMax(minmax + 1, r.mx); }
  }
}

cudaError_t launch_factorized(const BottleneckDev& bn, const float* x, int64_t n_vox, int C, float bound,
                              float* x_hat, float* p, double* bits, int32_t* minmax, double* scratch,
                              cudaStream_t s, int64_t* launches, int noise, uint64_t seed) {
  const int64_t n = n_vox * C;
  if (C % 4 != 0 || C != bn.channels) return cudaErrorInvalidValue;
  int64_t want = (n / ENT_VEC + ENT_THREADS - 1) / ENT_THREADS;
  const int blocks = (int)(want < 1 ? 1 : (want > 148 * 8 ? 148 * 8 : want));
  PCGC_CARVEOUT_ONCE(init_minmax_kernel); PCGC_CARVEOUT_ONCE(factorized_kernel); PCGC_CARVEOUT_ONCE(finalize_bits_kernel);
  if (minmax) { init_minmax_kernel<<<1, 32, 0, s>>>(minmax, 1); if (launches) ++*launches; }
  factorized_kernel<<<blocks, ENT_THREADS, C * BN_PARAMS * sizeof(float), s>>>(x, n, C, bn.params, bound, x_hat, p,
                                                                              bits ? scratch : nullptr, minmax, noise, seed);
  if (launches) ++*launches;
  if (bits) { finalize_bits_kernel<<<1, 32, 0, s>>>(scratch, blocks, bits); if (launches) ++*launches; }
  return cudaGetLastError();
}

// pmf of EntropyBottleneck._get_cdf (:195-215): [C, N] likelihoods of the integers min_v..max_v.
__global__ void factorized_pmf_kernel(const float* __restrict__ params, int C, int min_v, int N, float bound,
                                      float* __restrict__ pmf) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= C * N) return;
  const int c = i / N, k = i - c * N;
  pmf[i] = fmaxf(bn_likelihood((float)(min_v + k), params + c * BN_PARAMS), bound);
}

cudaError_t launch_factorized_pmf(const BottleneckDev& bn, int min_v, int max_v, float bound, float* pmf,
                                  cudaStream_t s, int64_t* launches) {
  const int N = max_v - min_v + 1;
  const int tot = bn.channels * N;
  PCGC_CARVEOUT_ONCE(factorized_pmf_kernel);
  factorized_pmf_kernel<<<(tot + 127) / 128, 128, 0, s>>>(bn.params, bn.channels, min_v, N, bound, pmf);
  if (launches) ++*launches;
  return cudaGetLastError();
}

// ---- conditional: grid (blocks_per_cube, B); per-cube min/max and bits ------------------------
__global__ void __launch_bounds__(ENT_THREADS)
laplace_kernel(const float* __restrict__ y, const float* __restrict__ loc, const float* __restrict__ scale,
               int64_t E, float bound, float* __restrict__ y_hat, float* __restrict__ p_out,
               double* __restrict__ partial, int32_t* __restrict__ minmax, int noise, uint64_t seed) {
  const int b = blockIdx.y;
  const size_t base = (size_t)b * E;
  double bits = 0.0;
  int mn = INT_MAX, mx = INT_MIN;
  const int64_t nvec = E / ENT_VEC;
  for (int64_t v = (int64_t)blockIdx.x * ENT_THREADS + threadIdx.x; v < nvec; v += (int64_t)gridDim.x * ENT_THREADS) {
    const size_t o = base / ENT_VEC + v;
    const float4 yv = __ldg(reinterpret_cast<const float4*>(y) + o);
    const float4 lv = __ldg(reinterpret_cast<const float4*>(loc) + o);
    const float4 sv = __ldg(reinterpret_cast<const float4*>(scale) + o);
    const float ys[4] = {yv.x, yv.y, yv.z, yv.w}, ls[4] = {lv.x, lv.y, lv.z, lv.w}, ss[4] = {sv.x, sv.y, sv.z, sv.w};
    float q[4], pr[4], u[4] = {0.f, 0.f, 0.f, 0.f};
    if (noise) noise4(seed, (uint64_t)o, u);
#pragma unroll
    for (int k = 0; k < 4; ++k) {
      q[k] = noise ? ys[k] + u[k] : rintf(ys[k]);               // "noise" (conditional_entropy_model.py:62-64) | round
      pr[k] = fmaxf(laplace_likelihood(q[k], ls[k], ss[k]), bound);
      bits -= (double)log2f(pr[k]);
      const int qi = (int)q[k];
      mn = min(mn, qi); mx = max(mx, qi);
    }
    if (y_hat) reinterpret_cast<float4*>(y_hat)[o] = make_float4(q[0], q[1], q[2], q[3]);
    if (p_out) reinterpret_cast<float4*>(p_out)[o] = make_float4(pr[0], pr[1], pr[2], pr[3]);
  }
  const BlockStats r = block_reduce<ENT_THREADS>(bits, mn, mx);
  if (threadIdx.x == 0) {
    if (partial) partial[(size_t)b * gridDim.x + blockIdx.x] = r.bits;
    if (minmax && r.mn <= r.mx) { atomicMin(minmax + 2 * b, r.mn); atomicMax(minmax + 2 * b + 1, r.mx); }
  }
}

cudaError_t launch_laplace(const float* y, const float* loc, const float* scale, int B, int64_t E, float bound,
                           float* y_hat, float* p, double* bits, int32_t* minmax, double* scratch, cudaStream_t s,
                           int64_t* launches, int noise, uint64_t seed) {
  if (E % ENT_VEC != 0) return cudaErrorInvalidValue;
  int64_t per = (E / ENT_VEC + ENT_THREADS - 1) / ENT_THREADS;
  if (per > 16) per = 16;                          // 16 blocks x 256 threads x 4 elements x 4 iterations per cube
  PCGC_CARVEOUT_ONCE(init_minmax_kernel); PCGC_CARVEOUT_ONCE(laplace_kernel); PCGC_CARVEOUT_ONCE(finalize_bits_kernel);
  if (minmax) { init_minmax_kernel<<<(B + 127) / 128, 128, 0, s>>>(minmax, B); if (launches) ++*launches; }
  dim3 grid((unsigned)per, (unsigned)B);
  laplace_kernel<<<grid, ENT_THREADS, 0, s>>>(y, loc, scale, E, bound, y_hat, p, bits ? scratch : nullptr, minmax, noise, seed);
  if (launches) ++*launches;
  if (bits) { finalize_bits_kernel<<<B, 32, 0, s>>>(scratch, (int)per, bits); if (launches) ++*launches; }
  return cudaGetLastError();
}

// ---- per-element quantised CDF rows (SymmetricConditional._get_cdf, :95-124) -------------------
// One thread per element: pmf over min_v..max_v -> quantize_pmf_row (cdf_norm.h, shared with the host) -> cumulative
// sums.  MODE 0: uint16 rows for the decoder, 1: the interval of the element's own symbol for the encoder,
// 2: test hook (pmf given, int32 cdf rows out).
// r01 note: an 8-lanes-per-row variant (all state in registers, shuffle reductions) was measured 2x SLOWER on the real
// symbol ranges (N = 5..12): most lanes idle and every greedy step pays 9 shuffles.  The cost that mattered was the
// water-filling pass of the few heavy-tail rows that almost every warp contains; it is now a closed form (cdf_last_u).
// r02 experiment, kept as a note: moving the three per-row arrays (pmf, counts, scores) from per-thread local memory (38 M local
// loads per 64 cubes at a 10 % L1 hit rate, ncu) into shared memory interleaved over the block ([entry][thread], 48 KiB per 128
// threads) made the kernel SLOWER (3.78 -> 4.90 ms per 191 cubes): 16 instead of 32 resident warps hide the exp / FP64 latencies
// of the normaliser worse than the L2 hits of the local arrays cost.  Keeping them in registers instead (NMAX-wide predicated loops,
// select subscripts, no local memory) was slower still (5.57 against 3.36 ms per 191 cubes): the kernel is bound by instruction
// issue, and that form executes about twice the instructions.
constexpr int CDF_THREADS = 128;
template <int MODE>
__global__ void __launch_bounds__(CDF_THREADS, 12)
laplace_cdf_kernel(const float* __restrict__ y_hat, const float* __restrict__ loc, const float* __restrict__ scale,
                   const float* __restrict__ pmf_in, int64_t E, const int32_t* __restrict__ minmax,
                   const int64_t* __restrict__ row_offset, float bound, int precision, uint32_t* __restrict__ intervals,
                   uint16_t* __restrict__ cdf, int32_t* __restrict__ cdf32, int* __restrict__ err) {
  const int b = blockIdx.y;
  const int min_v = minmax[2 * b], max_v = minmax[2 * b + 1];
  const int N = max_v - min_v + 1;
  if (N < 2 || N > PCGC_MAX_SYMBOLS) { if (threadIdx.x == 0 && blockIdx.x == 0) atomicExch(err, PCGC_ERR_BAD_RANGE); return; }
  float pmf[PCGC_MAX_SYMBOLS];
  int32_t v[PCGC_MAX_SYMBOLS];
  float g[PCGC_MAX_SYMBOLS];
  for (int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; e < E; e += (int64_t)gridDim.x * blockDim.x) {
    const size_t o = (size_t)b * E + e;
    if (MODE == 2) {
      for (int k = 0; k < N; ++k) pmf[k] = __ldg(pmf_in + o * N + k);
    } else {
      const float l = __ldg(loc + o), s = __ldg(scale + o);
      det_laplace_pmf_row(min_v, N, l, s, bound, pmf);         // == max(laplace_likelihood(min_v + k), bound), shared edge evaluations
    }
    if (quantize_pmf_row(pmf, N, precision, v, g) != 0) { atomicExch(err, PCGC_ERR_BAD_RANGE); continue; }
    if (MODE == 1) {
      const int sym = (int)__ldg(y_hat + o) - min_v;
      if (sym < 0 || sym >= N) { atomicExch(err, PCGC_ERR_BAD_RANGE); intervals[o] = 0; continue; }
      uint32_t lower = 0;
      for (int k = 0; k < sym; ++k) lower += (uint32_t)v[k];
      intervals[o] = lower | ((uint32_t)(v[sym] - 1) << 16);
    } else if (MODE == 0) {
      uint16_t* row = cdf + row_offset[b] + (size_t)e * N;
      uint32_t acc = 0;
      for (int k = 0; k < N; ++k) { row[k] = (uint16_t)acc; acc += (uint32_t)v[k]; }
    } else {
      int32_t* row = cdf32 + o * (N + 1);
      int32_t acc = 0;
      for (int k = 0; k < N; ++k) { row[k] = acc; acc += v[k]; }
      row[N] = acc;
    }
  }
}

// The shared carveout of the rest of the library leaves these kernels ~28 KB of L1 for their local arrays; the all-L1 carveout made
// them faster alone but gained nothing inside the step (r02, profiles/r02_ncu_cdf_last.txt).
template <int MODE>
static cudaError_t cdf_prepare() {
  static const cudaError_t once = [] {
    prefer_shared_carveout(laplace_cdf_kernel<MODE>);
    return cudaFuncSetAttribute(laplace_cdf_kernel<MODE>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)(96 * 1024));
  }();
  return once;
}

static inline dim3 cdf_grid(int64_t E, int B) {
  int64_t gx = (E + CDF_THREADS - 1) / CDF_THREADS;
  if (gx > 2048) gx = 2048;
  return dim3((unsigned)gx, (unsigned)B);
}

cudaError_t launch_laplace_intervals(const float* y_hat, const float* loc, const float* scale, int B, int64_t E,
                                     const int32_t* minmax, float bound, int precision, uint32_t* intervals,
                                     int* err_flag, cudaStream_t s, int64_t* launches) {
  cudaError_t pe = cdf_prepare<1>();
  if (pe != cudaSuccess) return pe;
  laplace_cdf_kernel<1><<<cdf_grid(E, B), CDF_THREADS, 0, s>>>(y_hat, loc, scale, nullptr, E, minmax, nullptr, bound, precision,
                                                               intervals, nullptr, nullptr, err_flag);
  if (launches) ++*launches;
  return cudaGetLastError();
}

cudaError_t launch_laplace_cdf(const float* loc, const float* scale, int B, int64_t E, const int32_t* minmax_dev,
                               const int64_t* row_offset_dev, float bound, int precision, uint16_t* cdf,
                               int* err_flag, cudaStream_t s, int64_t* launches) {
  cudaError_t pe = cdf_prepare<0>();
  if (pe != cudaSuccess) return pe;
  laplace_cdf_kernel<0><<<cdf_grid(E, B), CDF_THREADS, 0, s>>>(nullptr, loc, scale, nullptr, E, minmax_dev, row_offset_dev, bound,
                                                               precision, nullptr, cdf, nullptr, err_flag);
  if (launches) ++*launches;
  return cudaGetLastError();
}

// pmf [rows, N] (device) -> int32 cdf [rows, N+1] with the device copy of the normaliser (test hook).  minmax_dev = {0, N-1}.
cudaError_t launch_debug_quantize_pmf(const float* pmf, int64_t rows, const int32_t* minmax_dev, int precision,
                                      int32_t* cdf32, int* err_flag, cudaStream_t s, int64_t* launches) {
  cudaError_t pe = cdf_prepare<2>();
  if (pe != cudaSuccess) return pe;
  laplace_cdf_kernel<2><<<cdf_grid(rows, 1), CDF_THREADS, 0, s>>>(nullptr, nullptr, nullptr, pmf, rows, minmax_dev, nullptr, 0.f,
                                                                  precision, nullptr, nullptr, cdf32, err_flag);
  if (launches) ++*launches;
  return cudaGetLastError();
}

}  // namespace pcgc

// Test hook (host): the noise of elements 4*v .. 4*v+3 exactly as the kernels draw it.
extern "C" int pcgc_debug_noise(uint64_t seed, uint64_t v, float* out4) {
  if (!out4) return PCGC_ERR_BAD_ARG;
  pcgc::noise4(seed, v, out4);
  return PCGC_OK;
}
