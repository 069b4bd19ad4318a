// pmf -> 16-bit quantised CDF normaliser shared by the host coder (coder.cpp) and the CDF kernels
// (entropy.cu).  Replaces coder_ops.pmf_to_quantized_cdf (call sites models/entropy_model.py:218,
// models/conditional_entropy_model.py:122; upstream tensorflow/contrib/coder/kernels/pmf_to_cdf_op.cc,
// not vendored -- see oracle/coder.py for the restated contract).
//
// Contract (identical to the oracle's greedy definition):
//   v_i = max(rint(pmf_i * 2^precision), 1)
//   sum > target: repeatedly decrement the entry with the smallest penalty
//                 pmf_i*(log2 v_i - log2(v_i-1)), entries at 1 excluded, lowest index on ties;
//   sum < target: repeatedly increment the entry with the largest gain
//                 pmf_i*(log2(v_i+1) - log2 v_i), lowest index on ties.
// The deficit case can need thousands of steps (Laplace tails cut at min_v/max_v), so it is done
// as an exact water-filling: every increment whose gain is >= a threshold lambda that provably
// admits at most `deficit` increments is granted at once (counts verified with exact gain
// evaluations), and only the remainder runs the step-by-step greedy.  Because per-entry gains
// are strictly decreasing, the result equals the step-by-step greedy's.
#pragma once
#include <math.h>
#include <stdint.h>

#if defined(__CUDACC__)
#define PCGC_HD __host__ __device__ __forceinline__
#define PCGC_HD_NOINLINE static __host__ __device__ __noinline__      // big bodies: keep ptxas compile time sane
#else
#define PCGC_HD inline
#define PCGC_HD_NOINLINE inline
#endif

namespace pcgc {

// log2(v+1) - log2(v) for v = 1..32 and ln(1 + 1/v) for v = 1..15 as constants (hex doubles = what glibc's log2 / log1p give):
// one source of truth for host and device, and no libm call on paths that only one or two lanes of a warp take at a time
// (ncu r01: the v < 16 score and the small-u walk of cdf_last_u were 30 percent of the CDF kernels' warp instructions at 1-2
// active lanes).
#if defined(__CUDA_ARCH__)
#define PCGC_TABLE_QUAL __constant__
#else
#define PCGC_TABLE_QUAL
#endif
static PCGC_TABLE_QUAL const double pcgc_gain_tab[33] = {0x0.0p+0, 0x1.0000000000000p+0, 0x1.2b803473f7ad0p-1, 0x1.a8ff971810a60p-2, 0x1.49a784bcd1b88p-2, 0x1.0d58e42b1da18p-2, 0x1.c775ad8425790p-3, 0x1.8a8980abfbd30p-3, 0x1.5c01a39fbd680p-3, 0x1.374d65d9e6090p-3, 0x1.199b728cb9d10p-3, 0x1.011655c981720p-3, 0x1.d8fea38406fe0p-4, 0x1.b5ecb78443f40p-4, 0x1.97b2b7eafbf20p-4, 0x1.7d60496cfbb40p-4, 0x1.663f6fac91300p-4, 0x1.51c3d792e9a00p-4, 0x1.3f7f8fe0d2300p-4, 0x1.2f1b3bd2f9e40p-4, 0x1.20508f547ee00p-4, 0x1.12e655c4f4c00p-4, 0x1.06ad885e62d00p-4, 0x1.f6fe466940280p-5, 0x1.e275048da0b80p-5, 0x1.cf88427a6d400p-5, 0x1.be094776e7a80p-5, 0x1.add02791a0400p-5, 0x1.9eba920522280p-5, 0x1.90aaddd0d5c00p-5, 0x1.8387463c61d80p-5, 0x1.77394c9d95900p-5, 0x1.6bad3758efd80p-5};
static PCGC_TABLE_QUAL const double pcgc_ln1p_tab[16] = {0x0.0p+0, 0x1.62e42fefa39efp-1, 0x1.9f323ecbf984cp-2, 0x1.269621134db92p-2, 0x1.c8ff7c79a9a22p-3, 0x1.7565011e49676p-3, 0x1.3bb35a041d2a9p-3, 0x1.1178e8227e47cp-3, 0x1.e27076e2af2e6p-4, 0x1.af8e8210a415dp-4, 0x1.8663f793c46c7p-4, 0x1.64660aa8ce626p-4, 0x1.47dadcbbdba83p-4, 0x1.2f8bd74c5eacfp-4, 0x1.1a9844eb18ef1p-4, 0x1.08598b59e3a06p-4};

// log2(1 + 1/v) for v > 32 from correctly rounded IEEE operations only.  The first version called log2() twice: glibc's and
// libdevice's log2 differ in the last ulp now and then, the difference log2(v+1) - log2(v) amplifies that to ~1e-10 relative, and
// two entries whose gains are closer than that were ranked differently on host and device (r02: 2 of 5 M rows of the vox10 cloud
// one unit apart).  ln(1 + x) = x (1 - x (1/2 - x (1/3 - ...))), x = 1/v < 1/32: 15 terms leave < 1e-23 relative.  entropy.cu is
// compiled with -fmad=false and the host with -ffp-contract=off, so the same operations run on both sides.
PCGC_HD double cdf_log2_ratio(int v) {
  const double x = 1.0 / (double)v;
  double p = 1.0 / 15.0;
  for (int k = 14; k >= 1; --k) p = 1.0 / (double)k - x * p;
  return (x * p) * 1.4426950408889634;
}

PCGC_HD double cdf_gain(double m, int v) {
  if (v <= 32) return m * pcgc_gain_tab[v];
  return m * cdf_log2_ratio(v);
}

// Float SCORE used to shortlist candidates: score = cdf_gain(m, v) * 2^precision / log2(e) - 1, a strictly increasing
// function of the gain.  All large entries have gains within ~1/v of each other, so the gain itself cannot be ranked
// in float; the score can: with r = m*2^p - v (exact in float) and x = 1/v,
//     score = (v + r) * ln(1 + x) - 1 = P + r*x*(1 + P),   P = -x/2 + x^2/3 - x^3/4 + ...
// is evaluated without cancellation (relative error ~3e-7 OF THE SCORE, i.e. ~1e-12 of the gain).  Entries whose
// scores are within PCGC_SCORE_TOL of the best are re-ranked on the exact double gains, so every decision equals the
// all-double greedy of the oracle.
PCGC_HD float cdf_score(float m, int v, float scale) {
  if (v >= 16) {
    const float x = 1.0f / (float)v, r = m * scale - (float)v;
    const float P = x * (-0.5f + x * (1.0f / 3 + x * (-0.25f + x * (0.2f + x * (-1.0f / 6 + x * (1.0f / 7))))));
    return P + r * x * (1.0f + P);
  }
  return (float)((double)m * (double)scale * pcgc_ln1p_tab[v] - 1.0);
}
#define PCGC_SCORE_TOL(mx) (4e-6f * fabsf(mx) + 1e-9f)

// Largest u >= 1 with cdf_gain(m, u) >= lambda (0 if none), i.e. u <= 1 / (2^(lambda/m) - 1).  Closed form with a short
// exact check only when the bound is within rounding distance of an integer.
PCGC_HD_NOINLINE long long cdf_last_u(double m, double lambda) {
  if (!(m >= lambda)) return 0;                               // gain(m, u) <= gain(m, 1) = m
  const double t = lambda / m * 0.6931471805599453;          // gain >= lambda  <=>  ln(1 + 1/u) >= t
  if (t > 0.05) {                                            // u < 20: walk the few candidates exactly
    long long u = 0;
    while (u < 32 && cdf_gain(m, (int)(u + 1)) >= lambda) ++u;
    return u;
  }
  // expm1(t) by its series (t <= 0.05: truncation error < 1e-15 relative)
  const double em1 = t * (1.0 + t * (0.5 + t * (1.0 / 6 + t * (1.0 / 24 + t * (1.0 / 120 + t * (1.0 / 720 + t * (1.0 / 5040)))))));
  const double U = 1.0 / em1;
  if (U >= 4.0e9) return 4000000000LL;
  long long fu = (long long)U;
  const double frac = U - (double)fu, tol = 1e-9 * U + 1e-9;
  if (frac < tol) { if (!(cdf_gain(m, (int)fu) >= lambda)) --fu; }
  else if (1.0 - frac < tol) { if (cdf_gain(m, (int)(fu + 1)) >= lambda) ++fu; }
  return fu;
}

// pmf[n] -> v[n] (counts, sum == 2^precision).  g: scratch float[n].  Returns 0, or -2 if the row
// cannot be shrunk (all ones and n > target).
//
// One loop serves both directions (dir = +1: grow the entry with the largest gain; dir = -1: shrink the entry with
// the smallest penalty = largest negated gain at v-1) so that the 32 rows of a warp do not serialise two code paths.
PCGC_HD_NOINLINE int quantize_pmf_row(const float* pmf, int n, int precision, int32_t* v, float* g) {
  const int target = 1 << precision;
  const float scale = (float)target;
  long long sum = 0;
  for (int i = 0; i < n; ++i) {
    int q = (int)rintf(pmf[i] * scale);
    q = q < 1 ? 1 : q;
    v[i] = q;
    sum += q;
  }
  long long todo = sum > target ? sum - target : target - sum;
  if (todo == 0) return 0;
  const int dir = sum > target ? -1 : 1;

  // ---- water-filling for large deficits (Laplace tails cut at min_v / max_v: up to thousands of steps) ----
  // Every increment whose gain is >= lambda is granted at once, for a lambda that admits at most `todo` increments;
  // per-entry gains are strictly decreasing, so these are exactly the greedy's first picks.  lambda comes from the
  // continuous solution gain_i(u) ~ m_i*log2(e)/(u + 0.5), aimed a little short so that the pass is feasible.
  // Deficits above n + 2 take this pass, a pure speed choice: both routes give the step-by-step greedy's counts.  On the GPU the
  // threshold is set by the WARP, not by the row: some lane of almost every warp takes the water-filling pass anyway, so what a lower
  // threshold buys is a shorter greedy loop for the slowest lane (r02, 64 cubes of the vox10 cloud, intervals / rows kernel:
  // 2n + 8 -> 1.26 / 1.24 ms, n + 2 -> 1.15 / 1.12 ms, n/2 + 2 -> 1.16 / 1.13 ms, 4 -> 2.10 / 2.05 ms; identical bits).
  for (int pass = 0; pass < 8 && dir > 0 && todo > n + 2; ++pass) {
    const double L = 1.4426950408889634;
    double m_act = 0.0, t_act = (double)target;
    int n_act = n;
    for (int i = 0; i < n; ++i) m_act += (double)pmf[i];
    double inv_lambda = 0.0;
    for (int it = 0; it < 4 && m_act > 0.0; ++it) {           // active set = entries that grow at the solution
      const double slack = 2.0 * sqrt((double)n_act / 12.0) + 1.0;
      inv_lambda = (t_act - slack) / (L * m_act);
      double t2 = (double)target, m2 = 0.0;
      int n2 = 0;
      for (int i = 0; i < n; ++i) {
        if ((double)pmf[i] * L * inv_lambda >= (double)v[i]) { m2 += (double)pmf[i]; ++n2; } else { t2 -= (double)v[i]; }
      }
      if (n2 == n_act && m2 == m_act) break;
      t_act = t2; m_act = m2; n_act = n2;
      if (n2 == 0) break;
    }
    if (!(inv_lambda > 0.0) || n_act == 0) break;
    double lambda = 1.0 / inv_lambda;
    bool done = false;
    for (int attempt = 0; attempt < 8 && !done; ++attempt) {
      long long granted = 0;
      for (int i = 0; i < n; ++i) {
        long long lu = cdf_last_u((double)pmf[i], lambda);
        if (lu > 2 * (long long)target) lu = 2 * (long long)target;
        g[i] = (float)lu;                                     // <= 2^17: exact in float
        if (lu >= v[i]) granted += lu - v[i] + 1;
      }
      if (granted <= todo) {
        for (int i = 0; i < n; ++i) { const int32_t lu = (int32_t)g[i]; if (lu >= v[i]) v[i] = lu + 1; }
        todo -= granted;
        done = true;
      } else {
        lambda *= 1.0 + ((double)(granted - todo) + 2.0 * sqrt((double)n_act) + 2.0) / (double)target;
      }
    }
    if (!done) break;
  }

  // scores: dir > 0: gain(v);  dir < 0: -gain(v-1) (= -penalty), entries at 1 can not shrink
  for (int i = 0; i < n; ++i)
    g[i] = dir > 0 ? cdf_score(pmf[i], v[i], scale) : (v[i] > 1 ? -cdf_score(pmf[i], v[i] - 1, scale) : -INFINITY);
  while (todo > 0) {
    // one pass: the best score, its (first) index and the runner-up; only a runner-up within the tolerance needs the exact path
    float mx = -INFINITY, second = -INFINITY;
    int best = -1;
#pragma unroll 4
    for (int i = 0; i < n; ++i) {             // branch-free: (gi > mx) ? shift the leader down : second = max(second, gi)
      const float gi = g[i];
      const bool lead = gi > mx;
      second = lead ? mx : (gi > second ? gi : second);
      best = lead ? i : best;
      mx = lead ? gi : mx;
    }
    if (!(mx > -INFINITY)) return -2;
    const float thr = mx - PCGC_SCORE_TOL(mx);
    if (second >= thr) {                    // near tie: decide on the exact gains, lowest index first
      double bs = -INFINITY;
      for (int i = 0; i < n; ++i)
        if (g[i] >= thr) {
          const double e = dir > 0 ? cdf_gain((double)pmf[i], v[i]) : -cdf_gain((double)pmf[i], v[i] - 1);
          if (e > bs) { bs = e; best = i; }
        }
    }
    v[best] += dir;
    g[best] = dir > 0 ? cdf_score(pmf[best], v[best], scale) : (v[best] > 1 ? -cdf_score(pmf[best], v[best] - 1, scale) : -INFINITY);
    --todo;
  }
  return 0;
}

}  // namespace pcgc
