// Equivalence check of the shared-edge likelihood row (host build of the same header the CUDA kernels compile):
// det_laplace_pmf_row == per-symbol det_laplace_likelihood, bit for bit, on random Laplace rows over all symbol counts up to 32.
// g++ -O2 -ffp-contract=off -I pcgcv1_b200/csrc tools/cdf_check.cpp; exit code 0 = equal.
#include <cstdio>
#include <cstring>
#include <cmath>
#include <random>
#include "det_math.h"
using namespace pcgc;
int main() {
  long long n_rows = 0, n_bad = 0;
  std::mt19937_64 rng(99); std::uniform_real_distribution<double> U(0, 1);
  for (int it = 0; it < 300000; ++it) {
    int min_v = -(int)(U(rng) * 16), max_v = (int)(U(rng) * 16); if (max_v == min_v) max_v++;
    int N = max_v - min_v + 1; if (N > 32) continue;
    float l = (float)((U(rng) - 0.5) * 12), s = (float)std::exp((U(rng) - 0.6) * 7);
    float pm[32];
    det_laplace_pmf_row(min_v, N, l, s, 1e-9f, pm);
    ++n_rows;
    for (int k = 0; k < N; ++k) {
      const float ref = fmaxf(det_laplace_likelihood((float)(min_v + k), l, s), 1e-9f);
      if (memcmp(&ref, &pm[k], 4)) { if (n_bad++ < 5) printf("LIKELIHOOD MISMATCH N=%d k=%d\n", N, k); }
    }
  }
  printf("random Laplace rows: %lld checks, %lld mismatches\n", n_rows, n_bad);
  return n_bad != 0;
}
