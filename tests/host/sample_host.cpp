// Host build of the sampler of the continuous smoothed SDF (rho2sdf.jl_b200/csrc/r2s_sample.cuh), for tests/test_sample_host.py and the
// GPU tests (tests/test_sample_sdf.py).  Built with -ffp-contract=off, so every product and sum rounds where the header writes it.
#include <math.h>
#include <stdint.h>
#include "../../rho2sdf.jl_b200/csrc/r2s_sample.cuh"

extern "C" {

void smp_host_exp(const float *x, long n, float *out) {
  for (long i = 0; i < n; i++) out[i] = exp_f32(x[i]);
}

// every float in [lo, hi] (lo < 0 <= hi or both <= 0): the largest |exp_f32(x) - exp(x)| / exp(x), and the argument where it occurs
void smp_host_exp_scan(float lo, float hi, double *max_rel, float *worst) {
  uint32_t blo, bhi;
  // the negative floats from -0 down to lo are the bit patterns 0x80000000 .. bits(lo); the non-negative ones 0 .. bits(hi)
  memcpy(&blo, &lo, 4); memcpy(&bhi, &hi, 4);
  double best = 0.0; float arg = 0.0f;
#pragma omp parallel
  {
    double b = 0.0; float a = 0.0f;
#pragma omp for schedule(static)
    for (long long u = 0x80000000ll; u <= (long long)blo; u++) {
      uint32_t bits = (uint32_t)u; float x; memcpy(&x, &bits, 4);
      const double ref = exp((double)x), err = fabs((double)exp_f32(x) - ref) / ref;
      if (err > b) { b = err; a = x; }
    }
    if (hi >= 0.0f) {
#pragma omp for schedule(static)
      for (long long u = 0; u <= (long long)bhi; u++) {
        uint32_t bits = (uint32_t)u; float x; memcpy(&x, &bits, 4);
        const double ref = exp((double)x), err = fabs((double)exp_f32(x) - ref) / ref;
        if (err > b) { b = err; a = x; }
      }
    }
#pragma omp critical
    if (b > best) { best = b; arg = a; }
  }
  *max_rel = best; *worst = arg;
}

float smp_host_maxd(double rbf_cut, double cell) { return smp_maxd(rbf_cut, cell); }
float smp_host_t2(float maxd) { return smp_t2(maxd); }
void smp_host_range(double amin, double amax, int n, float *out) { smp_range(amin, amax, n, out); }

// the sampler on a whole-grid weight array w[(k * ny + j) * nx + i] (unpitched) of the grid amin, amax, N = n - 1
void smp_host_eval(const float *w, const int n[3], const double amin[3], const double amax[3], double cell, double rbf_cut, float th, const double *pts,
                   long np, float *val, float *grad) {
  float *tab[3];
  for (int d = 0; d < 3; d++) { tab[d] = new float[(size_t)n[d]]; smp_range(amin[d], amax[d], n[d], tab[d]); }
  SampleGrid G;
  smp_setup(&G, w, n[0], tab, n, cell, rbf_cut, th);
#pragma omp parallel for schedule(dynamic, 256)
  for (long t = 0; t < np; t++) {
    const float x = (float)pts[3 * t], y = (float)pts[3 * t + 1], z = (float)pts[3 * t + 2];
    if (grad) val[t] = sample_point<true>(G, x, y, z, grad + 3 * t);
    else val[t] = sample_point<false>(G, x, y, z, nullptr);
  }
  for (int d = 0; d < 3; d++) delete[] tab[d];
}

}  // extern "C"
