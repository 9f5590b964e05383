// Host build of the block classifier of r2s_isosurface_band (rho2sdf.jl_b200/csrc/r2s_band.cuh) over the host sampler (r2s_sample.cuh),
// for tests/test_isosurface_band_host.py.  Built with -ffp-contract=off, so every Float32 operation rounds where the headers write it.
#include <math.h>
#include <stdint.h>
#include "../../rho2sdf.jl_b200/csrc/r2s_sample.cuh"
#include "../../rho2sdf.jl_b200/csrc/r2s_band.cuh"

extern "C" {

int band_host_block() { return R2S_BAND_B; }

// boxes[6 b ..] = lo x y z, hi x y z (lattice indices) of the lattice o + float(i) h on the field of a whole-grid weight array
// w[(k * ny + j) * nx + i] (unpitched) of the grid amin, amax with n points per axis, at iso[b].  cls[b]: the classifier's answer, with the library's
// margins (exact = 1) or with none (exact = 0); wrong[b]: the box's lattice points on the other side of iso than cls[b] states (every
// point evaluated when cls[b] != 0), vmin / vmax[b]: their smallest and largest value (NaN when not evaluated)
void band_host_classify(const float *w, const int n[3], const double amin[3], const double amax[3], double cell, double rbf_cut, float th, const float o[3],
                        const float h[3], const int64_t *boxes, long nbox, const float *iso, int exact, int check, int *cls, long *wrong, float *vmin, float *vmax) {
  float *tab[3];
  for (int d = 0; d < 3; d++) { tab[d] = new float[(size_t)n[d]]; smp_range(amin[d], amax[d], n[d], tab[d]); }
  SampleGrid G;
  smp_setup(&G, w, n[0], tab, n, cell, rbf_cut, th);
  const BandMargin M = exact ? band_margin() : BandMargin{1.0, 1.0, 1.0, 1.0, 0.0};
#pragma omp parallel for schedule(dynamic, 16)
  for (long b = 0; b < nbox; b++) {
    const long long lo[3] = {boxes[6 * b], boxes[6 * b + 1], boxes[6 * b + 2]}, hi[3] = {boxes[6 * b + 3], boxes[6 * b + 4], boxes[6 * b + 5]};
    const int c = band_classify(G, o, h, lo, hi, iso[b], M);
    cls[b] = c;
    long bad = 0;
    float mn = NAN, mx = NAN;
    if (c || check)
      for (long long k = lo[2]; k <= hi[2]; k++)
        for (long long j = lo[1]; j <= hi[1]; j++)
          for (long long i = lo[0]; i <= hi[0]; i++) {
            const float v = sample_point<false>(G, smp_add(o[0], smp_mul((float)i, h[0])), smp_add(o[1], smp_mul((float)j, h[1])), smp_add(o[2], smp_mul((float)k, h[2])), nullptr);
            bad += (c == 1 && !(v >= iso[b])) || (c == 2 && !(v < iso[b]));
            mn = isnan(mn) || v < mn ? v : mn;
            mx = isnan(mx) || v > mx ? v : mx;
          }
    wrong[b] = bad; vmin[b] = mn; vmax[b] = mx;
  }
  for (int d = 0; d < 3; d++) delete[] tab[d];
}

}  // extern "C"
