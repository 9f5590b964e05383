// Host build of the per-element volume fractions of r2s_element_volume_fractions (rho2sdf.jl_b200/csrc/r2s_elemfrac.cuh) over the host
// sampler (r2s_sample.cuh) and the block classifier (r2s_band.cuh), for tests/test_element_fractions_host.py and the GPU tests' replay.
// Built with -ffp-contract=off, so every operation rounds where the headers write it.
#include <math.h>
#include <stdint.h>
#include "../../rho2sdf.jl_b200/csrc/r2s_elemfrac.cuh"

static EfElem load(int nen, const double *X, const int64_t *IEN, long e) {
  EfElem E;
  E.nen = nen;
  for (int a = 0; a < nen; a++)
    for (int d = 0; d < 3; d++) E.xe[d][a] = X[3 * IEN[(long)nen * e + a] + d];
  return E;
}

struct HostField {
  float *tab[3];
  SampleGrid G;
  HostField(const float *w, const int n[3], const double amin[3], const double amax[3], double cell, double cut, float th) {
    for (int d = 0; d < 3; d++) { tab[d] = new float[(size_t)n[d]]; smp_range(amin[d], amax[d], n[d], tab[d]); }
    smp_setup(&G, w, n[0], tab, n, cell, cut, th);
  }
  ~HostField() { for (int d = 0; d < 3; d++) delete[] tab[d]; }
};

extern "C" {

// every element of the mesh X (nnp x 3), IEN (nel x nen, 0-based) on the field of a whole-grid weight array w[(k * ny + j) * nx + i]
// (unpitched): fractions, volumes (V_e), and cls[e] = the classifier's answer on the element's box (0 sample, 1 inside, 2 outside).  Every
// point is evaluated, whatever cls says.
void ef_host_eval(const float *w, const int n[3], const double amin[3], const double amax[3], double cell, double cut, float th, int nen, const double *X,
                  const int64_t *IEN, long nel, int q, float iso, double *frac, double *vol, int *cls) {
  HostField F(w, n, amin, amax, cell, cut, th);
  const GaussTab G = gauss_legendre_host(q);
  const int npts = q * q * q;
#pragma omp parallel for schedule(dynamic, 64)
  for (long e = 0; e < nel; e++) {
    const EfElem E = load(nen, X, IEN, e);
    float a[3], b[3];
    ef_box(E, a, b);
    cls[e] = band_classify_box(F.G, a, b, iso, band_margin());
    double pv[R2S_EF_LANES], ps[R2S_EF_LANES];
    for (int l = 0; l < R2S_EF_LANES; l++) {
      double v = 0.0, s = 0.0;
      for (int t = l; t < npts; t += R2S_EF_LANES) {
        double x[3], W;
        if (!ef_point(E, G, t, x, &W)) continue;
        v += W;
        s += ef_inside(F.G, x, iso) ? W : 0.0;
      }
      pv[l] = v; ps[l] = s;
    }
    const double V = ef_tree(pv), S = ef_tree(ps);
    vol[e] = V; frac[e] = ef_fraction(S, V);
  }
}

// the Gauss points of element e: x[3 t ..], W[t], ok[t] (0: a dropped TET4 point)
void ef_host_points(int nen, const double *X, const int64_t *IEN, long e, int q, double *x, double *W, int *ok) {
  const EfElem E = load(nen, X, IEN, e);
  const GaussTab G = gauss_legendre_host(q);
  for (int t = 0; t < q * q * q; t++) ok[t] = ef_point(E, G, t, x + 3 * t, W + t);
}

// the element boxes a[3 e ..], b[3 e ..]; widen = 0 without the one-step widening
void ef_host_box(int nen, const double *X, const int64_t *IEN, long nel, int widen, float *a, float *b) {
  for (long e = 0; e < nel; e++) ef_box(load(nen, X, IEN, e), a + 3 * e, b + 3 * e, widen != 0);
}

// the classifier on m boxes: the box form on [a, b] (lattice = 0), or the lattice form on the index boxes lo, hi of o + float(i) h
void ef_host_classify(const float *w, const int n[3], const double amin[3], const double amax[3], double cell, double cut, float th, int lattice,
                      const float *a, const float *b, const float o[3], const float h[3], const int64_t *lo, const int64_t *hi, long m, const float *iso,
                      int *cls) {
  HostField F(w, n, amin, amax, cell, cut, th);
#pragma omp parallel for schedule(dynamic, 16)
  for (long k = 0; k < m; k++) {
    if (lattice) {
      const long long l[3] = {lo[3 * k], lo[3 * k + 1], lo[3 * k + 2]}, u[3] = {hi[3 * k], hi[3 * k + 1], hi[3 * k + 2]};
      cls[k] = band_classify(F.G, o, h, l, u, iso[k], band_margin());
    } else {
      cls[k] = band_classify_box(F.G, a + 3 * k, b + 3 * k, iso[k], band_margin());
    }
  }
}

}  // extern "C"
