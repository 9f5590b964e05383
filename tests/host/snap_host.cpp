// Host build of the vertex search of r2s_isosurface_lattice (rho2sdf.jl_b200/csrc/r2s_snap.cuh) on the host sampler (r2s_sample.cuh), for
// tests/test_isosurface_lattice_host.py and the GPU tests (tests/test_isosurface_lattice.py).  Built with -ffp-contract=off, so every
// operation rounds where the headers write it.
#include <math.h>
#include <stdint.h>
#include "../../rho2sdf.jl_b200/csrc/r2s_sample.cuh"
#include "../../rho2sdf.jl_b200/csrc/r2s_snap.cuh"

extern "C" {

int snap_host_max_evals() { return R2S_SNAP_MAX_EVALS; }

// a constructed edge function: f(x) = float(c0 + x (c1 + x (c2 + x c3)) + amp * noise(x)) in double, noise(x) in [-1, 1] a hash of the
// bits of x (amp > 0 makes f non-monotone at every scale); tr: lo, hi, flo, fhi (float) and the evaluation count
static float poly_f(const double c[4], double amp, float x) {
  uint32_t h = snap_key(x) * 2654435761u;
  h ^= h >> 15; h *= 2246822519u; h ^= h >> 13;
  const double noise = (double)(h & 0xffffu) / 32767.5 - 1.0;
  return (float)(c[0] + (double)x * (c[1] + (double)x * (c[2] + (double)x * c[3])) + amp * noise);
}
float snap_host_poly_f(const double c[4], double amp, float x) { return poly_f(c, amp, x); }
float snap_host_poly(const double c[4], double amp, float xa, float xb, float va, float vb, float iso, float *tr4, int *evals) {
  SnapTrace t;
  const float x = snap_search([&](float v) { return poly_f(c, amp, v); }, xa, xb, va, vb, iso, &t);
  tr4[0] = t.lo; tr4[1] = t.hi; tr4[2] = t.flo; tr4[3] = t.fhi; *evals = t.evals;
  return x;
}

// the vertices of lattice edges edges[4 q ..] = (i, j, k, axis) of the lattice o + float(i) h, on the field of a whole-grid weight array
// w[(k * ny + j) * nx + i] (unpitched) of the grid amin, amax, N = n - 1: V[3 q ..] and the final brackets tr[4 q ..], evals[q]
void snap_host_lattice(const float *w, const int n[3], const double amin[3], const double amax[3], double cell, double rbf_cut, float th, const float o[3],
                       const float h[3], const int64_t *edges, long ne, float iso, float *V, float *tr, int *evals) {
  float *tab[3];
  for (int d = 0; d < 3; d++) { tab[d] = new float[(size_t)n[d]]; smp_range(amin[d], amax[d], n[d], tab[d]); }
  SampleGrid G;
  smp_setup(&G, w, n[0], tab, n, cell, rbf_cut, th);
#pragma omp parallel for schedule(dynamic, 64)
  for (long q = 0; q < ne; q++) {
    const int64_t *e = edges + 4 * q;
    const int ax = (int)e[3];
    float p[3], b[3];
    for (int d = 0; d < 3; d++) {
      p[d] = smp_add(o[d], smp_mul((float)e[d], h[d]));
      b[d] = d == ax ? smp_add(o[d], smp_mul((float)(e[d] + 1), h[d])) : p[d];
    }
    const float va = sample_point<false>(G, p[0], p[1], p[2], nullptr), vb = sample_point<false>(G, b[0], b[1], b[2], nullptr);
    SnapTrace t;
    const float x = snap_search([&](float v) {
      float r[3] = {p[0], p[1], p[2]};
      r[ax] = v;
      return sample_point<false>(G, r[0], r[1], r[2], nullptr);
    }, p[ax], b[ax], va, vb, iso, &t);
    for (int d = 0; d < 3; d++) V[3 * q + d] = d == ax ? x : p[d];
    tr[4 * q] = t.lo; tr[4 * q + 1] = t.hi; tr[4 * q + 2] = t.flo; tr[4 * q + 3] = t.fhi; evals[q] = t.evals;
  }
  for (int d = 0; d < 3; d++) delete[] tab[d];
}

}  // extern "C"
