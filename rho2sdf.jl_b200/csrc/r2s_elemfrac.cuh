// r2s_elemfrac.cuh -- the solid volume fraction of one FE element in the continuous smoothed SDF (r2s_element_volume_fractions,
// r2s_elemfrac.cu): the Gauss points and weights of an element, the point rule, the ordered sums and the element's box for the classifier.
// Shared by the kernels and the host build (tests/host/elemfrac_host.cpp, g++ -ffp-contract=off); the kernels' TU is built with
// -fmad=false, like r2s_mesh.cu, whose calculate_mesh_volume uses the same shape functions and operation order.
//
// Gauss point t = (k q + j) q + i of an element, nodes g (ascending, gauss_legendre_host(q)) and weights w:
//   HEX8: xi = (g_i, g_j, g_k); x_d = sum_a N_a(xi) X_a,d (from 0, a ascending); W = ((w_i w_j) w_k) |det J(xi)|, J[r][c] = sum_a X_a,r
//         dN_a/dxi_c -- hex8_shape_d / det3 (r2s_tables.cuh), the order of k_mesh_volume
//   TET4: the collapsed cube of k_mesh_volume: xi = (g_i + 1) / 2, eta = (g_j + 1) / 2 (1 - xi), zeta = (g_k + 1) / 2 ((1 - xi) - eta);
//         a point with a negative coordinate or xi + eta + zeta > 1 is dropped (none is for nodes inside (-1, 1));
//         N = (xi, eta, zeta, ((1 - xi) - eta) - zeta) for nodes 0..3 (J's columns are X_0 - X_3, X_1 - X_3, X_2 - X_3);
//         W = (((w_i w_j) w_k) |det J|) ((1 - xi) ((1 - xi) - eta) / 8).  This is the Duffy factor of the map, so sum W = |det J| / 6; the
//         reference's calculate_mesh_volume multiplies by (1 - xi)^2 (MeshVolume.jl:107) and gets 3/4 of the volume -- a fraction is a
//         ratio of two integrals, and that factor would bias it.
// Every double operation is rounded where written.  At the point p = float(x) per coordinate the value f is the sampler's (r2s_sample.cuh,
// rules 2-5 of include/r2s.h); the point is inside iff f >= iso (a NaN value is outside).
// Sums: 32 lane partials, partial l = the sum of W (V) or of (inside ? W : +0) (S) over the points t = l mod 32 in ascending t, from +0;
// then the tree p[l] += p[l + o] for o = 16, 8, 4, 2, 1 (l < o); the element's sum is p[0].  V and S take the same order, so an element
// whose points are all inside has S == V bit for bit.  fraction = S / V, or 0 when V == 0.
//
// The element's box (ef_box) holds every p of its Gauss points: the exact N_a(xi) of a node xi in [-1, 1]^3 (TET4: of the simplex) are
// >= 0 and sum to 1, so the exact x_d lies in [min_a X_a,d, max_a X_a,d].  The rounded shape functions (a few roundings each; TET4: the
// rounded simplex test admits a sum over 1 by 2 ulps) and the rounded sum of at most 8 terms move x_d by less than 2^-48 M_d, M_d =
// max_a |X_a,d|.  The box per axis is [band_down(min - s), band_up(max + s)] with s = 2^-40 M_d (the double rounding
// of min - s is below 2^-53 M_d), widened by one Float32 step on each side; rounding to nearest is monotone, so every float(x_d) lies in it.
#pragma once
#include <math.h>
#include <stdint.h>
#include "r2s_tables.cuh"
#include "r2s_sample.cuh"
#include "r2s_band.cuh"

#define R2S_EF_LANES 32

// the nodes of one element, coordinates per axis
struct EfElem { double xe[3][8]; int nen; };

// Gauss point t of element E at the rule G (q = G.n): its coordinates x and weight W; false for a dropped TET4 point (W = 0)
R2S_HD bool ef_point(const EfElem &E, const GaussTab &G, int t, double x[3], double *W) {
  const int q = G.n, i = t % q, j = (t / q) % q, k = t / (q * q);
  if (E.nen == 8) {
    double N[8], dN[8][3];
    const double xi[3] = {G.x[i], G.x[j], G.x[k]};
    hex8_shape_d(xi, N, dN);
    double J[3][3];
    for (int r = 0; r < 3; r++)
      for (int c = 0; c < 3; c++) {
        double s = 0;
        for (int a = 0; a < 8; a++) s += E.xe[r][a] * dN[a][c];
        J[r][c] = s;
      }
    for (int d = 0; d < 3; d++) {
      double s = 0;
      for (int a = 0; a < 8; a++) s += N[a] * E.xe[d][a];
      x[d] = s;
    }
    *W = G.w[i] * G.w[j] * G.w[k] * fabs(det3(J));
    return true;
  }
  double J[3][3];
  for (int r = 0; r < 3; r++) { J[r][0] = E.xe[r][0] - E.xe[r][3]; J[r][1] = E.xe[r][1] - E.xe[r][3]; J[r][2] = E.xe[r][2] - E.xe[r][3]; }
  const double adet = fabs(det3(J));
  const double xi = (G.x[i] + 1.0) / 2.0, eta = (G.x[j] + 1.0) / 2.0 * (1.0 - xi), zeta = (G.x[k] + 1.0) / 2.0 * (1.0 - xi - eta);
  if (xi < 0 || eta < 0 || zeta < 0 || xi + eta + zeta > 1.0) { x[0] = x[1] = x[2] = 0.0; *W = 0.0; return false; }
  const double N[4] = {xi, eta, zeta, 1.0 - xi - eta - zeta};
  for (int d = 0; d < 3; d++) {
    double s = 0;
    for (int a = 0; a < 4; a++) s += N[a] * E.xe[d][a];
    x[d] = s;
  }
  const double jt = (1.0 - xi) * (1.0 - xi - eta) / 8.0;
  *W = G.w[i] * G.w[j] * G.w[k] * adet * jt;
  return true;
}

// the Float32 box of the element's Gauss points (see above); widen = false drops the one-step widening (host tests only)
R2S_HD void ef_box(const EfElem &E, float a[3], float b[3], bool widen = true) {
  for (int d = 0; d < 3; d++) {
    double mn = E.xe[d][0], mx = E.xe[d][0];
    for (int n = 1; n < E.nen; n++) { mn = fmin(mn, E.xe[d][n]); mx = fmax(mx, E.xe[d][n]); }
    const double s = fmax(fabs(mn), fabs(mx)) * 0x1p-40;
    a[d] = band_down(mn - s); b[d] = band_up(mx + s);
    if (widen) { a[d] = nextafterf(a[d], -INFINITY); b[d] = nextafterf(b[d], INFINITY); }
  }
}

// the point's value on the field G (the caller picked the slab's weights) and whether it is inside
R2S_HD bool ef_inside(const SampleGrid &G, const double x[3], float iso) {
  return sample_point<false>(G, (float)x[0], (float)x[1], (float)x[2], nullptr) >= iso;
}

R2S_HD double ef_fraction(double S, double V) { return V == 0.0 ? 0.0 : S / V; }

// host replay of the combination of the 32 lane partials (the kernels combine them with __shfl_down_sync in the same order)
static inline double ef_tree(double p[R2S_EF_LANES]) {
  for (int o = R2S_EF_LANES / 2; o > 0; o >>= 1)
    for (int l = 0; l < o; l++) p[l] = p[l] + p[l + o];
  return p[0];
}
