// r2s_bound.cuh -- lower bounds of the distance from a grid point to the iso-patch of an axis-aligned box element, shared by the pair
// scans of the box projection (r2s_dist.cu) and the points path (r2s_points.cu), with the per-element set-up of the HEX8 projection, and
// compiled for the host by tests/host/bound_host.cpp.
//
// The element maps xi in [-1, 1]^3 to X_d = org_d + c_d + h_d xi_d; rho - rho_t is trilinear in xi.  box_iso_bounds gives two sets that
// contain every point the solver (r2s_iso.cuh) can return for the element, i.e. every point of the element where |rho - rho_t| is at
// most its tolerance:
//   tight box  per axis the hull of the slices xi_d = s whose four corner densities straddle rho_t within tol = 1e-12 gs (a bilinear
//              field takes its extrema over a slice at the corners; the candidates for the hull's ends are s = +-1 and the crossings of
//              the four edges along d with rho_t +- tol), widened by 1e-9 in xi and by a few ulps in x.  With tol, and not only the iso
//              crossings, the box holds the solver's points also in elements whose densities differ by little more than tol;
//   slab       A <= n.y <= B.  On the tight box (xi-box [s0, s1]^3) rho - rho_t is again trilinear: in centred variables u in [-1, 1]^3
//              it is d0 + g.u + d4 u0u1 + d5 u0u2 + d6 u1u2 + d7 u0u1u2, and the remainder is at most R = |d4| + |d5| + |d6| + |d7|.
//              So the iso-patch has |d0 + g.u| <= R; with u_d = (y_d - m_d) / s_d (m, s: centre and signed half-width in x) that is a
//              slab in x with normal n = w / |w|, w_d = g_d / s_d.
// lb_box_slab(P, ...) is the Euclidean distance from P to (tight box) /\ (slab), rounded down: a lower bound of every distance the
// solver can report for P.
//
// Margins (u = 2^-53):
//   * rho: the solver stops at |rho - rho_t| <= 1e-14 gs (gs >= max(|rho_t|, |rho_e|, 1)); the corner values and the eight centred
//     coefficients are sums of at most 8 products of terms below gs and carry less than 32 u gs each, so the eight coefficients
//     together less than 3e-14 gs.  The slab takes E = 1e-12 gs, the tolerance of the tight box: |d0 + g.u| <= R + E.
//   * x: w.m / |w| and n.y are sums of three products of terms of magnitude <= |m|_1 + |s|_1 (= the scale of every point of the box);
//     their rounding, and that of n itself, stays below 16 u of that scale.  A and B are widened by 1e-14 (|m|_1 + |s|_1) ~ 90 u.
//   * lb_box_slab: the root mu of the piecewise-linear equation is taken from below (mu <= mu*, see there) and the distance is a
//     non-decreasing function of mu, so rounding only has to be covered in the final distance: 1e-14 (|P|_1 + |tlo|_1 + |thi|_1)
//     absolute (the ulps of the coordinates, including the ulp by which the scans' amin + cell i may differ from the tabulated point)
//     and 1e-14 relative.
// If |g| <= R + E the slab cannot be narrower than the box along g (near a saddle, or with no gradient) and it is left unbounded
// (n = 0, A = -inf, B = +inf): lb_box_slab is then the distance to the tight box.
#pragma once
#include <math.h>
#include "r2s_iso.cuh"

#ifndef R2S_HD
#if defined(__CUDACC__)
#define R2S_HD __host__ __device__ __forceinline__
#else
#define R2S_HD inline
#endif
#endif

namespace bnd {

// re: nodal densities in the node order of hex8_shape.jl:27-34; c, h: the box map in element-local coordinates (iso::make_box), org: node 0
R2S_HD void box_iso_bounds(const double re[8], double rho_t, double gs, const double org[3], const double c[3], const double h[3],
                           double tlo[3], double thi[3], double n[3], double &A, double &B) {
  const int ea[3][4] = {{0, 3, 4, 7}, {0, 1, 4, 5}, {0, 1, 2, 3}}, eb[3][4] = {{1, 2, 5, 6}, {3, 2, 7, 6}, {4, 5, 6, 7}};
  double s0[3], s1[3];
  for (int d = 0; d < 3; d++) {
    // S = {s : the slice's corner values have min <= tol and max >= -tol} holds every slice through a point with |rho - rho_t| <= tol;
    // its ends are +-1 or where an edge value crosses +tol or -tol, so those are the candidates (tested with 2 tol against their rounding)
    const double tol = 1e-12 * gs;
    double va[4], vb[4], cand[10]; int nc = 0;
    cand[nc++] = -1.0; cand[nc++] = 1.0;
    for (int q = 0; q < 4; q++) {
      va[q] = re[ea[d][q]] - rho_t; vb[q] = re[eb[d][q]] - rho_t;
      for (int sd = -1; sd <= 1; sd += 2) {
        const double ua = va[q] - sd * tol, ub = vb[q] - sd * tol;
        if ((ua < 0.0) != (ub < 0.0) && ua != ub) cand[nc++] = fmin(1.0, fmax(-1.0, -1.0 + 2.0 * ua / (ua - ub)));
      }
    }
    double smin = 1.0, smax = -1.0; bool any = false;
    for (int t = 0; t < nc; t++) {
      const double s = cand[t], w = 0.5 * (s + 1.0);
      double mn = 1e300, mx = -1e300;
      for (int q = 0; q < 4; q++) { const double val = va[q] + (vb[q] - va[q]) * w; mn = fmin(mn, val); mx = fmax(mx, val); }
      if (mn <= 2.0 * tol && mx >= -2.0 * tol) { smin = fmin(smin, s); smax = fmax(smax, s); any = true; }
    }
    if (!any) { smin = -1.0; smax = 1.0; }      // cannot happen for a crossing element; stay safe
    const double pad = 1e-9;                    // widen in xi: the bound only has to be a lower bound
    smin = fmax(-1.0, smin - pad); smax = fmin(1.0, smax + pad);
    s0[d] = smin; s1[d] = smax;
    const double x0 = c[d] + h[d] * smin + org[d], x1 = c[d] + h[d] * smax + org[d];
    const double wid = 4e-16 * (fabs(org[d]) + fabs(c[d]) + fabs(h[d]));
    tlo[d] = fmin(x0, x1) - wid; thi[d] = fmax(x0, x1) + wid;
  }
  // slab: the 8 corner values of rho - rho_t on the xi-box [s0, s1] (trilinear interpolation of the nodal values), then the centred
  // coefficients.  v[k], k = i + 2 j + 4 l, is the corner with u = (2i - 1, 2j - 1, 2l - 1).
  const double sg[8][3] = {{-1, -1, -1}, {1, -1, -1}, {1, 1, -1}, {-1, 1, -1}, {-1, -1, 1}, {1, -1, 1}, {1, 1, 1}, {-1, 1, 1}};
  double v[8];
  for (int k = 0; k < 8; k++) {
    const double xi[3] = {(k & 1) ? s1[0] : s0[0], (k & 2) ? s1[1] : s0[1], (k & 4) ? s1[2] : s0[2]};
    double acc = 0.0;
    for (int a = 0; a < 8; a++) acc += 0.125 * ((1.0 + sg[a][0] * xi[0]) * (1.0 + sg[a][1] * xi[1]) * (1.0 + sg[a][2] * xi[2])) * (re[a] - rho_t);
    v[k] = acc;
  }
  double dc[8] = {0, 0, 0, 0, 0, 0, 0, 0};      // 1, u0, u1, u2, u0u1, u0u2, u1u2, u0u1u2
  for (int k = 0; k < 8; k++) {
    const double u0 = (k & 1) ? 1.0 : -1.0, u1 = (k & 2) ? 1.0 : -1.0, u2 = (k & 4) ? 1.0 : -1.0;
    dc[0] += v[k]; dc[1] += u0 * v[k]; dc[2] += u1 * v[k]; dc[3] += u2 * v[k];
    dc[4] += u0 * u1 * v[k]; dc[5] += u0 * u2 * v[k]; dc[6] += u1 * u2 * v[k]; dc[7] += u0 * u1 * u2 * v[k];
  }
  for (int k = 0; k < 8; k++) dc[k] *= 0.125;
  const double E = 1e-12 * gs, R = fabs(dc[4]) + fabs(dc[5]) + fabs(dc[6]) + fabs(dc[7]) + E;
  double w[3], m[3], ww = 0.0, wm = 0.0, scale = 0.0; bool ok = sqrt(dc[1] * dc[1] + dc[2] * dc[2] + dc[3] * dc[3]) > R;
  for (int d = 0; d < 3; d++) {
    const double md = 0.5 * (s0[d] + s1[d]), sd = h[d] * (0.5 * (s1[d] - s0[d]));
    m[d] = c[d] + h[d] * md + org[d];
    ok = ok && sd != 0.0;
    w[d] = ok ? dc[1 + d] / sd : 0.0;
    ww += w[d] * w[d]; wm += w[d] * m[d]; scale += fabs(m[d]) + fabs(sd);
  }
  const double wn = sqrt(ww);
  ok = ok && wn > 0.0 && isfinite(wn) && isfinite(wm);
  if (!ok) { n[0] = n[1] = n[2] = 0.0; A = -INFINITY; B = INFINITY; return; }
  for (int d = 0; d < 3; d++) n[d] = w[d] / wn;
  // w.u-terms: g.u = w.y - w.m, and -R <= d0 + g.u <= R
  const double mx = 1e-14 * scale;
  A = (wm - dc[0] - R) / wn - mx;
  B = (wm - dc[0] + R) / wn + mx;
}

// Squared lower bound of the same distance, without the root: c = clamp(P) is the projection of P onto the box, so for every y of the
// box (y - c).(c - P) >= 0 and |y - P|^2 >= |c - P|^2 + |y - c|^2 >= |c - P|^2 + gap(c)^2, gap(c) = the distance from c to the slab.
// The gap is shortened by lb_box_slab's rounding margin.  A cheap test before lb_box_slab.
R2S_HD double lb2_box_gap(const double P[3], const double tlo[3], const double thi[3], const double n[3], double A, double B) {
  double t = 0.0, e2 = 0.0, scale = 0.0;
  for (int d = 0; d < 3; d++) {
    const double c = fmin(fmax(P[d], tlo[d]), thi[d]), e = c - P[d];
    t += n[d] * c; e2 += e * e; scale += fabs(P[d]) + fabs(tlo[d]) + fabs(thi[d]);
  }
  const double gap = fmax(0.0, fmax(A - t, t - B) - 1e-14 * scale);
  return (e2 + gap * gap) * (1.0 - 1e-14);
}

// Euclidean distance from P to {y : tlo <= y <= thi, A <= n.y <= B} (|n| = 1 or n = 0 with an unbounded slab), rounded down.
// By KKT the nearest point is clamp(P + mu n) for one scalar mu: mu = 0 if n.clamp(P) is in [A, B]; otherwise phi(mu) = n.clamp(P + mu n)
// is non-decreasing and piecewise linear in mu, with its breakpoints where a coordinate reaches a face of the box (at most 6), and mu
// is its root at the violated end of the slab.
R2S_HD double lb_box_slab(const double P[3], const double tlo[3], const double thi[3], const double n[3], double A, double B) {
  double y[3], t = 0.0, scale = 0.0;
  for (int d = 0; d < 3; d++) { y[d] = fmin(fmax(P[d], tlo[d]), thi[d]); t += n[d] * y[d]; scale += fabs(P[d]) + fabs(tlo[d]) + fabs(thi[d]); }
  const double dlt = 1e-14 * scale;      // covers the rounding of every value of phi below
  if (t < A || t > B) {
    // walk towards the violated end: m = -+n turns it into "phi(mu) >= target, mu >= 0", phi(0) = sgn t < target
    const double sgn = t < A ? 1.0 : -1.0, target = t < A ? A : -B;
    const double m[3] = {sgn * n[0], sgn * n[1], sgn * n[2]};
    // breakpoints (+inf where there is none), sorted by a 12-comparator network: everything stays in registers
    double bp[6];
    for (int d = 0; d < 3; d++) {
      const double a = m[d] != 0.0 ? (tlo[d] - P[d]) / m[d] : -1.0, b = m[d] != 0.0 ? (thi[d] - P[d]) / m[d] : -1.0;
      bp[2 * d] = a > 0.0 ? a : INFINITY; bp[2 * d + 1] = b > 0.0 ? b : INFINITY;
    }
    const int net[12][2] = {{0, 5}, {1, 3}, {2, 4}, {1, 2}, {3, 4}, {0, 3}, {2, 5}, {0, 1}, {2, 3}, {4, 5}, {1, 2}, {3, 4}};
    for (int q = 0; q < 12; q++) { const double lo = fmin(bp[net[q][0]], bp[net[q][1]]), hi = fmax(bp[net[q][0]], bp[net[q][1]]); bp[net[q][0]] = lo; bp[net[q][1]] = hi; }
    // mu is taken from below: the first segment whose end reaches target - dlt holds mu* or lies before it, and on it mu* is at least
    // mu0 + (target - phi(mu0) - dlt) / slope.  If no segment reaches it, the last breakpoint is below mu* as well.
    double mu0 = 0.0, f0 = sgn * t, mu = 0.0;
    bool found = false, end = false;
    for (int k = 0; k < 6; k++) {
      if (found || end) continue;
      if (bp[k] == INFINITY) { end = true; continue; }
      double f1 = 0.0, slope = 0.0;
      const double mid = 0.5 * (mu0 + bp[k]);
      for (int d = 0; d < 3; d++) {
        f1 += m[d] * fmin(fmax(P[d] + bp[k] * m[d], tlo[d]), thi[d]);
        const double z = P[d] + mid * m[d];
        if (z > tlo[d] && z < thi[d]) slope += m[d] * m[d];
      }
      if (f1 >= target - dlt) {
        found = true;
        const double r = target - f0 - dlt;
        mu = (r > 0.0 && slope > 0.0) ? fmin(bp[k], mu0 + (r / slope) * (1.0 - 1e-15)) : mu0;
      } else { mu0 = bp[k]; f0 = f1; }
    }
    if (!found) mu = mu0;
    for (int d = 0; d < 3; d++) y[d] = fmin(fmax(P[d] + mu * m[d], tlo[d]), thi[d]);
  }
  const double e0 = y[0] - P[0], e1 = y[1] - P[1], e2 = y[2] - P[2];
  const double dist = sqrt(e0 * e0 + e1 * e1 + e2 * e2);
  return fmax(0.0, dist * (1.0 - 1e-14) - dlt);
}

// The pair bound against box /\ slab: true if the distance from P to it, squared, exceeds the running value c squared with a relative margin
// of 1e-10 (the scans take P as amin + cell i, an ulp or so from the tabulated point) -- the gap bound first, lb_box_slab only if it fails
R2S_HD bool box_slab_prunes(const double P[3], const double tlo[3], const double thi[3], const double n[3], double A, double B, double c) {
  const double c2 = c * c * (1.0 + 1e-10);
  if (lb2_box_gap(P, tlo, thi, n, A, B) > c2) return true;
  const double lb = lb_box_slab(P, tlo, thi, n, A, B);
  return lb * lb > c2;
}

// The per-element set-up of a crossing HEX8 element's projection (k_box_records, the points path's solver records): node 0 subtracted
// from the coordinates, the monomial coefficients A of the local x, y, z and of rho, the tolerance scale gs, phase 1 (Newton projection of
// xi = 0 onto the iso-surface: xi0, ok0) and, for a box element (iso::HexBox), the tight box and slab of its iso-patch; otherwise (general
// trilinear element, iso::HexTri) an unbounded box and slab.  nv: x, y, z and rho of the 8 nodes; the coordinates become element-local.
struct __align__(16) HexSetup {
  double A[4][8];
  double org[3], xi0[3], gs;
  double tlo[3], thi[3], sn[3], sA, sB;      // global coordinates
  int box, ok0;
};
__device__ inline void hex8_setup(double nv[4][8], double rho_t, bool box, HexSetup &P) {
#pragma unroll
  for (int d = 0; d < 3; d++) {
    P.org[d] = nv[d][0];
#pragma unroll
    for (int k = 0; k < 8; k++) nv[d][k] -= P.org[d];
  }
#pragma unroll
  for (int c = 0; c < 4; c++) iso::monomial8(nv[c], P.A[c]);
  double gs = fabs(rho_t);
#pragma unroll
  for (int k = 0; k < 8; k++) gs = fmax(gs, fabs(nv[3][k]));
  P.gs = fmax(gs, 1.0);
  P.box = box ? 1 : 0;
  iso::ProjState S0;
  if (box) {
    iso::HexBox H; iso::make_box(P.A, H);
    P.ok0 = iso::proj_init_element<iso::HexBox, PMODE>(H, rho_t, P.gs, S0) ? 1 : 0;
    box_iso_bounds(nv[3], rho_t, P.gs, P.org, H.c, H.h, P.tlo, P.thi, P.sn, P.sA, P.sB);
  } else {
    iso::HexTri H; H.A = P.A;
    P.ok0 = iso::proj_init_element<iso::HexTri, PMODE>(H, rho_t, P.gs, S0) ? 1 : 0;
#pragma unroll
    for (int d = 0; d < 3; d++) { P.tlo[d] = -INFINITY; P.thi[d] = INFINITY; P.sn[d] = 0.0; }
    P.sA = -INFINITY; P.sB = INFINITY;
  }
#pragma unroll
  for (int d = 0; d < 3; d++) P.xi0[d] = S0.xi[d];
}

}  // namespace bnd
