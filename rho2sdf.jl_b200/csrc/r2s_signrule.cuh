// r2s_signrule.cuh -- one candidate element of Sign_Detection's per-point rule (SignDetection.jl:40-59 HEX8, :120-140 TET4), shared by the
// grid path (r2s_sign.cu) and the points path (r2s_points.cu).  Bit-exact arithmetic (r2s_exact.cuh).
#pragma once
#include "r2s_common.cuh"
#include "r2s_exact.cuh"

typedef ex::AffineInv SignEl;      // per-element affine inverse-map data (r2s_exact.cuh)

// point_to_grid_index (SignDetection.jl:256-268): clamp(floor((x - amin) / cell) + 1, 1, N + 1), clamped before the conversion
__device__ __forceinline__ int pt_bin(double x, double amin, double cell, int n1) {
  const double f = floor(ex::dvd(ex::sub(x, amin), cell)) + 1.0;
  return f < 1.0 ? 1 : (f > (double)n1 ? n1 : (int)f);
}
// The element prologue of both sign binnings (k_sign_ranges on the grid, k_pt_sign_records for points): closed AABB lo <= x <= hi
// (sdfOnDensityField.jl:60-69); hot = some nodal density >= rho_t (the skip rule, :36; every TET4 element); the density class of a HEX8
// element for k_sign<8, true> (see k_sign_ranges); for TET4 per axis fl = floor((lo - amin) / cell) and cu = ceil((hi - amin) / cell), the
// cell range of create_grid_tetrahedra_mapping_TET4 (:195-196) before its -1 / +1 and its clamps.
struct SignElem { double lo[3], hi[3], fl[3], cu[3]; int hot, dcls; };
__device__ __forceinline__ void sign_element(i64 e, int nen, const int *__restrict__ IEN, const double *__restrict__ X, const double *__restrict__ rn, double rho_t,
                                             const GridDev &g, SignElem &E) {
  double rmax = -1e300, rmin = 1e300;
  for (int d = 0; d < 3; d++) { E.lo[d] = 1e300; E.hi[d] = -1e300; }
  for (int a = 0; a < nen; a++) {
    const i64 n = IEN[nen * e + a]; rmax = fmax(rmax, rn[n]); rmin = fmin(rmin, rn[n]);
    for (int d = 0; d < 3; d++) { const double c = X[3 * n + d]; E.lo[d] = fmin(E.lo[d], c); E.hi[d] = fmax(E.hi[d], c); }
  }
  // HEX8 density class: for max|xi| < 1.01 every shape function is above -0.01 * 2.01^2 / 8 and they sum to one, so the interpolated density
  // stays within [rmin - 0.05 range, rmax + 0.05 range].  1: it is >= rho_t for every admissible xi (the test "rho >= rho_t" is known to
  // hold), 2: it is < rho_t, 0: undecided.
  E.dcls = 0;
  if (nen == 8) {
    const double range = rmax - rmin, tolc = 1e-9 * fmax(1.0, fabs(rho_t));
    if (rmin - 0.05 * range >= rho_t + tolc) E.dcls = 1; else if (rmax + 0.05 * range < rho_t - tolc) E.dcls = 2;
  }
  E.hot = (nen == 4 || !(rmax < rho_t)) ? 1 : 0;
  if (nen == 4)
    for (int d = 0; d < 3; d++) { E.fl[d] = floor(ex::dvd(ex::sub(E.lo[d], g.amin[d]), g.cell)); E.cu[d] = ceil(ex::dvd(ex::sub(E.hi[d], g.amin[d]), g.cell)); }
}
// the affine inverse-map data of HEX8 element e
__device__ __forceinline__ SignEl sign_affine(i64 e, const int *__restrict__ IEN, const double *__restrict__ X) {
  double A[3][8];
  for (int d = 0; d < 3; d++) { double v[8]; for (int a = 0; a < 8; a++) v[a] = X[3 * (i64)IEN[8 * e + a] + d]; ex::mono8(v, A[d]); }
  SignEl S; ex::affine_inverse_prepare(A, S);
  return S;
}

// HEX8 candidate e in the loop over the point's candidates: sign and max_local carry the loop state; returns true at the loop's break
// (:51-59).  dcls = density class of the element (k_sign_ranges: 1 rho >= rho_t, 2 rho < rho_t wherever max|xi| < 1.01) or 0 = evaluate.
__device__ __forceinline__ bool sign_hex8_candidate(const SignEl &S, int e, const int *__restrict__ IEN, const double *__restrict__ X, const double *__restrict__ rn,
                                                    double rho_t, const double x[3], int dcls, double &sign, double &max_local) {
  double xi[3];
  if (S.affine) ex::affine_inverse_apply(S, x, xi);
  else {
    double A[3][8];
#pragma unroll
    for (int d = 0; d < 3; d++) {      // one coordinate at a time: only the monomial coefficients stay live
      double v[8];
#pragma unroll
      for (int a = 0; a < 8; a++) v[a] = X[3 * (i64)IEN[8 * (i64)e + a] + d];
      ex::mono8(v, A[d]);
    }
    ex::inverse_map_hex8_mono(A, false, x, xi);
  }
  double mn = ex::max3abs(xi[0], xi[1], xi[2]);
  if (mn < 1.01 && max_local > mn) {                         // SignDetection.jl:48
    if (dcls == 1) sign = 1.0;
    else if (dcls == 0) {
      double N[8], re[8];
#pragma unroll
      for (int a = 0; a < 8; a++) re[a] = rn[IEN[8 * (i64)e + a]];
      ex::hex8_shape(xi, N);
      double rho = ex::dot8(N, re);
      if (rho >= rho_t) sign = 1.0;
    }
    if (mn < 0.95) return true;                              // :51-59 break
    max_local = mn;
  }
  return false;
}

// TET4 candidate e: returns true (and sets sign = +1) when the point lies in the tetrahedron and its density there is >= rho_t
__device__ __forceinline__ bool sign_tet4_candidate(int e, const int *__restrict__ IEN, const double *__restrict__ X, const double *__restrict__ rn, double rho_t,
                                                    const double x[3], double &sign) {
  double Xe[3][4], re[4], lo[3] = {1e300, 1e300, 1e300}, hi[3] = {-1e300, -1e300, -1e300};
#pragma unroll
  for (int a = 0; a < 4; a++) { i64 nd = IEN[4 * (i64)e + a]; re[a] = rn[nd];
#pragma unroll
    for (int d = 0; d < 3; d++) { double c = X[3 * nd + d]; Xe[d][a] = c; lo[d] = fmin(lo[d], c); hi[d] = fmax(hi[d], c); } }
  // is_point_in_tetrahedron (:220-242), tolerance 1e-10
  const double tol = 1e-10;
#pragma unroll
  for (int d = 0; d < 3; d++) if (x[d] < ex::sub(lo[d], tol) || x[d] > ex::add(hi[d], tol)) return false;
  using namespace ex;
  double A[3][3], b[3];
#pragma unroll
  for (int d = 0; d < 3; d++) { A[d][0] = sub(Xe[d][1], Xe[d][0]); A[d][1] = sub(Xe[d][2], Xe[d][0]); A[d][2] = sub(Xe[d][3], Xe[d][0]); b[d] = sub(x[d], Xe[d][0]); }
  double c00 = sub(mul(A[1][1], A[2][2]), mul(A[1][2], A[2][1])), c01 = sub(mul(A[1][2], A[2][0]), mul(A[1][0], A[2][2])), c02 = sub(mul(A[1][0], A[2][1]), mul(A[1][1], A[2][0]));
  double det = add(add(mul(A[0][0], c00), mul(A[0][1], c01)), mul(A[0][2], c02));
  if (!(fabs(det) > 0.0)) return false;
  double c10 = sub(mul(A[0][2], A[2][1]), mul(A[0][1], A[2][2])), c11 = sub(mul(A[0][0], A[2][2]), mul(A[0][2], A[2][0])), c12 = sub(mul(A[0][1], A[2][0]), mul(A[0][0], A[2][1]));
  double c20 = sub(mul(A[0][1], A[1][2]), mul(A[0][2], A[1][1])), c21 = sub(mul(A[0][2], A[1][0]), mul(A[0][0], A[1][2])), c22 = sub(mul(A[0][0], A[1][1]), mul(A[0][1], A[1][0]));
  double l2 = dvd(add(add(mul(c00, b[0]), mul(c10, b[1])), mul(c20, b[2])), det), l3 = dvd(add(add(mul(c01, b[0]), mul(c11, b[1])), mul(c21, b[2])), det),
         l4 = dvd(add(add(mul(c02, b[0]), mul(c12, b[1])), mul(c22, b[2])), det);
  double l1 = sub(1.0, add(add(l2, l3), l4));
  if (!(l1 >= -tol && l2 >= -tol && l3 >= -tol && l4 >= -tol && l1 <= 1.0 + tol && l2 <= 1.0 + tol && l3 <= 1.0 + tol && l4 <= 1.0 + tol)) return false;
  double lc[3];
  if (!inverse_map_tet4(Xe, x, lc)) return false;            // found (:132)
  double l4b = sub(1.0, add(add(lc[0], lc[1]), lc[2]));
  double rho = add(add(add(mul(lc[0], re[0]), mul(lc[1], re[1])), mul(lc[2], re[2])), mul(l4b, re[3]));
  if (rho >= rho_t) { sign = 1.0; return true; }
  return false;
}
