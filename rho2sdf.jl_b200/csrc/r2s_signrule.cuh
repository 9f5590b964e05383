// r2s_signrule.cuh -- one candidate element of Sign_Detection's per-point rule (SignDetection.jl:40-59 HEX8, :120-140 TET4), shared by the
// grid path (r2s_sign.cu) and the points path (r2s_points.cu).  Bit-exact arithmetic (r2s_exact.cuh).
#pragma once
#include "r2s_common.cuh"
#include "r2s_exact.cuh"

typedef ex::AffineInv SignEl;      // per-element affine inverse-map data (r2s_exact.cuh)

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
