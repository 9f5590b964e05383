// r2s_iso.cuh -- closest point on the in-element iso-surface of a HEX8 / TET4 (device functions)
//
//   min ||x - X(xi)||^2   s.t.   rho(xi) = rho_t,   -1 <= xi <= 1          (SignedDistances/ComputeCoordsOnIso.jl:16-87)
//
// The reference hands this to NLopt :LD_SLSQP from xi = 0.  Here: a feasible-path SQP from the same start
//   phase 1  Newton-project xi = 0 onto {g = 0} inside the box (fallback: iso-crossing of an element edge closest to x)
//   phase 2  Newton steps in the tangent space of g on the current face of the box (exact Hessian of the Lagrangian,
//            Gauss-Newton fallback), ratio test against the bounds, restoration onto g = 0, Armijo on f;
//            bounds are released by multiplier sign once the face problem has converged.
// The trilinear fields are held in monomial form  v = A0 + A1 x + A2 e + A3 z + A4 xe + A5 ez + A6 zx + A7 xez  so that a
// value costs 7 FMAs and a gradient 9; FMA contraction is allowed here (this is the FP64-bound hot loop) -- the result is
// converged to |step| <= 1e-11 in xi, far below the 1e-9 h parity tolerance.
#pragma once
#include <cuda_runtime.h>
#include <math.h>
#include <type_traits>

// Host build (tests/host/iso_host.cpp) only: operation counters for the offline cost studies; nothing on the device.
#ifdef R2S_ISO_HOST
static long iso_counts[8];      // 0 eval_full, 1 eval_g, 2 eval_f, 3 tangent steps, 4 line-search trials, 5 active-set passes
#define ISO_COUNT(k) (iso_counts[k]++)
// optional event trace of one projection (tools/divergence_model.py): codes 1 eval_g inside restore, 2 line-search trial, 3 eval_full
// (= start of a phase-2 iteration), 10..12 tangent3<K>, 13..15 tangent2 (fixed variable 0,1,2), 16 fewer than two free variables,
// 17 Gauss-Newton fallback of the multiplier branch, 18 the single-path tangent step (MODE bit 1)
static int *iso_trace = nullptr; static long iso_trace_n = 0, iso_trace_cap = 0;
#define ISO_TRACE(c) do { if (iso_trace && iso_trace_n < iso_trace_cap) iso_trace[iso_trace_n++] = (c); } while (0)
#else
#define ISO_COUNT(k) ((void)0)
#define ISO_TRACE(c) ((void)0)
#endif

namespace iso {

struct Eval {
  double f, g, F[3], c[3], a[3];
  double Hgn[3][3];   // 2 J^T J
  double m[3];        // extra off-diagonal terms of Hess f: pairs (0,1),(1,2),(2,0)
  double hg[3];       // off-diagonal terms of Hess g, same pair order (its diagonal is zero)
};

__device__ __forceinline__ double tri_val(const double A[8], double X, double E, double Z, double xe, double ez, double zx, double xez) {
  return fma(A[7], xez, fma(A[6], zx, fma(A[5], ez, fma(A[4], xe, fma(A[3], Z, fma(A[2], E, fma(A[1], X, A[0])))))));
}
// g and grad g only
__device__ __forceinline__ void eval_g(const double A[4][8], double rho_t, const double xi[3], double &g, double a[3]) {
  ISO_COUNT(1); ISO_TRACE(1);
  double X = xi[0], E = xi[1], Z = xi[2], xe = X * E, ez = E * Z, zx = Z * X, xez = xe * Z;
  g = tri_val(A[3], X, E, Z, xe, ez, zx, xez) - rho_t;
  a[0] = fma(A[3][7], ez, fma(A[3][6], Z, fma(A[3][4], E, A[3][1])));
  a[1] = fma(A[3][7], zx, fma(A[3][5], Z, fma(A[3][4], X, A[3][2])));
  a[2] = fma(A[3][7], xe, fma(A[3][6], X, fma(A[3][5], E, A[3][3])));
}
__device__ __forceinline__ void eval_pos(const double A[4][8], const double xi[3], double p[3]) {
  double X = xi[0], E = xi[1], Z = xi[2], xe = X * E, ez = E * Z, zx = Z * X, xez = xe * Z;
#pragma unroll
  for (int d = 0; d < 3; d++) p[d] = tri_val(A[d], X, E, Z, xe, ez, zx, xez);
}
__device__ __forceinline__ double eval_f(const double A[4][8], const double x[3], const double xi[3]) {
  ISO_COUNT(2);
  double p[3]; eval_pos(A, xi, p);
  double F0 = p[0] - x[0], F1 = p[1] - x[1], F2 = p[2] - x[2];
  return fma(F2, F2, fma(F1, F1, F0 * F0));
}
__device__ __forceinline__ void eval_full(const double A[4][8], const double x[3], double rho_t, const double xi[3], Eval &E_) {
  ISO_COUNT(0); ISO_TRACE(3);
  double X = xi[0], E = xi[1], Z = xi[2], xe = X * E, ez = E * Z, zx = Z * X, xez = xe * Z;
  double J[3][3], mx[3][3];
#pragma unroll
  for (int d = 0; d < 3; d++) {
    E_.F[d] = tri_val(A[d], X, E, Z, xe, ez, zx, xez) - x[d];
    J[d][0] = fma(A[d][7], ez, fma(A[d][6], Z, fma(A[d][4], E, A[d][1])));
    J[d][1] = fma(A[d][7], zx, fma(A[d][5], Z, fma(A[d][4], X, A[d][2])));
    J[d][2] = fma(A[d][7], xe, fma(A[d][6], X, fma(A[d][5], E, A[d][3])));
    mx[d][0] = fma(A[d][7], Z, A[d][4]);   // d2/dxi deta
    mx[d][1] = fma(A[d][7], X, A[d][5]);   // d2/deta dzeta
    mx[d][2] = fma(A[d][7], E, A[d][6]);   // d2/dzeta dxi
  }
  E_.f = fma(E_.F[2], E_.F[2], fma(E_.F[1], E_.F[1], E_.F[0] * E_.F[0]));
  eval_g(A, rho_t, xi, E_.g, E_.a);
  E_.hg[0] = fma(A[3][7], Z, A[3][4]); E_.hg[1] = fma(A[3][7], X, A[3][5]); E_.hg[2] = fma(A[3][7], E, A[3][6]);
#pragma unroll
  for (int j = 0; j < 3; j++) {
    E_.c[j] = 2.0 * fma(J[2][j], E_.F[2], fma(J[1][j], E_.F[1], J[0][j] * E_.F[0]));
    E_.m[j] = 2.0 * fma(E_.F[2], mx[2][j], fma(E_.F[1], mx[1][j], E_.F[0] * mx[0][j]));
#pragma unroll
    for (int i = 0; i < 3; i++) E_.Hgn[i][j] = 2.0 * fma(J[2][i], J[2][j], fma(J[1][i], J[1][j], J[0][i] * J[0][j]));
  }
}
// full Hessian entry of the Lagrangian
__device__ __forceinline__ double Hl(const Eval &E, double lam, int i, int j) {
  if (i == j) return E.Hgn[i][i];
  int p = (i + j == 1) ? 0 : ((i + j == 3) ? 1 : 2);
  return E.Hgn[i][j] + fma(lam, E.hg[p], E.m[p]);
}

// ----------------------------------------------------------------------------------------------------------------
// Element types of the solver.  HexTri: general trilinear geometry, monomial coefficients [x,y,z,rho][8].  HexBox: the
// element is an axis-aligned box in canonical node order, X_d(xi) = c_d + h_d xi_d (every mixed coefficient of the three
// geometry fields is EXACTLY zero -- true for every voxel-type SIMP mesh, since each nodal coordinate then takes one of two
// values per axis and the differences in monomial8 cancel exactly).  Dropping the exact-zero terms changes no finite value:
// F, c, f and the diagonal of 2 J^T J are what the general formulas give; m and the off-diagonal of 2 J^T J vanish.  The
// iteration then needs 17 element constants instead of 32 (registers) and about half the FP64 work.
struct HexTri {
  const double (*A)[8];
  typedef Eval EvalT;
};
struct HexBox {
  double R[8];            // monomial coefficients of rho
  double c[3], h[3];      // X_d = c_d + h_d xi_d
  double hh[3];           // 2 h_d^2 = diagonal of 2 J^T J
  struct EvalT {
    double f, g, F[3], c[3], a[3];
    double hh[3];         // diagonal of Hess f (constant)
    double hg[3];         // off-diagonal terms of Hess g, pairs (0,1),(1,2),(2,0)
  };
};
// true when the geometry coefficients A[0..2] describe a box in canonical orientation
__device__ __forceinline__ bool is_box(const double A[4][8]) {
  bool ok = true;
#pragma unroll
  for (int d = 0; d < 3; d++)
#pragma unroll
    for (int k = 1; k < 8; k++) if (k != d + 1 && A[d][k] != 0.0) ok = false;
  return ok;
}
__device__ __forceinline__ void make_box(const double A[4][8], HexBox &B) {
#pragma unroll
  for (int k = 0; k < 8; k++) B.R[k] = A[3][k];
#pragma unroll
  for (int d = 0; d < 3; d++) { B.c[d] = A[d][0]; B.h[d] = A[d][d + 1]; B.hh[d] = 2.0 * (A[d][d + 1] * A[d][d + 1]); }
}
// rho-field part shared by both element types (R = monomial coefficients of rho)
__device__ __forceinline__ void eval_g_R(const double R[8], double rho_t, const double xi[3], double &g, double a[3]) {
  ISO_COUNT(1); ISO_TRACE(1);
  double X = xi[0], E = xi[1], Z = xi[2], xe = X * E, ez = E * Z, zx = Z * X, xez = xe * Z;
  g = tri_val(R, X, E, Z, xe, ez, zx, xez) - rho_t;
  a[0] = fma(R[7], ez, fma(R[6], Z, fma(R[4], E, R[1])));
  a[1] = fma(R[7], zx, fma(R[5], Z, fma(R[4], X, R[2])));
  a[2] = fma(R[7], xe, fma(R[6], X, fma(R[5], E, R[3])));
}
// HexTri overloads: the array forms above, unchanged
__device__ __forceinline__ void eval_g(const HexTri &T, double rho_t, const double xi[3], double &g, double a[3]) { eval_g(T.A, rho_t, xi, g, a); }
__device__ __forceinline__ void eval_pos(const HexTri &T, const double xi[3], double p[3]) { eval_pos(T.A, xi, p); }
__device__ __forceinline__ double eval_f(const HexTri &T, const double x[3], const double xi[3]) { return eval_f(T.A, x, xi); }
__device__ __forceinline__ void eval_full(const HexTri &T, const double x[3], double rho_t, const double xi[3], Eval &E) { eval_full(T.A, x, rho_t, xi, E); }
__device__ __forceinline__ double hdiag(const Eval &E, int i) { return E.Hgn[i][i]; }
// HexBox overloads
__device__ __forceinline__ void eval_g(const HexBox &B, double rho_t, const double xi[3], double &g, double a[3]) { eval_g_R(B.R, rho_t, xi, g, a); }
__device__ __forceinline__ void eval_pos(const HexBox &B, const double xi[3], double p[3]) {
#pragma unroll
  for (int d = 0; d < 3; d++) p[d] = fma(B.h[d], xi[d], B.c[d]);
}
__device__ __forceinline__ double eval_f(const HexBox &B, const double x[3], const double xi[3]) {
  ISO_COUNT(2);
  double F0 = fma(B.h[0], xi[0], B.c[0]) - x[0], F1 = fma(B.h[1], xi[1], B.c[1]) - x[1], F2 = fma(B.h[2], xi[2], B.c[2]) - x[2];
  return fma(F2, F2, fma(F1, F1, F0 * F0));
}
__device__ __forceinline__ void eval_full(const HexBox &B, const double x[3], double rho_t, const double xi[3], HexBox::EvalT &E_) {
  ISO_COUNT(0); ISO_TRACE(3);
#pragma unroll
  for (int d = 0; d < 3; d++) {
    E_.F[d] = fma(B.h[d], xi[d], B.c[d]) - x[d];
    E_.c[d] = 2.0 * (B.h[d] * E_.F[d]);
    E_.hh[d] = B.hh[d];
  }
  E_.f = fma(E_.F[2], E_.F[2], fma(E_.F[1], E_.F[1], E_.F[0] * E_.F[0]));
  eval_g_R(B.R, rho_t, xi, E_.g, E_.a);
  E_.hg[0] = fma(B.R[7], xi[2], B.R[4]); E_.hg[1] = fma(B.R[7], xi[0], B.R[5]); E_.hg[2] = fma(B.R[7], xi[1], B.R[6]);
}
__device__ __forceinline__ double hdiag(const HexBox::EvalT &E, int i) { return E.hh[i]; }
// Solver variants (template parameter MODE).  The kernels run MODE 3 = FAST restoration + one tangent-step code path; MODE 0 (every
// step confirmed by an evaluation, one template instance per tangent-step case) and MODE 1 (FAST only) are instantiated by the host
// build (tests/host/iso_host.cpp), where MODE 3 is checked against them and against the oracle pair by pair.
// FAST: restore() leaves without the confirming evaluation once the step
// just taken is so short that the remainder of the trilinear field is below tolg:
//   g(xi + D) - g(xi) - a.D = R4 D0 D1 + R5 D1 D2 + R6 D2 D0 + R7 (xi0 D1 D2 + xi1 D2 D0 + xi2 D0 D1 + D0 D1 D2),
// so |g_new| <= (|R4| + |R5| + |R6| + 4 |R7|) |D|^2 for |xi|, |D| <= 1 when D is the full Newton step (no variable clamped).
// (A reciprocal-based replacement of the divisions was tried and dropped: the fast path of the IEEE division is itself
// MUFU.RCP64H + Newton, about 9 FP64 instructions, so there is little to gain.)
__device__ __forceinline__ const double *rho_coeffs(const HexTri &T) { return T.A[3]; }
__device__ __forceinline__ const double *rho_coeffs(const HexBox &B) { return B.R; }

// Newton restoration onto g = 0 moving only variables with fix[i] == 0; variables leaving the box are clamped and fixed
template <class EL, int MODE = 0>
__device__ __forceinline__ bool restore(const EL &A, double rho_t, double xi[3], int fix[3], double tolg) {
  constexpr bool FAST = (MODE & 1) != 0;
  double cq = 0.0;
  if (FAST) { const double *R = rho_coeffs(A); cq = (fabs(R[4]) + fabs(R[5])) + (fabs(R[6]) + 4.0 * fabs(R[7])); }
  for (int it = 0; it < 40; it++) {
    double g, a[3]; eval_g(A, rho_t, xi, g, a);
    if (fabs(g) <= tolg) return true;
    double den = 0;
#pragma unroll
    for (int i = 0; i < 3; i++) if (!fix[i]) den = fma(a[i], a[i], den);
    if (!(den > 0.0)) return false;
    double s = g / den;
    bool hit = false;
#pragma unroll
    for (int i = 0; i < 3; i++) if (!fix[i]) {
      xi[i] = fma(-s, a[i], xi[i]);
      if (xi[i] >= 1.0) { xi[i] = 1.0; fix[i] = 1; hit = true; } else if (xi[i] <= -1.0) { xi[i] = -1.0; fix[i] = -1; hit = true; }
    }
    if (FAST && !hit && cq * (s * s * den) <= 0.5 * tolg) return true;      // the remainder after this full Newton step is below tolg
  }
  return false;
}

// tangent step, two free variables (I,J), K fixed
template <int I, int J>
__device__ __forceinline__ void tangent2(const Eval &E, double lam, double d[3]) {
  double zi = -E.a[J], zj = E.a[I];
  double zz = fma(zi, zi, zj * zj);
  if (!(zz > 0.0)) return;
  double hii = Hl(E, lam, I, I), hij = Hl(E, lam, I, J), hjj = Hl(E, lam, J, J);
  double kap = zi * fma(hii, zi, hij * zj) + zj * fma(hij, zi, hjj * zj);
  double kgn = zi * fma(E.Hgn[I][I], zi, E.Hgn[I][J] * zj) + zj * fma(E.Hgn[I][J], zi, E.Hgn[J][J] * zj);
  if (!(kap > 1e-8 * kgn)) kap = kgn;
  if (!(kap > 0.0)) return;
  double t = -fma(zi, E.c[I], zj * E.c[J]) / kap;
  d[I] = t * zi; d[J] = t * zj;
}
// tangent step, all three free; null-space basis built around component K (largest |a_K|), U=(K+1)%3, V=(K+2)%3
template <int K>
__device__ __forceinline__ void tangent3(const Eval &E, double lam, double d[3]) {
  constexpr int U = (K + 1) % 3, V = (K + 2) % 3;
  double z1[3] = {0, 0, 0}, z2[3] = {0, 0, 0};
  z1[U] = E.a[K]; z1[K] = -E.a[U]; z2[V] = E.a[K]; z2[K] = -E.a[V];
  double Hz1[3], Hz2[3], Gz1[3], Gz2[3];
#pragma unroll
  for (int i = 0; i < 3; i++) {
    Hz1[i] = fma(Hl(E, lam, i, 2), z1[2], fma(Hl(E, lam, i, 1), z1[1], Hl(E, lam, i, 0) * z1[0]));
    Hz2[i] = fma(Hl(E, lam, i, 2), z2[2], fma(Hl(E, lam, i, 1), z2[1], Hl(E, lam, i, 0) * z2[0]));
    Gz1[i] = fma(E.Hgn[i][2], z1[2], fma(E.Hgn[i][1], z1[1], E.Hgn[i][0] * z1[0]));
    Gz2[i] = fma(E.Hgn[i][2], z2[2], fma(E.Hgn[i][1], z2[1], E.Hgn[i][0] * z2[0]));
  }
  double m11 = fma(z1[2], Hz1[2], fma(z1[1], Hz1[1], z1[0] * Hz1[0])), m12 = fma(z1[2], Hz2[2], fma(z1[1], Hz2[1], z1[0] * Hz2[0])),
         m22 = fma(z2[2], Hz2[2], fma(z2[1], Hz2[1], z2[0] * Hz2[0]));
  double g11 = fma(z1[2], Gz1[2], fma(z1[1], Gz1[1], z1[0] * Gz1[0])), g12 = fma(z1[2], Gz2[2], fma(z1[1], Gz2[1], z1[0] * Gz2[0])),
         g22 = fma(z2[2], Gz2[2], fma(z2[1], Gz2[1], z2[0] * Gz2[0]));
  double r1 = -fma(z1[2], E.c[2], fma(z1[1], E.c[1], z1[0] * E.c[0])), r2 = -fma(z2[2], E.c[2], fma(z2[1], E.c[1], z2[0] * E.c[0]));
  double det = m11 * m22 - m12 * m12, detg = g11 * g22 - g12 * g12;
  if (!(m11 > 1e-8 * g11 && det > 1e-8 * detg)) { m11 = g11; m12 = g12; m22 = g22; det = detg; }
  if (!(det > 0.0 && m11 > 0.0)) return;
  double y1 = (m22 * r1 - m12 * r2) / det, y2 = (m11 * r2 - m12 * r1) / det;
#pragma unroll
  for (int i = 0; i < 3; i++) d[i] = fma(y1, z1[i], y2 * z2[i]);
}
// HexBox: Hess f = diag(hh), Hess of the Lagrangian = diag(hh) + lam * (off-diagonal hg); the null-space vectors
// z1 = a_K e_U - a_U e_K, z2 = a_K e_V - a_V e_K have one zero component each, which is used explicitly
__device__ __forceinline__ int pair_of(int i, int j) { return (i + j == 1) ? 0 : ((i + j == 3) ? 1 : 2); }
template <int I, int J>
__device__ __forceinline__ void tangent2(const HexBox::EvalT &E, double lam, double d[3]) {
  double zi = -E.a[J], zj = E.a[I];
  double zz = fma(zi, zi, zj * zj);
  if (!(zz > 0.0)) return;
  double hii = E.hh[I], hij = lam * E.hg[pair_of(I, J)], hjj = E.hh[J];
  double kap = zi * fma(hii, zi, hij * zj) + zj * fma(hij, zi, hjj * zj);
  double kgn = zi * (hii * zi) + zj * (hjj * zj);
  if (!(kap > 1e-8 * kgn)) kap = kgn;
  if (!(kap > 0.0)) return;
  double t = -fma(zi, E.c[I], zj * E.c[J]) / kap;
  d[I] = t * zi; d[J] = t * zj;
}
template <int K>
__device__ __forceinline__ void tangent3(const HexBox::EvalT &E, double lam, double d[3]) {
  constexpr int U = (K + 1) % 3, V = (K + 2) % 3;
  const double aK = E.a[K], aU = E.a[U], aV = E.a[V];
  const double HUK = lam * E.hg[pair_of(U, K)], HUV = lam * E.hg[pair_of(U, V)], HKV = lam * E.hg[pair_of(K, V)];
  const double Hz1U = fma(E.hh[U], aK, -(HUK * aU)), Hz1K = fma(HUK, aK, -(E.hh[K] * aU));
  const double Hz2U = fma(HUV, aK, -(HUK * aV)), Hz2K = fma(HKV, aK, -(E.hh[K] * aV)), Hz2V = fma(E.hh[V], aK, -(HKV * aV));
  double m11 = fma(aK, Hz1U, -(aU * Hz1K)), m12 = fma(aK, Hz2U, -(aU * Hz2K)), m22 = fma(aK, Hz2V, -(aV * Hz2K));
  const double kK = E.hh[K] * aU;
  double g11 = fma(E.hh[U] * aK, aK, kK * aU), g12 = kK * aV, g22 = fma(E.hh[V] * aK, aK, (E.hh[K] * aV) * aV);
  const double r1 = -fma(aK, E.c[U], -(aU * E.c[K])), r2 = -fma(aK, E.c[V], -(aV * E.c[K]));
  double det = m11 * m22 - m12 * m12, detg = g11 * g22 - g12 * g12;
  if (!(m11 > 1e-8 * g11 && det > 1e-8 * detg)) { m11 = g11; m12 = g12; m22 = g22; det = detg; }
  if (!(det > 0.0 && m11 > 0.0)) return;
  const double y1 = (m22 * r1 - m12 * r2) / det, y2 = (m11 * r2 - m12 * r1) / det;
  d[U] = y1 * aK; d[V] = y2 * aK; d[K] = -fma(y1, aU, y2 * aV);
}
// MODE bit 1: ONE code path for every tangent-step case.  The three tangent3<K> and the three tangent2<I,J> variants
// differ only by a cyclic rotation of the indices: (K,U,V) = (K,K+1,K+2) with K = argmax |a_k| when all three variables are free,
// K = L+1 when variable L is fixed (then V = L, the second null-space vector is dropped: m12 = r2 = 0, m22 = 1 turns the 2x2 solve
// into tangent2's scalar step).  Lanes of a warp sit on different faces of the box; with the template variants every distinct
// case is issued separately (the offline SIMT model, tools/divergence_model.py, attributes half of the issued work of the
// projection kernel to that), here the rotation is a handful of selects.  Same mathematics, rounding differs in the last bits.
__device__ __forceinline__ double rot3(int k, double x0, double x1, double x2) { return k == 0 ? x0 : (k == 1 ? x1 : x2); }
// quadratic forms z1'S z1, z1'S z2, z2'S z2 of a symmetric S (diagonal SK, SU, SV; off-diagonal SUK, SUV, SKV in rotated indices) with
// z1 = aK e_U - aU e_K, z2 = aK e_V - aV e_K; with3 = false leaves the z2 forms at (0, 1) (two free variables)
__device__ __forceinline__ void null_forms(double SK, double SU, double SV, double SUK, double SUV, double SKV, double aK, double aU, double aV, bool with3,
                                           double &s11, double &s12, double &s22) {
  const double z1U = fma(SU, aK, -(SUK * aU)), z1K = fma(SUK, aK, -(SK * aU));
  s11 = fma(aK, z1U, -(aU * z1K));
  s12 = 0.0; s22 = 1.0;
  if (with3) {
    const double z2U = fma(SUV, aK, -(SUK * aV)), z2K = fma(SKV, aK, -(SK * aV)), z2V = fma(SV, aK, -(SKV * aV));
    s12 = fma(aK, z2U, -(aU * z2K)); s22 = fma(aK, z2V, -(aV * z2K));
  }
}
template <class EV>
__device__ __forceinline__ void tangent_step_rot(const EV &E, const int fix[3], double lam, double d[3]) {
  constexpr bool BOXE = std::is_same<EV, HexBox::EvalT>::value;
  d[0] = d[1] = d[2] = 0.0;
  const int nf = (fix[0] == 0) + (fix[1] == 0) + (fix[2] == 0);
  if (nf < 2) { ISO_TRACE(16); return; }
  int K;
  if (nf == 2) K = fix[0] ? 1 : (fix[1] ? 2 : 0);
  else { K = 0; if (fabs(E.a[1]) > fabs(E.a[K])) K = 1; if (fabs(E.a[2]) > fabs(K == 0 ? E.a[0] : E.a[1])) K = 2; }
  ISO_TRACE(18);
  const int U = K == 2 ? 0 : K + 1, V = K == 0 ? 2 : K - 1;
  const bool with3 = nf == 3;
  const double aK = rot3(K, E.a[0], E.a[1], E.a[2]), aU = rot3(U, E.a[0], E.a[1], E.a[2]), aV = rot3(V, E.a[0], E.a[1], E.a[2]);
  const double cK = rot3(K, E.c[0], E.c[1], E.c[2]), cU = rot3(U, E.c[0], E.c[1], E.c[2]), cV = rot3(V, E.c[0], E.c[1], E.c[2]);
  double m11, m12, m22, g11, g12, g22;
  // pair (U,K) is entry K, pair (U,V) entry U, pair (K,V) entry V of the cyclic pair numbering (0,1),(1,2),(2,0)
  if constexpr (BOXE) {
    const double hK = rot3(K, E.hh[0], E.hh[1], E.hh[2]), hU = rot3(U, E.hh[0], E.hh[1], E.hh[2]), hV = rot3(V, E.hh[0], E.hh[1], E.hh[2]);
    const double HUK = lam * rot3(K, E.hg[0], E.hg[1], E.hg[2]), HUV = lam * rot3(U, E.hg[0], E.hg[1], E.hg[2]), HKV = lam * rot3(V, E.hg[0], E.hg[1], E.hg[2]);
    null_forms(hK, hU, hV, HUK, HUV, HKV, aK, aU, aV, with3, m11, m12, m22);
    const double kK = hK * aU;      // Gauss-Newton part: diagonal only
    g11 = fma(hU * aK, aK, kK * aU); g12 = 0.0; g22 = 1.0;
    if (with3) { g12 = kK * aV; g22 = fma(hV * aK, aK, (hK * aV) * aV); }
  } else {
    const double hK = rot3(K, E.Hgn[0][0], E.Hgn[1][1], E.Hgn[2][2]), hU = rot3(U, E.Hgn[0][0], E.Hgn[1][1], E.Hgn[2][2]), hV = rot3(V, E.Hgn[0][0], E.Hgn[1][1], E.Hgn[2][2]);
    const double G0 = E.Hgn[0][1], G1 = E.Hgn[1][2], G2 = E.Hgn[2][0];
    const double M0 = G0 + fma(lam, E.hg[0], E.m[0]), M1 = G1 + fma(lam, E.hg[1], E.m[1]), M2 = G2 + fma(lam, E.hg[2], E.m[2]);
    null_forms(hK, hU, hV, rot3(K, M0, M1, M2), rot3(U, M0, M1, M2), rot3(V, M0, M1, M2), aK, aU, aV, with3, m11, m12, m22);
    null_forms(hK, hU, hV, rot3(K, G0, G1, G2), rot3(U, G0, G1, G2), rot3(V, G0, G1, G2), aK, aU, aV, with3, g11, g12, g22);
  }
  const double r1 = -fma(aK, cU, -(aU * cK)), r2 = with3 ? -fma(aK, cV, -(aV * cK)) : 0.0;
  double det = m11 * m22 - m12 * m12, detg = g11 * g22 - g12 * g12;
  if (!(m11 > 1e-8 * g11 && det > 1e-8 * detg)) { m11 = g11; m12 = g12; m22 = g22; det = detg; }
  if (!(det > 0.0 && m11 > 0.0)) return;
  // Two free variables: m12 = 0, m22 = 1, r2 = 0, so y2 = (+0) / det = +0 exactly -- and a zero numerator sends nvcc's FP64 division
  // down its out-of-line slow path (ncu, k_project_list: 11.7 % of all executed instructions at 7.5 of 32 lanes came from there).
  const double y1 = (m22 * r1 - m12 * r2) / det, y2 = with3 ? (m11 * r2 - m12 * r1) / det : 0.0;
  const double dU = y1 * aK, dV = y2 * aK, dK = -fma(y1, aU, y2 * aV);
  // rotate back: component i receives dK / dU / dV according to its role
#pragma unroll
  for (int i = 0; i < 3; i++) d[i] = (i == K) ? dK : ((i == U) ? dU : dV);
}
template <class EV, int MODE = 0>
__device__ __forceinline__ void tangent_step(const EV &E, const int fix[3], double lam, double d[3]) {
  if constexpr ((MODE & 2) != 0) { tangent_step_rot(E, fix, lam, d); return; }
  d[0] = d[1] = d[2] = 0.0;
  int nf = (fix[0] == 0) + (fix[1] == 0) + (fix[2] == 0);
  if (nf < 2) { ISO_TRACE(16); return; }
  if (nf == 2) {
    ISO_TRACE(fix[0] ? 13 : (fix[1] ? 14 : 15));
    if (fix[0]) tangent2<1, 2>(E, lam, d);
    else if (fix[1]) tangent2<0, 2>(E, lam, d);
    else tangent2<0, 1>(E, lam, d);
    return;
  }
  int k = 0;
  if (fabs(E.a[1]) > fabs(E.a[k])) k = 1;
  if (fabs(E.a[2]) > fabs(k == 0 ? E.a[0] : E.a[1])) k = 2;
  ISO_TRACE(10 + k);
  if (k == 0) { if (fabs(E.a[0]) > 0.0) tangent3<0>(E, lam, d); }
  else if (k == 1) { if (fabs(E.a[1]) > 0.0) tangent3<1>(E, lam, d); }
  else { if (fabs(E.a[2]) > 0.0) tangent3<2>(E, lam, d); }
}

// HEX8 projection as a resumable state machine: proj_init (phase 1) + proj_iter (ONE phase-2 iteration).  A: monomial
// coefficients [x,y,z,rho][8]; re: nodal densities (for the edge fallback).  project_hex8 below is init + iterate-to-the-end;
// the lane-refill kernel drives the two pieces itself so that the lanes of a warp can be at different iterations of
// different grid points.  The arithmetic and its order are the same in both drivers (bit-identical results).
struct ProjState { double xi[3]; double lam; double f; int it, stall; bool force; };      // f = |X(xi) - x|^2 at the current xi (valid once proj_iter has run)

template <class EL, int MODE = 0>
__device__ __forceinline__ bool proj_init(const EL &A, const double re[8], const double sg[8][3], const int edges[12][2],
                                          const double x[3], double rho_t, double gs, ProjState &S) {
  const double tolg = 1e-14 * gs;
  int fix[3] = {0, 0, 0};
  S.xi[0] = S.xi[1] = S.xi[2] = 0.0; S.lam = 0.0; S.f = 0.0; S.it = 0; S.stall = 0; S.force = false;
  bool ok = restore<EL, MODE>(A, rho_t, S.xi, fix, tolg);
  if (!ok) {
    double best = INFINITY;
    for (int e = 0; e < 12; e++) {
      int a = edges[e][0], b = edges[e][1]; double ra = re[a] - rho_t, rb = re[b] - rho_t;
      if ((ra <= 0 && rb >= 0) || (ra >= 0 && rb <= 0)) {
        double t = (ra == rb) ? 0.5 : ra / (ra - rb), cand[3];
#pragma unroll
        for (int d = 0; d < 3; d++) cand[d] = sg[a][d] + t * (sg[b][d] - sg[a][d]);
        double dd = eval_f(A, x, cand);
        if (dd < best) { best = dd; S.xi[0] = cand[0]; S.xi[1] = cand[1]; S.xi[2] = cand[2]; }
      }
    }
    if (!(best < INFINITY)) { S.xi[0] = S.xi[1] = S.xi[2] = 0.0; S.it = -1; return false; }
  }
  return true;
}
// Phase 1 without the edge fallback: the Newton projection of xi = 0 onto {g = 0} does not depend on the grid point, so a
// warp that works on one element computes it once and hands the state to every point (same arithmetic as proj_init).
template <class EL, int MODE = 0>
__device__ __forceinline__ bool proj_init_element(const EL &A, double rho_t, double gs, ProjState &S) {
  int fix[3] = {0, 0, 0};
  S.xi[0] = S.xi[1] = S.xi[2] = 0.0; S.lam = 0.0; S.f = 0.0; S.it = 0; S.stall = 0; S.force = false;
  return restore<EL, MODE>(A, rho_t, S.xi, fix, 1e-14 * gs);
}
// one phase-2 iteration; returns 0 = continue, 1 = converged, 2 = failed (line search exhausted)
template <class EL, int MODE = 0>
__device__ __forceinline__ int proj_iter(const EL &A, const double x[3], double rho_t, double gs, ProjState &S) {
  const double tolg = 1e-14 * gs, tolx = 1e-11, atol2 = 1e-24 * gs * gs;
  double *xi = S.xi; double lam = S.lam, dm = 0.0; bool force = S.force;
  int fix[3];
  {
    int bnd[3], tried[3] = {0, 0, 0};
#pragma unroll
    for (int i = 0; i < 3; i++) { bnd[i] = xi[i] >= 1.0 ? 1 : (xi[i] <= -1.0 ? -1 : 0); fix[i] = bnd[i]; }
    typename EL::EvalT E; eval_full(A, x, rho_t, xi, E);
    S.f = E.f;
    double d[3] = {0, 0, 0}; bool have_step = false; int status = 0;
    for (int pass = 0; pass < 8; pass++) {
      double num = 0, den = 0;
#pragma unroll
      for (int i = 0; i < 3; i++) if (!fix[i]) { num = fma(E.a[i], E.c[i], num); den = fma(E.a[i], E.a[i], den); }
      ISO_COUNT(5);
      if (den > atol2) { lam = -num / den; ISO_COUNT(3); tangent_step<typename EL::EvalT, MODE>(E, fix, lam, d); }
      else {
        ISO_TRACE(17);
        double llo = -INFINITY, lhi = INFINITY, akk = 0.0, ckk = 0.0; bool anyk = false;
#pragma unroll
        for (int i = 0; i < 3; i++) if (fix[i]) {
          double as = E.a[i] * fix[i], cs = E.c[i] * fix[i];
          if (as > 0) { double b = -cs / as; if (b < lhi) lhi = b; } else if (as < 0) { double b = -cs / as; if (b > llo) llo = b; }
          if (!anyk || fabs(E.a[i]) > fabs(akk)) { akk = E.a[i]; ckk = E.c[i]; anyk = true; }
        }
        if (llo <= lhi) lam = (llo > -INFINITY && lhi < INFINITY) ? 0.5 * (llo + lhi) : (llo > -INFINITY ? llo : (lhi < INFINITY ? lhi : 0.0));
        else if (anyk && akk != 0.0) lam = -ckk / akk;
        d[0] = d[1] = d[2] = 0.0;
#pragma unroll
        for (int i = 0; i < 3; i++) if (!fix[i]) {
          double h = hdiag(E, i); if (h > 0.0) d[i] = -E.c[i] / h;    // Hess g has a zero diagonal
        }
      }
      bool refix = false;
#pragma unroll
      for (int i = 0; i < 3; i++) if (!fix[i] && bnd[i] && d[i] * bnd[i] > 0.0) { if (fabs(d[i]) <= tolx) d[i] = 0.0; else { fix[i] = bnd[i]; refix = true; } }      // a numerically zero outward component is noise, not a reason to re-fix
      if (refix) continue;
      dm = fmax(fabs(d[0]), fmax(fabs(d[1]), fabs(d[2])));
      if (dm > tolx && !force) { have_step = true; break; }
      int worst = -1; double wv = 0.0;
#pragma unroll
      for (int i = 0; i < 3; i++) if (fix[i] && !tried[i]) {
        double gain = fma(lam, E.a[i], E.c[i]) * (double)fix[i];
        if (gain > 1e-10 * (fabs(E.c[i]) + fabs(lam * E.a[i]) + 1e-300) && gain > wv) { wv = gain; worst = i; }
      }
      if (worst < 0) { status = 1; break; }
#pragma unroll
      for (int i = 0; i < 3; i++) if (i == worst) { fix[i] = 0; tried[i] = 1; }
      force = false;
    }
    S.lam = lam; S.force = force;
    if (status) return 1;
    if (!have_step) return 1;
    double amax = 1.0; int blk = -1;
#pragma unroll
    for (int i = 0; i < 3; i++) if (!fix[i]) {
      // ties between blocking bounds (within 1e-12) go to the lower index, so that round-off cannot choose the face
      if (d[i] > 0 && xi[i] + d[i] > 1.0) { double t = (1.0 - xi[i]) / d[i]; if (t < amax * (1.0 - 1e-12)) { amax = t; blk = i; } }
      if (d[i] < 0 && xi[i] + d[i] < -1.0) { double t = (-1.0 - xi[i]) / d[i]; if (t < amax * (1.0 - 1e-12)) { amax = t; blk = i; } }
    }
    double slope = fma(E.c[2], d[2], fma(E.c[1], d[1], E.c[0] * d[0]));
    if (!(slope < 0.0)) { S.force = true; S.it++; return 0; }      // no descent left on this face: go to the multiplier test
    double alpha = amax; bool acc = false;
    for (int ls = 0; ls < 40; ls++) {
      double xt[3]; int fx[3];
#pragma unroll
      for (int i = 0; i < 3; i++) {
        fx[i] = fix[i]; xt[i] = fma(alpha, d[i], xi[i]);
        if (i == blk && alpha == amax) { xt[i] = d[i] > 0 ? 1.0 : -1.0; fx[i] = d[i] > 0 ? 1 : -1; }
        if (xt[i] >= 1.0) { xt[i] = 1.0; fx[i] = 1; }
        if (xt[i] <= -1.0) { xt[i] = -1.0; fx[i] = -1; }
      }
      ISO_COUNT(4); ISO_TRACE(2);
      if (restore<EL, MODE>(A, rho_t, xt, fx, tolg)) {
        double ft = eval_f(A, x, xt);
        // steps below 1e-7 are in Newton's quadratic regime: accepted without the Armijo test (decrease below noise)
        if (dm <= 1e-7 || ft <= E.f + 1e-4 * alpha * slope + 1e-15 * E.f) {
          if (E.f - ft <= 1e-15 * E.f) S.stall++; else S.stall = 0;
          xi[0] = xt[0]; xi[1] = xt[1]; xi[2] = xt[2]; acc = true; S.f = ft;
          // A full Newton step of size dm <= 1e-6 that ends strictly inside the box leaves an error of O(dm^2) <= 1e-12: the
          // next iteration would only confirm |step| <= tolx, so it is skipped (saves one evaluation of ~3.5 per pair; the CPU
          // oracle keeps the confirming iteration -- the two agree to ~1e-12 in xi, far inside the 1e-9 h tolerance).
          if (dm <= 1e-6 && alpha == 1.0 && fx[0] == 0 && fx[1] == 0 && fx[2] == 0) { S.it++; return 1; }
          break;
        }
      }
      alpha *= 0.5;
    }
    if (!acc) { if (dm < 1e-6) { S.force = true; S.it++; return 0; } return 2; }
    if (S.stall >= 3) { S.force = true; S.stall = 0; }
  }
  S.it++;
  return 0;
}
// Returns true when converged; xi receives the local coordinates; nit the phase-2 iteration count.
template <class EL, int MODE = 0>
__device__ __forceinline__ bool project_hex8(const EL &A, const double re[8], const double sg[8][3], const int edges[12][2],
                                             const double x[3], double rho_t, double gs, double xi[3], int &nit) {
  ProjState S;
  if (!proj_init<EL, MODE>(A, re, sg, edges, x, rho_t, gs, S)) { xi[0] = xi[1] = xi[2] = 0.0; nit = -1; return false; }
  int status = 0;
  while (S.it < 100 && status == 0) status = proj_iter<EL, MODE>(A, x, rho_t, gs, S);
  xi[0] = S.xi[0]; xi[1] = S.xi[1]; xi[2] = S.xi[2];
  nit = S.it;
  return status == 1;
}
// The same with phase 1 taken from a per-element table (xi0 = Newton projection of xi = 0 onto {g = 0}, ok0 = it converged): phase 1
// does not depend on the grid point, so one thread per element can compute it once instead of every (element, point) pair.
template <class EL, int MODE = 0>
__device__ __forceinline__ bool project_hex8_from(const EL &A, const double re[8], const double sg[8][3], const int edges[12][2],
                                                  const double x[3], double rho_t, double gs, const double xi0[3], bool ok0, double xi[3], int &nit) {
  ProjState S;
  S.xi[0] = xi0[0]; S.xi[1] = xi0[1]; S.xi[2] = xi0[2]; S.lam = 0.0; S.f = 0.0; S.it = 0; S.stall = 0; S.force = false;
  if (!ok0 && !proj_init<EL, MODE>(A, re, sg, edges, x, rho_t, gs, S)) { xi[0] = xi[1] = xi[2] = 0.0; nit = -1; return false; }
  int status = 0;
  while (S.it < 100 && status == 0) status = proj_iter<EL, MODE>(A, x, rho_t, gs, S);
  xi[0] = S.xi[0]; xi[1] = S.xi[1]; xi[2] = S.xi[2];
  nit = S.it;
  return status == 1;
}

// monomial coefficients of a trilinear field from its 8 nodal values (node order of hex8_shape.jl:27-34)
__device__ __forceinline__ void monomial8(const double v[8], double A[8]) {
  double s01 = v[0] + v[1], d01 = v[1] - v[0], s32 = v[3] + v[2], d32 = v[2] - v[3];
  double s45 = v[4] + v[5], d45 = v[5] - v[4], s76 = v[7] + v[6], d76 = v[6] - v[7];
  // bottom (z=-1) and top (z=+1) bilinear coefficients
  double b0 = s01 + s32, b1 = d01 + d32, b2 = s32 - s01, b3 = d32 - d01;     // 4*(c, x, e, xe) on bottom
  double t0 = s45 + s76, t1 = d45 + d76, t2 = s76 - s45, t3 = d76 - d45;     // on top
  A[0] = 0.125 * (b0 + t0); A[1] = 0.125 * (b1 + t1); A[2] = 0.125 * (b2 + t2); A[4] = 0.125 * (b3 + t3);
  A[3] = 0.125 * (t0 - b0); A[6] = 0.125 * (t1 - b1); A[5] = 0.125 * (t2 - b2); A[7] = 0.125 * (t3 - b3);
}

// ----------------------------------------------------------------------------------------------------------------
// TET4 (ComputeCoordsOnIso.jl:90-181): rho is affine on the tet -> projection of x onto the convex polygon {rho=rho_t}
// ----------------------------------------------------------------------------------------------------------------
__device__ __forceinline__ double det3(const double M[3][3]) {
  return M[0][0] * (M[1][1] * M[2][2] - M[1][2] * M[2][1]) - M[0][1] * (M[1][0] * M[2][2] - M[1][2] * M[2][0]) + M[0][2] * (M[1][0] * M[2][1] - M[1][1] * M[2][0]);
}
__device__ __forceinline__ void closest_on_segment(const double a[3], const double b[3], const double x[3], double q[3]) {
  double e[3] = {b[0] - a[0], b[1] - a[1], b[2] - a[2]}, ee = (e[0] * e[0] + e[1] * e[1]) + e[2] * e[2];
  double t = ee > 0 ? (((x[0] - a[0]) * e[0] + (x[1] - a[1]) * e[1]) + (x[2] - a[2]) * e[2]) / ee : 0.0;
  t = fmin(fmax(t, 0.0), 1.0);
#pragma unroll
  for (int d = 0; d < 3; d++) q[d] = a[d] + t * e[d];
}
__device__ inline bool project_tet4(const double Xe[3][4], const double re[4], const int isn[4][3], const double x[3], double rho_t, double xp[3]) {
  double M[3][3], r[3] = {re[1] - re[0], re[2] - re[0], re[3] - re[0]}, G[3];
#pragma unroll
  for (int d = 0; d < 3; d++) { M[0][d] = Xe[d][1] - Xe[d][0]; M[1][d] = Xe[d][2] - Xe[d][0]; M[2][d] = Xe[d][3] - Xe[d][0]; }
  double det = det3(M);
  if (!(fabs(det) > 0.0)) return false;
#pragma unroll
  for (int c = 0; c < 3; c++) {
    double B[3][3];
#pragma unroll
    for (int k = 0; k < 3; k++)
#pragma unroll
      for (int l = 0; l < 3; l++) B[k][l] = (l == c) ? r[k] : M[k][l];
    G[c] = det3(B) / det;
  }
  double gg = (G[0] * G[0] + G[1] * G[1]) + G[2] * G[2];
  if (!(gg > 0.0)) return false;
  double rx = re[0] + ((G[0] * (x[0] - Xe[0][0]) + G[1] * (x[1] - Xe[1][0])) + G[2] * (x[2] - Xe[2][0]));
  double s = (rx - rho_t) / gg, q[3] = {x[0] - s * G[0], x[1] - s * G[1], x[2] - s * G[2]};
  {  // barycentrics of q (columns of M^T are the edge vectors)
    double A[3][3], b[3], l[4];
#pragma unroll
    for (int d = 0; d < 3; d++) { A[d][0] = M[0][d]; A[d][1] = M[1][d]; A[d][2] = M[2][d]; b[d] = q[d] - Xe[d][0]; }
    double dA = det3(A);
#pragma unroll
    for (int c = 0; c < 3; c++) {
      double B[3][3];
#pragma unroll
      for (int k = 0; k < 3; k++)
#pragma unroll
        for (int m = 0; m < 3; m++) B[k][m] = (m == c) ? b[k] : A[k][m];
      l[c + 1] = det3(B) / dA;
    }
    l[0] = 1.0 - ((l[1] + l[2]) + l[3]);
    if (l[0] >= 0.0 && l[1] >= 0.0 && l[2] >= 0.0 && l[3] >= 0.0) { xp[0] = q[0]; xp[1] = q[1]; xp[2] = q[2]; return true; }
  }
  double best = INFINITY;
  for (int f = 0; f < 4; f++) {
    double P[3][3]; int np = 0;
    for (int e = 0; e < 3 && np < 3; e++) {
      int a = isn[f][e], b = isn[f][(e + 1) % 3]; double ra = re[a] - rho_t, rb = re[b] - rho_t;
      if ((ra <= 0 && rb > 0) || (ra > 0 && rb <= 0) || (ra < 0 && rb >= 0) || (ra >= 0 && rb < 0)) {
        double t = ra / (ra - rb);
        for (int d = 0; d < 3; d++) P[np][d] = Xe[d][a] + t * (Xe[d][b] - Xe[d][a]);
        np++;
      }
    }
    if (np < 2) continue;
    for (int i = 0; i < np; i++) {
      if (np == 2 && i == 1) break;
      int j = (i + 1) % np; double c[3]; closest_on_segment(P[i], P[j], x, c);
      double dd = ((x[0] - c[0]) * (x[0] - c[0]) + (x[1] - c[1]) * (x[1] - c[1])) + (x[2] - c[2]) * (x[2] - c[2]);
      if (dd < best) { best = dd; xp[0] = c[0]; xp[1] = c[1]; xp[2] = c[2]; }
    }
  }
  return best < INFINITY;
}
}  // namespace iso

// solver variant the distance kernels use (r2s_dist.cu, r2s_points.cu): FAST restoration, one code path for all tangent-step cases
#define PMODE 3
