// r2s_replay.cuh -- the per-point replay of evalDistances' running minimum (sdfOnDensityField.jl:44-119, :489-815), shared by the grid
// path (r2s_dist.cu) and the points path (r2s_points.cu): boundary-face triangles and their candidate tests, bit-exact (r2s_exact.cuh).
#pragma once
#include "r2s_common.cuh"
#include "r2s_tables.cuh"
#include "r2s_exact.cuh"

struct VoxState { double c; double xp[3]; };
template <bool WANT_XP>
__device__ __forceinline__ void write_value(VoxState &s, double dt, const double xp[3]) {   // WriteValue :44-57
  if (fabs(dt) < fabs(s.c)) { s.c = dt; if (WANT_XP) { s.xp[0] = xp[0]; s.xp[1] = xp[1]; s.xp[2] = xp[2]; } }
}
// IsProjectedOnFullSegment (:78-119)
template <bool WANT_XP, int NEN>
__device__ inline bool projected_on_full_segment(const double Xe[3][NEN], const double re[NEN], double rho_t, const double xp[3], const double x[3], VoxState &s,
                                                 const ex::AffineInv *pre = nullptr) {
  double rho;
  if (NEN == 8) {
    double xi[3], N[8];
    if (pre && pre->affine) ex::affine_inverse_apply(*pre, xp, xi);      // same arithmetic as the general path on an affine element
    else ex::inverse_map_hex8((const double(*)[8])Xe, xp, xi);
    if (!(ex::max3abs(xi[0], xi[1], xi[2]) < 1.001)) return false;
    ex::hex8_shape(xi, N);
    rho = ex::dot8(N, re);
  } else {
    double lc[3];
    if (!ex::inverse_map_tet4((const double(*)[4])Xe, xp, lc)) return false;
    if (!(lc[0] >= 0 && lc[1] >= 0 && lc[2] >= 0 && ex::add(ex::add(lc[0], lc[1]), lc[2]) <= 1.0)) return false;
    double l4 = ex::sub(1.0, ex::add(ex::add(lc[0], lc[1]), lc[2]));
    rho = ex::add(ex::add(ex::add(ex::mul(lc[0], re[0]), ex::mul(lc[1], re[1])), ex::mul(lc[2], re[2])), ex::mul(l4, re[3]));
  }
  if (rho >= rho_t) { write_value<WANT_XP>(s, ex::norm3(ex::sub(x[0], xp[0]), ex::sub(x[1], xp[1]), ex::sub(x[2], xp[2])), xp); return true; }
  return false;
}
// process_triangle_projection! (:628-815) for one grid point
template <bool WANT_XP, int NEN>
__device__ inline void triangle_point(const double Xe[3][NEN], const double re[NEN], double rho_t, bool solid, const double Xt[3][3], const double Et[3][3],
                                      const double n[3], const double x[3], VoxState &s, const ex::AffineInv *pre = nullptr) {
  double lam[3]; ex::barycentric(Xt[0], Xt[1], Xt[2], n, x, lam);
  double xp[3]; bool ok = false;
  double lmin = lam[0]; if (lam[1] < lmin) lmin = lam[1]; if (lam[2] < lmin) lmin = lam[2];
  if (lmin >= 0.0) {
#pragma unroll
    for (int d = 0; d < 3; d++) xp[d] = ex::add(ex::add(ex::mul(lam[0], Xt[0][d]), ex::mul(lam[1], Xt[1][d])), ex::mul(lam[2], Xt[2][d]));
    double dt = ex::norm3(ex::sub(x[0], xp[0]), ex::sub(x[1], xp[1]), ex::sub(x[2], xp[2]));
    if (solid) { if (fabs(dt) < fabs(s.c)) { write_value<WANT_XP>(s, dt, xp); ok = true; } }
    else ok = projected_on_full_segment<WANT_XP, NEN>(Xe, re, rho_t, xp, x, s, pre);
  } else {
#pragma unroll
    for (int j = 0; j < 3; j++) {
      if (ok) continue;      // "break" on the first successful edge
      double L = ex::norm3(Et[j][0], Et[j][1], Et[j][2]);
      double u[3] = {ex::dvd(Et[j][0], L), ex::dvd(Et[j][1], L), ex::dvd(Et[j][2], L)};
      double P = ex::add(ex::add(ex::mul(ex::sub(x[0], Xt[j][0]), u[0]), ex::mul(ex::sub(x[1], Xt[j][1]), u[1])), ex::mul(ex::sub(x[2], Xt[j][2]), u[2]));
      if (P >= 0 && P <= L) {
#pragma unroll
        for (int d = 0; d < 3; d++) xp[d] = ex::add(Xt[j][d], ex::mul(u[d], P));
        double dt = ex::norm3(ex::sub(x[0], xp[0]), ex::sub(x[1], xp[1]), ex::sub(x[2], xp[2]));
        if (solid) { if (fabs(dt) < fabs(s.c)) { write_value<WANT_XP>(s, dt, xp); ok = true; } }
        else ok = projected_on_full_segment<WANT_XP, NEN>(Xe, re, rho_t, xp, x, s, pre);
      }
    }
  }
  if (!ok) {
    double dd[3];
#pragma unroll
    for (int j = 0; j < 3; j++) dd[j] = ex::norm3(ex::sub(x[0], Xt[j][0]), ex::sub(x[1], Xt[j][1]), ex::sub(x[2], Xt[j][2]));
    int idx = 0; if (dd[1] < dd[idx]) idx = 1; if (dd[2] < dd[idx]) idx = 2;
    double dmin = idx == 0 ? dd[0] : (idx == 1 ? dd[1] : dd[2]);
#pragma unroll
    for (int d = 0; d < 3; d++) xp[d] = idx == 0 ? Xt[0][d] : (idx == 1 ? Xt[1][d] : Xt[2][d]);
    if (solid) write_value<WANT_XP>(s, dmin, xp);
    else projected_on_full_segment<WANT_XP, NEN>(Xe, re, rho_t, xp, x, s, pre);
  }
}
// Boundary-face triangles (process_boundary_faces! :489-558): every boundary face of an active element is split into nsn
// triangles around its centroid (:520-529).  The triangles and the grid-point range of their (AABB +- delta) cell range
// (Grid.jl:122-154) do not depend on the grid point, so they are built ONCE per call into a table (one thread per active
// element) instead of once per (grid point, candidate element) inside the assemble kernel.
struct TriRec {
  int ps[3], pe[3];      // candidate grid-point range per axis [ps, pe)
  double Xt[3][3];       // vertices (x1, x2, centroid)
  double n[3];           // unit normal
  double lo[3], hi[3];   // bounding box of the three vertices (lower bound of every candidate distance, k_assemble)
  double rlo[3], rhi[3]; // in the FIRST triangle of an element: bounding box of all its boundary triangles (record-level bound)
};
// The nsn triangles of every boundary face of one element (fmask bit sg = face sg), in the reference's order, with the candidate range of
// each: grid-point ranges [cstart[I0], cstart[I1 + 1]) for the grid path (CELLS = false), the cell ranges [I0, I1 + 1) themselves for
// arbitrary points (CELLS = true).  tri[0] also gets the box around all of them (rlo, rhi).
template <int NEN, bool CELLS>
__device__ void face_triangles(const double Xe[3][NEN], int fmask, const GridDev &g, double delta, TriRec *__restrict__ tri) {
  constexpr int NSN = NEN == 8 ? 4 : 3, NES = NEN == 8 ? 6 : 4;
  int o = 0;
  double rlo[3] = {1e300, 1e300, 1e300}, rhi[3] = {-1e300, -1e300, -1e300};
  for (int sg = 0; sg < NES; sg++) {
    if (!((fmask >> sg) & 1)) continue;
    double Xs[NSN][3], Xc[3];
    for (int q = 0; q < NSN; q++) { int ln = NEN == 8 ? c_hex_isn[sg][q] : c_tet_isn[sg][q]; for (int d = 0; d < 3; d++) Xs[q][d] = Xe[d][ln]; }
    for (int d = 0; d < 3; d++) { double t = Xs[0][d]; for (int q = 1; q < NSN; q++) t = ex::add(t, Xs[q][d]); Xc[d] = ex::dvd(t, (double)NSN); }
    for (int q = 0; q < NSN; q++) {
      int q2 = (q + 1) % NSN; TriRec T; double Et[2][3];
      for (int d = 0; d < 3; d++) { T.Xt[0][d] = Xs[q][d]; T.Xt[1][d] = Xs[q2][d]; T.Xt[2][d] = Xc[d]; }
      bool ok = true;
      for (int d = 0; d < 3; d++) {
        double lo = fmin(T.Xt[0][d], fmin(T.Xt[1][d], T.Xt[2][d])), hi = fmax(T.Xt[0][d], fmax(T.Xt[1][d], T.Xt[2][d])); int I0 = 0, I1 = -1;
        T.lo[d] = lo; T.hi[d] = hi; rlo[d] = fmin(rlo[d], lo); rhi[d] = fmax(rhi[d], hi); T.rlo[d] = 0.0; T.rhi[d] = 0.0;
        ok = ok && ex::cell_range_axis(lo, hi, delta, g.amin[d], g.amax[d], g.N[d], I0, I1);
        if (ok) {
          if (CELLS) { T.ps[d] = I0; T.pe[d] = I1 + 1; }
          else { T.ps[d] = g.cstart[g.cs_off[d] + I0]; T.pe[d] = g.cstart[g.cs_off[d] + I1 + 1]; }
        } else { T.ps[d] = 0; T.pe[d] = 0; }
      }
      if (!ok) { for (int d = 0; d < 3; d++) { T.ps[d] = 0; T.pe[d] = 0; } }
      for (int d = 0; d < 3; d++) { Et[0][d] = ex::sub(T.Xt[1][d], T.Xt[0][d]); Et[1][d] = ex::sub(T.Xt[2][d], T.Xt[1][d]); }
      T.n[0] = ex::sub(ex::mul(Et[0][1], Et[1][2]), ex::mul(Et[0][2], Et[1][1]));
      T.n[1] = ex::sub(ex::mul(Et[0][2], Et[1][0]), ex::mul(Et[0][0], Et[1][2]));
      T.n[2] = ex::sub(ex::mul(Et[0][0], Et[1][1]), ex::mul(Et[0][1], Et[1][0]));
      double nn = ex::norm3(T.n[0], T.n[1], T.n[2]);
      T.n[0] = ex::dvd(T.n[0], nn); T.n[1] = ex::dvd(T.n[1], nn); T.n[2] = ex::dvd(T.n[2], nn);
      tri[o++] = T;
    }
  }
  for (int d = 0; d < 3; d++) { tri[0].rlo[d] = rlo[d]; tri[0].rhi[d] = rhi[d]; }
}
