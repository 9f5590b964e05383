// bound_host.cpp -- the lower bounds of the box projection's pair scans (rho2sdf.jl_b200/csrc/r2s_bound.cuh) and the projection of
// k_project_list (r2s_iso.cuh, element-local coordinates, phase 1 once per element) compiled for the HOST, for
// tests/test_proj_bound_host.py and tools/prune_study.py.  Test infrastructure only.
#include <math.h>
#ifndef __device__
#define __device__
#endif
#ifndef __forceinline__
#define __forceinline__ inline __attribute__((always_inline))
#endif
#include "../../rho2sdf.jl_b200/csrc/r2s_iso.cuh"
#include "../../rho2sdf.jl_b200/csrc/r2s_bound.cuh"

static const double sg[8][3] = {{-1, -1, -1}, {1, -1, -1}, {1, 1, -1}, {-1, 1, -1}, {-1, -1, 1}, {1, -1, 1}, {1, 1, 1}, {-1, 1, 1}};
static const int edges[12][2] = {{0, 1}, {1, 2}, {2, 3}, {3, 0}, {4, 5}, {5, 6}, {6, 7}, {7, 4}, {0, 4}, {1, 5}, {2, 6}, {3, 7}};

// the element set-up of k_box_records: node 0 as origin, monomial coefficients, HexBox, tolerance scale.  Returns false if not a box.
static bool setup(const double *Xe /*[8][3]*/, const double *re, double rho_t, double org[3], iso::HexBox &H, double &gs) {
  double A[4][8];
  for (int d = 0; d < 3; d++) {
    org[d] = Xe[d];
    double nv[8];
    for (int k = 0; k < 8; k++) nv[k] = Xe[3 * k + d] - org[d];
    iso::monomial8(nv, A[d]);
  }
  iso::monomial8(re, A[3]);
  if (!iso::is_box(A)) return false;
  iso::make_box(A, H);
  gs = fabs(rho_t);
  for (int k = 0; k < 8; k++) gs = fmax(gs, fabs(re[k]));
  gs = fmax(gs, 1.0);
  return true;
}

extern "C" {
// out[11]: tlo[3], thi[3], n[3], A, B as k_box_records stores them.  Returns 0 when the element is not an axis-aligned box.
int bnd_host_element(const double *Xe, const double *re, double rho_t, double *out) {
  double org[3], gs; iso::HexBox H;
  if (!setup(Xe, re, rho_t, org, H, gs)) return 0;
  bnd::box_iso_bounds(re, rho_t, gs, org, H.c, H.h, out, out + 3, out + 6, out[9], out[10]);
  return 1;
}
// lower bound of n points P[n][3] for the element record rec[11] of bnd_host_element
void bnd_host_lb(long n, const double *P, const double *rec, double *out) {
  for (long q = 0; q < n; q++) out[q] = bnd::lb_box_slab(P + 3 * q, rec, rec + 3, rec + 6, rec[9], rec[10]);
}
// lb2_box_gap (squared) of n points
void bnd_host_lb2gap(long n, const double *P, const double *rec, double *out) {
  for (long q = 0; q < n; q++) out[q] = bnd::lb2_box_gap(P + 3 * q, rec, rec + 3, rec + 6, rec[9], rec[10]);
}
// the distance k_project_list reports for n points P[n][3] of one box element; ok[q] = 1 when the solver converged.  Returns -1 when
// the element is not a box.
int bnd_host_project(const double *Xe, const double *re, double rho_t, long n, const double *P, double *dist, int *ok, int *its) {
  double org[3], gs; iso::HexBox H;
  if (!setup(Xe, re, rho_t, org, H, gs)) return -1;
  iso::ProjState S0; const bool ok0 = iso::proj_init_element<iso::HexBox, 3>(H, rho_t, gs, S0);
  for (long q = 0; q < n; q++) {
    const double x[3] = {P[3 * q] - org[0], P[3 * q + 1] - org[1], P[3 * q + 2] - org[2]};
    iso::ProjState S; S.xi[0] = S0.xi[0]; S.xi[1] = S0.xi[1]; S.xi[2] = S0.xi[2]; S.lam = 0.0; S.f = 0.0; S.it = 0; S.stall = 0; S.force = false;
    bool okc = true;
    if (!ok0) okc = iso::proj_init<iso::HexBox, 3>(H, re, sg, edges, x, rho_t, gs, S);
    double xi[3] = {0.0, 0.0, 0.0}, p[3];
    if (okc) {
      int status = 0;
      while (S.it < 100 && status == 0) status = iso::proj_iter<iso::HexBox, 3>(H, x, rho_t, gs, S);
      okc = status == 1;
      xi[0] = S.xi[0]; xi[1] = S.xi[1]; xi[2] = S.xi[2];
    }
    iso::eval_pos(H, xi, p);
    const double d0 = x[0] - p[0], d1 = x[1] - p[1], d2 = x[2] - p[2];
    dist[q] = sqrt(fma(d2, d2, fma(d1, d1, d0 * d0))); ok[q] = okc ? 1 : 0; its[q] = S.it;
  }
  return 0;
}
}
