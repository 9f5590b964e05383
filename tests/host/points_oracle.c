/*
 * points_oracle.c -- CPU reference of evalDistances / Sign_Detection at a list of points, for the tests of the points entry points
 * (r2s_eval_distances_points / r2s_sign_detection_points).  TEST INFRASTRUCTURE: it restates the reference with a point list on top of
 * the CPU oracle (oracle/r2s_oracle.c, included whole so that every per-point step -- triangle_point, project_iso_hex8, inverse maps,
 * cell_range -- is the oracle's own), literal and serial apart from OpenMP over the points of the sign rule.  Built by
 * tests/points_oracle.py with the oracle's flags (-ffp-contract=off).
 */
#include "../../oracle/r2s_oracle.c"

/* ------------------------------------------------------------------------------------------------
 * evalDistances / Sign_Detection at a list of points (the reference's `points` argument, LinkedList(grid, points), Grid.jl:47-69).
 * Distances: a point's cell per axis is floor(N (x - amin) / (amax - amin)) (the expression of grid_init's cellof), not clamped; a point
 * whose cell lies outside [0, N] on some axis is in no element's range.  The loops over cstart ranges of the grid functions become loops
 * over the points whose cell lies in the range (points binned by linear cell id, ascending point id within a cell); every per-point
 * step is the grid functions' own.  Signs: the per-point candidate rules of r2so_sign_detection, candidates in ascending element order.
 * ---------------------------------------------------------------------------------------------- */
typedef struct { i64 n; const double *P; i64 *cptr, *pid; i64 nc[3]; } opts;     /* points by cell: pid[cptr[c] .. cptr[c+1]) */
static int point_cell(const ogrid *g, const double x[3], i64 c[3]) {
  for (int d = 0; d < 3; d++) {
    double f = floor((double)g->N[d] * (x[d] - g->amin[d]) / (g->amax[d] - g->amin[d]));
    if (!(f >= 0 && f <= (double)g->N[d])) return 0;
    c[d] = (i64)f;
  }
  return 1;
}
static void pts_bin(const ogrid *g, const double *P, i64 n, opts *o) {
  o->n = n; o->P = P;
  for (int d = 0; d < 3; d++) o->nc[d] = g->N[d] + 1;
  i64 ncell = o->nc[0] * o->nc[1] * o->nc[2], *cid = (i64 *)malloc(sizeof(i64) * (size_t)(n > 0 ? n : 1));
  o->cptr = (i64 *)calloc((size_t)ncell + 1, sizeof(i64)); o->pid = (i64 *)malloc(sizeof(i64) * (size_t)(n > 0 ? n : 1));
  for (i64 v = 0; v < n; v++) {
    i64 c[3]; cid[v] = point_cell(g, P + 3 * v, c) ? (c[2] * o->nc[1] + c[1]) * o->nc[0] + c[0] : -1;
    if (cid[v] >= 0) o->cptr[cid[v] + 1]++;
  }
  for (i64 c = 0; c < ncell; c++) o->cptr[c + 1] += o->cptr[c];
  i64 *fill = (i64 *)calloc((size_t)ncell, sizeof(i64));
  for (i64 v = 0; v < n; v++) if (cid[v] >= 0) o->pid[o->cptr[cid[v]] + fill[cid[v]]++] = v;
  free(fill); free(cid);
}
#define FOR_POINTS_IN(o, I0, I1, v)                                                                       \
  for (i64 ck = I0[2]; ck <= I1[2]; ck++) for (i64 cj = I0[1]; cj <= I1[1]; cj++) for (i64 ci = I0[0]; ci <= I1[0]; ci++) \
  for (i64 q = (o)->cptr[(ck * (o)->nc[1] + cj) * (o)->nc[0] + ci], qe = (o)->cptr[(ck * (o)->nc[1] + cj) * (o)->nc[0] + ci + 1], v = 0; q < qe && ((v = (o)->pid[q]), 1); q++)
static void pts_boundary_faces(const omesh *m, const ogrid *g, const opts *o, i64 el, const double *rho_n, double rho_t, double delta, int solid, double *dist, double *xpo) {
  for (int sg = 0; sg < m->nes; sg++) {
    if (!face_is_boundary(m, el, sg)) continue;
    const int *fn = m->nen == 8 ? HEX_ISN[sg] : TET_ISN[sg];
    double Xs[4][3], Xc[3];
    for (int a = 0; a < m->nsn; a++) for (int d = 0; d < 3; d++) Xs[a][d] = m->X[3 * (m->IEN[m->nen * el + fn[a]] - 1) + d];
    for (int d = 0; d < 3; d++) { double s = Xs[0][d]; for (int a = 1; a < m->nsn; a++) s = s + Xs[a][d]; Xc[d] = s / (double)m->nsn; }
    for (int a = 0; a < m->nsn; a++) {
      double Xt[3][3], Et[3][3], n[3], lo[3], hi[3];
      int a2 = (a + 1) % m->nsn;
      for (int d = 0; d < 3; d++) { Xt[0][d] = Xs[a][d]; Xt[1][d] = Xs[a2][d]; Xt[2][d] = Xc[d]; }
      for (int d = 0; d < 3; d++) { Et[0][d] = Xt[1][d] - Xt[0][d]; Et[1][d] = Xt[2][d] - Xt[1][d]; Et[2][d] = Xt[0][d] - Xt[2][d]; }
      n[0] = Et[0][1] * Et[1][2] - Et[0][2] * Et[1][1]; n[1] = Et[0][2] * Et[1][0] - Et[0][0] * Et[1][2]; n[2] = Et[0][0] * Et[1][1] - Et[0][1] * Et[1][0];
      double nn = norm3(n); n[0] = n[0] / nn; n[1] = n[1] / nn; n[2] = n[2] / nn;
      for (int d = 0; d < 3; d++) { lo[d] = fmin(Xt[0][d], fmin(Xt[1][d], Xt[2][d])); hi[d] = fmax(Xt[0][d], fmax(Xt[1][d], Xt[2][d])); }
      i64 I0[3], I1[3]; if (!cell_range(g, lo, hi, delta, I0, I1)) continue;
      FOR_POINTS_IN(o, I0, I1, v) triangle_point(m, el, rho_n, rho_t, solid, (const double(*)[3])Xt, (const double(*)[3])Et, n, o->P + 3 * v, dist, xpo, v);
    }
  }
}
static void pts_isocontour_element(const omesh *m, const ogrid *g, const opts *o, i64 el, const double *rho_n, double rho_t, double delta, double *dist, double *xpo, i64 *stats) {
  pts_boundary_faces(m, g, o, el, rho_n, rho_t, delta, 0, dist, xpo);
  double Xe8[3][8], Xe4[3][4], re[8], lo[3] = {DBL_MAX, DBL_MAX, DBL_MAX}, hi[3] = {-DBL_MAX, -DBL_MAX, -DBL_MAX};
  for (int a = 0; a < m->nen; a++) {
    i64 n = m->IEN[m->nen * el + a] - 1; re[a] = rho_n[n];
    for (int d = 0; d < 3; d++) { double c = m->X[3 * n + d]; if (m->nen == 8) Xe8[d][a] = c; else Xe4[d][a] = c; if (c < lo[d]) lo[d] = c; if (c > hi[d]) hi[d] = c; }
  }
  i64 I0[3], I1[3]; if (!cell_range(g, lo, hi, delta, I0, I1)) return;
  FOR_POINTS_IN(o, I0, I1, v) {
    const double *x = o->P + 3 * v; double xp[3];
    if (m->nen == 8) {
      double xi[3], N[8]; int nit = 0;
      int ok = project_iso_hex8(x, rho_t, (const double(*)[8])Xe8, re, xi, &nit);
      if (stats) { stats[0]++; stats[1] += nit > 0 ? nit : 0; if (!ok) stats[2]++; }
      hex8_shape(xi, N);
      for (int d = 0; d < 3; d++) { double s = 0; for (int a = 0; a < 8; a++) s += Xe8[d][a] * N[a]; xp[d] = s; }
    } else {
      int ok = project_iso_tet4(x, rho_t, (const double(*)[4])Xe4, re, xp);
      if (stats) { stats[0]++; if (!ok) stats[2]++; }
      if (!ok) continue;
    }
    double dv[3] = {x[0] - xp[0], x[1] - xp[1], x[2] - xp[2]};
    write_value(norm3(dv), xp, dist, xpo, v);
  }
}
API int r2so_eval_distances_points(i64 nnp, const double *X, i64 nel, int nen, const i64 *IEN, const double *amin, const double *amax, const i64 *N, double cell,
                                   const double *rho_n, double rho_t, double delta_factor, const double *P, i64 n, double *dist, double *xp, i64 *stats) {
  omesh m = {nnp, nel, nen, nen == 8 ? 6 : 4, nen == 8 ? 4 : 3, X, IEN, build_ine(nnp, nel, nen, IEN)};
  ogrid g; grid_init(&g, amin, amax, N, cell);
  opts o; pts_bin(&g, P, n, &o);
  double delta = delta_factor * cell;
  if (stats) stats[0] = stats[1] = stats[2] = 0;
  for (i64 v = 0; v < n; v++) dist[v] = -BIG;
  if (xp) memset(xp, 0, sizeof(double) * 3 * (size_t)n);
  for (i64 el = 0; el < nel; el++) {
    double mn = DBL_MAX, mx = -DBL_MAX;
    for (int a = 0; a < nen; a++) { double r = rho_n[IEN[nen * el + a] - 1]; if (r < mn) mn = r; if (r > mx) mx = r; }
    if (mn >= rho_t) pts_boundary_faces(&m, &g, &o, el, rho_n, rho_t, delta, 1, dist, xp);
    else if (mx > rho_t) pts_isocontour_element(&m, &g, &o, el, rho_n, rho_t, delta, dist, xp, stats);
  }
  for (i64 v = 0; v < n; v++) dist[v] = fabs(dist[v]);
  free(o.cptr); free(o.pid); grid_free(&g); free_ine(&m.ine); return 0;
}
/* HEX8: candidates = elements whose closed AABB holds the point; TET4: elements whose create_grid_tetrahedra_mapping_TET4 cell range
 * holds point_to_grid_index(x) = clamp(floor((x - amin) / cell) + 1, 1, N + 1) per axis.  Ascending element order, -1 without one. */
API int r2so_sign_detection_points(i64 nnp, const double *X, i64 nel, int nen, const i64 *IEN, const double *amin, const double *amax, const i64 *N, double cell,
                                   const double *rho_n, double rho_t, const double *P, i64 n, int nthreads, double *signs) {
  (void)nnp; (void)amax;
  double *box = (double *)malloc(sizeof(double) * 6 * (size_t)(nel > 0 ? nel : 1)); i64 *rg = (i64 *)malloc(sizeof(i64) * 6 * (size_t)(nel > 0 ? nel : 1));
  for (i64 e = 0; e < nel; e++) {
    double *b = box + 6 * e;
    for (int d = 0; d < 3; d++) { b[d] = DBL_MAX; b[3 + d] = -DBL_MAX; }
    for (int a = 0; a < nen; a++) for (int d = 0; d < 3; d++) { double c = X[3 * (IEN[nen * e + a] - 1) + d]; if (c < b[d]) b[d] = c; if (c > b[3 + d]) b[3 + d] = c; }
    for (int d = 0; d < 3; d++) {      /* create_grid_tetrahedra_mapping_TET4 :195-196 */
      double mi = floor((b[d] - amin[d]) / cell) - 1, ma = ceil((b[3 + d] - amin[d]) / cell) + 1;
      if (mi < 1) mi = 1;
      if (ma > (double)(N[d] + 1)) ma = (double)(N[d] + 1);
      rg[6 * e + d] = mi > (double)(N[d] + 2) ? N[d] + 2 : (i64)mi; rg[6 * e + 3 + d] = ma < 0 ? 0 : (i64)ma;
    }
  }
  if (nthreads < 1) nthreads = 1;
#ifdef _OPENMP
#pragma omp parallel for num_threads(nthreads) schedule(dynamic, 256)
#endif
  for (i64 v = 0; v < n; v++) {
    const double *x = P + 3 * v; signs[v] = -1.0;
    if (nen == 8) {
      double mx = -DBL_MAX; int any = 0;
      for (i64 e = 0; e < nel; e++) {
        const double *b = box + 6 * e;
        if (!(x[0] >= b[0] && x[0] <= b[3] && x[1] >= b[1] && x[1] <= b[4] && x[2] >= b[2] && x[2] <= b[5])) continue;
        any = 1; for (int a = 0; a < 8; a++) { double r = rho_n[IEN[8 * e + a] - 1]; if (r > mx) mx = r; }
      }
      if (!any || mx < rho_t) continue;                                    /* :36 */
      double max_local = 10.0;
      for (i64 e = 0; e < nel; e++) {
        const double *b = box + 6 * e;
        if (!(x[0] >= b[0] && x[0] <= b[3] && x[1] >= b[1] && x[1] <= b[4] && x[2] >= b[2] && x[2] <= b[5])) continue;
        double Xe[3][8], re[8], xi[3], Nn[8];
        for (int a = 0; a < 8; a++) { i64 nd = IEN[8 * e + a] - 1; re[a] = rho_n[nd]; for (int d = 0; d < 3; d++) Xe[d][a] = X[3 * nd + d]; }
        inverse_map_hex8((const double(*)[8])Xe, x, xi);
        double mn = fmax(fabs(xi[0]), fmax(fabs(xi[1]), fabs(xi[2])));
        if (mn < 1.01 && max_local > mn) {                                 /* :48 */
          hex8_shape(xi, Nn);
          double rho = Nn[0] * re[0]; for (int a = 1; a < 8; a++) rho = rho + Nn[a] * re[a];
          if (rho >= rho_t) signs[v] = 1.0;
          if (mn < 0.95) break;                                            /* :51-59 */
          max_local = mn;
        }
      }
    } else {
      i64 idx[3];
      for (int d = 0; d < 3; d++) { double f = floor((x[d] - amin[d]) / cell) + 1; if (f < 1) f = 1; if (f > (double)(N[d] + 1)) f = (double)(N[d] + 1); idx[d] = (i64)f; }
      for (i64 e = 0; e < nel; e++) {
        const i64 *r = rg + 6 * e;
        if (idx[0] < r[0] || idx[0] > r[3] || idx[1] < r[1] || idx[1] > r[4] || idx[2] < r[2] || idx[2] > r[5]) continue;
        double Xe[3][4], re[4]; const double *b = box + 6 * e;
        for (int a = 0; a < 4; a++) { i64 nd = IEN[4 * e + a] - 1; re[a] = rho_n[nd]; for (int d = 0; d < 3; d++) Xe[d][a] = X[3 * nd + d]; }
        /* is_point_in_tetrahedron :220-242 (tol 1e-10), as r2so_sign_detection */
        const double tol = 1e-10; int out = 0;
        for (int d = 0; d < 3; d++) if (x[d] < b[d] - tol || x[d] > b[3 + d] + tol) out = 1;
        if (out) continue;
        double A[3][3], bb[3];
        for (int d = 0; d < 3; d++) { A[d][0] = Xe[d][1] - Xe[d][0]; A[d][1] = Xe[d][2] - Xe[d][0]; A[d][2] = Xe[d][3] - Xe[d][0]; bb[d] = x[d] - Xe[d][0]; }
        double c00 = A[1][1] * A[2][2] - A[1][2] * A[2][1], c01 = A[1][2] * A[2][0] - A[1][0] * A[2][2], c02 = A[1][0] * A[2][1] - A[1][1] * A[2][0];
        double det = (A[0][0] * c00 + A[0][1] * c01) + A[0][2] * c02; if (!(fabs(det) > 0.0)) continue;
        double c10 = A[0][2] * A[2][1] - A[0][1] * A[2][2], c11 = A[0][0] * A[2][2] - A[0][2] * A[2][0], c12 = A[0][1] * A[2][0] - A[0][0] * A[2][1];
        double c20 = A[0][1] * A[1][2] - A[0][2] * A[1][1], c21 = A[0][2] * A[1][0] - A[0][0] * A[1][2], c22 = A[0][0] * A[1][1] - A[0][1] * A[1][0];
        double l2 = ((c00 * bb[0] + c10 * bb[1]) + c20 * bb[2]) / det, l3 = ((c01 * bb[0] + c11 * bb[1]) + c21 * bb[2]) / det, l4 = ((c02 * bb[0] + c12 * bb[1]) + c22 * bb[2]) / det;
        double l1 = 1.0 - ((l2 + l3) + l4);
        if (!(l1 >= -tol && l2 >= -tol && l3 >= -tol && l4 >= -tol && l1 <= 1.0 + tol && l2 <= 1.0 + tol && l3 <= 1.0 + tol && l4 <= 1.0 + tol)) continue;
        double lc[3]; if (!inverse_map_tet4((const double(*)[4])Xe, x, lc)) continue;
        double l4b = 1.0 - ((lc[0] + lc[1]) + lc[2]);
        double rho = ((lc[0] * re[0] + lc[1] * re[1]) + lc[2] * re[2]) + l4b * re[3];
        if (rho >= rho_t) { signs[v] = 1.0; break; }
      }
    }
  }
  free(box); free(rg); return 0;
}
