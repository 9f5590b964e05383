// r2s_points.cu -- evalDistances and Sign_Detection at arbitrary points (the reference's `points` argument, binned by LinkedList(grid,
// points), Grid.jl:47-69) on the GPU.  The rule is written out in include/r2s.h.
//
// Distances, once per call: the active elements (solid with boundary faces, crossing) get the CELL range of their AABB +- delta
// (calculateMiniAABB_grid, Grid.jl:122-154) over the whole grid -- no slab clipping -- and are binned into tiles of cells, (tile, element)
// keys radix-sorted into per-tile lists in ascending element order; the boundary-face triangles get cell ranges too (face_triangles<.., true>),
// and every crossing HEX8 element a solver record (phase 1 of the projection done once).  Per chunk of points: each point's cell, its
// tile, the point ids sorted by tile; one thread per point walks its tile's list in element order and replays the running minimum
// (r2s_replay.cuh) with the per-pair solvers of the grid path's closest-point (xp) kernels.  A triangle or an iso pair is skipped when a
// lower bound of everything it could write is not below the running |value| (triangle box; box /\ slab of r2s_bound.cuh for box elements):
// the strict `<` of WriteValue could not take it, so the distance and xp are unchanged.
//
// Signs, once per call: every element's bin range -- bins b = clamp(floor((x - amin) / cell) + 1, 1, N + 1) per axis (point_to_grid_index,
// SignDetection.jl:256-268) -- over the bins of its closed AABB (HEX8) or the padded range of create_grid_tetrahedra_mapping_TET4 (TET4),
// binned into tiles of bins.  The bin expression is monotone in x, so an AABB that holds x has bin(lo) <= bin(x) <= bin(hi) and binning
// cannot miss a candidate; the exact closed-AABB test decides.  Per point the candidates of its tile's list, in element order, go through
// the per-candidate rule of the grid path (r2s_signrule.cuh).
#include <algorithm>
#include <cmath>
#include <type_traits>
#include "r2s_common.cuh"
#include "r2s_tables.cuh"
#include "r2s_exact.cuh"
#include "r2s_iso.cuh"
#include "r2s_bound.cuh"
#include "r2s_replay.cuh"
#include "r2s_signrule.cuh"

#define PT_CHUNK (1ll << 22)      // points per chunk: the bounded device buffer (as r2s_sample_sdf)
#define PT_IDX_BITS 22            // sort key = tile << PT_IDX_BITS | point index in the chunk

// crossing HEX8 element: the solver constants of k_project_hex8 (element-local coordinates, node 0 subtracted) and phase 1
struct __align__(16) PtHex {
  double A[4][8];            // monomial coefficients of x, y, z (local) and rho
  double org[3], xi0[3], gs;
  double tlo[3], thi[3], sn[3], sA, sB;      // box elements: tight box and slab of the iso-patch, global coordinates (r2s_bound.cuh)
  int box, ok0;
};
// element of the sign binning: closed AABB, inclusive bin range per axis (1-based bins), hot = some nodal density >= rho_t (:36)
struct SPRec { double lo[3], hi[3]; int b0[3], b1[3]; int hot, pad; };

// cell of a point per axis (the oracle's cellof, Grid.jl:58), false if outside [0, N] on some axis
__device__ __forceinline__ bool pt_cell(const GridDev &g, const double x[3], int c[3]) {
  bool ok = true;
#pragma unroll
  for (int d = 0; d < 3; d++) {
    const double f = floor(ex::dvd(ex::mul((double)g.N[d], ex::sub(x[d], g.amin[d])), ex::sub(g.amax[d], g.amin[d])));
    if (f >= 0.0 && f <= (double)g.N[d]) c[d] = (int)f; else { ok = false; c[d] = 0; }
  }
  return ok;
}
// point_to_grid_index (SignDetection.jl:256-268): clamp(floor((x - amin) / cell) + 1, 1, N + 1), clamped before the conversion
__device__ __forceinline__ int pt_bin(double x, double amin, double cell, int n1) {
  const double f = floor(ex::dvd(ex::sub(x, amin), cell)) + 1.0;
  return f < 1.0 ? 1 : (f > (double)n1 ? n1 : (int)f);
}
__device__ __forceinline__ i64 tile_of(const GridDev &g, int c0, int c1, int c2) {
  return ((i64)(c2 / TILE_Z) * g.nt[1] + c1 / TILE_Y) * g.nt[0] + c0 / TILE_X;
}

// ------------------------------------------------------------------------------------------------ distances: once per call
__global__ void k_pt_classify(i64 nel, int nen, const int *__restrict__ IEN, const double *__restrict__ rn, const unsigned char *__restrict__ fb, double rho_t,
                              unsigned char *__restrict__ cls, int *__restrict__ flag, u64 *__restrict__ ctr) {
  const i64 e = blockIdx.x * (i64)blockDim.x + threadIdx.x;
  int c = 0;
  if (e < nel) {
    double mn = 1e300, mx = -1e300;
    for (int a = 0; a < nen; a++) { const double r = rn[IEN[nen * e + a]]; mn = fmin(mn, r); mx = fmax(mx, r); }
    c = mn >= rho_t ? 1 : (mx > rho_t ? 2 : 0);      // :199-201, :312
    cls[e] = (unsigned char)c;
    flag[e] = (c == 2 || (c == 1 && fb[e] != 0)) ? 1 : 0;
  }
  const unsigned m1 = __ballot_sync(0xffffffffu, c == 1), m2 = __ballot_sync(0xffffffffu, c == 2);      // class counters (report): one atomic per warp
  if ((threadIdx.x & 31) == 0) { if (m1) atomicAdd(&ctr[0], (u64)__popc(m1)); if (m2) atomicAdd(&ctr[1], (u64)__popc(m2)); }
}
// active record with CELL ranges [ps, pe) (ActRec's fields hold cells here, not grid points), its tile and triangle counts
__global__ void k_pt_records(i64 nel, int nen, int nsn, const int *__restrict__ IEN, const double *__restrict__ X, const unsigned char *__restrict__ cls,
                             const unsigned char *__restrict__ fb, const int *__restrict__ flag, const int *__restrict__ idx, GridDev g, double delta,
                             ActRec *__restrict__ rec, i64 *__restrict__ ntile, int *__restrict__ ntri) {
  const i64 e = blockIdx.x * (i64)blockDim.x + threadIdx.x;
  if (e >= nel || !flag[e]) return;
  double lo[3] = {1e300, 1e300, 1e300}, hi[3] = {-1e300, -1e300, -1e300};
  for (int a = 0; a < nen; a++) { const i64 n = IEN[nen * e + a]; for (int d = 0; d < 3; d++) { const double c = X[3 * n + d]; lo[d] = fmin(lo[d], c); hi[d] = fmax(hi[d], c); } }
  ActRec r; r.el = (int)e; r.cls = cls[e]; r.fmask = fb[e]; r.tri_off = 0; r.pair_off = 0;
  bool ok = true;
  for (int d = 0; d < 3; d++) {
    int I0 = 0, I1 = -1;
    ok = ok && ex::cell_range_axis(lo[d], hi[d], delta, g.amin[d], g.amax[d], g.N[d], I0, I1);
    r.ps[d] = ok ? I0 : 0; r.pe[d] = ok ? I1 + 1 : 0;
  }
  const int a = idx[e];
  if (!ok) { for (int d = 0; d < 3; d++) r.pe[d] = r.ps[d]; }
  rec[a] = r;
  ntile[a] = ok ? (i64)((r.pe[0] - 1) / TILE_X - r.ps[0] / TILE_X + 1) * ((r.pe[1] - 1) / TILE_Y - r.ps[1] / TILE_Y + 1) * ((r.pe[2] - 1) / TILE_Z - r.ps[2] / TILE_Z + 1) : 0;
  ntri[a] = __popc((unsigned)r.fmask) * nsn;
}
template <int NEN>
__global__ void k_pt_emit(i64 nact, ActRec *__restrict__ rec, const i64 *__restrict__ toff, const int *__restrict__ troff, const int *__restrict__ IEN,
                          const double *__restrict__ X, const double *__restrict__ rn, const unsigned char *__restrict__ ebox, int proj_box, GridDev g, double delta,
                          double rho_t, u64 *__restrict__ keys, int *__restrict__ tile_cnt, TriRec *__restrict__ tri, PtHex *__restrict__ hex) {
  const i64 a = blockIdx.x * (i64)blockDim.x + threadIdx.x;
  if (a >= nact) return;
  ActRec r = rec[a];
  rec[a].tri_off = troff[a];
  if (r.pe[0] > r.ps[0]) {
    i64 o = toff[a];
    for (int tz = r.ps[2] / TILE_Z; tz <= (r.pe[2] - 1) / TILE_Z; tz++)
      for (int ty = r.ps[1] / TILE_Y; ty <= (r.pe[1] - 1) / TILE_Y; ty++)
        for (int tx = r.ps[0] / TILE_X; tx <= (r.pe[0] - 1) / TILE_X; tx++) {
          const u64 t = ((u64)tz * g.nt[1] + ty) * g.nt[0] + tx;
          keys[o++] = (t << 32) | (u64)a;
          atomicAdd(&tile_cnt[t], 1);
        }
  }
  double Xe[3][NEN];
  for (int q = 0; q < NEN; q++) { const i64 n = IEN[NEN * (i64)r.el + q]; for (int d = 0; d < 3; d++) Xe[d][q] = X[3 * n + d]; }
  if (r.fmask) face_triangles<NEN, true>(Xe, r.fmask, g, delta, tri + troff[a]);
  if (NEN == 8 && r.cls == 2) {      // the arithmetic of k_project_hex8 / k_box_records
    PtHex P; double nv[4][8];
#pragma unroll
    for (int k = 0; k < 8; k++) { nv[0][k] = Xe[0][k]; nv[1][k] = Xe[1][k]; nv[2][k] = Xe[2][k]; nv[3][k] = rn[IEN[8 * (i64)r.el + k]]; }
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
    P.box = (proj_box && ebox[r.el]) ? 1 : 0;
    iso::ProjState S0;
    if (P.box) {
      iso::HexBox H; iso::make_box(P.A, H);
      P.ok0 = iso::proj_init_element<iso::HexBox, PMODE>(H, rho_t, P.gs, S0) ? 1 : 0;
      bnd::box_iso_bounds(nv[3], rho_t, P.gs, P.org, H.c, H.h, P.tlo, P.thi, P.sn, P.sA, P.sB);
    } else {
      iso::HexTri H; H.A = P.A;
      P.ok0 = iso::proj_init_element<iso::HexTri, PMODE>(H, rho_t, P.gs, S0) ? 1 : 0;
#pragma unroll
      for (int d = 0; d < 3; d++) { P.tlo[d] = -INFINITY; P.thi[d] = INFINITY; P.sn[d] = 0.0; }
      P.sA = -INFINITY; P.sB = INFINITY;
    }
#pragma unroll
    for (int d = 0; d < 3; d++) P.xi0[d] = S0.xi[d];
    hex[a] = P;
  }
}

// ------------------------------------------------------------------------------------------------ per chunk
// sort key of every point: (tile << PT_IDX_BITS) | index; kind 0 = distance cells (outside [0, N] -> tile ntiles), 1 = sign bins
__global__ void k_pt_keys(i64 m, const double *__restrict__ pts, GridDev g, int kind, u64 *__restrict__ keys, int *__restrict__ err) {
  const i64 i = blockIdx.x * (i64)blockDim.x + threadIdx.x;
  if (i >= m) return;
  const double x[3] = {pts[3 * i], pts[3 * i + 1], pts[3 * i + 2]};
  if (!isfinite(x[0]) || !isfinite(x[1]) || !isfinite(x[2])) { *err = 1; keys[i] = ((u64)g.ntiles << PT_IDX_BITS) | (u64)i; return; }
  i64 t;
  if (kind == 0) { int c[3]; t = pt_cell(g, x, c) ? tile_of(g, c[0], c[1], c[2]) : g.ntiles; }
  else t = tile_of(g, pt_bin(x[0], g.amin[0], g.cell, g.np[0]) - 1, pt_bin(x[1], g.amin[1], g.cell, g.np[1]) - 1, pt_bin(x[2], g.amin[2], g.cell, g.np[2]) - 1);
  keys[i] = ((u64)t << PT_IDX_BITS) | (u64)i;
}

// the iso distance of one (crossing HEX8 element, point) pair: k_project_hex8<true, BOX>'s arithmetic
template <bool BOX>
__device__ __forceinline__ double pt_project_hex8(const PtHex &P, const int *__restrict__ IEN, const double *__restrict__ rn, int el, double rho_t, const double xg[3],
                                                  double xp[3], int &nit, bool &ok) {
  double A[4][8], re[8];
#pragma unroll
  for (int c = 0; c < 4; c++)
#pragma unroll
    for (int k = 0; k < 8; k++) A[c][k] = P.A[c][k];
  const bool ok0 = P.ok0 != 0;
#pragma unroll
  for (int k = 0; k < 8; k++) re[k] = ok0 ? 0.0 : rn[IEN[8 * (i64)el + k]];      // only phase 1's edge fallback reads them
  typedef typename std::conditional<BOX, iso::HexBox, iso::HexTri>::type ElemT;
  ElemT EL;
  if constexpr (BOX) iso::make_box(A, EL); else EL.A = A;
  const double x[3] = {xg[0] - P.org[0], xg[1] - P.org[1], xg[2] - P.org[2]};
  const double xi0[3] = {P.xi0[0], P.xi0[1], P.xi0[2]};
  double xi[3], p[3];
  ok = iso::project_hex8_from<ElemT, PMODE>(EL, re, c_hex_sg, c_hex_edges, x, rho_t, P.gs, xi0, ok0, xi, nit);
  iso::eval_pos(EL, xi, p);
  const double d0 = x[0] - p[0], d1 = x[1] - p[1], d2 = x[2] - p[2];
#pragma unroll
  for (int d = 0; d < 3; d++) xp[d] = p[d] + P.org[d];
  return sqrt(fma(d2, d2, fma(d1, d1, d0 * d0)));
}
// lower bound of |point - y| over every y a triangle (or an element's triangles) can write, against the running value (k_assemble's margins)
__device__ __forceinline__ bool box_not_below(const double lo[3], const double hi[3], const double x[3], double c) {
  double lb2 = 0.0;
#pragma unroll
  for (int d = 0; d < 3; d++) { const double e = fmax(fmax(lo[d] - x[d], x[d] - hi[d]), 0.0); lb2 = fma(e, e, lb2); }
  const double cv = fabs(c) * (1.0 + 1e-12);
  return lb2 * (1.0 - 1e-12) > cv * cv;
}

// stats: [0] pairs (crossing element whose range holds the point), [1] pairs pruned, [2] Newton iterations, [3] not converged
template <bool WANT_XP, int NEN>
__global__ void __launch_bounds__(128) k_pt_dist(i64 m, const u64 *__restrict__ skeys, const double *__restrict__ pts, GridDev g, const int *__restrict__ tile_ptr,
                                                 const u64 *__restrict__ tkeys, const ActRec *__restrict__ rec, const TriRec *__restrict__ tri, const PtHex *__restrict__ hex,
                                                 const int *__restrict__ IEN, const double *__restrict__ X, const double *__restrict__ rn, double rho_t, int prune,
                                                 double *__restrict__ dist, double *__restrict__ xpo, u64 *__restrict__ stats) {
  constexpr int NSN = NEN == 8 ? 4 : 3;
  const i64 s = blockIdx.x * (i64)blockDim.x + threadIdx.x;
  u64 npair = 0, npruned = 0, nits = 0, nbad = 0;
  if (s < m) {
    const u64 key = skeys[s];
    const i64 i = (i64)(key & ((1ull << PT_IDX_BITS) - 1)), t = (i64)(key >> PT_IDX_BITS);
    const double x[3] = {pts[3 * i], pts[3 * i + 1], pts[3 * i + 2]};
    VoxState st; st.c = -R2S_BIG; st.xp[0] = st.xp[1] = st.xp[2] = 0.0;
    int c[3];
    if (t < g.ntiles && pt_cell(g, x, c)) {
      const int l1 = tile_ptr[t + 1];
      for (int l = tile_ptr[t]; l < l1; l++) {
        const int a = (int)(tkeys[l] & 0xffffffffull);
        const ActRec r = rec[a];
        if (c[0] < r.ps[0] || c[0] >= r.pe[0] || c[1] < r.ps[1] || c[1] >= r.pe[1] || c[2] < r.ps[2] || c[2] >= r.pe[2]) continue;
        // boundary faces first (process_isocontour_element! :584 / the solid elements' process_boundary_faces!)
        if (r.fmask && !(prune && box_not_below(tri[r.tri_off].rlo, tri[r.tri_off].rhi, x, st.c))) {
          double Xe[3][NEN], re[NEN];
          if (r.cls == 2)
            for (int q = 0; q < NEN; q++) { const i64 nd = IEN[NEN * (i64)r.el + q]; re[q] = rn[nd]; for (int d = 0; d < 3; d++) Xe[d][q] = X[3 * nd + d]; }
          const int ntri = __popc((unsigned)r.fmask) * NSN;
          for (int q = 0; q < ntri; q++) {
            const TriRec &T = tri[r.tri_off + q];
            if (c[0] < T.ps[0] || c[0] >= T.pe[0] || c[1] < T.ps[1] || c[1] >= T.pe[1] || c[2] < T.ps[2] || c[2] >= T.pe[2]) continue;
            if (prune && box_not_below(T.lo, T.hi, x, st.c)) continue;
            double Xt[3][3], Et[3][3], nn[3];
            for (int d = 0; d < 3; d++) { Xt[0][d] = T.Xt[0][d]; Xt[1][d] = T.Xt[1][d]; Xt[2][d] = T.Xt[2][d]; nn[d] = T.n[d]; }
            for (int d = 0; d < 3; d++) { Et[0][d] = ex::sub(Xt[1][d], Xt[0][d]); Et[1][d] = ex::sub(Xt[2][d], Xt[1][d]); Et[2][d] = ex::sub(Xt[0][d], Xt[2][d]); }
            triangle_point<WANT_XP, NEN>(Xe, re, rho_t, r.cls == 1, Xt, Et, nn, x, st);
          }
        }
        if (r.cls != 2) continue;
        // the element's iso distance (:617-621)
        npair++;
        double dt, p[3];
        if (NEN == 8) {
          const PtHex &P = hex[a];
          if (prune && P.box) {      // tight box, then box /\ slab (k_pair_scan<2>'s tests and margin)
            const double cur = fabs(st.c), c2 = cur * cur * (1.0 + 1e-10);
            double lb2 = 0.0;
#pragma unroll
            for (int d = 0; d < 3; d++) { const double e = fmax(fmax(P.tlo[d] - x[d], x[d] - P.thi[d]), 0.0); lb2 = fma(e, e, lb2); }
            bool prn = lb2 > c2;
            if (!prn && P.sA != -INFINITY) {
              const double n3[3] = {P.sn[0], P.sn[1], P.sn[2]};
              prn = bnd::lb2_box_gap(x, P.tlo, P.thi, n3, P.sA, P.sB) > c2;
              if (!prn) { const double lb = bnd::lb_box_slab(x, P.tlo, P.thi, n3, P.sA, P.sB); prn = lb * lb > c2; }
            }
            if (prn) { npruned++; continue; }
          }
          int nit = 0; bool ok = true;
          dt = P.box ? pt_project_hex8<true>(P, IEN, rn, r.el, rho_t, x, p, nit, ok) : pt_project_hex8<false>(P, IEN, rn, r.el, rho_t, x, p, nit, ok);
          nits += nit > 0 ? nit : 0; nbad += ok ? 0 : 1;
        } else {      // k_project_tet4's arithmetic; no projection = the running value stays
          double Xe[3][4], re[4];
          for (int q = 0; q < 4; q++) { const i64 nd = IEN[4 * (i64)r.el + q]; re[q] = rn[nd]; for (int d = 0; d < 3; d++) Xe[d][q] = X[3 * nd + d]; }
          const bool ok = iso::project_tet4(Xe, re, c_tet_isn, x, rho_t, p);
          dt = -1.0;
          if (ok) { const double d0 = x[0] - p[0], d1 = x[1] - p[1], d2 = x[2] - p[2]; dt = sqrt((d0 * d0 + d1 * d1) + d2 * d2); }
          else nbad++;
        }
        if (dt >= 0.0 && fabs(dt) < fabs(st.c)) {
          st.c = dt;
          if (WANT_XP) { st.xp[0] = p[0]; st.xp[1] = p[1]; st.xp[2] = p[2]; }
        }
      }
    }
    dist[i] = fabs(st.c);
    if (WANT_XP) { xpo[3 * i] = st.xp[0]; xpo[3 * i + 1] = st.xp[1]; xpo[3 * i + 2] = st.xp[2]; }
  }
  for (int o = 16; o > 0; o >>= 1) {
    npair += __shfl_down_sync(0xffffffffu, npair, o); npruned += __shfl_down_sync(0xffffffffu, npruned, o);
    nits += __shfl_down_sync(0xffffffffu, nits, o); nbad += __shfl_down_sync(0xffffffffu, nbad, o);
  }
  if ((threadIdx.x & 31) == 0) {
    u64 *cs = stats + 8 * (1 + (blockIdx.x & 127));
    if (npair) atomicAdd(&cs[0], npair); if (npruned) atomicAdd(&cs[1], npruned); if (nits) atomicAdd(&cs[2], nits); if (nbad) atomicAdd(&cs[3], nbad);
  }
}

// ------------------------------------------------------------------------------------------------ signs
__global__ void k_pt_sign_records(i64 nel, int nen, const int *__restrict__ IEN, const double *__restrict__ X, const double *__restrict__ rn, double rho_t, GridDev g,
                                  SPRec *__restrict__ rng, SignEl *__restrict__ sel, i64 *__restrict__ ntile) {
  const i64 e = blockIdx.x * (i64)blockDim.x + threadIdx.x;
  if (e >= nel) return;
  SPRec R; double rmax = -1e300;
  for (int d = 0; d < 3; d++) { R.lo[d] = 1e300; R.hi[d] = -1e300; }
  for (int a = 0; a < nen; a++) { const i64 n = IEN[nen * e + a]; rmax = fmax(rmax, rn[n]); for (int d = 0; d < 3; d++) { const double c = X[3 * n + d]; R.lo[d] = fmin(R.lo[d], c); R.hi[d] = fmax(R.hi[d], c); } }
  R.hot = (nen == 4 || !(rmax < rho_t)) ? 1 : 0; R.pad = 0;
  bool ok = true;
  for (int d = 0; d < 3; d++) {
    const int n1 = g.np[d];
    if (nen == 8) { R.b0[d] = pt_bin(R.lo[d], g.amin[d], g.cell, n1); R.b1[d] = pt_bin(R.hi[d], g.amin[d], g.cell, n1); }
    else {      // create_grid_tetrahedra_mapping_TET4 (:195-196), as k_sign_ranges, clamped before the conversion
      const double mi = floor(ex::dvd(ex::sub(R.lo[d], g.amin[d]), g.cell)) - 1.0, ma = ceil(ex::dvd(ex::sub(R.hi[d], g.amin[d]), g.cell)) + 1.0;
      R.b0[d] = mi < 1.0 ? 1 : (mi > (double)n1 ? n1 + 1 : (int)mi);
      R.b1[d] = ma > (double)n1 ? n1 : (ma < 1.0 ? 0 : (int)ma);
    }
    ok = ok && R.b0[d] <= R.b1[d];
  }
  if (!ok) { R.b0[0] = 1; R.b1[0] = 0; }
  rng[e] = R;
  if (nen == 8) {
    double A[3][8];
    for (int d = 0; d < 3; d++) { double v[8]; for (int a = 0; a < 8; a++) v[a] = X[3 * (i64)IEN[8 * e + a] + d]; ex::mono8(v, A[d]); }
    SignEl S; ex::affine_inverse_prepare(A, S);
    sel[e] = S;
  }
  ntile[e] = ok ? (i64)((R.b1[0] - 1) / TILE_X - (R.b0[0] - 1) / TILE_X + 1) * ((R.b1[1] - 1) / TILE_Y - (R.b0[1] - 1) / TILE_Y + 1) * ((R.b1[2] - 1) / TILE_Z - (R.b0[2] - 1) / TILE_Z + 1) : 0;
}
__global__ void k_pt_sign_emit(i64 nel, const SPRec *__restrict__ rng, const i64 *__restrict__ toff, GridDev g, u64 *__restrict__ keys, int *__restrict__ tile_cnt) {
  const i64 e = blockIdx.x * (i64)blockDim.x + threadIdx.x;
  if (e >= nel) return;
  const SPRec R = rng[e];
  if (R.b0[0] > R.b1[0]) return;
  i64 o = toff[e];
  for (int tz = (R.b0[2] - 1) / TILE_Z; tz <= (R.b1[2] - 1) / TILE_Z; tz++)
    for (int ty = (R.b0[1] - 1) / TILE_Y; ty <= (R.b1[1] - 1) / TILE_Y; ty++)
      for (int tx = (R.b0[0] - 1) / TILE_X; tx <= (R.b1[0] - 1) / TILE_X; tx++) {
        const u64 t = ((u64)tz * g.nt[1] + ty) * g.nt[0] + tx;
        keys[o++] = (t << 32) | (u64)e;
        atomicAdd(&tile_cnt[t], 1);
      }
}
template <int NEN>
__global__ void __launch_bounds__(128) k_pt_sign(i64 m, const u64 *__restrict__ skeys, const double *__restrict__ pts, GridDev g, const int *__restrict__ tile_ptr,
                                                 const u64 *__restrict__ tkeys, const SPRec *__restrict__ rng, const SignEl *__restrict__ sel, const int *__restrict__ IEN,
                                                 const double *__restrict__ X, const double *__restrict__ rn, double rho_t, double *__restrict__ signs) {
  const i64 s = blockIdx.x * (i64)blockDim.x + threadIdx.x;
  if (s >= m) return;
  const u64 key = skeys[s];
  const i64 i = (i64)(key & ((1ull << PT_IDX_BITS) - 1)), t = (i64)(key >> PT_IDX_BITS);
  const double x[3] = {pts[3 * i], pts[3 * i + 1], pts[3 * i + 2]};
  const int b[3] = {pt_bin(x[0], g.amin[0], g.cell, g.np[0]), pt_bin(x[1], g.amin[1], g.cell, g.np[1]), pt_bin(x[2], g.amin[2], g.cell, g.np[2])};
  const int p0 = tile_ptr[t], p1 = tile_ptr[t + 1];
  double sign = -1.0;
  if (NEN == 8) {
    // candidates: the elements whose closed AABB holds the point (compute_aabb / is_point_inside_aabb, sdfOnDensityField.jl:60-69)
    bool hot = false;
    for (int p = p0; p < p1 && !hot; p++) {
      const SPRec &R = rng[(int)(tkeys[p] & 0xffffffffull)];
      if (R.hot && x[0] >= R.lo[0] && x[0] <= R.hi[0] && x[1] >= R.lo[1] && x[1] <= R.hi[1] && x[2] >= R.lo[2] && x[2] <= R.hi[2]) hot = true;
    }
    if (hot) {      // else no candidate reaches rho_t: -1 (:36)
      double max_local = 10.0;
      for (int p = p0; p < p1; p++) {
        const int e = (int)(tkeys[p] & 0xffffffffull);
        const SPRec &R = rng[e];
        if (!(x[0] >= R.lo[0] && x[0] <= R.hi[0] && x[1] >= R.lo[1] && x[1] <= R.hi[1] && x[2] >= R.lo[2] && x[2] <= R.hi[2])) continue;
        if (sign_hex8_candidate(sel[e], e, IEN, X, rn, rho_t, x, 0, sign, max_local)) break;
      }
    }
  } else {
    for (int p = p0; p < p1; p++) {
      const int e = (int)(tkeys[p] & 0xffffffffull);
      const SPRec &R = rng[e];
      if (b[0] < R.b0[0] || b[0] > R.b1[0] || b[1] < R.b0[1] || b[1] > R.b1[1] || b[2] < R.b0[2] || b[2] > R.b1[2]) continue;
      if (sign_tet4_candidate(e, IEN, X, rn, rho_t, x, sign)) break;
    }
  }
  signs[i] = sign;
}

// ------------------------------------------------------------------------------------------------ host drivers
static int pt_check(r2s_ctx *ctx, const double *rho_n, const double *pts, i64 n, const void *out) {
  if (!ctx->has_grid) FAIL("r2s_set_grid has not been called");
  if (ctx->nel == 0) FAIL("r2s_set_mesh has not been called");
  if (n < 0) FAIL("points: n must be >= 0");
  if (!rho_n) FAIL("points: rho_n is required");
  if (n > 0 && (!pts || !out)) FAIL("points: a NULL points or result array with n > 0");
  CK(cudaSetDevice(ctx->device));
  CK(ctx->pt_rn.reserve(sizeof(double) * (size_t)ctx->nnp));
  CK(cudaMemcpyAsync(ctx->pt_rn.p, rho_n, sizeof(double) * (size_t)ctx->nnp, cudaMemcpyHostToDevice, ctx->stream));
  return 0;
}
// per-tile lists from (tile << 32 | id) keys: sort, then the counts tile_cnt (at tile_ptr + 1) scanned into offsets
static int pt_tile_lists(r2s_ctx *ctx, i64 nkeys, u64 **sorted) {
  const GridDev &g = ctx->g; cudaStream_t st = ctx->stream;
  int tbits = 1; while ((1ll << tbits) < g.ntiles) tbits++;
  *sorted = ctx->pt_tkeys.as<u64>();
  if (nkeys > 0 && r2s_sort_keys_u64(ctx, ctx->pt_tkeys.as<u64>(), ctx->pt_tkeys_alt.as<u64>(), nkeys, 32 + tbits, sorted)) return 1;
  CK(ctx->pt_off.reserve(sizeof(int) * (size_t)(g.ntiles + 2)));
  if (r2s_scan_exclusive_i32(ctx, ctx->pt_tile_ptr.as<int>() + 1, ctx->pt_off.as<int>(), g.ntiles + 1)) return 1;
  CK(cudaMemcpyAsync(ctx->pt_tile_ptr.as<int>(), ctx->pt_off.as<int>(), sizeof(int) * (size_t)(g.ntiles + 1), cudaMemcpyDeviceToDevice, st));
  return 0;
}
// the chunk loop both calls share: upload, key, sort, run(m, sorted keys, device points), download, check the coordinates
template <class RUN>
static int pt_chunks(r2s_ctx *ctx, const double *pts, i64 n, int kind, RUN run) {
  const GridDev &g = ctx->g; cudaStream_t st = ctx->stream;
  int tbits = 1; while ((1ll << tbits) < g.ntiles + 1) tbits++;
  const i64 ch = std::min<i64>(PT_CHUNK, std::max<i64>(n, 1));
  CK(ctx->pt_in.reserve(sizeof(double) * 3 * (size_t)ch));
  CK(ctx->pt_keys.reserve(sizeof(u64) * (size_t)ch));
  CK(ctx->pt_keys_alt.reserve(sizeof(u64) * (size_t)ch));
  CK(ctx->pt_ctr.reserve(sizeof(u64) * 8 * 129 + sizeof(int)));
  int *err = (int *)(ctx->pt_ctr.as<u64>() + 8 * 129);
  for (i64 s0 = 0; s0 < n; s0 += ch) {
    const i64 m = std::min(ch, n - s0);
    CK(cudaMemsetAsync(err, 0, sizeof(int), st));
    CK(cudaMemcpyAsync(ctx->pt_in.p, pts + 3 * s0, sizeof(double) * 3 * (size_t)m, cudaMemcpyHostToDevice, st));
    k_pt_keys<<<cdiv(m, 256), 256, 0, st>>>(m, ctx->pt_in.as<double>(), g, kind, ctx->pt_keys.as<u64>(), err); LAUNCH_CHECK();
    u64 *sorted = nullptr;
    if (r2s_sort_keys_u64(ctx, ctx->pt_keys.as<u64>(), ctx->pt_keys_alt.as<u64>(), m, PT_IDX_BITS + tbits, &sorted)) return 1;
    int herr = 0;
    if (r2s_readback(ctx, &herr, err, sizeof(int))) return 1;
    if (herr) FAIL("points: a point coordinate is NaN or infinite");
    if (run(s0, m, sorted)) return 1;
  }
  return 0;
}

int r2s_points_distances(r2s_ctx *ctx, const double *rho_n, double rho_t, double delta_factor, const double *pts, i64 n, double *dist, double *xp) {
  if (pt_check(ctx, rho_n, pts, n, dist)) return 1;
  const GridDev &g = ctx->g; cudaStream_t st = ctx->stream;
  const i64 nel = ctx->nel; const int nen = ctx->nen;
  const double delta = delta_factor * g.cell;
  const bool want_xp = xp != nullptr;
  CK(cudaEventRecord(ctx->ev[0], st));
  CK(ctx->pt_ctr.reserve(sizeof(u64) * 8 * 129 + sizeof(int)));
  u64 *ctr = ctx->pt_ctr.as<u64>();
  CK(cudaMemsetAsync(ctr, 0, sizeof(u64) * 8 * 129, st));
  CK(ctx->pt_cls.reserve((size_t)nel));
  CK(ctx->pt_flag.reserve(sizeof(int) * (size_t)(nel + 1)));
  CK(ctx->pt_idx.reserve(sizeof(int) * (size_t)(nel + 1)));
  CK(cudaMemsetAsync(ctx->pt_flag.as<int>() + nel, 0, sizeof(int), st));
  k_pt_classify<<<cdiv(nel, 256), 256, 0, st>>>(nel, nen, ctx->IEN32.as<int>(), ctx->pt_rn.as<double>(), ctx->fbnd.as<unsigned char>(), rho_t, ctx->pt_cls.as<unsigned char>(),
                                                ctx->pt_flag.as<int>(), ctr); LAUNCH_CHECK();
  if (r2s_scan_exclusive_i32(ctx, ctx->pt_flag.as<int>(), ctx->pt_idx.as<int>(), nel + 1)) return 1;
  int nact_i = 0;
  if (r2s_readback(ctx, &nact_i, ctx->pt_idx.as<int>() + nel, sizeof(int))) return 1;
  const i64 nact = nact_i;
  CK(ctx->pt_tile_ptr.reserve(sizeof(int) * (size_t)(g.ntiles + 2)));
  CK(cudaMemsetAsync(ctx->pt_tile_ptr.p, 0, sizeof(int) * (size_t)(g.ntiles + 2), st));
  i64 nkeys = 0; int ntri = 0;
  u64 *tsorted = ctx->pt_tkeys.as<u64>();
  if (nact > 0) {
    CK(ctx->pt_rec.reserve(sizeof(ActRec) * (size_t)nact));
    CK(ctx->pt_cnt.reserve((sizeof(i64) + sizeof(int)) * 2 * (size_t)(nact + 1)));
    i64 *ntile = ctx->pt_cnt.as<i64>(), *toff = ntile + (nact + 1);
    int *ntr = (int *)(toff + (nact + 1)), *troff = ntr + (nact + 1);
    CK(cudaMemsetAsync(ntile + nact, 0, sizeof(i64), st));
    CK(cudaMemsetAsync(ntr + nact, 0, sizeof(int), st));
    k_pt_records<<<cdiv(nel, 256), 256, 0, st>>>(nel, nen, ctx->nsn, ctx->IEN32.as<int>(), ctx->X.as<double>(), ctx->pt_cls.as<unsigned char>(), ctx->fbnd.as<unsigned char>(),
                                                 ctx->pt_flag.as<int>(), ctx->pt_idx.as<int>(), g, delta, ctx->pt_rec.as<ActRec>(), ntile, ntr); LAUNCH_CHECK();
    if (r2s_scan_exclusive_i64(ctx, ntile, toff, nact + 1)) return 1;
    if (r2s_scan_exclusive_i32(ctx, ntr, troff, nact + 1)) return 1;
    const size_t o0 = r2s_rb_put(ctx, toff + nact, sizeof(i64)), o1 = r2s_rb_put(ctx, troff + nact, sizeof(int));
    if (o0 == (size_t)-1 || o1 == (size_t)-1 || r2s_rb_sync(ctx)) return 1;
    nkeys = *(const i64 *)r2s_rb_at(ctx, o0); ntri = *(const int *)r2s_rb_at(ctx, o1);
    if (nkeys >= (1ll << 31)) FAIL("points: too many (tile, element) pairs");
    CK(ctx->pt_tkeys.reserve(sizeof(u64) * (size_t)(nkeys + 1)));
    CK(ctx->pt_tkeys_alt.reserve(sizeof(u64) * (size_t)(nkeys + 1)));
    CK(ctx->pt_tri.reserve(sizeof(TriRec) * (size_t)(ntri + 1)));
    if (nen == 8) CK(ctx->pt_hex.reserve(sizeof(PtHex) * (size_t)nact));
#define EMIT(NEN) k_pt_emit<NEN><<<cdiv(nact, 128), 128, 0, st>>>(nact, ctx->pt_rec.as<ActRec>(), toff, troff, ctx->IEN32.as<int>(), ctx->X.as<double>(), ctx->pt_rn.as<double>(), \
      ctx->ebox.as<unsigned char>(), ctx->knobs.proj_box, g, delta, rho_t, ctx->pt_tkeys.as<u64>(), ctx->pt_tile_ptr.as<int>() + 1, ctx->pt_tri.as<TriRec>(), ctx->pt_hex.as<PtHex>())
    if (nen == 8) EMIT(8); else EMIT(4);
#undef EMIT
    LAUNCH_CHECK();
  }
  if (pt_tile_lists(ctx, nkeys, &tsorted)) return 1;
  CK(cudaEventRecord(ctx->ev[1], st));
  CK(ctx->pt_out.reserve(sizeof(double) * 4 * (size_t)std::min<i64>(PT_CHUNK, std::max<i64>(n, 1))));
  double *dd = ctx->pt_out.as<double>(), *dx = dd + std::min<i64>(PT_CHUNK, std::max<i64>(n, 1));
  const int prune = ctx->knobs.proj_prune ? 1 : 0;
  auto run = [&](i64 s0, i64 m, const u64 *sk) -> int {
#define DIST(XP, NEN) k_pt_dist<XP, NEN><<<cdiv(m, 128), 128, 0, st>>>(m, sk, ctx->pt_in.as<double>(), g, ctx->pt_tile_ptr.as<int>(), tsorted, ctx->pt_rec.as<ActRec>(), \
      ctx->pt_tri.as<TriRec>(), ctx->pt_hex.as<PtHex>(), ctx->IEN32.as<int>(), ctx->X.as<double>(), ctx->pt_rn.as<double>(), rho_t, prune, dd, dx, ctr)
    if (nen == 8) { if (want_xp) DIST(true, 8); else DIST(false, 8); }
    else { if (want_xp) DIST(true, 4); else DIST(false, 4); }
#undef DIST
    LAUNCH_CHECK();
    CK(cudaMemcpyAsync(dist + s0, dd, sizeof(double) * (size_t)m, cudaMemcpyDeviceToHost, st));
    if (want_xp) CK(cudaMemcpyAsync(xp + 3 * s0, dx, sizeof(double) * 3 * (size_t)m, cudaMemcpyDeviceToHost, st));
    CK(cudaStreamSynchronize(st));
    return 0;
  };
  if (pt_chunks(ctx, pts, n, 0, run)) return 1;
  CK(cudaEventRecord(ctx->ev[2], st));
  u64 hall[8 * 129];
  if (r2s_readback(ctx, hall, ctr, sizeof(hall))) return 1;
  u64 hc[4] = {0, 0, 0, 0};
  for (int q = 0; q < 4; q++) for (int sl = 1; sl <= 128; sl++) hc[q] += hall[8 * sl + q];
  ctx->rep.n_solid = (i64)hall[0]; ctx->rep.n_crossing = (i64)hall[1]; ctx->rep.n_active = nact;
  ctx->rep.n_pairs = (i64)hc[0]; ctx->rep.n_pairs_pruned = (i64)hc[1]; ctx->rep.n_newton_iters = (i64)hc[2]; ctx->rep.n_not_converged = (i64)hc[3];
  CK(cudaEventElapsedTime(&ctx->rep.ms_bin, ctx->ev[0], ctx->ev[1]));
  CK(cudaEventElapsedTime(&ctx->rep.ms_project, ctx->ev[0], ctx->ev[2]));
  return 0;
}

int r2s_points_signs(r2s_ctx *ctx, const double *rho_n, double rho_t, const double *pts, i64 n, double *signs) {
  if (pt_check(ctx, rho_n, pts, n, signs)) return 1;
  const GridDev &g = ctx->g; cudaStream_t st = ctx->stream;
  const i64 nel = ctx->nel; const int nen = ctx->nen;
  CK(cudaEventRecord(ctx->ev[0], st));
  // sign records in pt_hex (SPRec per element), the affine inverse-map data in pt_rec, tile counts / offsets in pt_cnt
  CK(ctx->pt_hex.reserve(sizeof(SPRec) * (size_t)nel));
  if (nen == 8) CK(ctx->pt_rec.reserve(sizeof(SignEl) * (size_t)nel));
  CK(ctx->pt_cnt.reserve(sizeof(i64) * 2 * (size_t)(nel + 1)));
  CK(ctx->pt_tile_ptr.reserve(sizeof(int) * (size_t)(g.ntiles + 2)));
  CK(cudaMemsetAsync(ctx->pt_tile_ptr.p, 0, sizeof(int) * (size_t)(g.ntiles + 2), st));
  i64 *ntile = ctx->pt_cnt.as<i64>(), *toff = ntile + (nel + 1);
  CK(cudaMemsetAsync(ntile + nel, 0, sizeof(i64), st));
  SPRec *rng = ctx->pt_hex.as<SPRec>(); SignEl *sel = ctx->pt_rec.as<SignEl>();
  k_pt_sign_records<<<cdiv(nel, 256), 256, 0, st>>>(nel, nen, ctx->IEN32.as<int>(), ctx->X.as<double>(), ctx->pt_rn.as<double>(), rho_t, g, rng, sel, ntile); LAUNCH_CHECK();
  if (r2s_scan_exclusive_i64(ctx, ntile, toff, nel + 1)) return 1;
  i64 nkeys = 0;
  if (r2s_readback(ctx, &nkeys, toff + nel, sizeof(i64))) return 1;
  if (nkeys >= (1ll << 31)) FAIL("points: too many (tile, element) pairs");
  CK(ctx->pt_tkeys.reserve(sizeof(u64) * (size_t)(nkeys + 1)));
  CK(ctx->pt_tkeys_alt.reserve(sizeof(u64) * (size_t)(nkeys + 1)));
  if (nkeys > 0) { k_pt_sign_emit<<<cdiv(nel, 128), 128, 0, st>>>(nel, rng, toff, g, ctx->pt_tkeys.as<u64>(), ctx->pt_tile_ptr.as<int>() + 1); LAUNCH_CHECK(); }
  u64 *tsorted = nullptr;
  if (pt_tile_lists(ctx, nkeys, &tsorted)) return 1;
  CK(cudaEventRecord(ctx->ev[1], st));
  CK(ctx->pt_out.reserve(sizeof(double) * (size_t)std::min<i64>(PT_CHUNK, std::max<i64>(n, 1))));
  double *ds = ctx->pt_out.as<double>();
  auto run = [&](i64 s0, i64 m, const u64 *sk) -> int {
    if (nen == 8) k_pt_sign<8><<<cdiv(m, 128), 128, 0, st>>>(m, sk, ctx->pt_in.as<double>(), g, ctx->pt_tile_ptr.as<int>(), tsorted, rng, sel, ctx->IEN32.as<int>(), ctx->X.as<double>(), ctx->pt_rn.as<double>(), rho_t, ds);
    else k_pt_sign<4><<<cdiv(m, 128), 128, 0, st>>>(m, sk, ctx->pt_in.as<double>(), g, ctx->pt_tile_ptr.as<int>(), tsorted, rng, sel, ctx->IEN32.as<int>(), ctx->X.as<double>(), ctx->pt_rn.as<double>(), rho_t, ds);
    LAUNCH_CHECK();
    CK(cudaMemcpyAsync(signs + s0, ds, sizeof(double) * (size_t)m, cudaMemcpyDeviceToHost, st));
    CK(cudaStreamSynchronize(st));
    return 0;
  };
  if (pt_chunks(ctx, pts, n, 1, run)) return 1;
  CK(cudaEventRecord(ctx->ev[2], st));
  CK(cudaEventSynchronize(ctx->ev[2]));
  CK(cudaEventElapsedTime(&ctx->rep.ms_bin, ctx->ev[0], ctx->ev[1]));
  CK(cudaEventElapsedTime(&ctx->rep.ms_sign, ctx->ev[0], ctx->ev[2]));
  return 0;
}

extern "C" {
int r2s_eval_distances_points(r2s_ctx *ctx, const double *rho_n, double rho_t, double delta_factor, const double *points, int64_t n, double *dist, double *xp) {
  if (!ctx) return 1;
  ctx->launches = 0;
  if (r2s_points_distances(ctx, rho_n, rho_t, delta_factor, points, n, dist, xp)) return 1;
  ctx->rep.launches = ctx->launches;
  return 0;
}
int r2s_sign_detection_points(r2s_ctx *ctx, const double *rho_n, double rho_t, const double *points, int64_t n, double *signs) {
  if (!ctx) return 1;
  ctx->launches = 0;
  if (r2s_points_signs(ctx, rho_n, rho_t, points, n, signs)) return 1;
  ctx->rep.launches = ctx->launches;
  return 0;
}
}  // extern "C"
