// r2s_dist.cu -- evalDistances (SignedDistances/sdfOnDensityField.jl:139-486) on the GPU
//
//  1. binning   : classify elements (solid / crossing / void, :199-201,:312), give every active element the grid-point
//                 range of its AABB +- delta cell range (MeshGrid/Grid.jl:122-154) and bin it into the voxel tiles it
//                 overlaps: (tile, element) keys -> radix sort -> per-tile element lists in ascending element order.
//  2. project   : element-centric, one warp per 32 grid points of a crossing element: closest point on the in-element
//                 iso-surface (r2s_iso.cuh), distance written to a per-(element, point) pair buffer.  FP64-bound.
//  3. assemble  : voxel-centric, one thread per grid point: walks its tile's element list IN ELEMENT ORDER and replays
//                 the reference's running-min logic exactly (boundary-face triangles with their state-dependent
//                 early-outs, then the element's iso distance from the pair buffer).  Bit-exact decisions (r2s_exact.cuh).
//                 No atomics: every voxel is owned by one thread, the result is deterministic.
#include <stdlib.h>
#include <type_traits>
#include "r2s_common.cuh"
#include "r2s_tables.cuh"
#include "r2s_exact.cuh"
#include "r2s_iso.cuh"
#include "r2s_bound.cuh"
#include "r2s_replay.cuh"

// ------------------------------------------------------------------------------------------------ binning
// [zlo, zhi]: z-extent of the slab's planes grown by a safe margin; elements entirely outside cannot reach a plane of this rank
// and are left inactive without touching their nodes (single rank: the interval is infinite).  The class counters then
// count the elements near the slab only.
__global__ void k_classify(i64 nel, int nen, const int *__restrict__ IEN, const double *__restrict__ rn, const unsigned char *__restrict__ fb,
                           const double2 *__restrict__ ezr, double zlo, double zhi,
                           double rho_t, unsigned char *__restrict__ cls, int *__restrict__ flag, i64 *__restrict__ counts) {
  i64 e = blockIdx.x * (i64)blockDim.x + threadIdx.x;
  int c = 0;
  if (e < nel) { const double2 z = ezr[e]; if (z.y < zlo || z.x > zhi) { cls[e] = 0; flag[e] = 0; e = nel; } }
  if (e < nel) {
    double mn = 1e300, mx = -1e300;
    for (int a = 0; a < nen; a++) { double r = rn[IEN[nen * e + a]]; mn = fmin(mn, r); mx = fmax(mx, r); }
    if (mn >= rho_t) c = 1; else if (mx > rho_t) c = 2;
    cls[e] = (unsigned char)c;
    flag[e] = (c == 2 || (c == 1 && fb[e] != 0)) ? 1 : 0;
  }
  // class counters (report only): one pair of atomics per CTA
  __shared__ int s1, s2;
  if (threadIdx.x == 0) { s1 = 0; s2 = 0; }
  __syncthreads();
  unsigned m1 = __ballot_sync(0xffffffffu, c == 1), m2 = __ballot_sync(0xffffffffu, c == 2);
  if ((threadIdx.x & 31) == 0) { if (m1) atomicAdd(&s1, __popc(m1)); if (m2) atomicAdd(&s2, __popc(m2)); }
  __syncthreads();
  if (threadIdx.x == 0) { if (s1) atomicAdd((u64 *)&counts[0], (u64)s1); if (s2) atomicAdd((u64 *)&counts[1], (u64)s2); }
}
// compacted active list: record with point ranges, tile count, pair count
__global__ void k_act_records(i64 nel, int nen, const int *__restrict__ IEN, const double *__restrict__ X, const unsigned char *__restrict__ cls,
                              const unsigned char *__restrict__ fb, const int *__restrict__ flag, const int *__restrict__ idx, GridDev g, double delta,
                              int kz0, int kz1, ActRec *__restrict__ rec, i64 *__restrict__ ntile, i64 *__restrict__ npair, i64 *__restrict__ nchunk) {
  i64 e = blockIdx.x * (i64)blockDim.x + threadIdx.x;
  if (e >= nel || !flag[e]) return;
  double lo[3] = {1e300, 1e300, 1e300}, hi[3] = {-1e300, -1e300, -1e300};
  for (int a = 0; a < nen; a++) { i64 n = IEN[nen * e + a]; for (int d = 0; d < 3; d++) { double c = X[3 * n + d]; lo[d] = fmin(lo[d], c); hi[d] = fmax(hi[d], c); } }
  ActRec r; r.el = (int)e; r.cls = cls[e]; r.fmask = fb[e]; r.tri_off = 0; r.pair_off = 0;
  bool ok = true;
  for (int d = 0; d < 3; d++) {
    int I0 = 0, I1 = -1;
    ok = ok && ex::cell_range_axis(lo[d], hi[d], delta, g.amin[d], g.amax[d], g.N[d], I0, I1);
    if (ok) { r.ps[d] = g.cstart[g.cs_off[d] + I0]; r.pe[d] = g.cstart[g.cs_off[d] + I1 + 1]; } else { r.ps[d] = 0; r.pe[d] = 0; }
  }
  // z-slab restriction (multi-GPU): only planes [kz0,kz1)
  if (r.ps[2] < kz0) r.ps[2] = kz0;
  if (r.pe[2] > kz1) r.pe[2] = kz1;
  i64 vol = 0, nt = 0;
  if (ok && r.pe[0] > r.ps[0] && r.pe[1] > r.ps[1] && r.pe[2] > r.ps[2]) {
    vol = (i64)(r.pe[0] - r.ps[0]) * (r.pe[1] - r.ps[1]) * (r.pe[2] - r.ps[2]);
    nt = (i64)((r.pe[0] - 1) / TILE_X - r.ps[0] / TILE_X + 1) * ((r.pe[1] - 1) / TILE_Y - r.ps[1] / TILE_Y + 1) * ((r.pe[2] - 1) / TILE_Z - r.ps[2] / TILE_Z + 1);
  } else { r.pe[0] = r.ps[0]; r.pe[1] = r.ps[1]; r.pe[2] = r.ps[2]; }
  int a = idx[e];
  rec[a] = r; ntile[a] = nt;
  i64 np = (r.cls == 2) ? vol : 0;
  npair[a] = np; nchunk[a] = (np + 31) / 32;
}
__global__ void k_emit_keys(i64 nact, ActRec *__restrict__ rec, const i64 *__restrict__ toff, const i64 *__restrict__ poff, GridDev g,
                            u64 *__restrict__ keys, int *__restrict__ tile_cnt, unsigned char *__restrict__ tile_faces) {
  i64 a = blockIdx.x * (i64)blockDim.x + threadIdx.x;
  if (a >= nact) return;
  ActRec r = rec[a];
  rec[a].pair_off = poff[a];
  if (r.pe[0] <= r.ps[0]) return;
  i64 o = toff[a];
  for (int tz = r.ps[2] / TILE_Z; tz <= (r.pe[2] - 1) / TILE_Z; tz++)
    for (int ty = r.ps[1] / TILE_Y; ty <= (r.pe[1] - 1) / TILE_Y; ty++)
      for (int tx = r.ps[0] / TILE_X; tx <= (r.pe[0] - 1) / TILE_X; tx++) {
        u64 t = ((u64)tz * g.nt[1] + ty) * g.nt[0] + tx;
        keys[o++] = (t << 32) | (u64)a;
        atomicAdd(&tile_cnt[t], 1);
        if (r.fmask) tile_faces[t] = 1;       // this tile needs the boundary-face path of the assemble kernel
      }
}

// ------------------------------------------------------------------------------------------------ project (hot, FP64)
// Solver variant of every HEX8 kernel (r2s_iso.cuh): FAST restoration (no confirming evaluation) + ONE code path for all tangent-step
// cases; phase 1 (Newton projection of xi = 0 onto the iso-surface, the same for every point of an element) is computed once per
// warp / per element.  The kernels work in element-local coordinates (node 0 subtracted from the nodes and from the grid point: exact
// in floating point), so X(xi) - x does not cancel the mesh offset.
__global__ void k_fill_f64(i64 n, double *__restrict__ a, double v) {
  i64 i = blockIdx.x * (i64)blockDim.x + threadIdx.x;
  if (i < n) a[i] = v;
}
__device__ __forceinline__ void proj_stats(u64 *counters, int its, bool bad, int lane) {      // one atomic per warp, spread over 128 slots
  for (int o = 16; o > 0; o >>= 1) its += __shfl_down_sync(0xffffffffu, its, o);
  const unsigned mb = __ballot_sync(0xffffffffu, bad);
  if (lane == 0) { u64 *cs = counters + 8 * (1 + (blockIdx.x & 127)); atomicAdd(&cs[2], (u64)its); if (mb) atomicAdd(&cs[3], (u64)__popc(mb)); }
}
// Chunk kernel: one warp per 32-point chunk of a crossing element (general trilinear elements, and every element when the closest
// points xp are wanted).  BOX: the element is an axis-aligned box (iso::HexBox: 17 element constants instead of 32, about half the FP64
// work per iteration); kind_check: the mesh holds both kinds and this launch leaves the chunks of the other kind alone (ebox[e] = 1 for
// boxes).  Without xp the distance of a point in a tile WITHOUT boundary-face elements goes straight into dist[] by a 64-bit atomicMin
// on the bit pattern of the non-negative double (the minimum over the pairs is order independent there); pairs of the other tiles go to
// the pair buffer for the exact replay of k_assemble.
template <bool WANT_XP, bool BOX>
__global__ void __launch_bounds__(128, WANT_XP ? (BOX ? 4 : 2) : 4) k_project_hex8(i64 nitems, i64 nact, const ActRec *__restrict__ rec, const i64 *__restrict__ choff,
                                                      const int *__restrict__ IEN, const double *__restrict__ X, const double *__restrict__ rn, GridDev g,
                                                      double rho_t, double *__restrict__ pairbuf, double *__restrict__ pairxp, u64 *__restrict__ counters,
                                                      const unsigned char *__restrict__ ebox, int kind_check, int skip_box,
                                                      const unsigned char *__restrict__ tile_faces, double *__restrict__ dist) {
  i64 item = (blockIdx.x * (i64)blockDim.x + threadIdx.x) >> 5; int lane = threadIdx.x & 31;
  if (item >= nitems) return;
  // binary search: last a with choff[a] <= item
  i64 lo = 0, hi = nact - 1;
  while (lo < hi) { i64 mid = (lo + hi + 1) >> 1; if (choff[mid] <= item) lo = mid; else hi = mid - 1; }
  const ActRec r = rec[lo];
  if (kind_check && (ebox[r.el] != 0) != BOX) return;
  if (skip_box && ebox[r.el] != 0) return;      // box elements are handled by the pair-list path
  int chunk = (int)(item - choff[lo]);
  // element data: lane l < 8 loads node l; monomial coefficients assembled through shuffles
  double v[4] = {0, 0, 0, 0};
  if (lane < 8) { i64 n = IEN[8 * (i64)r.el + lane]; v[0] = X[3 * n]; v[1] = X[3 * n + 1]; v[2] = X[3 * n + 2]; v[3] = rn[n]; }
  double org[3];
#pragma unroll
  for (int d = 0; d < 3; d++) { org[d] = __shfl_sync(0xffffffffu, v[d], 0); v[d] -= org[d]; }
  double A[4][8], re[8];
#pragma unroll
  for (int c = 0; c < 4; c++) {
    double nv[8];
#pragma unroll
    for (int k = 0; k < 8; k++) nv[k] = __shfl_sync(0xffffffffu, v[c], k);
    iso::monomial8(nv, A[c]);
    if (c == 3) {
#pragma unroll
      for (int k = 0; k < 8; k++) re[k] = nv[k];
    }
  }
  double gs = fabs(rho_t);
#pragma unroll
  for (int k = 0; k < 8; k++) gs = fmax(gs, fabs(re[k]));
  gs = fmax(gs, 1.0);
  int nx = r.pe[0] - r.ps[0], ny = r.pe[1] - r.ps[1], nz = r.pe[2] - r.ps[2];
  i64 vol = (i64)nx * ny * nz, li = (i64)chunk * 32 + lane;
  int nit = 0; bool okc = true;
  typedef typename std::conditional<BOX, iso::HexBox, iso::HexTri>::type ElemT;
  ElemT EL;
  if constexpr (BOX) iso::make_box(A, EL); else EL.A = A;
  iso::ProjState S0; const bool ok0 = iso::proj_init_element<ElemT, PMODE>(EL, rho_t, gs, S0);      // warp-uniform
  if (li < vol) {
    int i = (int)(li % nx), j = (int)((li / nx) % ny), k = (int)(li / ((i64)nx * ny));
    const int pi0 = r.ps[0] + i, pi1 = r.ps[1] + j, pi2 = r.ps[2] + k;
    const double x[3] = {g.pc[g.pc_off[0] + pi0] - org[0], g.pc[g.pc_off[1] + pi1] - org[1], g.pc[g.pc_off[2] + pi2] - org[2]};
    double xi[3], p[3];
    okc = iso::project_hex8_from<ElemT, PMODE>(EL, re, c_hex_sg, c_hex_edges, x, rho_t, gs, S0.xi, ok0, xi, nit);
    iso::eval_pos(EL, xi, p);
    double d0 = x[0] - p[0], d1 = x[1] - p[1], d2 = x[2] - p[2];
    const double dd = sqrt(fma(d2, d2, fma(d1, d1, d0 * d0)));
    bool direct = false;
    if constexpr (!WANT_XP) {
      direct = tile_faces[((i64)(pi2 / TILE_Z) * g.nt[1] + pi1 / TILE_Y) * g.nt[0] + pi0 / TILE_X] == 0;
      if (direct) atomicMin((u64 *)&dist[((i64)pi2 * g.np[1] + pi1) * g.np[0] + pi0], (u64)__double_as_longlong(dd));
    }
    if (!direct) pairbuf[r.pair_off + li] = dd;
    if (WANT_XP) { pairxp[3 * (r.pair_off + li)] = p[0] + org[0]; pairxp[3 * (r.pair_off + li) + 1] = p[1] + org[1]; pairxp[3 * (r.pair_off + li) + 2] = p[2] + org[2]; }
  }
  proj_stats(counters, nit > 0 ? nit : 0, !okc, lane);
}

// ---- pair-list path for box elements (the headline workload: every voxel-type SIMP mesh) ----------------------------------------
// evalDistances keeps, per grid point, the MINIMUM over the crossing elements whose candidate range holds the point
// (sdfOnDensityField.jl:606-621).  A pair whose lower bound -- the distance from the point to a set that contains the element's
// iso-patch -- is not below the point's current minimum cannot change the result, so it is never projected (exact: the result is a
// minimum).  Organisation:
//   k_box_records  per crossing box element: solver constants (iso::HexBox in element-local coordinates), phase 1, the TIGHT box of its
//                  iso-patch and a slab that holds the patch (r2s_bound.cuh); the bound of a pair is the distance to box /\ slab
//   k_pair_scan<0> seed: for every pair that does not go to the pair buffer, atomicMin of (float tight-box distance rounded down) << 32
//                  | element on a per-point key -- each point's nearest element box, ties to the smaller active index (the seed only
//                  chooses which pair pass A solves; seeding by box /\ slab solved 0.7 % of the pairs fewer on the replica of
//                  tools/prune_study.py and cost an exact bound for every pair)
//   k_pair_scan<1> pass A: every pair of a tile with boundary-face elements (those go to the pair buffer un-pruned: k_assemble replays
//                  them in element order) and, for each other point, the one pair its key names
//   k_pair_scan<2> pass B, after pass A has been projected: the other pairs, kept only if their bound is below dist[] so far (the cheap
//                  tight-box bound first, then box distance + slab gap (lb2_box_gap), box /\ slab only for the pairs both leave)
//   k_project_list one LANE per listed pair (dense warps whatever was pruned), result by atomicMin / into the pair buffer.
struct __align__(16) BoxRec {      // 16-byte aligned: the projection kernel reads its doubles two at a time
  double R[8];               // monomial coefficients of rho
  double c[3], h[3];         // X_d = c_d + h_d xi_d in element-local coordinates (node 0 at the origin)
  double org[3];             // node 0
  double xi0[3];             // phase 1: Newton projection of xi = 0 onto the iso-surface
  double gs;                 // scale of the tolerances
  double tlo[3], thi[3];     // tight box of the iso-patch, GLOBAL coordinates (slightly widened)
  double sn[3], sA, sB;      // slab sA <= sn.y <= sB that holds the iso-patch, GLOBAL coordinates (r2s_bound.cuh; sn = 0: unbounded)
  i64 pair_off;
  int ps[3], nx, ny, vol, ok0, el;
  int ftile, pad_;           // 1 = some tile overlapped by the candidate range holds boundary-face elements (its pairs may go to the pair buffer)
};
__global__ void k_box_records(i64 nact, const ActRec *__restrict__ rec, const int *__restrict__ IEN, const double *__restrict__ X, const double *__restrict__ rn,
                              const unsigned char *__restrict__ ebox, double rho_t, GridDev g, const unsigned char *__restrict__ tile_faces, BoxRec *__restrict__ box, u64 *__restrict__ too_big) {
  const i64 a = blockIdx.x * (i64)blockDim.x + threadIdx.x;
  if (a >= nact) return;
  const ActRec r = rec[a];
  BoxRec B; B.el = r.el; B.pair_off = r.pair_off; B.vol = 0; B.ok0 = 0;
  if (r.cls != 2 || !ebox[r.el]) { box[a].vol = 0; return; }
  double nv[4][8];
#pragma unroll
  for (int k = 0; k < 8; k++) { const i64 n = IEN[8 * (i64)r.el + k]; nv[0][k] = X[3 * n]; nv[1][k] = X[3 * n + 1]; nv[2][k] = X[3 * n + 2]; nv[3][k] = rn[n]; }
  double A[4][8];
#pragma unroll
  for (int d = 0; d < 3; d++) {
    B.org[d] = nv[d][0];
#pragma unroll
    for (int k = 0; k < 8; k++) nv[d][k] -= B.org[d];
    iso::monomial8(nv[d], A[d]);
  }
  iso::monomial8(nv[3], A[3]);
  iso::HexBox H; iso::make_box(A, H);
#pragma unroll
  for (int k = 0; k < 8; k++) B.R[k] = H.R[k];
  double gs = fabs(rho_t);
#pragma unroll
  for (int k = 0; k < 8; k++) gs = fmax(gs, fabs(nv[3][k]));
  B.gs = fmax(gs, 1.0);
  iso::ProjState S0; B.ok0 = iso::proj_init_element<iso::HexBox, PMODE>(H, rho_t, B.gs, S0) ? 1 : 0;
#pragma unroll
  for (int d = 0; d < 3; d++) { B.c[d] = H.c[d]; B.h[d] = H.h[d]; B.xi0[d] = S0.xi[d]; B.ps[d] = r.ps[d]; }
  B.nx = r.pe[0] - r.ps[0]; B.ny = r.pe[1] - r.ps[1]; B.vol = B.nx * B.ny * (r.pe[2] - r.ps[2]);
  if ((i64)B.nx * B.ny * (r.pe[2] - r.ps[2]) >= (1ll << 24)) { B.vol = 0; atomicAdd(too_big, 1ull); }      // a pair-list entry holds 24 bits of local point index (PL_LI_BITS)
  B.ftile = 0; B.pad_ = 0;
  if (B.vol > 0)
    for (int tz = r.ps[2] / TILE_Z; tz <= (r.pe[2] - 1) / TILE_Z; tz++)
      for (int ty = r.ps[1] / TILE_Y; ty <= (r.pe[1] - 1) / TILE_Y; ty++)
        for (int tx = r.ps[0] / TILE_X; tx <= (r.pe[0] - 1) / TILE_X; tx++)
          if (tile_faces[((i64)tz * g.nt[1] + ty) * g.nt[0] + tx]) B.ftile = 1;
  bnd::box_iso_bounds(nv[3], rho_t, B.gs, B.org, H.c, H.h, B.tlo, B.thi, B.sn, B.sA, B.sB);
  box[a] = B;
}
// one warp per active element; lanes stride over its candidate points.  plist entry: bit 63 = goes to the pair buffer, bits 24..62 =
// active-element index, bits 0..23 = local point index.  cnt[0] = list length.  seed: per grid point the key of k_pair_scan<0>.
#define PL_LI_BITS 24
#ifndef R2S_SCAN_MINB
#define R2S_SCAN_MINB 4      // pair scan: 64 registers (a few spills), 4 CTAs of 256 threads per SM: project 43.8 -> 42.7 ms against the unconstrained 94-register build
#endif
#ifndef R2S_PL_MINB
#define R2S_PL_MINB 4      // resident CTAs per SM the projection kernel is compiled for: 4 = 128 registers (solve 36.1 ms), 5 = 96 registers with spills (37.5), 3 = 167 registers (42.3); tools/gpu_ab_libs.sh
#endif
template <int PASS>
__global__ void __launch_bounds__(256, R2S_SCAN_MINB) k_pair_scan(i64 nact, const BoxRec *__restrict__ box, GridDev g, const unsigned char *__restrict__ tile_faces, const double *__restrict__ dist,
                                                   int prune, u64 *__restrict__ seed, u64 *__restrict__ plist, u64 *__restrict__ cnt, u64 *__restrict__ stats) {
  const i64 a = (blockIdx.x * (i64)blockDim.x + threadIdx.x) >> 5; const int lane = threadIdx.x & 31;
  if (a >= nact) return;
  const int vol = box[a].vol;
  if (vol == 0) return;
  const BoxRec &B = box[a];
  const int nx = B.nx, ny = B.ny, ps0 = B.ps[0], ps1 = B.ps[1], ps2 = B.ps[2];
  const bool ftile = B.ftile != 0;
  // The point coordinates are taken as amin + cell * i here (no table look-up; at most an ulp from the tabulated value): the seed is
  // free to choose, and the bounds are compared with a relative margin of 1e-10 (lb_box_slab's own margin covers the ulp as well).
  double tlo[3], thi[3];
#pragma unroll
  for (int d = 0; d < 3; d++) { tlo[d] = B.tlo[d]; thi[d] = B.thi[d]; }
  // local point index li = lane, lane + 32, ... -> (ci, cj, ck), advanced by 32 per round without divisions (runtime divisors cost ~25
  // instructions each and were 40 % of this kernel's instructions)
  int ci = lane % nx, cj = (lane / nx) % ny, ck = lane / (nx * ny);
  const int r32 = 32 % nx, q32 = 32 / nx, jq = q32 % ny, kq = q32 / ny;
  if (PASS == 0) {      // seed: no list; the key is read first and the atomic only issued when it would lower it (keys only decrease,
                        // so a stale read only costs an atomic)
    for (int li = lane; li < vol; li += 32) {
      const int pi0 = ps0 + ci, pi1 = ps1 + cj, pi2 = ps2 + ck;
      { ci += r32; const int c = ci >= nx ? 1 : 0; ci -= c ? nx : 0; cj += jq + c; ck += kq; if (cj >= ny) { cj -= ny; ck++; } }
      if (ftile && tile_faces[((i64)(pi2 / TILE_Z) * g.nt[1] + pi1 / TILE_Y) * g.nt[0] + pi0 / TILE_X] != 0) continue;
      const double x0 = fma(g.cell, (double)pi0, g.amin[0]), x1 = fma(g.cell, (double)pi1, g.amin[1]), x2 = fma(g.cell, (double)pi2, g.amin[2]);
      const double e0 = fmax(fmax(tlo[0] - x0, x0 - thi[0]), 0.0), e1 = fmax(fmax(tlo[1] - x1, x1 - thi[1]), 0.0), e2 = fmax(fmax(tlo[2] - x2, x2 - thi[2]), 0.0);
      const u64 key = ((u64)__float_as_uint(__double2float_rd(sqrt(fma(e2, e2, fma(e1, e1, e0 * e0))))) << 32) | (u64)a;
      u64 *sp = &seed[((i64)pi2 * g.np[1] + pi1) * g.np[0] + pi0];
      if (key < *sp) atomicMin((unsigned long long *)sp, key);
    }
    return;
  }
  constexpr int RB = 7;      // rounds handled as one batch: all loads of a batch are issued before the first decision (32 * 7 >= 6^3 points)
  const bool slab = B.sA != -INFINITY;
  int npruned = 0;
  for (int base0 = 0; base0 < vol; base0 += 32 * RB) {
    double lb2[RB], cur[RB]; int flags[RB];      // flags: bit 0 valid candidate of this pass, bit 1 to_buf, bit 2 needs the bound test
#pragma unroll
    for (int r = 0; r < RB; r++) {
      const int li = base0 + r * 32 + lane;
      flags[r] = 0; lb2[r] = 0.0; cur[r] = R2S_BIG;
      const int i = ci, j = cj, k = ck;
      { ci += r32; const int c = ci >= nx ? 1 : 0; ci -= c ? nx : 0; cj += jq + c; ck += kq; if (cj >= ny) { cj -= ny; ck++; } }
      if (li < vol) {
        const int pi0 = ps0 + i, pi1 = ps1 + j, pi2 = ps2 + k;
        const i64 v = ((i64)pi2 * g.np[1] + pi1) * g.np[0] + pi0;
        const bool to_buf = ftile && tile_faces[((i64)(pi2 / TILE_Z) * g.nt[1] + pi1 / TILE_Y) * g.nt[0] + pi0 / TILE_X] != 0;
        const bool seeded = !to_buf && prune && (unsigned)seed[v] == (unsigned)a;      // this pair is its point's seed (pass A)
        if (PASS == 1) { if (to_buf || seeded || !prune) flags[r] = 1 | (to_buf ? 2 : 0); }
        else if (!to_buf && !seeded) {
          const double x0 = fma(g.cell, (double)pi0, g.amin[0]), x1 = fma(g.cell, (double)pi1, g.amin[1]), x2 = fma(g.cell, (double)pi2, g.amin[2]);
          const double e0 = fmax(fmax(tlo[0] - x0, x0 - thi[0]), 0.0), e1 = fmax(fmax(tlo[1] - x1, x1 - thi[1]), 0.0), e2 = fmax(fmax(tlo[2] - x2, x2 - thi[2]), 0.0);
          lb2[r] = fma(e2, e2, fma(e1, e1, e0 * e0));
          cur[r] = dist[v];
          flags[r] = 1 | 4;
        }
      }
    }
    // pass B: the tight box first; the two slab bounds only for the pairs it leaves, in a rolled loop (one copy of lb_box_slab; the point
    // and its dist[] entry, unchanged since the batch read it, are fetched again)
    unsigned keepb = 0, need = 0;
#pragma unroll
    for (int r = 0; r < RB; r++) {
      bool keep = (flags[r] & 1) != 0;
      if (PASS == 2 && keep) {
        if (lb2[r] > cur[r] * cur[r] * (1.0 + 1e-10)) { keep = false; npruned++; }
        else if (slab) need |= 1u << r;
      }
      keepb |= (keep ? 1u : 0u) << r;
    }
    while (PASS == 2 && need) {
      const int r = __ffs(need) - 1; need &= need - 1;
      const int li = base0 + r * 32 + lane;
      const int pi0 = ps0 + li % nx, pi1 = ps1 + (li / nx) % ny, pi2 = ps2 + li / (nx * ny);
      const double c = dist[((i64)pi2 * g.np[1] + pi1) * g.np[0] + pi0], c2 = c * c * (1.0 + 1e-10);
      const double P[3] = {fma(g.cell, (double)pi0, g.amin[0]), fma(g.cell, (double)pi1, g.amin[1]), fma(g.cell, (double)pi2, g.amin[2])};
      const double n[3] = {B.sn[0], B.sn[1], B.sn[2]};
      bool prn = bnd::lb2_box_gap(P, tlo, thi, n, B.sA, B.sB) > c2;
      if (!prn) { const double lb = bnd::lb_box_slab(P, tlo, thi, n, B.sA, B.sB); prn = lb * lb > c2; }
      if (prn) { keepb &= ~(1u << r); npruned++; }
    }
    // ONE list-slot claim per warp and batch: a single global counter serves the whole grid, and same-address atomics retire at about one
    // per clock -- a claim per 32-point round (7 per element) made this kernel atomic-bound (ncu: 3.4 + 7.2 ms)
    unsigned keepm[RB]; int total = 0;
#pragma unroll
    for (int r = 0; r < RB; r++) {
      keepm[r] = __ballot_sync(0xffffffffu, (keepb >> r) & 1u);
      total += __popc(keepm[r]);
    }
    if (total) {
      u64 pos = 0;
      if (lane == 0) pos = atomicAdd(&cnt[0], (u64)total);
      pos = __shfl_sync(0xffffffffu, pos, 0);
#pragma unroll
      for (int r = 0; r < RB; r++) {
        if ((keepm[r] >> lane) & 1u) plist[pos + __popc(keepm[r] & ((1u << lane) - 1))] = ((u64)((flags[r] >> 1) & 1) << 63) | ((u64)a << PL_LI_BITS) | (u64)(base0 + r * 32 + lane);
        pos += __popc(keepm[r]);
      }
    }
  }
  if (PASS == 2) {      // statistics: spread over the 128 counter slots (summed on the host)
    for (int o = 16; o > 0; o >>= 1) npruned += __shfl_down_sync(0xffffffffu, npruned, o);
    if (lane == 0 && npruned) atomicAdd(&stats[8 * (1 + (blockIdx.x & 127)) + 4], (u64)npruned);
  }
}
// grid-stride over the list: consecutive lanes take consecutive entries (mostly the same element: broadcast loads of its record)
__global__ void __launch_bounds__(128, R2S_PL_MINB) k_project_list(const u64 *__restrict__ plist, const u64 *__restrict__ cnt, const BoxRec *__restrict__ box, const int *__restrict__ IEN,
                                                         const double *__restrict__ rn, GridDev g, double rho_t, double *__restrict__ pairbuf, double *__restrict__ dist,
                                                         u64 *__restrict__ counters) {
  const u64 n = cnt[0];
  const int lane = threadIdx.x & 31;
  const u64 stride = (u64)gridDim.x * blockDim.x;
  int its = 0, nbad = 0;
  for (u64 base = (u64)blockIdx.x * blockDim.x + (threadIdx.x & ~31u); base < n; base += stride) {      // warp-uniform trip count
    const u64 it = base + lane;
    if (it < n) {
      const u64 ent = plist[it];
      const bool to_buf = (ent >> 63) != 0; const i64 a = (i64)((ent & 0x7fffffffffffffffull) >> PL_LI_BITS); const int li = (int)(ent & ((1u << PL_LI_BITS) - 1));
      const BoxRec &B = box[a];
      iso::HexBox H;
#pragma unroll
      for (int k = 0; k < 8; k++) H.R[k] = B.R[k];
#pragma unroll
      for (int d = 0; d < 3; d++) { H.c[d] = B.c[d]; H.h[d] = B.h[d]; H.hh[d] = 2.0 * (H.h[d] * H.h[d]); }
      const int nx = B.nx, ny = B.ny;
      const int i = li % nx, j = (li / nx) % ny, k = li / (nx * ny);
      const int pi0 = B.ps[0] + i, pi1 = B.ps[1] + j, pi2 = B.ps[2] + k;
      const double x[3] = {g.pc[g.pc_off[0] + pi0] - B.org[0], g.pc[g.pc_off[1] + pi1] - B.org[1], g.pc[g.pc_off[2] + pi2] - B.org[2]};
      const double gs = B.gs; const bool ok0 = B.ok0 != 0;
      double xi0[3] = {B.xi0[0], B.xi0[1], B.xi0[2]}, xi[3], p[3]; int nit = 0;
      iso::ProjState S;
      S.xi[0] = xi0[0]; S.xi[1] = xi0[1]; S.xi[2] = xi0[2]; S.lam = 0.0; S.f = 0.0; S.it = 0; S.stall = 0; S.force = false;
      bool okc = true;
      if (!ok0) {      // rare: phase 1 failed for this element -> per-point edge fallback (needs the nodal densities)
        double re[8];
#pragma unroll
        for (int q = 0; q < 8; q++) re[q] = rn[IEN[8 * (i64)B.el + q]];
        okc = iso::proj_init<iso::HexBox, PMODE>(H, re, c_hex_sg, c_hex_edges, x, rho_t, gs, S);
      }
      if (okc) {
        int status = 0;
        while (S.it < 100 && status == 0) status = iso::proj_iter<iso::HexBox, PMODE>(H, x, rho_t, gs, S);
        okc = status == 1; nit = S.it;
        xi[0] = S.xi[0]; xi[1] = S.xi[1]; xi[2] = S.xi[2];
      } else { xi[0] = xi[1] = xi[2] = 0.0; nit = -1; }
      iso::eval_pos(H, xi, p);
      const double d0 = x[0] - p[0], d1 = x[1] - p[1], d2 = x[2] - p[2];
      const double dd = sqrt(fma(d2, d2, fma(d1, d1, d0 * d0)));
      if (to_buf) pairbuf[B.pair_off + li] = dd;
      else atomicMin((u64 *)&dist[((i64)pi2 * g.np[1] + pi1) * g.np[0] + pi0], (u64)__double_as_longlong(dd));
      its += nit > 0 ? nit : 0; nbad += okc ? 0 : 1;
    }
  }
  for (int o = 16; o > 0; o >>= 1) { its += __shfl_down_sync(0xffffffffu, its, o); nbad += __shfl_down_sync(0xffffffffu, nbad, o); }
  if (lane == 0) { u64 *cs = counters + 8 * (1 + (blockIdx.x & 127)); atomicAdd(&cs[2], (u64)its); if (nbad) atomicAdd(&cs[3], (u64)nbad); }
}
template <bool WANT_XP>
__global__ void __launch_bounds__(128) k_project_tet4(i64 nitems, i64 nact, const ActRec *__restrict__ rec, const i64 *__restrict__ choff,
                                                      const int *__restrict__ IEN, const double *__restrict__ X, const double *__restrict__ rn, GridDev g,
                                                      double rho_t, double *__restrict__ pairbuf, double *__restrict__ pairxp, u64 *__restrict__ counters) {
  i64 item = (blockIdx.x * (i64)blockDim.x + threadIdx.x) >> 5; int lane = threadIdx.x & 31;
  if (item >= nitems) return;
  i64 lo = 0, hi = nact - 1;
  while (lo < hi) { i64 mid = (lo + hi + 1) >> 1; if (choff[mid] <= item) lo = mid; else hi = mid - 1; }
  const ActRec r = rec[lo];
  int chunk = (int)(item - choff[lo]);
  double Xe[3][4], re[4];
  for (int a = 0; a < 4; a++) { i64 n = IEN[4 * (i64)r.el + a]; re[a] = rn[n]; for (int d = 0; d < 3; d++) Xe[d][a] = X[3 * n + d]; }
  int nx = r.pe[0] - r.ps[0], ny = r.pe[1] - r.ps[1], nz = r.pe[2] - r.ps[2];
  i64 vol = (i64)nx * ny * nz, li = (i64)chunk * 32 + lane;
  if (li < vol) {
    int i = (int)(li % nx), j = (int)((li / nx) % ny), k = (int)(li / ((i64)nx * ny));
    double x[3] = {g.pc[g.pc_off[0] + r.ps[0] + i], g.pc[g.pc_off[1] + r.ps[1] + j], g.pc[g.pc_off[2] + r.ps[2] + k]}, p[3];
    bool ok = iso::project_tet4(Xe, re, c_tet_isn, x, rho_t, p);
    double dist = -1.0;     // negative = "no projection" (the reference would keep the running value)
    if (ok) { double d0 = x[0] - p[0], d1 = x[1] - p[1], d2 = x[2] - p[2]; dist = sqrt((d0 * d0 + d1 * d1) + d2 * d2); }
    else atomicAdd(&counters[3], 1ull);
    pairbuf[r.pair_off + li] = dist;
    if (WANT_XP) { pairxp[3 * (r.pair_off + li)] = p[0]; pairxp[3 * (r.pair_off + li) + 1] = p[1]; pairxp[3 * (r.pair_off + li) + 2] = p[2]; }
  }
}

__global__ void k_tri_count(i64 nact, const ActRec *__restrict__ rec, int nsn, int *__restrict__ cnt) {
  i64 a = blockIdx.x * (i64)blockDim.x + threadIdx.x;
  if (a >= nact) return;
  cnt[a] = __popc((unsigned)rec[a].fmask) * nsn;
}
template <int NEN>
__global__ void k_tri_records(i64 nact, ActRec *__restrict__ rec, const int *__restrict__ toff, const int *__restrict__ IEN, const double *__restrict__ X, GridDev g,
                              double delta, TriRec *__restrict__ tri, int *__restrict__ fc_list, u64 *__restrict__ fc_count) {
  i64 a = blockIdx.x * (i64)blockDim.x + threadIdx.x;
  if (a >= nact) return;
  ActRec r = rec[a];
  rec[a].tri_off = toff[a];
  if (!r.fmask) return;
  if (r.cls == 2) fc_list[atomicAdd(fc_count, 1ull)] = (int)a;      // crossing element with boundary faces: work list of k_faces_crossing (a few 10^4 entries)
  double Xe[3][NEN];
  for (int q = 0; q < NEN; q++) { i64 n = IEN[NEN * (i64)r.el + q]; for (int d = 0; d < 3; d++) Xe[d][q] = X[3 * n + d]; }
  face_triangles<NEN, false>(Xe, r.fmask, g, delta, tri + toff[a]);
}
// Boundary faces of CROSSING elements (process_boundary_faces!(..., false), :584).  For a crossing element every candidate of
// process_triangle_projection! is accepted or rejected by the rho-test alone (IsProjectedOnFullSegment, :78-119) -- never by
// the running minimum -- and accepted candidates only ever lower the minimum.  So the element's face contribution to a grid
// point is ONE number, min over its boundary triangles, independent of the order of anything else, and it can be folded into
// the element's entry of the pair buffer: pair = min(iso distance, face candidates).  One warp per crossing element with
// boundary faces, lanes over the element's candidate points; the order-dependent replay (k_assemble) is then left with the
// faces of SOLID elements only, which need no inverse map.
template <int NEN>
__global__ void __launch_bounds__(128) k_faces_crossing(const int *__restrict__ fc_list, const u64 *__restrict__ fc_count, const ActRec *__restrict__ rec, const TriRec *__restrict__ tri,
                                                        const int *__restrict__ IEN, const double *__restrict__ X, const double *__restrict__ rn, GridDev g, double rho_t,
                                                        double *__restrict__ pairbuf) {
  constexpr int NSN = NEN == 8 ? 4 : 3;
  const int lane = threadIdx.x & 31; const i64 nlist = (i64)*fc_count;
  for (i64 w = (blockIdx.x * (i64)blockDim.x + threadIdx.x) >> 5; w < nlist; w += ((i64)gridDim.x * blockDim.x) >> 5) {
  const ActRec r = rec[fc_list[w]];
  double Xe[3][NEN], re[NEN];
  for (int q = 0; q < NEN; q++) { i64 n = IEN[NEN * (i64)r.el + q]; re[q] = rn[n]; for (int d = 0; d < 3; d++) Xe[d][q] = X[3 * n + d]; }
  ex::AffineInv pre; pre.affine = 0;
  if (NEN == 8) {      // element-only part of the inverse map, once per warp instead of once per candidate
    double A[3][8];
#pragma unroll
    for (int d = 0; d < 3; d++) ex::mono8((const double *)Xe[d], A[d]);
    ex::affine_inverse_prepare(A, pre);
  }
  const int ntri = __popc((unsigned)r.fmask) * NSN;
  const int nx = r.pe[0] - r.ps[0], ny = r.pe[1] - r.ps[1], nz = r.pe[2] - r.ps[2], vol = nx * ny * nz;
  for (int li = lane; li < vol; li += 32) {
    const int pi[3] = {r.ps[0] + li % nx, r.ps[1] + (li / nx) % ny, r.ps[2] + li / (nx * ny)};
    const double x[3] = {g.pc[g.pc_off[0] + pi[0]], g.pc[g.pc_off[1] + pi[1]], g.pc[g.pc_off[2] + pi[2]]};
    VoxState s; s.c = -R2S_BIG; s.xp[0] = s.xp[1] = s.xp[2] = 0.0;
    for (int t = 0; t < ntri; t++) {
      const TriRec &T = tri[r.tri_off + t];
      if (pi[0] < T.ps[0] || pi[0] >= T.pe[0] || pi[1] < T.ps[1] || pi[1] >= T.pe[1] || pi[2] < T.ps[2] || pi[2] >= T.pe[2]) continue;
      double Xt[3][3], Et[3][3], n[3];
      for (int d = 0; d < 3; d++) { Xt[0][d] = T.Xt[0][d]; Xt[1][d] = T.Xt[1][d]; Xt[2][d] = T.Xt[2][d]; n[d] = T.n[d]; }
      for (int d = 0; d < 3; d++) { Et[0][d] = ex::sub(Xt[1][d], Xt[0][d]); Et[1][d] = ex::sub(Xt[2][d], Xt[1][d]); Et[2][d] = ex::sub(Xt[0][d], Xt[2][d]); }
      triangle_point<false, NEN>(Xe, re, rho_t, false, Xt, Et, n, x, s, &pre);
    }
    if (s.c != -R2S_BIG) {
      const i64 idx = r.pair_off + li;
      const double cur = pairbuf[idx];
      if (!(cur >= 0.0 && cur <= s.c)) pairbuf[idx] = s.c;
    }
  }
  }
}

// ------------------------------------------------------------------------------------------------ assemble (exact)
// One CTA per tile, one thread per grid point; the tile's element list is culled per warp (footprint 8x4x1 points) into
// shared memory in list order, then every lane replays ITS candidates in ascending element order (a warp-uniform walk over the
// culled records was measured: 13.5 vs 8.4 ms -- the per-lane cursors keep 32 different triangles in flight per round).
#define ACULL_CAP 96
// FACES = false: tiles whose list holds no element with boundary faces (the vast majority; only needed when xp is wanted or for
// TET4) -- one CTA per tile, tiles of the other kind exit.  FACES = true: the tiles with boundary-face elements, taken from the
// compacted list k_face_tile_list wrote (a few per cent of all tiles), grid-stride.
__global__ void k_face_tile_list(int ntiles, const unsigned char *__restrict__ tile_faces, int *__restrict__ list, u64 *__restrict__ count) {
  const int t = blockIdx.x * blockDim.x + threadIdx.x, lane = threadIdx.x & 31;
  const bool f = t < ntiles && tile_faces[t] != 0;
  const unsigned m = __ballot_sync(0xffffffffu, f);
  if (!m) return;
  u64 base = 0;
  if (lane == 0) base = atomicAdd(count, (u64)__popc(m));
  base = __shfl_sync(0xffffffffu, base, 0);
  if (f) list[base + __popc(m & ((1u << lane) - 1))] = t;
}
template <bool WANT_XP, int NEN, bool FACES>
__global__ void __launch_bounds__(TILE_VOX) k_assemble(GridDev g, int kz0, int kz1, const unsigned char *__restrict__ tile_faces, const int *__restrict__ face_list, u64 *__restrict__ nface,
                                                       const int *__restrict__ tile_ptr, const u64 *__restrict__ keys,
                                                       const ActRec *__restrict__ rec, const TriRec *__restrict__ tri, const int *__restrict__ IEN, const double *__restrict__ X,
                                                       const double *__restrict__ rn, double rho_t, double delta, const double *__restrict__ pairbuf,
                                                       const double *__restrict__ pairxp, double *__restrict__ dist, double *__restrict__ xpo) {
  __shared__ ActRec srec[TILE_VOX / 32][ACULL_CAP];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  __shared__ int s_next;
  const int nlist = FACES ? (int)nface[0] : (int)gridDim.x;
  for (int it = blockIdx.x;;) {
  if (FACES) {        // tiles differ a lot in work (edges and corners of the domain): fetch them dynamically
    __syncthreads();
    if (threadIdx.x == 0) s_next = (int)atomicAdd((u64 *)&nface[1], 1ull);
    __syncthreads();
    it = s_next;
  }
  if (it >= nlist) return;
  const int t = FACES ? face_list[it] : it;
  if (!FACES && tile_faces[t] != 0) return;
  const int tx = t % g.nt[0], ty = (t / g.nt[0]) % g.nt[1], tz = t / (g.nt[0] * g.nt[1]);
  const int li = threadIdx.x % TILE_X, lj = (threadIdx.x / TILE_X) % TILE_Y, lk = threadIdx.x / (TILE_X * TILE_Y);
  const int pi[3] = {tx * TILE_X + li, ty * TILE_Y + lj, tz * TILE_Z + lk};
  const bool valid = pi[0] < g.np[0] && pi[1] < g.np[1] && pi[2] < g.np[2] && pi[2] >= kz0 && pi[2] < kz1;
  const int wx0 = tx * TILE_X, wx1 = wx0 + TILE_X - 1, wy0 = ty * TILE_Y + (warp % (TILE_Y / 4)) * 4, wy1 = wy0 + 3, wz = tz * TILE_Z + warp / (TILE_Y / 4);
  double x[3] = {0, 0, 0};
  if (valid) { x[0] = g.pc[g.pc_off[0] + pi[0]]; x[1] = g.pc[g.pc_off[1] + pi[1]]; x[2] = g.pc[g.pc_off[2] + pi[2]]; }
  VoxState s; s.c = -R2S_BIG; s.xp[0] = s.xp[1] = s.xp[2] = 0.0;
  const int p0 = tile_ptr[t], p1 = tile_ptr[t + 1];
  int p = p0;
  while (p < p1) {
    int n = 0;
    while (p < p1 && n <= ACULL_CAP - 32) {
      int idx = p + lane; bool ov = false; ActRec r;
      if (idx < p1) {
        r = rec[(int)(keys[idx] & 0xffffffffull)];
        ov = r.ps[0] <= wx1 && r.pe[0] > wx0 && r.ps[1] <= wy1 && r.pe[1] > wy0 && r.ps[2] <= wz && r.pe[2] > wz;
      }
      unsigned m = __ballot_sync(0xffffffffu, ov);
      if (ov) srec[warp][n + __popc(m & ((1u << lane) - 1))] = r;
      n += __popc(m); p += 32;
    }
    __syncwarp();
    // which culled records contain THIS lane's point: one uniform sweep (broadcast reads)
    unsigned mk0 = 0, mk1 = 0, mk2 = 0;
    for (int q = 0; q < n; q++) {
      const ActRec &r = srec[warp][q];
      if (valid && pi[0] >= r.ps[0] && pi[0] < r.pe[0] && pi[1] >= r.ps[1] && pi[1] < r.pe[1] && pi[2] >= r.ps[2] && pi[2] < r.pe[2]) {
        if (q < 32) mk0 |= 1u << q; else if (q < 64) mk1 |= 1u << (q - 32); else mk2 |= 1u << (q - 64);
      }
    }
    // Every lane walks ITS records in list order (= ascending element index) and, inside a record, its boundary triangles in
    // order, then takes the record's pair-buffer entry -- exactly the reference's sequence for that grid point.  The lanes do
    // not wait for each other's records: in each round every lane brings its own next triangle to triangle_point, so the
    // expensive part runs with (nearly) full warps instead of only the lanes that happen to share the current element.
    constexpr int NSN = NEN == 8 ? 4 : 3;
    int w = 0, pos = -1, t = 0, ntri = 0; unsigned cur = mk0; bool more = valid;
    ActRec r; r.cls = 0; r.tri_off = 0; r.pair_off = 0; r.fmask = 0; r.el = 0;
    double Xe[3][NEN], re[NEN]; bool loaded = false;
    while (true) {
      int ti = -1;                                   // index of this lane's next triangle (work item of this round)
      while (more && ti < 0) {
        if (t < ntri) {
          const TriRec &T = tri[r.tri_off + t]; const int tcur = t; t++;
          if (pi[0] < T.ps[0] || pi[0] >= T.pe[0] || pi[1] < T.ps[1] || pi[1] >= T.pe[1] || pi[2] < T.ps[2] || pi[2] >= T.pe[2]) continue;
          if (r.cls == 1) {
            // solid element: no candidate of this triangle can be below the distance to its bounding box; if that is not
            // below the running value the triangle changes nothing (exact; the margin covers the rounding of the candidates)
            double lb2 = 0.0;
#pragma unroll
            for (int d = 0; d < 3; d++) {
              const double e = fmax(fmax(T.lo[d] - x[d], x[d] - T.hi[d]), 0.0);
              lb2 = fma(e, e, lb2);
            }
            const double cv = fabs(s.c) * (1.0 + 1e-12);
            if (lb2 * (1.0 - 1e-12) > cv * cv) continue;
          }
          ti = tcur;
        } else {
          if (pos >= 0 && r.cls == 2) {              // the record's faces are done: now its iso distance (:617-621)
            i64 idx = r.pair_off + ((i64)(pi[2] - r.ps[2]) * (r.pe[1] - r.ps[1]) + (pi[1] - r.ps[1])) * (r.pe[0] - r.ps[0]) + (pi[0] - r.ps[0]);
            double dt = pairbuf[idx];
            if (dt >= 0.0 && fabs(dt) < fabs(s.c)) {
              s.c = dt;
              if (WANT_XP) { s.xp[0] = pairxp[3 * idx]; s.xp[1] = pairxp[3 * idx + 1]; s.xp[2] = pairxp[3 * idx + 2]; }
            }
          }
          while (w < 3 && cur == 0) { w++; cur = (w == 1) ? mk1 : (w == 2 ? mk2 : 0u); }
          if (w >= 3) { more = false; pos = -1; break; }
          const int bq = __ffs(cur) - 1; cur &= cur - 1; pos = w * 32 + bq;
          r = srec[warp][pos];
          t = 0; loaded = false;
          ntri = (FACES && r.fmask && (WANT_XP || r.cls == 1)) ? __popc((unsigned)r.fmask) * NSN : 0;      // crossing faces are folded into the pair buffer unless xp is wanted
          if (ntri && r.cls == 1) {
            // solid element: if even the box around all its boundary triangles is not closer than the running value, none of them can
            // change it (same bound and margin as per triangle below) -- skip the record without touching its triangles
            const TriRec &T0 = tri[r.tri_off];
            double lb2 = 0.0;
#pragma unroll
            for (int d = 0; d < 3; d++) { const double e = fmax(fmax(T0.rlo[d] - x[d], x[d] - T0.rhi[d]), 0.0); lb2 = fma(e, e, lb2); }
            const double cv = fabs(s.c) * (1.0 + 1e-12);
            if (lb2 * (1.0 - 1e-12) > cv * cv) ntri = 0;
          }
        }
      }
      if (!__any_sync(0xffffffffu, ti >= 0)) break;
      if (ti >= 0) {
        const TriRec &T = tri[r.tri_off + ti];
        if (WANT_XP && r.cls != 1 && !loaded) {      // the element itself is only needed for the rho-test of crossing elements (:92-113), replayed here only when xp is wanted
          for (int a = 0; a < NEN; a++) { i64 nd = IEN[NEN * (i64)r.el + a]; re[a] = rn[nd]; for (int d = 0; d < 3; d++) Xe[d][a] = X[3 * nd + d]; }
          loaded = true;
        }
        double Xt[3][3], Et[3][3], nn[3];
        for (int d = 0; d < 3; d++) { Xt[0][d] = T.Xt[0][d]; Xt[1][d] = T.Xt[1][d]; Xt[2][d] = T.Xt[2][d]; nn[d] = T.n[d]; }
        for (int d = 0; d < 3; d++) { Et[0][d] = ex::sub(Xt[1][d], Xt[0][d]); Et[1][d] = ex::sub(Xt[2][d], Xt[1][d]); Et[2][d] = ex::sub(Xt[0][d], Xt[2][d]); }
        triangle_point<WANT_XP, NEN>(Xe, re, rho_t, WANT_XP ? r.cls == 1 : true, Xt, Et, nn, x, s);
      }
    }
    __syncwarp();
  }
  if (valid) {
    i64 v = ((i64)pi[2] * g.np[1] + pi[1]) * g.np[0] + pi[0];
    dist[v] = fabs(s.c);
    if (WANT_XP) { xpo[3 * v] = s.xp[0]; xpo[3 * v + 1] = s.xp[1]; xpo[3 * v + 2] = s.xp[2]; }
  }
  __syncwarp();
  if (!FACES) return;
  }
}

// ------------------------------------------------------------------------------------------------ host driver
int r2s_dev_eval_distances(r2s_ctx *ctx, double rho_t, double delta_factor, bool want_xp) {
  if (!ctx->has_grid) FAIL("r2s_set_grid has not been called");
  if (ctx->nel == 0) FAIL("r2s_set_mesh has not been called");
  const GridDev &g = ctx->g; cudaStream_t st = ctx->stream;
  i64 nel = ctx->nel; int nen = ctx->nen;
  double delta = delta_factor * g.cell;
  int kz0 = (int)ctx->k0, kz1 = (int)ctx->k1;
  CK(cudaEventRecord(ctx->ev[0], st));
  CK(ctx->cls.reserve((size_t)nel));
  CK(ctx->act_flag.reserve(sizeof(int) * (size_t)(nel + 1)));
  CK(ctx->act_idx.reserve(sizeof(int) * (size_t)(nel + 1)));
  constexpr int NCTR = 8 * 129;      // slot 0: element classes; slots 1..128: projection statistics; 8 more words: pair-list counters
  CK(ctx->counters.reserve(sizeof(u64) * (NCTR + 8)));
  CK(cudaMemsetAsync(ctx->counters.p, 0, sizeof(u64) * (NCTR + 8), st));
  CK(cudaMemsetAsync(ctx->act_flag.as<int>() + nel, 0, sizeof(int), st));
  // z-interval of this rank's planes with a margin of (delta + 2 cells): only elements that can reach them are classified
  double zlo = -1e300, zhi = 1e300;
  if (kz0 > 0 || kz1 < g.np[2]) { const double m = delta + 2.0 * g.cell; zlo = ctx->h_pc[2][(size_t)kz0] - m; zhi = ctx->h_pc[2][(size_t)kz1 - 1] + m; }
  k_classify<<<cdiv(nel, 256), 256, 0, st>>>(nel, nen, ctx->IEN32.as<int>(), ctx->rho_n.as<double>(), ctx->fbnd.as<unsigned char>(), ctx->ezr.as<double2>(), zlo, zhi, rho_t,
                                             ctx->cls.as<unsigned char>(), ctx->act_flag.as<int>(), ctx->counters.as<i64>()); LAUNCH_CHECK();
  if (r2s_scan_exclusive_i32(ctx, ctx->act_flag.as<int>(), ctx->act_idx.as<int>(), nel + 1)) return 1;
  int nact_i = 0;
  if (r2s_readback(ctx, &nact_i, ctx->act_idx.as<int>() + nel, sizeof(int))) return 1;
  i64 nact = nact_i;
  CK(ctx->dist.reserve(sizeof(double) * (size_t)g.ngp));
  if (want_xp) CK(ctx->xp.reserve(sizeof(double) * 3 * (size_t)g.ngp));
  CK(ctx->tile_ptr.reserve(sizeof(int) * (size_t)(g.ntiles + 2)));
  CK(cudaMemsetAsync(ctx->tile_ptr.p, 0, sizeof(int) * (size_t)(g.ntiles + 2), st));
  CK(ctx->tile_faces.reserve((size_t)g.ntiles + 16));
  CK(cudaMemsetAsync(ctx->tile_faces.p, 0, (size_t)g.ntiles, st));
  i64 npairs = 0, nkeys = 0, nitems = 0; int ntri = 0;
  u64 *sorted = nullptr;
  if (nact > 0) {
    CK(ctx->act_rec.reserve(sizeof(ActRec) * (size_t)nact));
    CK(ctx->cnt_a.reserve(sizeof(i64) * 3 * (size_t)(nact + 1)));
    CK(ctx->cnt_b.reserve(sizeof(i64) * 3 * (size_t)(nact + 1)));
    i64 *ntile = ctx->cnt_a.as<i64>(), *npair = ntile + (nact + 1), *nchunk = npair + (nact + 1);
    i64 *toff = ctx->cnt_b.as<i64>(), *poff = toff + (nact + 1), *choff = poff + (nact + 1);
    CK(cudaMemsetAsync(ctx->cnt_a.p, 0, sizeof(i64) * 3 * (size_t)(nact + 1), st));
    k_act_records<<<cdiv(nel, 256), 256, 0, st>>>(nel, nen, ctx->IEN32.as<int>(), ctx->X.as<double>(), ctx->cls.as<unsigned char>(), ctx->fbnd.as<unsigned char>(),
                                                  ctx->act_flag.as<int>(), ctx->act_idx.as<int>(), g, delta, kz0, kz1, ctx->act_rec.as<ActRec>(), ntile, npair, nchunk);
    LAUNCH_CHECK();
    if (r2s_scan_exclusive_i64(ctx, ntile, toff, nact + 1)) return 1;
    if (r2s_scan_exclusive_i64(ctx, npair, poff, nact + 1)) return 1;
    if (r2s_scan_exclusive_i64(ctx, nchunk, choff, nact + 1)) return 1;
    {
      const size_t o0 = r2s_rb_put(ctx, toff + nact, sizeof(i64)), o1 = r2s_rb_put(ctx, poff + nact, sizeof(i64)), o2 = r2s_rb_put(ctx, choff + nact, sizeof(i64));
      if (o0 == (size_t)-1 || o1 == (size_t)-1 || o2 == (size_t)-1) return 1;
      // the triangle count of the boundary-face table is read back with the same synchronisation
      CK(ctx->tri_cnt.reserve(sizeof(int) * 2 * (size_t)(nact + 1)));
      int *tcnt = ctx->tri_cnt.as<int>(), *toff32 = tcnt + (nact + 1);
      CK(cudaMemsetAsync(tcnt + nact, 0, sizeof(int), st));
      k_tri_count<<<cdiv(nact, 256), 256, 0, st>>>(nact, ctx->act_rec.as<ActRec>(), ctx->nsn, tcnt); LAUNCH_CHECK();
      if (r2s_scan_exclusive_i32(ctx, tcnt, toff32, nact + 1)) return 1;
      const size_t o3 = r2s_rb_put(ctx, toff32 + nact, sizeof(int));
      if (o3 == (size_t)-1) return 1;
      if (r2s_rb_sync(ctx)) return 1;
      nkeys = *(const i64 *)r2s_rb_at(ctx, o0); npairs = *(const i64 *)r2s_rb_at(ctx, o1); nitems = *(const i64 *)r2s_rb_at(ctx, o2); ntri = *(const int *)r2s_rb_at(ctx, o3);
    }
    if (nkeys >= (1ll << 31) || npairs >= (1ll << 40)) FAIL("distance binning: problem too large for one slab (key/pair count overflow)");
    CK(ctx->keys.reserve(sizeof(u64) * (size_t)(nkeys + 1)));
    CK(ctx->keys_alt.reserve(sizeof(u64) * (size_t)(nkeys + 1)));
    CK(ctx->pairbuf.reserve(sizeof(double) * (size_t)(npairs + 1)));
    if (want_xp) CK(ctx->pairxp.reserve(sizeof(double) * 3 * (size_t)(npairs + 1)));
    k_emit_keys<<<cdiv(nact, 128), 128, 0, st>>>(nact, ctx->act_rec.as<ActRec>(), toff, poff, g, ctx->keys.as<u64>(), ctx->tile_ptr.as<int>() + 1, ctx->tile_faces.as<unsigned char>()); LAUNCH_CHECK();
    int tbits = 1; while ((1ll << tbits) < g.ntiles) tbits++;
    if (nkeys > 0) { if (r2s_sort_keys_u64(ctx, ctx->keys.as<u64>(), ctx->keys_alt.as<u64>(), nkeys, 32 + tbits, &sorted)) return 1; }
    // boundary-face triangle table
    int *toff32 = ctx->tri_cnt.as<int>() + (nact + 1);
    CK(ctx->tri_rec.reserve(sizeof(TriRec) * (size_t)(ntri + 1)));
    CK(ctx->fc_list.reserve(sizeof(int) * (size_t)(nact + 16)));
    u64 *fc_count = ctx->counters.as<u64>() + NCTR + 5;
    if (nen == 8) k_tri_records<8><<<cdiv(nact, 128), 128, 0, st>>>(nact, ctx->act_rec.as<ActRec>(), toff32, ctx->IEN32.as<int>(), ctx->X.as<double>(), g, delta, ctx->tri_rec.as<TriRec>(), ctx->fc_list.as<int>(), fc_count);
    else k_tri_records<4><<<cdiv(nact, 128), 128, 0, st>>>(nact, ctx->act_rec.as<ActRec>(), toff32, ctx->IEN32.as<int>(), ctx->X.as<double>(), g, delta, ctx->tri_rec.as<TriRec>(), ctx->fc_list.as<int>(), fc_count);
    LAUNCH_CHECK();
  }
  // tile_ptr[t+1] currently holds the count of tile t (tile_ptr[0] = 0): inclusive scan in place == exclusive offsets
  {
    DevBuf &tmp = ctx->s_cnt;   // reuse as scratch
    CK(tmp.reserve(sizeof(int) * (size_t)(g.ntiles + 2)));
    if (r2s_scan_exclusive_i32(ctx, ctx->tile_ptr.as<int>() + 1, tmp.as<int>(), g.ntiles + 1)) return 1;
    CK(cudaMemcpyAsync(ctx->tile_ptr.as<int>(), tmp.as<int>(), sizeof(int) * (size_t)(g.ntiles + 1), cudaMemcpyDeviceToDevice, st));
  }
  CK(cudaEventRecord(ctx->ev[1], st));
  // Without xp, dist[] starts at BIG and receives the minima of the face-free tiles by atomicMin; k_assemble then replays only the tiles
  // with boundary-face elements.  With xp everything goes through the pair buffer (the closest point of a voxel is tie-order dependent).
  bool timed_list = false;
  if (!want_xp) {
    i64 v0 = (i64)kz0 * g.np[0] * g.np[1], nv = (i64)(kz1 - kz0) * g.np[0] * g.np[1];
    k_fill_f64<<<cdiv(nv, 256), 256, 0, st>>>(nv, ctx->dist.as<double>() + v0, R2S_BIG); LAUNCH_CHECK();
  }
  if (nitems > 0) {
    i64 *choff = ctx->cnt_b.as<i64>() + 2 * (nact + 1);
    const int nb = cdiv(nitems * 32, 128);
    if (nen == 8) {
      // axis-aligned box elements (flag + count built with the mesh): pair-list path without xp, HexBox chunk kernel with xp; the others
      // take the general trilinear chunk kernel.  R2S_PROJ_BOX=0 sends everything through the general kernel.
      const i64 nbx = ctx->knobs.proj_box ? ctx->n_box : 0; const int kc = (nbx > 0 && nbx < nel) ? 1 : 0;
      const bool list_path = !want_xp && nbx > 0;
#define PROJH(XP, BX, SKIP) k_project_hex8<XP, BX><<<nb, 128, 0, st>>>(nitems, nact, ctx->act_rec.as<ActRec>(), choff, ctx->IEN32.as<int>(), ctx->X.as<double>(), ctx->rho_n.as<double>(), g, rho_t, \
        ctx->pairbuf.as<double>(), ctx->pairxp.as<double>(), ctx->counters.as<u64>(), ctx->ebox.as<unsigned char>(), kc, SKIP, ctx->tile_faces.as<unsigned char>(), ctx->dist.as<double>())
      if (nbx < nel) { if (want_xp) PROJH(true, false, 0); else PROJH(false, false, list_path ? 1 : 0); LAUNCH_CHECK(); }
      if (nbx > 0 && want_xp) { PROJH(true, true, 0); LAUNCH_CHECK(); }
#undef PROJH
      if (list_path) {
        CK(ctx->box_rec.reserve(sizeof(BoxRec) * (size_t)nact));
        CK(ctx->plist.reserve(sizeof(u64) * (size_t)(npairs + 1)));
        u64 *pc = ctx->counters.as<u64>() + NCTR;      // 4 words behind the statistics slots: [0],[1] pass A, [2],[3] pass B
        BoxRec *box = ctx->box_rec.as<BoxRec>(); u64 *pl = ctx->plist.as<u64>();
        CK(cudaEventRecord(ctx->ev_k[0], st));
        k_box_records<<<cdiv(nact, 128), 128, 0, st>>>(nact, ctx->act_rec.as<ActRec>(), ctx->IEN32.as<int>(), ctx->X.as<double>(), ctx->rho_n.as<double>(), ctx->ebox.as<unsigned char>(), rho_t, g, ctx->tile_faces.as<unsigned char>(), box, ctx->counters.as<u64>() + NCTR + 4); LAUNCH_CHECK();
        const int prune = ctx->knobs.proj_prune ? 1 : 0, pgrid = 148 * R2S_PL_MINB * 4;
        u64 *seed = nullptr;
        if (prune) {      // per-point seed keys: all ones = no pair yet
          CK(ctx->pseed.reserve(sizeof(u64) * (size_t)g.ngp));
          seed = ctx->pseed.as<u64>();
          const i64 v0 = (i64)kz0 * g.np[0] * g.np[1], nv = (i64)(kz1 - kz0) * g.np[0] * g.np[1];
          CK(cudaMemsetAsync(seed + v0, 0xff, sizeof(u64) * (size_t)nv, st));
          k_pair_scan<0><<<cdiv(nact * 32, 256), 256, 0, st>>>(nact, box, g, ctx->tile_faces.as<unsigned char>(), ctx->dist.as<double>(), prune, seed, pl, pc, ctx->counters.as<u64>()); LAUNCH_CHECK();
        }
        k_pair_scan<1><<<cdiv(nact * 32, 256), 256, 0, st>>>(nact, box, g, ctx->tile_faces.as<unsigned char>(), ctx->dist.as<double>(), prune, seed, pl, pc, ctx->counters.as<u64>()); LAUNCH_CHECK();
        CK(cudaEventRecord(ctx->ev_k[1], st));
        k_project_list<<<pgrid, 128, 0, st>>>(pl, pc, box, ctx->IEN32.as<int>(), ctx->rho_n.as<double>(), g, rho_t, ctx->pairbuf.as<double>(), ctx->dist.as<double>(), ctx->counters.as<u64>()); LAUNCH_CHECK();
        CK(cudaEventRecord(ctx->ev_k[2], st));
        if (prune) {
          k_pair_scan<2><<<cdiv(nact * 32, 256), 256, 0, st>>>(nact, box, g, ctx->tile_faces.as<unsigned char>(), ctx->dist.as<double>(), prune, seed, pl, pc + 2, ctx->counters.as<u64>()); LAUNCH_CHECK();
          CK(cudaEventRecord(ctx->ev_k[3], st));
          k_project_list<<<pgrid, 128, 0, st>>>(pl, pc + 2, box, ctx->IEN32.as<int>(), ctx->rho_n.as<double>(), g, rho_t, ctx->pairbuf.as<double>(), ctx->dist.as<double>(), ctx->counters.as<u64>()); LAUNCH_CHECK();
        } else CK(cudaEventRecord(ctx->ev_k[3], st));
        CK(cudaEventRecord(ctx->ev_k[4], st));
        timed_list = true;
      }
    } else {
      if (want_xp) k_project_tet4<true><<<nb, 128, 0, st>>>(nitems, nact, ctx->act_rec.as<ActRec>(), choff, ctx->IEN32.as<int>(), ctx->X.as<double>(), ctx->rho_n.as<double>(), g, rho_t, ctx->pairbuf.as<double>(), ctx->pairxp.as<double>(), ctx->counters.as<u64>());
      else k_project_tet4<false><<<nb, 128, 0, st>>>(nitems, nact, ctx->act_rec.as<ActRec>(), choff, ctx->IEN32.as<int>(), ctx->X.as<double>(), ctx->rho_n.as<double>(), g, rho_t, ctx->pairbuf.as<double>(), ctx->pairxp.as<double>(), ctx->counters.as<u64>());
      LAUNCH_CHECK();
    }
  }
  if (!want_xp && nact > 0 && npairs > 0) {
    const u64 *fc_count = ctx->counters.as<u64>() + NCTR + 5;
    const unsigned fcg = (unsigned)std::min<i64>(cdiv(nact * 32, 128), 148 * 32);
    if (nen == 8) k_faces_crossing<8><<<fcg, 128, 0, st>>>(ctx->fc_list.as<int>(), fc_count, ctx->act_rec.as<ActRec>(), ctx->tri_rec.as<TriRec>(), ctx->IEN32.as<int>(), ctx->X.as<double>(), ctx->rho_n.as<double>(), g, rho_t, ctx->pairbuf.as<double>());
    else k_faces_crossing<4><<<fcg, 128, 0, st>>>(ctx->fc_list.as<int>(), fc_count, ctx->act_rec.as<ActRec>(), ctx->tri_rec.as<TriRec>(), ctx->IEN32.as<int>(), ctx->X.as<double>(), ctx->rho_n.as<double>(), g, rho_t, ctx->pairbuf.as<double>());
    LAUNCH_CHECK();
  }
  CK(cudaEventRecord(ctx->ev[2], st));
  {
    // the tiles that hold boundary-face elements, as a list (order irrelevant: tiles are independent)
    u64 *nface = ctx->counters.as<u64>() + NCTR + 6;      // [0] list length, [1] next tile to fetch
    CK(ctx->face_tiles.reserve(sizeof(int) * ((size_t)g.ntiles + 16)));
    k_face_tile_list<<<cdiv(g.ntiles, 256), 256, 0, st>>>((int)g.ntiles, ctx->tile_faces.as<unsigned char>(), ctx->face_tiles.as<int>(), nface); LAUNCH_CHECK();
    const unsigned fgrid = (unsigned)std::min<i64>(g.ntiles, (i64)148 * 64);
#define ASM(XP, NEN, F) k_assemble<XP, NEN, F><<<(F) ? fgrid : (unsigned)g.ntiles, TILE_VOX, 0, st>>>(g, kz0, kz1, ctx->tile_faces.as<unsigned char>(), ctx->face_tiles.as<int>(), nface, ctx->tile_ptr.as<int>(), sorted, \
        ctx->act_rec.as<ActRec>(), ctx->tri_rec.as<TriRec>(), ctx->IEN32.as<int>(), ctx->X.as<double>(), ctx->rho_n.as<double>(), rho_t, delta, ctx->pairbuf.as<double>(), ctx->pairxp.as<double>(), \
        ctx->dist.as<double>(), ctx->xp.as<double>()); LAUNCH_CHECK()
    if (nen == 8) { if (want_xp) { ASM(true, 8, false); ASM(true, 8, true); } else { ASM(false, 8, true); } }      // without xp the face-free tiles are final already
    else { if (want_xp) { ASM(true, 4, false); ASM(true, 4, true); } else { ASM(false, 4, false); ASM(false, 4, true); } }
#undef ASM
  }
  CK(cudaEventRecord(ctx->ev[3], st));
  u64 hall[NCTR + 8], hc[8];
  if (r2s_readback(ctx, hall, ctx->counters.p, sizeof(hall))) return 1;
  for (int q = 0; q < 8; q++) { hc[q] = hall[q]; for (int sl = 1; sl <= 128; sl++) hc[q] += hall[8 * sl + q]; }
  ctx->rep.n_solid = (i64)hc[0]; ctx->rep.n_crossing = (i64)hc[1]; ctx->rep.n_active = nact; ctx->rep.n_pairs = npairs;
  ctx->rep.n_newton_iters = (i64)hc[2]; ctx->rep.n_not_converged = (i64)hc[3];
  ctx->rep.n_pairs_pruned = (i64)hc[4];
  if (hall[NCTR + 4] != 0) FAIL("evalDistances: the grid is so much finer than the mesh that one element's candidate range exceeds 2^24 grid points");
  ctx->rep.ms_solve = ctx->rep.ms_scan = 0.0f;
  if (timed_list) {      // the read-back above synchronised the stream: the events are complete
    float t[4];
    for (int q = 0; q < 4; q++) CK(cudaEventElapsedTime(&t[q], ctx->ev_k[q], ctx->ev_k[q + 1]));
    ctx->rep.ms_scan = t[0] + t[2]; ctx->rep.ms_solve = t[1] + t[3];
  }
  CK(cudaEventElapsedTime(&ctx->rep.ms_bin, ctx->ev[0], ctx->ev[1]));
  CK(cudaEventElapsedTime(&ctx->rep.ms_project, ctx->ev[1], ctx->ev[2]));
  CK(cudaEventElapsedTime(&ctx->rep.ms_assemble, ctx->ev[2], ctx->ev[3]));
  return 0;
}
