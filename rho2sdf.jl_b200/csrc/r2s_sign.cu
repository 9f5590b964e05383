// r2s_sign.cu -- Sign_Detection (SignedDistances/SignDetection.jl:6-81 HEX8, :88-268 TET4) on the GPU, fused with
// sdf_dists = dists .* signs (RhoToSDF.jl:171).
//
// The reference scans all nel element AABBs per grid point (O(ngp*nel)).  Here every element is binned into the voxel
// tiles its candidate point range overlaps ((tile, element) keys, radix sort); a CTA owns one tile, stages the tile's
// element list (ascending element index = the reference's candidate order) through shared memory together with the
// element's nodal coordinates/densities, and every thread replays the reference's per-point rule exactly.
#include <stdlib.h>
#include "r2s_common.cuh"
#include "r2s_tables.cuh"
#include "r2s_exact.cuh"
#include "r2s_signrule.cuh"

struct SRange { int a[3], b[3]; int hot, pad; };   // inclusive grid-point index range of the candidate points of one element; pad = density class (sign_element);
                                                   // hot = some nodal density >= rho_t (HEX8 skip rule, SignDetection.jl:36)

__global__ void k_sign_ranges(i64 nel, int nen, const int *__restrict__ IEN, const double *__restrict__ X, const double *__restrict__ rn, double rho_t,
                              GridDev g, int kz0, int kz1, const double2 *__restrict__ ezr, double zlo, double zhi, SRange *__restrict__ rng, i64 *__restrict__ ntile,
                              SignEl *__restrict__ sel) {
  i64 e = blockIdx.x * (i64)blockDim.x + threadIdx.x;
  if (e >= nel) return;
  { const double2 z = ezr[e];      // z-slab: elements that cannot reach this rank's planes get an empty range without touching their nodes
    if (z.y < zlo || z.x > zhi) { SRange r; r.a[0] = 1; r.b[0] = 0; r.a[1] = r.a[2] = 1; r.b[1] = r.b[2] = 0; r.hot = 0; r.pad = 0; rng[e] = r; ntile[e] = 0; return; } }
  SignElem E; sign_element(e, nen, IEN, X, rn, rho_t, g, E);
  SRange r; bool ok = true;
  r.pad = E.dcls; r.hot = E.hot;
  for (int d = 0; d < 3; d++) {
    const double *pc = g.pc + g.pc_off[d]; int n1 = g.np[d], a, b;
    if (nen == 8) {
      // the grid points in the closed AABB: first point >= lo, last point <= hi (pc is monotone)
      int l = 0, h = n1;
      while (l < h) { int m = (l + h) >> 1; if (pc[m] < E.lo[d]) l = m + 1; else h = m; }
      a = l; l = 0; h = n1;
      while (l < h) { int m = (l + h) >> 1; if (pc[m] <= E.hi[d]) l = m + 1; else h = m; }
      b = l - 1;
    } else {
      // create_grid_tetrahedra_mapping_TET4 (:195-196): cells max(1, floor((lo-min)/cell)-1) .. min(dims, ceil((hi-min)/cell)+1)
      int mi = (int)E.fl[d] - 1; if (mi < 1) mi = 1;
      int ma = (int)E.cu[d] + 1; if (ma > n1) ma = n1;
      a = n1; b = -1;
      int p0 = max(0, mi - 4), p1 = min(n1 - 1, ma + 3);
      for (int p = p0; p <= p1; p++) { int idx = pt_bin(pc[p], g.amin[d], g.cell, n1); if (idx >= mi && idx <= ma) { if (p < a) a = p; if (p > b) b = p; } }
    }
    if (d == 2) { if (a < kz0) a = kz0; if (b > kz1 - 1) b = kz1 - 1; }
    r.a[d] = a; r.b[d] = b; ok = ok && (a <= b);
  }
  if (!ok) { r.a[0] = 1; r.b[0] = 0; }
  rng[e] = r;
  if (nen == 8 && ok) sel[e] = sign_affine(e, IEN, X);      // only elements with candidate points in this slab
  ntile[e] = ok ? tile_span(r.a, r.b) : 0;
}
__global__ void k_sign_emit(i64 nel, const SRange *__restrict__ rng, const i64 *__restrict__ toff, GridDev g, u64 *__restrict__ keys, int *__restrict__ tile_cnt) {
  i64 e = blockIdx.x * (i64)blockDim.x + threadIdx.x;
  if (e >= nel) return;
  SRange r = rng[e];
  if (r.a[0] > r.b[0]) return;
  emit_tile_keys(g, r.a, r.b, e, keys + toff[e], tile_cnt);
}

// One CTA per tile, one thread per grid point.  Each WARP walks the tile's element list 32 entries at a time, keeps the
// entries whose candidate range overlaps the warp's 8x4x1 point footprint (ballot compaction into shared memory, order
// preserved), then every lane advances through that culled list on its own: all lanes run the expensive inverse map at
// the same time, each on its own next candidate, instead of serialising over elements.
#define CULL_CAP 96
// CLS: candidates whose element is of density class 1 / 2 (sign_element) skip the gather of the eight
// nodal densities and the shape functions -- the outcome of "rho >= rho_t" is known; the state updates (max_local, break) are the same.
template <int NEN, bool CLS>
__global__ void __launch_bounds__(TILE_VOX, 2) k_sign(GridDev g, int kz0, int kz1, const int *__restrict__ tile_ptr, const u64 *__restrict__ keys,
                                                   const SRange *__restrict__ rng, const SignEl *__restrict__ sel, const int *__restrict__ IEN, const double *__restrict__ X,
                                                   const double *__restrict__ rn, double rho_t, const double *__restrict__ dist,
                                                   double *__restrict__ signs, double *__restrict__ sdf) {
  __shared__ int s_el[TILE_VOX / 32][CULL_CAP];
  __shared__ SRange s_rg[TILE_VOX / 32][CULL_CAP];
  const int t = blockIdx.x, lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int tx = t % g.nt[0], ty = (t / g.nt[0]) % g.nt[1], tz = t / (g.nt[0] * g.nt[1]);
  const int li = threadIdx.x % TILE_X, lj = (threadIdx.x / TILE_X) % TILE_Y, lk = threadIdx.x / (TILE_X * TILE_Y);
  const int pi[3] = {tx * TILE_X + li, ty * TILE_Y + lj, tz * TILE_Z + lk};
  const bool valid = pi[0] < g.np[0] && pi[1] < g.np[1] && pi[2] < g.np[2] && pi[2] >= kz0 && pi[2] < kz1;
  // footprint of this warp (TILE_X = 8 points in x, 4 rows in y, one plane in z)
  const int wx0 = tx * TILE_X, wx1 = wx0 + TILE_X - 1, wy0 = ty * TILE_Y + (warp % (TILE_Y / 4)) * 4, wy1 = wy0 + 3, wz = tz * TILE_Z + warp / (TILE_Y / 4);
  double x[3] = {0, 0, 0};
  if (valid) { x[0] = g.pc[g.pc_off[0] + pi[0]]; x[1] = g.pc[g.pc_off[1] + pi[1]]; x[2] = g.pc[g.pc_off[2] + pi[2]]; }
  double sign = -1.0, max_local = 10.0; bool done = false;
  const int p0 = tile_ptr[t], p1 = tile_ptr[t + 1];
  // Skip rule (SignDetection.jl:36): a point none of whose candidates has a nodal density >= rho_t keeps sign -1 (TET4 elements
  // are all marked hot).  The tile's list is culled to the warp's footprint into shared memory; when it fits one round (the
  // normal case) the hot test comes from that same round, otherwise a separate pass over the list computes it first.
  bool hotany = false, hot_known = false, first = true;
  int p = p0;
  while (p < p1) {
    int n = 0; bool warp_hot = false;
    while (p < p1 && n <= CULL_CAP - 32) {
      int idx = p + lane; bool ov = false; int e = 0; SRange r; r.hot = 0;
      if (idx < p1) {
        e = (int)(keys[idx] & 0xffffffffull); r = rng[e];
        ov = r.a[0] <= wx1 && r.b[0] >= wx0 && r.a[1] <= wy1 && r.b[1] >= wy0 && r.a[2] <= wz && r.b[2] >= wz;
      }
      unsigned m = __ballot_sync(0xffffffffu, ov);
      warp_hot = warp_hot || __any_sync(0xffffffffu, ov && r.hot != 0);
      if (ov) { int slot = n + __popc(m & ((1u << lane) - 1)); s_el[warp][slot] = e; s_rg[warp][slot] = r; }
      n += __popc(m); p += 32;
    }
    __syncwarp();
    if (first && p >= p1 && !warp_hot) break;      // void region: no element near this warp reaches rho_t -> every lane keeps -1
    if (first && p < p1) {      // long list: the hot test needs all of it before the first candidate is processed
      for (int pp = p0; pp < p1; pp += 32) {
        int idx = pp + lane; bool ov = false; SRange r;
        if (idx < p1) {
          r = rng[(int)(keys[idx] & 0xffffffffull)];
          ov = r.hot && r.a[0] <= wx1 && r.b[0] >= wx0 && r.a[1] <= wy1 && r.b[1] >= wy0 && r.a[2] <= wz && r.b[2] >= wz;
        }
        unsigned m = __ballot_sync(0xffffffffu, ov);
        while (m) {
          int src = __ffs(m) - 1; m &= m - 1;
          int a0 = __shfl_sync(0xffffffffu, r.a[0], src), b0 = __shfl_sync(0xffffffffu, r.b[0], src), a1 = __shfl_sync(0xffffffffu, r.a[1], src),
              b1 = __shfl_sync(0xffffffffu, r.b[1], src), a2 = __shfl_sync(0xffffffffu, r.a[2], src), b2 = __shfl_sync(0xffffffffu, r.b[2], src);
          if (pi[0] >= a0 && pi[0] <= b0 && pi[1] >= a1 && pi[1] <= b1 && pi[2] >= a2 && pi[2] <= b2) hotany = true;
        }
      }
      hot_known = true;
    }
    // which entries of the culled list are candidates of THIS lane: one uniform sweep (broadcast reads, no bank conflicts)
    unsigned mk0 = 0, mk1 = 0, mk2 = 0; bool hotloc = false;
    for (int q = 0; q < n; q++) {
      const SRange &r = s_rg[warp][q];
      if (valid && pi[0] >= r.a[0] && pi[0] <= r.b[0] && pi[1] >= r.a[1] && pi[1] <= r.b[1] && pi[2] >= r.a[2] && pi[2] <= r.b[2]) {
        if (q < 32) mk0 |= 1u << q; else if (q < 64) mk1 |= 1u << (q - 32); else mk2 |= 1u << (q - 64);
        hotloc = hotloc || r.hot != 0;
      }
    }
    if (!hot_known) { hotany = hotloc; hot_known = true; }
    first = false;
    const bool live = valid && hotany;
    if (!__any_sync(0xffffffffu, live)) break;
    int w = 0; unsigned cur = mk0;
    while (true) {
      // this lane's next candidate (ascending list position = ascending element index)
      int pos = -1;
      if (live && !done) {
        while (w < 3 && cur == 0) { w++; cur = (w == 1) ? mk1 : (w == 2 ? mk2 : 0u); }
        if (w < 3) { int bq = __ffs(cur) - 1; cur &= cur - 1; pos = w * 32 + bq; }
      }
      bool act = pos >= 0;
      if (!__any_sync(0xffffffffu, act)) break;
      if (act) {
        const int e = s_el[warp][pos];
        if (NEN == 8) { if (sign_hex8_candidate(sel[e], e, IEN, X, rn, rho_t, x, CLS ? s_rg[warp][pos].pad : 0, sign, max_local)) done = true; }
        else if (sign_tet4_candidate(e, IEN, X, rn, rho_t, x, sign)) done = true;
      }
    }
    __syncwarp();
  }
  if (valid) {
    i64 v = ((i64)pi[2] * g.np[1] + pi[1]) * g.np[0] + pi[0];
    if (signs) signs[v] = sign;
    if (sdf) sdf[v] = dist[v] * sign;
  }
}


// ------------------------------------------------------------------------------------------------ lattice fast path
// Tensor-product lattice meshes (r2s_mesh_build_lattice): the elements whose closed AABB contains a grid point are the <= 2 x 2 x 2
// lattice cells around it, read from per-axis tables -- no keys, no sort, no list walk.  The reference's rule is replayed on those
// candidates in ascending element index with the arithmetic of the general path: for a box element the affine inverse map of
// ex::affine_inverse_apply reduces per axis to xi_d = -((cof_d * (ctr_d - x_d)) / det) with ctr_d = fl(lo + hi) / 2, half_d = fl(hi - lo) / 2
// (what ex::mono8 yields for a box, exactly), cof_0 = fl(h1 h2), cof_1 = fl(h0 h2), cof_2 = fl(h0 h1), det = fl(h0 cof_0); the terms
// the general formula adds are exact zeros.  Bit-identical signs (tests: lattice path vs. k_sign<8> vs. oracle).
// info[cell] = element id | density class << 29 | hot << 31, 0xffffffff = no element (hole, or irrelevant for this z-slab)
__global__ void k_lat_info(i64 nel, const int *__restrict__ IEN, const double *__restrict__ rn, double rho_t, const int *__restrict__ cell_of,
                           const double2 *__restrict__ ezr, double zlo, double zhi, unsigned *__restrict__ info) {
  i64 e = blockIdx.x * (i64)blockDim.x + threadIdx.x;
  if (e >= nel) return;
  const double2 z = ezr[e];
  if (z.y < zlo || z.x > zhi) return;
  double rmax = -1e300, rmin = 1e300;
#pragma unroll
  for (int a = 0; a < 8; a++) { const double r = rn[IEN[8 * e + a]]; rmax = fmax(rmax, r); rmin = fmin(rmin, r); }
  unsigned cls = 0;      // same density classes as sign_element
  const double range = rmax - rmin, tolc = 1e-9 * fmax(1.0, fabs(rho_t));
  if (rmin - 0.05 * range >= rho_t + tolc) cls = 1; else if (rmax + 0.05 * range < rho_t - tolc) cls = 2;
  const unsigned hot = !(rmax < rho_t) ? 1u : 0u;
  info[cell_of[e]] = (unsigned)e | (cls << 29) | (hot << 31);
}
// per grid axis point: first candidate cell and how many (0, 1 or 2): cells a with xs[a] <= x <= xs[a+1] (closed AABB, sdfOnDensityField.jl:60-69)
__global__ void k_lat_pt(GridDev g, const double *__restrict__ xs, int o0, int o1, int o2, int n0, int n1, int n2, int *__restrict__ pt) {
  const int t = blockIdx.x * blockDim.x + threadIdx.x;
  const int off[3] = {o0, o1, o2}, nd[3] = {n0, n1, n2};
  int d = 0, i = t;
  if (i >= g.np[0]) { i -= g.np[0]; d = 1; if (i >= g.np[1]) { i -= g.np[1]; d = 2; if (i >= g.np[2]) return; } }
  const double x = g.pc[g.pc_off[d] + i]; const double *tab = xs + off[d]; const int n = nd[d];
  int l = 0, h = n;
  while (l < h) { int m = (l + h) >> 1; if (tab[m] < x) l = m + 1; else h = m; }
  int a0, cnt;
  if (l < n && tab[l] == x) { a0 = l >= 1 ? l - 1 : 0; cnt = (l >= 1 ? 1 : 0) + (l <= n - 2 ? 1 : 0); }
  else { a0 = l - 1; cnt = (l >= 1 && l <= n - 1) ? 1 : 0; }
  pt[g.pc_off[d] + i] = (a0 << 2) | cnt;
}
// Two kernels.  k_sign_lattice looks at the density classes of the candidates only -- enough for nine points out of ten -- and lists
// the others (packed i | j << 21 | k << 42; per-warp staging, r2s_common.cuh); k_sign_lattice_hard replays the reference's rule for the
// listed points, one lane each, so its FP64 work runs in full warps instead of the few lanes per warp that sit next to the surface.
__global__ void __launch_bounds__(256) k_sign_lattice(GridDev g, int kz0, int kz1, const int *__restrict__ pt, int m0, int m1, const unsigned *__restrict__ info,
                                                      const double *__restrict__ dist, double *__restrict__ signs, double *__restrict__ sdf,
                                                      u64 *__restrict__ hard, u64 *__restrict__ nhard, i64 cap) {
  __shared__ u64 s_hard[8][WS_CAP];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5; int nh = 0;
  const i64 pl = (i64)g.np[0] * g.np[1];
  const int nrow = g.np[1] * (kz1 - kz0);
  // a warp owns grid ROWS (j, k): the candidate cells' row offsets are the same for the whole row, only the x cell differs per lane
  for (int row = blockIdx.x * 8 + warp; row < nrow; row += gridDim.x * 8) {
    const int j = row % g.np[1], k = kz0 + row / g.np[1];
    const int p1 = pt[g.pc_off[1] + j], p2 = pt[g.pc_off[2] + k];
    const int c1 = p1 >> 2, c2 = p2 >> 2, n1 = p1 & 3, n2 = p2 & 3;
    const i64 vrow = (i64)k * pl + (i64)j * g.np[0];
    const unsigned *__restrict__ rb[4];      // (jj, kk) candidate rows; a missing one repeats the first (its loads are predicated off)
#pragma unroll
    for (int q = 0; q < 4; q++) rb[q] = info + ((i64)(c2 + (q >> 1)) * m1 + (c1 + (q & 1))) * m0;
    for (int i0 = 0; i0 < g.np[0]; i0 += 32) {
      const int i = i0 + lane;
      const bool in = i < g.np[0];
      bool later = false; double sign = -1.0;
      if (in) {
        const int p0 = pt[g.pc_off[0] + i];
        const int c0 = p0 >> 2, n0 = p0 & 3;
        if (n0 * n1 * n2 != 0) {
          bool hotany = false; int nc = 0, nsolid = 0, nvoid = 0;
#pragma unroll
          for (int q = 0; q < 4; q++) {
            if ((q & 1) < n1 && (q >> 1) < n2) {      // warp-uniform
#pragma unroll
              for (int ii = 0; ii < 2; ii++) {
                if (ii < n0) {
                  const unsigned w = rb[q][c0 + ii];
                  if (w != 0xffffffffu) { hotany = hotany || (w >> 31); nc++; const unsigned cls = (w >> 29) & 3u; nsolid += cls == 1; nvoid += cls == 2; }
                }
              }
            }
          }
          // Every candidate holds the point in its closed AABB, so max|xi| <= 1 + O(eps) < 1.01 for each of them.  If ALL candidates are of
          // density class 2 (rho < rho_t wherever max|xi| < 1.01) no candidate can set the sign; if ALL are of class 1 (rho >= rho_t there)
          // the first candidate -- accepted whatever its max|xi|, because max_local starts at 10 -- sets it.  Only points next to an element
          // that may cross rho_t replay the rule (about 7 % of the elements of a SIMP field); skip rule (SignDetection.jl:36): and only if
          // some candidate has a nodal density >= rho_t.
          if (nc > 0 && nvoid == nc) sign = -1.0;
          else if (nc > 0 && nsolid == nc) sign = 1.0;
          else if (nc > 0 && hotany) later = true;
        }
        if (!later) {
          if (signs) signs[vrow + i] = sign;
          if (sdf) sdf[vrow + i] = dist[vrow + i] * sign;
        }
      }
      ws_push<u64>(s_hard[warp], nh, later, (u64)i | ((u64)j << 21) | ((u64)k << 42), hard, nhard, cap, lane);
    }
  }
  ws_flush<u64>(s_hard[warp], nh, hard, nhard, cap, lane);
}
#define CSWAP(a, b) do { const unsigned _lo = min(key[a], key[b]), _hi = max(key[a], key[b]); key[a] = _lo; key[b] = _hi; } while (0)
__global__ void __launch_bounds__(128) k_sign_lattice_hard(GridDev g, const u64 *__restrict__ hard, const u64 *__restrict__ nhard, const int *__restrict__ pt,
                                                           const double *__restrict__ xs, int o0, int o1, int o2, int m0, int m1, const unsigned *__restrict__ info,
                                                           const int *__restrict__ IEN, const double *__restrict__ rn, double rho_t, const double *__restrict__ dist,
                                                           double *__restrict__ signs, double *__restrict__ sdf) {
  const i64 pl = (i64)g.np[0] * g.np[1], n = (i64)*nhard;
  for (i64 h = blockIdx.x * (i64)blockDim.x + threadIdx.x; h < n; h += (i64)gridDim.x * blockDim.x) {
    const u64 w64 = hard[h];
    const int i = (int)(w64 & 0x1fffffu), j = (int)((w64 >> 21) & 0x1fffffu), k = (int)(w64 >> 42);
    const int p0 = pt[g.pc_off[0] + i], p1 = pt[g.pc_off[1] + j], p2 = pt[g.pc_off[2] + k];
    const int c0 = p0 >> 2, c1 = p1 >> 2, c2 = p2 >> 2, n0 = p0 & 3, n1 = p1 & 3, n2 = p2 & 3;
    double sign = -1.0;
    unsigned key[8]; int nc = 0;
#pragma unroll
    for (int q = 0; q < 8; q++) {
      const int ii = q & 1, jj = (q >> 1) & 1, kk = q >> 2;
      key[q] = 0xffffffffu;
      if (ii < n0 && jj < n1 && kk < n2) {
        const unsigned w = info[((i64)(c2 + kk) * m1 + (c1 + jj)) * m0 + (c0 + ii)];
        if (w != 0xffffffffu) { key[q] = ((w & 0x0fffffffu) << 3) | (unsigned)q; nc++; }
      }
    }
    // ascending element index = the reference's candidate order (missing candidates sort to the end)
    CSWAP(0, 1); CSWAP(2, 3); CSWAP(4, 5); CSWAP(6, 7); CSWAP(0, 2); CSWAP(1, 3); CSWAP(4, 6); CSWAP(5, 7); CSWAP(1, 2); CSWAP(5, 6);
    CSWAP(0, 4); CSWAP(1, 5); CSWAP(2, 6); CSWAP(3, 7); CSWAP(2, 4); CSWAP(3, 5); CSWAP(1, 2); CSWAP(3, 4); CSWAP(5, 6);
    const double x[3] = {g.pc[g.pc_off[0] + i], g.pc[g.pc_off[1] + j], g.pc[g.pc_off[2] + k]};
    double max_local = 10.0;
#pragma unroll 1
    for (int q = 0; q < nc; q++) {
      unsigned kq = key[0];
#pragma unroll
      for (int b = 1; b < 8; b++) if (q == b) kq = key[b];      // register select instead of a local-memory array
      const int e = (int)(kq >> 3), loc = (int)(kq & 7u);
      const int a[3] = {c0 + (loc & 1), c1 + ((loc >> 1) & 1), c2 + (loc >> 2)};
      const double l0 = xs[o0 + a[0]], h0 = xs[o0 + a[0] + 1], l1 = xs[o1 + a[1]], h1 = xs[o1 + a[1] + 1], l2 = xs[o2 + a[2]], h2 = xs[o2 + a[2] + 1];
      const double hx = ex::mul(0.5, ex::sub(h0, l0)), hy = ex::mul(0.5, ex::sub(h1, l1)), hz = ex::mul(0.5, ex::sub(h2, l2));
      const double cof0 = ex::mul(hy, hz), cof1 = ex::mul(hx, hz), cof2 = ex::mul(hx, hy), det = ex::mul(hx, cof0);
      double xi[3];
      if (!(fabs(det) > 0.0)) xi[0] = xi[1] = xi[2] = 10.0;
      else {
        const double d0 = ex::dvd(ex::mul(cof0, ex::sub(ex::mul(0.5, ex::add(l0, h0)), x[0])), det);
        const double d1 = ex::dvd(ex::mul(cof1, ex::sub(ex::mul(0.5, ex::add(l1, h1)), x[1])), det);
        const double d2 = ex::dvd(ex::mul(cof2, ex::sub(ex::mul(0.5, ex::add(l2, h2)), x[2])), det);
        xi[0] = ex::sub(0.0, d0); xi[1] = ex::sub(0.0, d1); xi[2] = ex::sub(0.0, d2);
        if (!(ex::max3abs(d0, d1, d2) < 1.0e3) || !(ex::max3abs(xi[0], xi[1], xi[2]) < 1.0e3)) xi[0] = xi[1] = xi[2] = 10.0;
      }
      const double mn = ex::max3abs(xi[0], xi[1], xi[2]);
      if (mn < 1.01 && max_local > mn) {                         // SignDetection.jl:48
        const unsigned cls = (info[((i64)a[2] * m1 + a[1]) * m0 + a[0]] >> 29) & 3u;
        if (cls == 1) sign = 1.0;
        else if (cls == 0) {
          double N[8], re[8];
#pragma unroll
          for (int b = 0; b < 8; b++) re[b] = rn[IEN[8 * (i64)e + b]];
          ex::hex8_shape(xi, N);
          if (ex::dot8(N, re) >= rho_t) sign = 1.0;
        }
        if (mn < 0.95) break;                                    // :51-59
        max_local = mn;
      }
    }
    const i64 v = (i64)k * pl + (i64)j * g.np[0] + i;
    if (signs) signs[v] = sign;
    if (sdf) sdf[v] = dist[v] * sign;
  }
}
#undef CSWAP

int r2s_dev_sign(r2s_ctx *ctx, double rho_t, bool write_signs, bool write_sdf) {
  if (!ctx->has_grid) FAIL("r2s_set_grid has not been called");
  if (ctx->nel == 0) FAIL("r2s_set_mesh has not been called");
  const GridDev &g = ctx->g; cudaStream_t st = ctx->stream; i64 nel = ctx->nel; int nen = ctx->nen;
  int kz0 = (int)ctx->k0, kz1 = (int)ctx->k1;
  if (ctx->lattice && ctx->knobs.sign_lattice && nen == 8) {
    double *signs = nullptr, *sdf = nullptr;
    if (write_signs) { CK(ctx->signs.reserve(sizeof(double) * (size_t)g.ngp)); signs = ctx->signs.as<double>(); }
    if (write_sdf) { CK(ctx->sdf.reserve(sizeof(double) * (size_t)g.ngp)); sdf = ctx->sdf.as<double>(); ctx->have_sdf = true; }
    const int npt = g.np[0] + g.np[1] + g.np[2];
    CK(ctx->lat_info.reserve(sizeof(unsigned) * (size_t)ctx->lat_ncell));
    CK(ctx->lat_pt.reserve(sizeof(int) * (size_t)npt));
    CK(cudaMemsetAsync(ctx->lat_info.p, 0xff, sizeof(unsigned) * (size_t)ctx->lat_ncell, st));
    double zlo = -1e300, zhi = 1e300;
    if (kz0 > 0 || kz1 < g.np[2]) { const double m = 3.0 * g.cell; zlo = ctx->h_pc[2][(size_t)kz0] - m; zhi = ctx->h_pc[2][(size_t)kz1 - 1] + m; }
    const int *lo = ctx->lat_off, *nd = ctx->lat_nd;
    k_lat_info<<<cdiv(nel, 256), 256, 0, st>>>(nel, ctx->IEN32.as<int>(), ctx->rho_n.as<double>(), rho_t, ctx->lat_cell.as<int>(), ctx->ezr.as<double2>(), zlo, zhi, ctx->lat_info.as<unsigned>()); LAUNCH_CHECK();
    k_lat_pt<<<cdiv(npt, 256), 256, 0, st>>>(g, ctx->lat_xs.as<double>(), lo[0], lo[1], lo[2], nd[0], nd[1], nd[2], ctx->lat_pt.as<int>()); LAUNCH_CHECK();
    // hard-point list: the pair list of the projection is free by now and large enough in all but degenerate cases
    const i64 cap = (i64)g.np[0] * g.np[1] * (kz1 - kz0);
    CK(ctx->plist.reserve(sizeof(u64) * (size_t)(cap + 16)));
    CK(ctx->counters.reserve(sizeof(u64) * 16));
    u64 *nhard = ctx->counters.as<u64>();
    CK(cudaMemsetAsync(nhard, 0, sizeof(u64), st));
    k_sign_lattice<<<148 * 8, 256, 0, st>>>(g, kz0, kz1, ctx->lat_pt.as<int>(), nd[0] - 1, nd[1] - 1, ctx->lat_info.as<unsigned>(), ctx->dist.as<double>(), signs, sdf,
                                            ctx->plist.as<u64>(), nhard, cap); LAUNCH_CHECK();
    k_sign_lattice_hard<<<148 * 16, 128, 0, st>>>(g, ctx->plist.as<u64>(), nhard, ctx->lat_pt.as<int>(), ctx->lat_xs.as<double>(), lo[0], lo[1], lo[2], nd[0] - 1, nd[1] - 1,
                                                  ctx->lat_info.as<unsigned>(), ctx->IEN32.as<int>(), ctx->rho_n.as<double>(), rho_t, ctx->dist.as<double>(), signs, sdf); LAUNCH_CHECK();
    return 0;
  }
  CK(ctx->s_rng.reserve(sizeof(SRange) * (size_t)nel));
  if (nen == 8) CK(ctx->s_el.reserve(sizeof(SignEl) * (size_t)nel));
  CK(ctx->cnt_a.reserve(sizeof(i64) * (size_t)(nel + 1)));
  CK(ctx->cnt_b.reserve(sizeof(i64) * (size_t)(nel + 1)));
  CK(ctx->s_tile_ptr.reserve(sizeof(int) * (size_t)(g.ntiles + 2)));
  CK(cudaMemsetAsync(ctx->s_tile_ptr.p, 0, sizeof(int) * (size_t)(g.ntiles + 2), st));
  CK(cudaMemsetAsync(ctx->cnt_a.as<i64>() + nel, 0, sizeof(i64), st));
  i64 *ntile = ctx->cnt_a.as<i64>(), *toff = ctx->cnt_b.as<i64>();
  double zlo = -1e300, zhi = 1e300;
  if (kz0 > 0 || kz1 < g.np[2]) { const double m = 3.0 * g.cell; zlo = ctx->h_pc[2][(size_t)kz0] - m; zhi = ctx->h_pc[2][(size_t)kz1 - 1] + m; }
  k_sign_ranges<<<cdiv(nel, 256), 256, 0, st>>>(nel, nen, ctx->IEN32.as<int>(), ctx->X.as<double>(), ctx->rho_n.as<double>(), rho_t, g, kz0, kz1, ctx->ezr.as<double2>(), zlo, zhi, ctx->s_rng.as<SRange>(), ntile, ctx->s_el.as<SignEl>()); LAUNCH_CHECK();
  if (r2s_scan_exclusive_i64(ctx, ntile, toff, nel + 1)) return 1;
  i64 nkeys = 0;
  if (r2s_readback(ctx, &nkeys, toff + nel, sizeof(i64))) return 1;
  if (nkeys >= (1ll << 31)) FAIL("sign binning: too many (tile, element) pairs for one slab");
  if (nkeys > 0) {
    CK(ctx->s_keys.reserve(sizeof(u64) * (size_t)nkeys));
    CK(ctx->s_keys_alt.reserve(sizeof(u64) * (size_t)nkeys));
    k_sign_emit<<<cdiv(nel, 128), 128, 0, st>>>(nel, ctx->s_rng.as<SRange>(), toff, g, ctx->s_keys.as<u64>(), ctx->s_tile_ptr.as<int>() + 1); LAUNCH_CHECK();
  }
  u64 *sorted = nullptr;
  if (r2s_tile_lists(ctx, ctx->s_keys.as<u64>(), ctx->s_keys_alt.as<u64>(), nkeys, ctx->s_tile_ptr.as<int>(), &sorted)) return 1;
  double *signs = nullptr, *sdf = nullptr;
  if (write_signs) { CK(ctx->signs.reserve(sizeof(double) * (size_t)g.ngp)); signs = ctx->signs.as<double>(); }
  if (write_sdf) { CK(ctx->sdf.reserve(sizeof(double) * (size_t)g.ngp)); sdf = ctx->sdf.as<double>(); ctx->have_sdf = true; }
  if (nen == 8)      // density-class shortcut: bit-identical to the plain rule (test_sign_density_class_shortcut), always on
    k_sign<8, true><<<(unsigned)g.ntiles, TILE_VOX, 0, st>>>(g, kz0, kz1, ctx->s_tile_ptr.as<int>(), sorted, ctx->s_rng.as<SRange>(), ctx->s_el.as<SignEl>(), ctx->IEN32.as<int>(), ctx->X.as<double>(),
                                                             ctx->rho_n.as<double>(), rho_t, ctx->dist.as<double>(), signs, sdf);
  else
    k_sign<4, false><<<(unsigned)g.ntiles, TILE_VOX, 0, st>>>(g, kz0, kz1, ctx->s_tile_ptr.as<int>(), sorted, ctx->s_rng.as<SRange>(), ctx->s_el.as<SignEl>(), ctx->IEN32.as<int>(), ctx->X.as<double>(),
                                                       ctx->rho_n.as<double>(), rho_t, ctx->dist.as<double>(), signs, sdf);
  LAUNCH_CHECK();
  return 0;
}
