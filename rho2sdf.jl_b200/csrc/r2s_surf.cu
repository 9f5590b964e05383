// r2s_surf.cu -- the zero surface of the smoothed SDF as a closed, oriented triangle mesh (marching cubes with the face rule of
// r2s_mc.cuh), and its STL / PLY writers.
//
// The reference leaves {fine_sdf = 0} to ParaView or a Makie isosurface plot (src/Visualizations).  Here it is two passes over the
// device-resident field; the mesh is a function of the field and iso alone:
//   vertices: one per grid edge whose ends lie on different sides of iso (inside iff value >= iso), ordered by (linear id of the
//             edge's lower point, axis x < y < z), coordinates mc_vertex() in the frame of r2s_export_vti (origin AABB_min,
//             spacing cell_size / smooth);
//   triangles: int32 vertex ids, ordered by linear cell id, then by table order within the cell; counter-clockwise seen from outside
//             the solid {value >= iso}.
// Pass 1 (k_surf_count): one warp per row of points (j, k) writes the row's vertex and triangle counts.  Two exclusive scans over the
// rows give every row its first vertex and first triangle.  Pass 2 (k_surf_emit): the same warps number their row's crossings with a
// warp prefix sum, and a cell finds the ids of its edges in the four point rows (j + dy, k + dz) it touches from those rows' bases
// and the same prefix sums.  No atomics, no per-point index array: scratch is four i64 per row, the output is sized from the counts.
//
// Several slabs (r2s_multi_isosurface): slab r owns point planes [z0, z1) and the cells of those planes.  Its cells also reference
// the x / y vertices of plane z1, which the next slab numbers; to number them itself the slab counts one plane beyond z1 (which needs
// plane z1 + 1: two halo planes), so its row bases run on into the next slab's first plane and agree with the next slab's numbering.
// The slab's global bases are an exclusive scan of the slab counts made on the host, so the concatenation of the slabs' arrays is
// bit-identical to one context on the whole field.
#include <math.h>
#include <stdio.h>
#include <string.h>
#include <algorithm>
#include <string>
#include <vector>
#include "r2s_common.cuh"
#include "r2s_mc.cuh"
#include "r2s_sample.cuh"
#include "r2s_snap.cuh"
#include "r2s_band.cuh"

__constant__ uint8_t c_mc[256][16];      // per case: triangle count, then 3 cube edges per triangle (mc_build_case)
__constant__ uint8_t c_mc_edge[12];      // per cube edge: start corner | axis << 4

#define SURF_WARPS 8                     // rows of points (consecutive j) per CTA
#define SURF_STEP 30                     // points owned per warp step: lane 30 supplies point i + 1 of lane 29, lane 31 its x-neighbour

struct SurfArgs {
  const float *f;                        // globally indexed field, plane stride nx * ny
  int nx, ny, nz;                        // points of the whole grid
  int z0, z1, zc;                        // owned point planes [z0, z1); counted planes [z0, zc), zc = z1 + 1 unless z1 = nz
  float iso;
  double origin[3], spacing[3];
  i64 *vcnt, *tcnt, *vbase, *tbase;      // per counted row, local row id (k - z0) * ny + j
  i64 vglob;                             // global id of this slab's first vertex
  float *V;                              // this slab's vertices (local ids)
  int *T;                                // this slab's triangles (global vertex ids)
  unsigned *bad;                         // set when an owned value is not finite
};

__device__ __forceinline__ float surf_load(const float *f, int nx, int ny, int nz, int i, int j, int k) {
  return (i < nx && j < ny && k < nz) ? __ldg(f + ((i64)k * ny + j) * nx + i) : 0.0f;
}

// counts of one row of points: crossings of every point of the row, triangles of the row's cells (owned planes only)
__global__ void __launch_bounds__(32 * SURF_WARPS) k_surf_count(SurfArgs a) {
  const int lane = threadIdx.x & 31, j = blockIdx.x * SURF_WARPS + (threadIdx.x >> 5), k = a.z0 + blockIdx.y;
  if (j >= a.ny) return;
  const bool cells_here = j + 1 < a.ny && k + 1 < a.nz && k < a.z1;
  i64 nv = 0, nt = 0;
  unsigned bad = 0;
  // the loads of step i0 + SURF_STEP are issued before step i0 is evaluated: a warp walks its row serially, so it keeps two steps in flight
  float n000 = surf_load(a.f, a.nx, a.ny, a.nz, lane, j, k), n010 = surf_load(a.f, a.nx, a.ny, a.nz, lane, j + 1, k);
  float n001 = surf_load(a.f, a.nx, a.ny, a.nz, lane, j, k + 1), n011 = surf_load(a.f, a.nx, a.ny, a.nz, lane, j + 1, k + 1);
  for (int i0 = 0; i0 < a.nx; i0 += SURF_STEP) {
    const int i = i0 + lane, ip = i + SURF_STEP;
    const float v000 = n000, v010 = n010, v001 = n001, v011 = n011;
    n000 = surf_load(a.f, a.nx, a.ny, a.nz, ip, j, k); n010 = surf_load(a.f, a.nx, a.ny, a.nz, ip, j + 1, k);
    n001 = surf_load(a.f, a.nx, a.ny, a.nz, ip, j, k + 1); n011 = surf_load(a.f, a.nx, a.ny, a.nz, ip, j + 1, k + 1);
    const unsigned b = (unsigned)(v000 >= a.iso) | (unsigned)(v010 >= a.iso) << 1 | (unsigned)(v001 >= a.iso) << 2 | (unsigned)(v011 >= a.iso) << 3;
    const unsigned bx = __shfl_down_sync(0xffffffffu, b, 1);      // the same four corners at i + 1
    const bool own = lane < SURF_STEP && i < a.nx;
    int c = 0, t = 0;
    if (own) {
      bad |= !isfinite(v000);
      c = (i + 1 < a.nx && ((b ^ bx) & 1)) + (j + 1 < a.ny && ((b ^ (b >> 1)) & 1)) + (k + 1 < a.nz && ((b ^ (b >> 2)) & 1));
      if (cells_here && i + 1 < a.nx) {
        const unsigned cs = (b & 1) | (bx & 1) << 1 | (b >> 1 & 1) << 2 | (bx >> 1 & 1) << 3 | (b >> 2 & 1) << 4 | (bx >> 2 & 1) << 5 | (b >> 3 & 1) << 6 | (bx >> 3 & 1) << 7;
        t = c_mc[cs][0];
      }
    }
    nv += __reduce_add_sync(0xffffffffu, (unsigned)c);
    nt += __reduce_add_sync(0xffffffffu, (unsigned)t);
  }
  if (__any_sync(0xffffffffu, bad) && lane == 0) atomicOr(a.bad, 1u);      // a flag, not an order: any writer gives the same result
  if (lane == 0) {
    const i64 r = (i64)(k - a.z0) * a.ny + j;
    a.vcnt[r] = nv; a.tcnt[r] = nt;
  }
}

// inclusive warp scan of four 8-bit counters packed in one word (each total stays below 256: at most 3 * SURF_STEP)
__device__ __forceinline__ unsigned warp_scan_u32(unsigned x, int lane) {
#pragma unroll
  for (int d = 1; d < 32; d <<= 1) {
    const unsigned y = __shfl_up_sync(0xffffffffu, x, d);
    if (lane >= d) x += y;
  }
  return x;
}

// REC = false: vertex coordinates by mc_vertex.  REC = true (r2s_isosurface_lattice): each vertex slot of V receives its edge instead, as
// three uint32 (i, j, (k - z0) << 2 | axis), which k_surf_snap reads and overwrites with the snapped vertex
template <bool REC>
__global__ void __launch_bounds__(32 * SURF_WARPS) k_surf_emit(SurfArgs a) {
  const int lane = threadIdx.x & 31, j = blockIdx.x * SURF_WARPS + (threadIdx.x >> 5), k = a.z0 + blockIdx.y;
  if (j >= a.ny) return;
  const i64 r0 = (i64)(k - a.z0) * a.ny + j;
  // the four point rows R = (j + dy, k + dz), R = dy | dz << 1, that the cells of this row touch: their first vertex (local id)
  i64 base[4];
#pragma unroll
  for (int R = 0; R < 4; R++) {
    const int jj = j + (R & 1), kk = k + (R >> 1);
    base[R] = (jj < a.ny && kk < a.zc) ? a.vbase[r0 + (R & 1) + (R >> 1) * (i64)a.ny] : 0;
  }
  i64 tb = a.tbase[r0];
  const bool cells_here = j + 1 < a.ny && k + 1 < a.nz;      // k < z1 here: the emitting grid covers the owned planes only
  // inside bits of the points (i, j + dy, k + dz), bit dy + 3 dz, dy, dz in 0..2 ((2, 2) is never needed); the values of step
  // i0 + SURF_STEP are loaded before step i0 is evaluated (two steps in flight per warp)
  float nv[8];
#pragma unroll
  for (int q = 0; q < 8; q++) nv[q] = surf_load(a.f, a.nx, a.ny, a.nz, lane, j + (q < 3 ? q : q < 6 ? q - 3 : q - 6), k + (q < 3 ? 0 : q < 6 ? 1 : 2));
  for (int i0 = 0; i0 < a.nx; i0 += SURF_STEP) {
    const int i = i0 + lane;
    unsigned b = 0;
#pragma unroll
    for (int q = 0; q < 8; q++) {
      const int dy = q < 3 ? q : q < 6 ? q - 3 : q - 6, dz = q < 3 ? 0 : q < 6 ? 1 : 2;
      b |= (unsigned)(nv[q] >= a.iso) << (dy + 3 * dz);
      nv[q] = surf_load(a.f, a.nx, a.ny, a.nz, i + SURF_STEP, j + dy, k + dz);
    }
    const unsigned bx = __shfl_down_sync(0xffffffffu, b, 1);
    // crossing masks (bit = axis) of point i in the four rows; lanes 0..30 have their x-neighbour's bits
    unsigned m4 = 0, cnt = 0;
    const bool own = lane < SURF_STEP && i < a.nx;
#pragma unroll
    for (int R = 0; R < 4; R++) {
      const int dy = R & 1, dz = R >> 1, s = dy + 3 * dz;
      if (i >= a.nx || j + dy >= a.ny || k + dz >= a.nz) continue;
      const unsigned me = b >> s & 1;
      unsigned m = 0;
      if (lane < 31 && i + 1 < a.nx && me != (bx >> s & 1)) m |= 1;
      if (j + dy + 1 < a.ny && me != (b >> (s + 1) & 1)) m |= 2;
      if (k + dz + 1 < a.nz && me != (b >> (s + 3) & 1)) m |= 4;
      m4 |= m << (3 * R);
      if (own) cnt |= (unsigned)__popc(m) << (8 * R);
    }
    const unsigned inc = warp_scan_u32(cnt, lane), exc = inc - cnt, tot = __shfl_sync(0xffffffffu, inc, 31);
    const unsigned m4x = __shfl_down_sync(0xffffffffu, m4, 1);      // masks of point i + 1 (lane 29 reads lane 30: complete)
    // vertices of this row
    if (REC && own && (m4 & 7)) {
      i64 id = base[0] + (exc & 255);
#pragma unroll
      for (int ax = 0; ax < 3; ax++) {
        if (!(m4 >> ax & 1)) continue;
        uint32_t *rec = (uint32_t *)(a.V + 3 * id);
        rec[0] = (uint32_t)i; rec[1] = (uint32_t)j; rec[2] = (uint32_t)(k - a.z0) << 2 | (uint32_t)ax;
        id++;
      }
    }
    if (!REC && own && (m4 & 7)) {
      i64 id = base[0] + (exc & 255);
      const i64 p = ((i64)k * a.ny + j) * a.nx + i;
      const float va = a.f[p];
#pragma unroll
      for (int ax = 0; ax < 3; ax++) {
        if (!(m4 >> ax & 1)) continue;
        const float vb = a.f[p + (ax == 0 ? 1 : ax == 1 ? (i64)a.nx : (i64)a.nx * a.ny)];
        float o[3];
        mc_vertex(a.origin, a.spacing, i, j, k, ax, va, vb, a.iso, o);
        a.V[3 * id] = o[0]; a.V[3 * id + 1] = o[1]; a.V[3 * id + 2] = o[2];
        id++;
      }
    }
    // triangles of this row's cells
    unsigned cs = 0, nt = 0;
    if (own && cells_here && i + 1 < a.nx) {
      cs = (b & 1) | (bx & 1) << 1 | (b >> 1 & 1) << 2 | (bx >> 1 & 1) << 3 | (b >> 3 & 1) << 4 | (bx >> 3 & 1) << 5 | (b >> 4 & 1) << 6 | (bx >> 4 & 1) << 7;
      nt = c_mc[cs][0];
    }
    const unsigned tinc = warp_scan_u32(nt, lane), ttot = __shfl_sync(0xffffffffu, tinc, 31);
    if (nt) {
      int *out = a.T + 3 * (tb + (tinc - nt));
      for (unsigned q = 0; q < 3 * nt; q++) {
        const int ce = c_mc_edge[c_mc[cs][1 + q]], c = ce & 15, ax = ce >> 4, dx = c & 1, R = c >> 1;
        const unsigned mm = ((dx ? m4x : m4) >> (3 * R)) & 7;
        const i64 bR = R == 0 ? base[0] : R == 1 ? base[1] : R == 2 ? base[2] : base[3];      // selects, not a local-memory array
        const i64 id = bR + ((exc >> (8 * R)) & 255) + (dx ? ((cnt >> (8 * R)) & 255) : 0) + __popc(mm & ((1u << ax) - 1));
        out[q] = (int)(a.vglob + id);
      }
    }
#pragma unroll
    for (int R = 0; R < 4; R++) base[R] += (tot >> (8 * R)) & 255;
    tb += ttot;
  }
}

// one thread per vertex of a lattice chunk: the edge record k_surf_emit<true> left in V -> the vertex on the continuous field's zero set
// (r2s_snap.cuh).  f: the chunk's lattice values (globally indexed planes, as SurfArgs::f); every evaluation reads the weights of the slab
// owning the point's floor plane (tab, nslab entries; nslab = 1: G's own weights)
struct SnapArgs {
  const float *f;
  int nx, ny, z0, nslab;
  float o[3], h[3], iso;
  i64 n;
  const SurfSlabW *tab;
  float *V;
};
__global__ void __launch_bounds__(128) k_surf_snap(SampleGrid G, SnapArgs s) {
  const i64 t = blockIdx.x * (i64)blockDim.x + threadIdx.x;
  if (t >= s.n) return;
  const uint32_t *rec = (const uint32_t *)(s.V + 3 * t);
  const int i = (int)rec[0], j = (int)rec[1], k = s.z0 + (int)(rec[2] >> 2), ax = (int)(rec[2] & 3);
  const float px = smp_add(s.o[0], smp_mul((float)i, s.h[0])), py = smp_add(s.o[1], smp_mul((float)j, s.h[1])), pz = smp_add(s.o[2], smp_mul((float)k, s.h[2]));
  const i64 p = ((i64)k * s.ny + j) * s.nx + i;
  const float va = s.f[p], vb = s.f[p + (ax == 0 ? 1 : ax == 1 ? (i64)s.nx : (i64)s.nx * s.ny)];
  const int q = ax == 0 ? i : ax == 1 ? j : k;
  const float xa = ax == 0 ? px : ax == 1 ? py : pz, xb = smp_add(s.o[ax], smp_mul((float)(q + 1), s.h[ax]));
  const float x = snap_search([&](float v) {
    const float qx = ax == 0 ? v : px, qy = ax == 1 ? v : py, qz = ax == 2 ? v : pz;
    SampleGrid g = G;
    if (s.nslab > 1) {
      const int c = smp_floor(G.C[2], G.n[2], G.c0[2], G.inv[2], qz);
      int r = 0;
      while (r + 1 < s.nslab && c >= s.tab[r].k1) r++;
      g.w = s.tab[r].w; g.px = s.tab[r].px;
    }
    return sample_point<false>(g, qx, qy, qz, nullptr);
  }, xa, xb, va, vb, s.iso, nullptr);
  s.V[3 * t] = ax == 0 ? x : px; s.V[3 * t + 1] = ax == 1 ? x : py; s.V[3 * t + 2] = ax == 2 ? x : pz;
}

// ---- r2s_isosurface_band: sample only the lattice blocks that can hold the surface (r2s_band.cuh) -------------------------------------
// Block (bx, by, bz) covers the lattice cells [b B, min(b B + B, dims - 1)) per axis and classifies the closed box of their points.  A point
// belongs to the closed boxes of at most two blocks per axis: its owner min(i / B, nb - 1), and owner - 1 when i is a multiple of B inside
// the lattice.  The chunk's points whose owner is skipped receive a fill value on the proven side (iso, or the float below iso); then every
// point that some sampled block holds is evaluated once, by the last sampled block (in (bz, by, bx) order) holding it, with the sampler's
// arithmetic.  A value marching cubes or the snap reads is therefore exact wherever it matters: every crossing edge lies in the closed box
// of its lower point's owner, which is sampled, and a fill value sits on its point's true side.
struct BandArgs {
  float o[3], h[3], iso, below;          // below: the float below iso (the fill of an outside block)
  i64 n[3], nb[3];                       // lattice points and blocks per axis
  i64 ka, kb, lz0, nblk;                 // chunk planes [ka, kb) written to out (plane ka first); block layers from lz0 on, nblk blocks
  i64 kown;                              // planes below kown are this context's: only their evaluations are counted
  int nslab;
  const SurfSlabW *tab;
  uint8_t *cls;                          // per block of the chunk's layers: 0 sampled, 1 inside, 2 outside
  i64 *list, *cnt;                       // the sampled blocks; cnt[0] = their number, cnt[1] += points evaluated
  float *out;
};

__device__ __forceinline__ int band_slab(const SampleGrid &G, const BandArgs &A, float z) {
  const int c = smp_floor(G.C[2], G.n[2], G.c0[2], G.inv[2], z);
  int r = 0;
  while (r + 1 < A.nslab && c >= A.tab[r].k1) r++;
  return r;
}

// one thread per block of the chunk's layers: classify, and list the sampled ones (in any order: the values do not depend on it)
__global__ void __launch_bounds__(128) k_band_classify(SampleGrid G, BandArgs A) {
  const i64 t = blockIdx.x * (i64)blockDim.x + threadIdx.x;
  if (t >= A.nblk) return;
  const i64 b[3] = {t % A.nb[0], (t / A.nb[0]) % A.nb[1], A.lz0 + t / (A.nb[0] * A.nb[1])};
  i64 lo[3], hi[3];
  for (int d = 0; d < 3; d++) { lo[d] = b[d] * R2S_BAND_B; hi[d] = lo[d] + R2S_BAND_B < A.n[d] - 1 ? lo[d] + R2S_BAND_B : A.n[d] - 1; }
  // a block whose points read two slabs' weights is sampled; otherwise every evaluation in it reads slab r's
  const int r = band_slab(G, A, smp_add(A.o[2], smp_mul((float)lo[2], A.h[2])));
  int c = 0;
  if (r == band_slab(G, A, smp_add(A.o[2], smp_mul((float)hi[2], A.h[2])))) {
    G.w = A.tab[r].w; G.px = A.tab[r].px;
    c = band_classify(G, A.o, A.h, lo, hi, A.iso, band_margin());
    if (c == 2 && !(A.below > -INFINITY)) c = 0;
  }
  A.cls[t] = (uint8_t)c;
  if (!c) A.list[atomicAdd((unsigned long long *)A.cnt, 1ull)] = t;
}

__device__ __forceinline__ i64 band_owner(i64 i, i64 nb) { return i / R2S_BAND_B < nb - 1 ? i / R2S_BAND_B : nb - 1; }

// one thread per point of planes [ka, kb): the fill value of a point whose owner is skipped
__global__ void __launch_bounds__(256) k_band_fill(BandArgs A) {
  const i64 t = blockIdx.x * (i64)blockDim.x + threadIdx.x, pl = A.n[0] * A.n[1];
  if (t >= (A.kb - A.ka) * pl) return;
  const i64 i = t % A.n[0], j = (t / A.n[0]) % A.n[1], k = A.ka + t / pl;
  const uint8_t c = A.cls[band_owner(i, A.nb[0]) + A.nb[0] * (band_owner(j, A.nb[1]) + A.nb[1] * (band_owner(k, A.nb[2]) - A.lz0))];
  if (c) A.out[t] = c == 1 ? A.iso : A.below;
}

// one CTA per sampled block: its closed box's points within planes [ka, kb) that it is the last sampled holder of
__global__ void __launch_bounds__(256) k_band_sample(SampleGrid G, BandArgs A) {
  constexpr int P = R2S_BAND_B + 1;
  const i64 me = A.list[blockIdx.x];
  const i64 b[3] = {me % A.nb[0], (me / A.nb[0]) % A.nb[1], A.lz0 + me / (A.nb[0] * A.nb[1])};
  unsigned long long n = 0;
  for (int q = threadIdx.x; q < P * P * P; q += blockDim.x) {
    const i64 p[3] = {b[0] * R2S_BAND_B + q % P, b[1] * R2S_BAND_B + (q / P) % P, b[2] * R2S_BAND_B + q / (P * P)};
    if (p[0] >= A.n[0] || p[1] >= A.n[1] || p[2] < A.ka || p[2] >= A.kb) continue;
    // the blocks holding p, owner first per axis; the first sampled one in descending (z, y, x) order evaluates p
    i64 c[3][2];
    int nc[3];
    for (int d = 0; d < 3; d++) {
      c[d][0] = band_owner(p[d], A.nb[d]); nc[d] = 1;
      if (p[d] % R2S_BAND_B == 0 && p[d] / R2S_BAND_B >= 1 && p[d] / R2S_BAND_B <= A.nb[d] - 1) c[d][nc[d]++] = p[d] / R2S_BAND_B - 1;
    }
    i64 first = -1;
    for (int z = 0; z < nc[2] && first < 0; z++)
      for (int y = 0; y < nc[1] && first < 0; y++)
        for (int x = 0; x < nc[0] && first < 0; x++) {
          const i64 id = c[0][x] + A.nb[0] * (c[1][y] + A.nb[1] * (c[2][z] - A.lz0));
          if (!A.cls[id]) first = id;
        }
    if (first != me) continue;
    const float x = smp_add(A.o[0], smp_mul((float)p[0], A.h[0])), y = smp_add(A.o[1], smp_mul((float)p[1], A.h[1]));
    const float z = smp_add(A.o[2], smp_mul((float)p[2], A.h[2]));
    SampleGrid g = G;
    if (A.nslab > 1) { const int r = band_slab(G, A, z); g.w = A.tab[r].w; g.px = A.tab[r].px; }
    A.out[((p[2] - A.ka) * A.n[1] + p[1]) * A.n[0] + p[0]] = sample_point<false>(g, x, y, z, nullptr);
    n += p[2] < A.kown;
  }
  n = __reduce_add_sync(0xffffffffu, (unsigned)n);
  if ((threadIdx.x & 31) == 0 && n) atomicAdd((unsigned long long *)A.cnt + 1, n);
}

__global__ void k_surf_totals(const i64 *vcnt, const i64 *tcnt, const i64 *vbase, const i64 *tbase, i64 nrows, i64 nown, const unsigned *bad, i64 *out) {
  out[0] = nown < nrows ? vbase[nown] : vbase[nrows - 1] + vcnt[nrows - 1];      // vertices of the owned rows
  out[1] = tbase[nrows - 1] + tcnt[nrows - 1];
  out[2] = *bad;
}

// ---- host side ----------------------------------------------------------------------------------------------------------------------
struct McTable {
  uint8_t t[256][16], e[12];
  McTable() {
    for (int q = 0; q < 12; q++) e[q] = (uint8_t)(mc_edge_corner(q) | mc_edge_axis(q) << 4);
    for (int c = 0; c < 256; c++) {
      const McCase m = mc_build_case(c);
      t[c][0] = m.n;
      memcpy(&t[c][1], m.e, 15);
    }
  }
};
static int upload_table(r2s_ctx *ctx) {
  static const McTable tab;      // built once, on first use (thread-safe initialisation)
  CK(cudaMemcpyToSymbolAsync(c_mc, tab.t, sizeof(tab.t), 0, cudaMemcpyHostToDevice, ctx->stream));
  CK(cudaMemcpyToSymbolAsync(c_mc_edge, tab.e, sizeof(tab.e), 0, cudaMemcpyHostToDevice, ctx->stream));
  return 0;
}

static SurfArgs surf_args(r2s_ctx *ctx, const float *f, i64 nx, i64 ny, i64 nz, i64 z0, i64 z1, const double origin[3], const double spacing[3], float iso) {
  SurfArgs a;
  a.f = f; a.nx = (int)nx; a.ny = (int)ny; a.nz = (int)nz; a.z0 = (int)z0; a.z1 = (int)z1; a.zc = (int)std::min(z1 + 1, nz); a.iso = iso;
  for (int d = 0; d < 3; d++) { a.origin[d] = origin[d]; a.spacing[d] = spacing[d]; }
  const i64 nrows = (i64)(a.zc - a.z0) * ny;
  a.vcnt = ctx->surf_rows.as<i64>(); a.tcnt = a.vcnt + nrows; a.vbase = a.tcnt + nrows; a.tbase = a.vbase + nrows;
  a.vglob = 0; a.V = nullptr; a.T = nullptr; a.bad = (unsigned *)(a.tbase + nrows + 3);
  return a;
}

// pass 1 + scans on the owned planes [z0, z1) of an nx x ny x nz field: per-row counts and bases in ctx->surf_rows, the owned totals
static int count_rows(r2s_ctx *ctx, const float *f, i64 nx, i64 ny, i64 nz, i64 z0, i64 z1, float iso, i64 *nv, i64 *nt) {
  const i64 zc = std::min(z1 + 1, nz), nrows = (zc - z0) * ny;
  CK(ctx->surf_rows.reserve(sizeof(i64) * (size_t)(4 * nrows + 4)));
  const double zero[3] = {0, 0, 0};
  SurfArgs a = surf_args(ctx, f, nx, ny, nz, z0, z1, zero, zero, iso);
  CK(cudaMemsetAsync(a.bad, 0, sizeof(unsigned), ctx->stream));
  k_surf_count<<<dim3(cdiv(ny, SURF_WARPS), (unsigned)(zc - z0)), 32 * SURF_WARPS, 0, ctx->stream>>>(a);
  LAUNCH_CHECK();
  if (r2s_scan_exclusive_i64(ctx, a.vcnt, a.vbase, nrows)) return 1;
  if (r2s_scan_exclusive_i64(ctx, a.tcnt, a.tbase, nrows)) return 1;
  i64 *tot = a.tbase + nrows;
  k_surf_totals<<<1, 1, 0, ctx->stream>>>(a.vcnt, a.tcnt, a.vbase, a.tbase, nrows, (z1 - z0) * ny, a.bad, tot);
  LAUNCH_CHECK();
  i64 h[3];
  if (r2s_readback(ctx, h, tot, sizeof(h))) return 1;
  if (h[2]) FAIL("isosurface: the field holds a non-finite value");
  *nv = h[0]; *nt = h[1];
  return 0;
}

// pass 1 + scans: this context's vertex / triangle counts (owned planes [z0, z1) of an nx x ny x nz field)
int r2s_surf_count(r2s_ctx *ctx, const float *f, i64 nx, i64 ny, i64 nz, i64 z0, i64 z1, const double origin[3], const double spacing[3], float iso,
                   i64 *nv, i64 *nt) {
  ctx->have_surface = false;
  if (!isfinite(iso)) FAIL("isosurface: iso must be finite");
  if (nx < 2 || ny < 2 || nz < 2) FAIL("isosurface: the field needs at least 2 points per axis");
  if ((nx - 1) * (ny - 1) * (nz - 1) >= (1ll << 31)) FAIL("isosurface: 2^31 or more cells");
  for (int d = 0; d < 3; d++) if (!isfinite(origin[d]) || !isfinite(spacing[d])) FAIL("isosurface: origin and spacing must be finite");
  CK(cudaSetDevice(ctx->device));
  if (upload_table(ctx)) return 1;
  i64 h[2];
  if (count_rows(ctx, f, nx, ny, nz, z0, z1, iso, &h[0], &h[1])) return 1;
  ctx->surf_f = f; ctx->surf_nx = nx; ctx->surf_ny = ny; ctx->surf_nz = nz; ctx->surf_z0 = z0; ctx->surf_z1 = z1; ctx->surf_iso = iso;
  for (int d = 0; d < 3; d++) { ctx->surf_origin[d] = origin[d]; ctx->surf_spacing[d] = spacing[d]; }
  ctx->surf_nv = h[0]; ctx->surf_nt = h[1];
  *nv = h[0]; *nt = h[1];
  return 0;
}

// pass 2: emit with this context's first global vertex id (the field and frame of the last r2s_surf_count)
int r2s_surf_emit(r2s_ctx *ctx, i64 vglob, i64 nv_total) {
  CK(cudaSetDevice(ctx->device));
  if (nv_total >= (1ll << 31)) FAIL("isosurface: 2^31 or more vertices (vertex ids are int32)");
  const i64 nv = ctx->surf_nv, nt = ctx->surf_nt;
  CK(ctx->surf_V.reserve(sizeof(float) * 3 * (size_t)std::max<i64>(nv, 1)));
  CK(ctx->surf_T.reserve(sizeof(int) * 3 * (size_t)std::max<i64>(nt, 1)));
  SurfArgs a = surf_args(ctx, ctx->surf_f, ctx->surf_nx, ctx->surf_ny, ctx->surf_nz, ctx->surf_z0, ctx->surf_z1, ctx->surf_origin, ctx->surf_spacing, ctx->surf_iso);
  a.vglob = vglob; a.V = ctx->surf_V.as<float>(); a.T = ctx->surf_T.as<int>();
  if (ctx->surf_z1 > ctx->surf_z0 && (nv > 0 || nt > 0)) {
    k_surf_emit<false><<<dim3(cdiv(a.ny, SURF_WARPS), (unsigned)(ctx->surf_z1 - ctx->surf_z0)), 32 * SURF_WARPS, 0, ctx->stream>>>(a);
    LAUNCH_CHECK();
  }
  CK(cudaStreamSynchronize(ctx->stream));
  ctx->surf_vglob = vglob; ctx->have_surface = true;
  return 0;
}

// ---- the surface of the continuous field on a lattice (r2s_isosurface_lattice) -------------------------------------------------------
// Lattice planes stream through ctx->surf_buf, `planes` owned planes per chunk plus the two planes above them that the count and emit
// kernels read; the field is never held whole.  Sweep 1 samples and counts every chunk (chunk totals); after the host scan of the totals
// (over the slabs too) sweep 2 samples again, counts again for the row bases, emits with the chunk's global bases and snaps the chunk's
// vertices.  The kernels of a chunk see its buffer through the plane-indexed SurfArgs::f, shifted by the chunk's first plane.  The two
// planes above a chunk are the next chunk's first two: they move to the front of the buffer instead of being sampled again.
#define SURF_LAT_BUDGET (1ll << 30)      // bytes of lattice values per chunk when R2S_SURF_PLANES is not set

int r2s_surf_lattice_check(r2s_ctx *ctx, const double origin[3], const double spacing[3], const int64_t dims[3], float iso, float o[3], float h[3],
                           bool band) {
  if (!isfinite(iso)) FAIL("isosurface: iso must be finite");
  if (r2s_sample_lattice_check(ctx, origin, spacing, dims, o, h)) return 1;
  if (dims[0] < 2 || dims[1] < 2 || dims[2] < 2) FAIL("isosurface: the field needs at least 2 points per axis");
  if (!band && (dims[0] - 1) * (dims[1] - 1) * (dims[2] - 1) >= (1ll << 31)) FAIL("isosurface: 2^31 or more cells");
  SampleGrid G;
  return r2s_sample_grid(ctx, &G, false);
}

// r2s_isosurface_band: the lattice planes [ka, kb) into out (plane ka first) -- classify the blocks of the layers holding them, fill the
// points of skipped owners, evaluate the points the sampled blocks hold.  cnt[1] of ctx->surf_band counts the evaluations.
static int band_planes(r2s_ctx *ctx, const SampleGrid &G, const SurfLattice &L, i64 ka, i64 kb, float *out) {
  BandArgs A;
  for (int d = 0; d < 3; d++) { A.o[d] = L.o[d]; A.h[d] = L.h[d]; A.n[d] = L.dims[d]; A.nb[d] = (L.dims[d] - 2) / R2S_BAND_B + 1; }
  A.iso = L.iso; A.below = nextafterf(L.iso, -INFINITY);
  A.ka = ka; A.kb = kb; A.kown = L.kb;
  A.lz0 = std::min((ka > 0 ? ka - 1 : 0) / R2S_BAND_B, A.nb[2] - 1);      // plane ka also lies in the layer below when ka is a multiple of B
  A.nblk = (std::min((kb - 1) / R2S_BAND_B, A.nb[2] - 1) - A.lz0 + 1) * A.nb[0] * A.nb[1];
  A.nslab = (int)L.slabs.size(); A.tab = ctx->surf_wtab.as<SurfSlabW>();
  A.cnt = ctx->surf_band.as<i64>(); A.list = A.cnt + 2; A.cls = (uint8_t *)(A.list + A.nblk);
  A.out = out;
  CK(cudaMemsetAsync(A.cnt, 0, sizeof(i64), ctx->stream));
  k_band_classify<<<cdiv(A.nblk, 128), 128, 0, ctx->stream>>>(G, A);
  LAUNCH_CHECK();
  const i64 np = (kb - ka) * A.n[0] * A.n[1];
  k_band_fill<<<cdiv(np, 256), 256, 0, ctx->stream>>>(A);
  LAUNCH_CHECK();
  i64 nact = 0;
  if (r2s_readback(ctx, &nact, A.cnt, sizeof(i64))) return 1;
  if (nact > 0) {
    k_band_sample<<<(unsigned)nact, 256, 0, ctx->stream>>>(G, A);
    LAUNCH_CHECK();
  }
  return 0;
}

static int lattice_sweep(r2s_ctx *ctx, bool emit, i64 vglob) {
  SurfLattice &L = ctx->surf_lat;
  CK(cudaSetDevice(ctx->device));
  SampleGrid G, Gh;
  if (r2s_sample_grid(ctx, &G, true) || r2s_sample_grid(ctx, &Gh, false)) return 1;
  const i64 nx = L.dims[0], ny = L.dims[1], nz = L.dims[2], pl = nx * ny, P = L.planes;
  CK(ctx->surf_buf.reserve(sizeof(float) * (size_t)((P + 2) * pl)));
  float *buf = ctx->surf_buf.as<float>();
  const int nslab = (int)L.slabs.size();
  CK(ctx->surf_wtab.reserve(sizeof(SurfSlabW) * (size_t)nslab));
  CK(cudaMemcpyAsync(ctx->surf_wtab.p, L.slabs.data(), sizeof(SurfSlabW) * (size_t)nslab, cudaMemcpyHostToDevice, ctx->stream));
  // the slab whose weights serve lattice plane k: the owner of the plane's floor plane (all planes of [ka, kb) are this context's)
  auto slab_of = [&](i64 k) {
    const int c = smp_floor(Gh.C[2], Gh.n[2], Gh.c0[2], Gh.inv[2], smp_add(L.o[2], smp_mul((float)k, L.h[2])));
    int r = 0;
    while (r + 1 < nslab && c >= L.slabs[(size_t)r].k1) r++;
    return r;
  };
  if (!emit) { L.cnv.clear(); L.cnt.clear(); }
  if (L.band) {      // per chunk: its block layers' classes, list and two counters
    const i64 nb = ((nx - 2) / R2S_BAND_B + 1) * ((ny - 2) / R2S_BAND_B + 1) * ((P + 2) / R2S_BAND_B + 2);
    CK(ctx->surf_band.reserve(sizeof(i64) * (size_t)(nb + 2) + (size_t)nb));
    CK(cudaMemsetAsync(ctx->surf_band.p, 0, 2 * sizeof(i64), ctx->stream));
  }
  i64 have = L.ka, vb = 0, tb = 0;
  for (i64 c0 = L.ka, ci = 0; c0 < L.kb; c0 += P, ci++) {
    const i64 c1 = std::min(c0 + P, L.kb), need = std::min(c1 + 2, nz);
    // planes [c0, have) are the previous chunk's top planes, at buffer positions P + (k - c0): one plane per copy (no overlap for P = 1)
    for (i64 k = c0; k < have; k++)
      CK(cudaMemcpyAsync(buf + (k - c0) * pl, buf + (P + k - c0) * pl, sizeof(float) * (size_t)pl, cudaMemcpyDeviceToDevice, ctx->stream));
    const i64 k0 = std::max(have, c0);
    if (L.band) {
      if (k0 < need && band_planes(ctx, G, L, k0, need, buf + (k0 - c0) * pl)) return 1;
    } else {
      for (i64 k = k0; k < need;) {      // runs of planes read with the same slab's weights
        const int r = slab_of(k);
        i64 e = k + 1;
        while (e < need && slab_of(e) == r) e++;
        SampleGrid Gr = G;
        Gr.w = L.slabs[(size_t)r].w; Gr.px = L.slabs[(size_t)r].px;
        if (r2s_sample_lattice_dev(ctx, Gr, L.o, L.h, L.dims, k, e, buf + (k - c0) * pl)) return 1;
        k = e;
      }
    }
    have = need;
    const float *f = buf - c0 * pl;      // plane k of the chunk at f + k * pl (only planes [c0, need) are read)
    i64 cv, ct;
    if (count_rows(ctx, f, nx, ny, nz, c0, c1, L.iso, &cv, &ct)) return 1;
    if (!emit) { L.cnv.push_back(cv); L.cnt.push_back(ct); }
    else {
      if (cv != L.cnv[(size_t)ci] || ct != L.cnt[(size_t)ci]) FAIL("isosurface: the lattice counts changed between the two sweeps");
      const double zero[3] = {0, 0, 0};
      SurfArgs a = surf_args(ctx, f, nx, ny, nz, c0, c1, zero, zero, L.iso);
      a.vglob = vglob + vb; a.V = ctx->surf_V.as<float>() + 3 * vb; a.T = ctx->surf_T.as<int>() + 3 * tb;
      if (cv > 0 || ct > 0) {
        k_surf_emit<true><<<dim3(cdiv(ny, SURF_WARPS), (unsigned)(c1 - c0)), 32 * SURF_WARPS, 0, ctx->stream>>>(a);
        LAUNCH_CHECK();
      }
      if (cv > 0) {
        SnapArgs s;
        s.f = f; s.nx = (int)nx; s.ny = (int)ny; s.z0 = (int)c0; s.nslab = nslab; s.iso = L.iso; s.n = cv; s.tab = ctx->surf_wtab.as<SurfSlabW>(); s.V = a.V;
        for (int d = 0; d < 3; d++) { s.o[d] = L.o[d]; s.h[d] = L.h[d]; }
        k_surf_snap<<<cdiv(cv, 128), 128, 0, ctx->stream>>>(G, s);
        LAUNCH_CHECK();
      }
    }
    vb += cv; tb += ct;
  }
  CK(cudaStreamSynchronize(ctx->stream));
  if (!emit) { ctx->surf_nv = vb; ctx->surf_nt = tb; }
  if (!emit && L.band && r2s_readback(ctx, &L.nsampled, ctx->surf_band.as<i64>() + 1, sizeof(i64))) return 1;
  return 0;
}

// sweep 1 over ctx->surf_lat (set by the caller): this context's vertex and triangle counts
int r2s_surf_lattice_count(r2s_ctx *ctx, i64 *nv, i64 *nt) {
  ctx->have_surface = false;
  SurfLattice &L = ctx->surf_lat;
  const i64 pl = L.dims[0] * L.dims[1];
  L.planes = ctx->knobs.surf_planes > 0 ? (i64)ctx->knobs.surf_planes : std::max<i64>(1, SURF_LAT_BUDGET / (i64)sizeof(float) / pl - 2);
  L.planes = std::max<i64>(1, std::min(L.planes, L.kb - L.ka));
  CK(cudaSetDevice(ctx->device));
  if (upload_table(ctx)) return 1;
  ctx->surf_nv = ctx->surf_nt = 0;
  if (L.kb > L.ka && lattice_sweep(ctx, false, 0)) { ctx->surf_buf.release(); return 1; }
  *nv = ctx->surf_nv; *nt = ctx->surf_nt;
  return 0;
}

// sweep 2: the mesh part of this context, its vertices from global id vglob on (nv_total vertices in the whole mesh)
int r2s_surf_lattice_emit(r2s_ctx *ctx, i64 vglob, i64 nv_total) {
  CK(cudaSetDevice(ctx->device));
  if (nv_total >= (1ll << 31)) { ctx->surf_buf.release(); FAIL("isosurface: 2^31 or more vertices (vertex ids are int32)"); }
  const i64 nv = ctx->surf_nv, nt = ctx->surf_nt;
  CK(ctx->surf_V.reserve(sizeof(float) * 3 * (size_t)std::max<i64>(nv, 1)));
  CK(ctx->surf_T.reserve(sizeof(int) * 3 * (size_t)std::max<i64>(nt, 1)));
  const SurfLattice &L = ctx->surf_lat;
  const int rc = L.kb > L.ka && (nv > 0 || nt > 0) ? lattice_sweep(ctx, true, vglob) : 0;
  ctx->surf_buf.release();
  if (rc) return 1;
  ctx->surf_f = nullptr; ctx->surf_vglob = vglob; ctx->have_surface = true;
  return 0;
}

// the fine field resident on this context: its planes, frame and the planes it owns
static int resident_field(r2s_ctx *ctx, const float **f, i64 n[3], i64 *z0, i64 *z1, double origin[3], double spacing[3]) {
  if (!ctx->has_grid) FAIL("r2s_set_grid has not been called");
  if (!ctx->have_fine) FAIL("isosurface: no fine_sdf for the current grid on the device yet (run the pipeline or the smoothing first)");
  const GridDev &g = ctx->g;
  const int s = ctx->smooth_last;
  for (int d = 0; d < 3; d++) { n[d] = g.N[d] * (i64)s + 1; origin[d] = g.amin[d]; spacing[d] = g.cell / s; }
  *f = ctx->f_fine.as<float>();
  *z0 = 0; *z1 = n[2];
  if (ctx->nranks > 1) { *z0 = s * ctx->k0; *z1 = ctx->k1 < g.np[2] ? s * ctx->k1 : n[2]; }
  return 0;
}

// ---- writers ------------------------------------------------------------------------------------------------------------------------
// Binary STL: 80-byte header, uint32 triangle count, 50 bytes per triangle (unit normal, three vertices, uint16 0); the normal is the
// cross product (v1 - v0) x (v2 - v0) in double, divided by its norm, 0 0 0 for a degenerate triangle.  Binary little-endian PLY:
// float x y z per vertex, `list uchar int vertex_indices` per face.  Both are written from host arrays, in chunks.
static int write_mesh_file(const char *path, int format, const float *V, i64 nv, const int *T, i64 nt, std::string *err) {
  if (format != 0 && format != 1) { *err = "isosurface export: format must be 0 (binary STL) or 1 (binary PLY)"; return 1; }
  if (format == 0 && nt > 0xffffffffll) { *err = "isosurface export: binary STL holds at most 2^32 - 1 triangles"; return 1; }
  FILE *fp = fopen(path, "wb");
  if (!fp) { *err = std::string("isosurface export: cannot open ") + path; return 1; }
  int rc = 0;
  const i64 CH = 1 << 20;
  std::vector<char> buf;
  if (format == 0) {
    char head[80];
    memset(head, 0, sizeof(head));
    snprintf(head, sizeof(head), "rho2sdf isosurface, %lld triangles", (long long)nt);
    const uint32_t n32 = (uint32_t)nt;
    if (fwrite(head, 1, 80, fp) != 80 || fwrite(&n32, 4, 1, fp) != 1) rc = 1;
    buf.resize((size_t)CH * 50);
    for (i64 t0 = 0; !rc && t0 < nt; t0 += CH) {
      const i64 m = std::min(CH, nt - t0);
      for (i64 t = 0; t < m; t++) {
        const int *tr = T + 3 * (t0 + t);
        const float *p[3] = {V + 3 * (i64)tr[0], V + 3 * (i64)tr[1], V + 3 * (i64)tr[2]};
        const double ux = (double)p[1][0] - p[0][0], uy = (double)p[1][1] - p[0][1], uz = (double)p[1][2] - p[0][2];
        const double wx = (double)p[2][0] - p[0][0], wy = (double)p[2][1] - p[0][1], wz = (double)p[2][2] - p[0][2];
        double nx = uy * wz - uz * wy, ny = uz * wx - ux * wz, nz = ux * wy - uy * wx;
        const double len = sqrt(nx * nx + ny * ny + nz * nz);
        if (len > 0) { nx /= len; ny /= len; nz /= len; } else nx = ny = nz = 0;
        float rec[12] = {(float)nx, (float)ny, (float)nz};
        for (int q = 0; q < 3; q++) for (int d = 0; d < 3; d++) rec[3 + 3 * q + d] = p[q][d];
        char *o = buf.data() + 50 * t;
        memcpy(o, rec, 48); o[48] = 0; o[49] = 0;
      }
      if (fwrite(buf.data(), 50, (size_t)m, fp) != (size_t)m) rc = 1;
    }
  } else {
    char head[256];
    const int hn = snprintf(head, sizeof(head),
                            "ply\nformat binary_little_endian 1.0\ncomment rho2sdf isosurface\nelement vertex %lld\nproperty float x\nproperty float y\nproperty float z\n"
                            "element face %lld\nproperty list uchar int vertex_indices\nend_header\n",
                            (long long)nv, (long long)nt);
    if (fwrite(head, 1, (size_t)hn, fp) != (size_t)hn) rc = 1;
    if (!rc && nv > 0 && fwrite(V, 12, (size_t)nv, fp) != (size_t)nv) rc = 1;
    buf.resize((size_t)CH * 13);
    for (i64 t0 = 0; !rc && t0 < nt; t0 += CH) {
      const i64 m = std::min(CH, nt - t0);
      for (i64 t = 0; t < m; t++) { char *o = buf.data() + 13 * t; o[0] = 3; memcpy(o + 1, T + 3 * (t0 + t), 12); }
      if (fwrite(buf.data(), 13, (size_t)m, fp) != (size_t)m) rc = 1;
    }
  }
  if (fclose(fp) != 0) rc = 1;
  if (rc) *err = std::string("isosurface export: write failed: ") + path;
  return rc;
}

// device -> host in chunks through two pinned staging buffers (the copy of chunk c + 1 overlaps the host copy of chunk c)
static int download_chunked(r2s_ctx *ctx, void *dst, const void *src, size_t bytes) {
  if (!bytes) return 0;
  const size_t CH = 64u << 20;
  void *stage[2] = {nullptr, nullptr};
  CK(cudaMallocHost(&stage[0], std::min(CH, bytes)));
  if (cudaMallocHost(&stage[1], std::min(CH, bytes)) != cudaSuccess) { cudaFreeHost(stage[0]); FAIL("isosurface download: cannot allocate pinned staging"); }
  int rc = 0, b = 0;
  if (cudaMemcpyAsync(stage[0], src, std::min(CH, bytes), cudaMemcpyDeviceToHost, ctx->stream) != cudaSuccess) rc = 1;
  for (size_t o = 0; !rc && o < bytes; o += CH, b ^= 1) {
    const size_t n = std::min(CH, bytes - o);
    if (cudaStreamSynchronize(ctx->stream) != cudaSuccess) { rc = 1; break; }
    if (o + n < bytes && cudaMemcpyAsync(stage[b ^ 1], (const char *)src + o + n, std::min(CH, bytes - o - n), cudaMemcpyDeviceToHost, ctx->stream) != cudaSuccess) { rc = 1; break; }
    memcpy((char *)dst + o, stage[b], n);
  }
  cudaStreamSynchronize(ctx->stream);
  cudaFreeHost(stage[0]); cudaFreeHost(stage[1]);
  if (rc) FAIL("isosurface download: copy failed");
  return 0;
}

// this context's part of the mesh into the caller's whole arrays (vertices from its first global id on), one copy each like
// r2s_download_fine_sdf; with staging = true (the file writers) through the pinned staging buffers of download_chunked
static int download_part(r2s_ctx *ctx, float *V, int32_t *T, i64 tglob, bool staging = false) {
  if (!ctx->have_surface) FAIL("isosurface: no surface on this context (call r2s_isosurface first)");
  CK(cudaSetDevice(ctx->device));
  if (staging) {
    if (V && download_chunked(ctx, V + 3 * ctx->surf_vglob, ctx->surf_V.p, sizeof(float) * 3 * (size_t)ctx->surf_nv)) return 1;
    return T && download_chunked(ctx, T + 3 * tglob, ctx->surf_T.p, sizeof(int) * 3 * (size_t)ctx->surf_nt) ? 1 : 0;
  }
  if (V && ctx->surf_nv) CK(cudaMemcpyAsync(V + 3 * ctx->surf_vglob, ctx->surf_V.p, sizeof(float) * 3 * (size_t)ctx->surf_nv, cudaMemcpyDeviceToHost, ctx->stream));
  if (T && ctx->surf_nt) CK(cudaMemcpyAsync(T + 3 * tglob, ctx->surf_T.p, sizeof(int) * 3 * (size_t)ctx->surf_nt, cudaMemcpyDeviceToHost, ctx->stream));
  CK(cudaStreamSynchronize(ctx->stream));
  return 0;
}

extern "C" {

int r2s_isosurface(r2s_ctx *ctx, float iso, int64_t *n_vertices, int64_t *n_triangles) {
  if (!ctx) return 1;
  if (ctx->nranks > 1)
    FAIL(ctx->lg ? "r2s_isosurface: this context is one slab of an r2s_multi group; use r2s_multi_isosurface"
                 : "r2s_isosurface: not available on a slab rank of the NCCL communicator (one process per GPU); extract on one context or with r2s_multi");
  const float *f; i64 n[3], z0, z1; double origin[3], spacing[3];
  if (resident_field(ctx, &f, n, &z0, &z1, origin, spacing)) return 1;
  i64 nv, nt;
  if (r2s_surf_count(ctx, f, n[0], n[1], n[2], z0, z1, origin, spacing, iso, &nv, &nt)) return 1;
  if (r2s_surf_emit(ctx, 0, nv)) return 1;
  ctx->surf_nv_all = nv; ctx->surf_nt_all = nt; ctx->surf_f = nullptr; ctx->surf_part = false;
  if (n_vertices) *n_vertices = nv;
  if (n_triangles) *n_triangles = nt;
  return 0;
}

int r2s_isosurface_from_sdf(r2s_ctx *ctx, const float *sdf, int64_t nx, int64_t ny, int64_t nz, const double origin[3], const double spacing[3], float iso,
                            int64_t *n_vertices, int64_t *n_triangles) {
  if (!ctx) return 1;
  ctx->have_surface = false;
  if (!sdf || !origin || !spacing) FAIL("r2s_isosurface_from_sdf: sdf, origin and spacing are required");
  if (nx < 2 || ny < 2 || nz < 2) FAIL("isosurface: the field needs at least 2 points per axis");
  if ((nx - 1) * (ny - 1) * (nz - 1) >= (1ll << 31)) FAIL("isosurface: 2^31 or more cells");
  CK(cudaSetDevice(ctx->device));
  DevBuf tmp;      // the caller's field; the pipeline's resident results are not touched
  CK(tmp.reserve(sizeof(float) * (size_t)(nx * ny * nz)));
  int rc = cudaMemcpyAsync(tmp.p, sdf, sizeof(float) * (size_t)(nx * ny * nz), cudaMemcpyHostToDevice, ctx->stream) != cudaSuccess;
  if (rc) ctx->err = "r2s_isosurface_from_sdf: upload failed";
  i64 nv = 0, nt = 0;
  if (!rc) rc = r2s_surf_count(ctx, tmp.as<float>(), nx, ny, nz, 0, nz, origin, spacing, iso, &nv, &nt);
  if (!rc) rc = r2s_surf_emit(ctx, 0, nv);
  cudaStreamSynchronize(ctx->stream);
  tmp.release();
  ctx->surf_f = nullptr;
  if (rc) { ctx->have_surface = false; return 1; }
  ctx->surf_nv_all = nv; ctx->surf_nt_all = nt; ctx->surf_part = false;
  if (n_vertices) *n_vertices = nv;
  if (n_triangles) *n_triangles = nt;
  return 0;
}

int r2s_isosurface_lattice(r2s_ctx *ctx, const double origin[3], const double spacing[3], const int64_t dims[3], float iso, int64_t *n_vertices,
                           int64_t *n_triangles) {
  if (!ctx) return 1;
  ctx->have_surface = false;
  if (ctx->nranks > 1)
    FAIL(ctx->lg ? "r2s_isosurface_lattice: this context is one slab of an r2s_multi group; use r2s_multi_isosurface_lattice"
                 : "r2s_isosurface_lattice: not available on a slab rank of the NCCL communicator (one process per GPU); extract on one context or with r2s_multi");
  SurfLattice &L = ctx->surf_lat;
  if (r2s_surf_lattice_check(ctx, origin, spacing, dims, iso, L.o, L.h)) return 1;
  for (int d = 0; d < 3; d++) L.dims[d] = dims[d];
  L.iso = iso; L.ka = 0; L.kb = dims[2]; L.band = false;
  L.slabs.assign(1, SurfSlabW{INT64_MAX, ctx->rbf_w, (long long)ctx->rbf_px});
  i64 nv, nt;
  if (r2s_surf_lattice_count(ctx, &nv, &nt) || r2s_surf_lattice_emit(ctx, 0, nv)) return 1;
  ctx->surf_nv_all = nv; ctx->surf_nt_all = nt; ctx->surf_part = false;
  if (n_vertices) *n_vertices = nv;
  if (n_triangles) *n_triangles = nt;
  return 0;
}

int r2s_isosurface_band(r2s_ctx *ctx, const double origin[3], const double spacing[3], const int64_t dims[3], float iso, int64_t *n_vertices,
                        int64_t *n_triangles, int64_t *n_sampled) {
  if (!ctx) return 1;
  ctx->have_surface = false;
  if (ctx->nranks > 1)
    FAIL(ctx->lg ? "r2s_isosurface_band: this context is one slab of an r2s_multi group; use r2s_multi_isosurface_band"
                 : "r2s_isosurface_band: not available on a slab rank of the NCCL communicator (one process per GPU); extract on one context or with r2s_multi");
  SurfLattice &L = ctx->surf_lat;
  if (r2s_surf_lattice_check(ctx, origin, spacing, dims, iso, L.o, L.h, true)) return 1;
  for (int d = 0; d < 3; d++) L.dims[d] = dims[d];
  L.iso = iso; L.ka = 0; L.kb = dims[2]; L.band = true; L.nsampled = 0;
  L.slabs.assign(1, SurfSlabW{INT64_MAX, ctx->rbf_w, (long long)ctx->rbf_px});
  i64 nv, nt;
  if (r2s_surf_lattice_count(ctx, &nv, &nt) || r2s_surf_lattice_emit(ctx, 0, nv)) { ctx->surf_band.release(); return 1; }
  ctx->surf_band.release();
  ctx->surf_nv_all = nv; ctx->surf_nt_all = nt; ctx->surf_part = false;
  if (n_vertices) *n_vertices = nv;
  if (n_triangles) *n_triangles = nt;
  if (n_sampled) *n_sampled = L.nsampled;
  return 0;
}

int r2s_download_isosurface(r2s_ctx *ctx, float *vertices, int32_t *triangles) {
  if (!ctx) return 1;
  if (ctx->have_surface && ctx->surf_part) FAIL("r2s_download_isosurface: this context holds one slab of a mesh; use r2s_multi_download_isosurface");
  return download_part(ctx, vertices, triangles, 0);
}

int r2s_export_isosurface(r2s_ctx *ctx, const char *path, int format) {
  if (!ctx) return 1;
  if (!path) FAIL("r2s_export_isosurface: path is required");
  if (!ctx->have_surface) FAIL("isosurface: no surface on this context (call r2s_isosurface first)");
  if (ctx->surf_part) FAIL("r2s_export_isosurface: this context holds one slab of a mesh; use r2s_multi_export_isosurface");
  std::vector<float> V((size_t)(3 * ctx->surf_nv_all));
  std::vector<int> T((size_t)(3 * ctx->surf_nt_all));
  if (download_part(ctx, V.data(), T.data(), 0, true)) return 1;
  std::string e;
  if (write_mesh_file(path, format, V.data(), ctx->surf_nv_all, T.data(), ctx->surf_nt_all, &e)) FAIL(e);
  return 0;
}

}  // extern "C"

// ---- several slabs (r2s_multi.cu calls these from its per-slab threads) ----------------------------------------------------------------
// pass 1 on one slab of the resident fine field: two halo planes above (plane z1 and z1 + 1) so that the slab can number plane z1's vertices
int r2s_surf_count_slab(r2s_ctx *ctx, float iso, i64 *nv, i64 *nt) {
  const float *f; i64 n[3], z0, z1; double origin[3], spacing[3];
  ctx->have_surface = false;
  if (resident_field(ctx, &f, n, &z0, &z1, origin, spacing)) return 1;
  CK(cudaSetDevice(ctx->device));
  if (ctx->nranks > 1 && r2s_halo_exchange_f32(ctx, ctx->f_fine.as<float>(), n[0] * n[1], (int)z0, (int)z1, (int)n[2], 0, 2)) return 1;
  ctx->surf_part = true;
  return r2s_surf_count(ctx, f, n[0], n[1], n[2], z0, z1, origin, spacing, iso, nv, nt);
}
int r2s_surf_download_slab(r2s_ctx *ctx, float *V, int32_t *T, i64 tglob, bool staging) { return download_part(ctx, V, T, tglob, staging); }
int r2s_surf_write_file(const char *path, int format, const float *V, i64 nv, const int *T, i64 nt, std::string *err) {
  return write_mesh_file(path, format, V, nv, T, nt, err);
}
