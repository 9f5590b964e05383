// r2s_mc.cuh -- the marching-cubes case table of the isosurface stage (r2s_surf.cu), generated from one rule, and the vertex formula.
// Host and device code: tests/host/mc_host.cpp compiles this header with g++ -ffp-contract=off.
//
// Cube corner c (0..7) sits at offset (c & 1, c >> 1 & 1, c >> 2 & 1); corner c is INSIDE iff its value >= iso (the convention of the
// volume stages and of remove_sdf_artifacts!).  The 12 cube edges are the corner pairs (a, b), a < b, that differ in one bit, numbered in
// lexicographic order; edge e starts at corner mc_edge_corner(e) and runs along axis mc_edge_axis(e).
//
// Face rule: on each cube face, each maximal cyclic run of inside corners is cut off by one segment, from the crossing on the edge that
// enters the run to the crossing on the edge that leaves it, the face's corners walked counter-clockwise as seen from outside the cube.
// An ambiguous face (two diagonal inside corners) therefore SEPARATES its inside corners.  The segments depend on the face's four corners
// only, so two cells sharing a face cut it identically (no cracks), and the surface separates {value >= iso} in its 6-connectivity.
// The segments chain into closed loops (each crossing edge ends one segment and starts the next).  Each loop is walked from its smallest
// edge id and fan-triangulated from the first of its vertices whose fan chords all cross the cube's interior: a chord between two edges of
// one face would lie in that face, and where the neighbouring cell drew the same chord the two cells' triangles would meet in a
// four-triangle edge (a flat double sheet in the face; random fields produce it).  17 of the 358 loops of the table need an apex other than
// the smallest edge; every loop has one (the exhaustive host test checks both).  With segments oriented entry -> exit, every triangle is
// counter-clockwise seen from the outside corners.
#pragma once
#include <stdint.h>
#ifdef __CUDACC__
#define MC_HD __host__ __device__
#else
#define MC_HD
#endif

#define MC_MAX_TRI 5      // most triangles of one case (the rule above never needs more; the exhaustive host test checks it)

// edge e = corner pair (mc_edge_corner(e), mc_edge_corner(e) + (1 << mc_edge_axis(e)))
MC_HD inline int mc_edge_corner(int e) { const int a[12] = {0, 0, 0, 1, 1, 2, 2, 3, 4, 4, 5, 6}; return a[e]; }
MC_HD inline int mc_edge_axis(int e) { const int a[12] = {0, 1, 2, 1, 2, 0, 2, 2, 0, 1, 1, 0}; return a[e]; }

struct McCase {
  uint8_t n;                       // triangles
  uint8_t e[3 * MC_MAX_TRI];       // their cube edges, three per triangle
};

// faces (bit 2 * axis + side) that contain edge e
MC_HD inline int mc_edge_faces(int e) {
  const int c = mc_edge_corner(e), a = mc_edge_axis(e);
  int m = 0;
  for (int d = 0; d < 3; d++) if (d != a) m |= 1 << (2 * d + (c >> d & 1));
  return m;
}

MC_HD inline int mc_edge_of(int a, int b) {
  if (a > b) { const int t = a; a = b; b = t; }
  const int ax = (b ^ a) == 1 ? 0 : (b ^ a) == 2 ? 1 : 2;
  for (int e = 0; e < 12; e++)
    if (mc_edge_corner(e) == a && mc_edge_axis(e) == ax) return e;
  return -1;
}

// face f = 2 * axis + side: its four corners in counter-clockwise order seen from outside the cube
MC_HD inline void mc_face(int f, int cyc[4]) {
  const int ax = f >> 1, s = f & 1, u = ax == 0 ? 1 : 0, v = ax == 2 ? 1 : 2;
  const int pu[4] = {0, 1, 1, 0}, pv[4] = {0, 0, 1, 1};
  for (int q = 0; q < 4; q++) cyc[q] = (s << ax) | (pu[q] << u) | (pv[q] << v);
  // (u, v, ax) is a cyclic permutation of (x, y, z) for ax = 0, 2: the walk above then turns about +ax; an outward normal is +ax iff s = 1
  const int turn = ax == 1 ? -1 : 1, out = s ? 1 : -1;
  if (turn != out) { const int t = cyc[1]; cyc[1] = cyc[3]; cyc[3] = t; }
}

// the face-rule segments of case c on face f: seg[2 * q] -> seg[2 * q + 1]; returns their number (0..2)
MC_HD inline int mc_face_segments(int c, int f, int seg[4]) {
  int cyc[4];
  mc_face(f, cyc);
  int in[4], n = 0;
  for (int q = 0; q < 4; q++) in[q] = (c >> cyc[q]) & 1;
  for (int q = 0; q < 4; q++) {
    if (!in[q] || in[(q + 3) & 3]) continue;      // a run of inside corners starts at q
    int r = q;
    while (in[(r + 1) & 3] && ((r + 1) & 3) != q) r = (r + 1) & 3;
    seg[2 * n] = mc_edge_of(cyc[(q + 3) & 3], cyc[q]);
    seg[2 * n + 1] = mc_edge_of(cyc[r], cyc[(r + 1) & 3]);
    n++;
  }
  return n;
}

// case c (bit k set iff corner k is inside) -> triangles in table order
MC_HD inline McCase mc_build_case(int c) {
  int nxt[12];
  for (int e = 0; e < 12; e++) nxt[e] = -1;
  for (int f = 0; f < 6; f++) {
    int seg[4];
    const int n = mc_face_segments(c, f, seg);
    for (int q = 0; q < n; q++) nxt[seg[2 * q]] = seg[2 * q + 1];
  }
  McCase out;
  out.n = 0;
  for (int q = 0; q < 3 * MC_MAX_TRI; q++) out.e[q] = 0;
  bool seen[12];
  for (int e = 0; e < 12; e++) seen[e] = false;
  for (int s = 0; s < 12; s++) {      // loops in order of their smallest edge, each walked from it
    if (nxt[s] < 0 || seen[s]) continue;
    int loop[12], m = 0, x = s;
    do { loop[m++] = x; seen[x] = true; x = nxt[x]; } while (x != s && m < 12);
    int apex = 0;      // the first loop vertex whose chords (to the loop vertices not next to it) share no face with it
    for (; apex < m; apex++) {
      bool ok = true;
      for (int q = 2; q + 1 < m; q++) ok = ok && !(mc_edge_faces(loop[apex]) & mc_edge_faces(loop[(apex + q) % m]));
      if (ok) break;
    }
    if (apex == m) apex = 0;      // not reached by any case (tested); keeps the table well defined
    for (int q = 1; q + 1 < m && out.n < MC_MAX_TRI; q++) {
      out.e[3 * out.n] = (uint8_t)loop[apex]; out.e[3 * out.n + 1] = (uint8_t)loop[(apex + q) % m]; out.e[3 * out.n + 2] = (uint8_t)loop[(apex + q + 1) % m];
      out.n++;
    }
  }
  return out;
}

// the vertex on the grid edge from point p to p + e_ax (values va at p, vb at the other end, on different sides of iso): coordinate
// d = origin[d] + spacing[d] * (p[d] + (d == ax ? t : 0)), t = (iso - va) / (vb - va), all in double without contraction, rounded to
// float once per coordinate.  The device build uses the round-to-nearest intrinsics (nvcc cannot fuse them); the host build relies on
// -ffp-contract=off.
#ifdef __CUDA_ARCH__
#define MC_ADD(a, b) __dadd_rn(a, b)
#define MC_SUB(a, b) __dsub_rn(a, b)
#define MC_MUL(a, b) __dmul_rn(a, b)
#define MC_DIV(a, b) __ddiv_rn(a, b)
#else
#define MC_ADD(a, b) ((a) + (b))
#define MC_SUB(a, b) ((a) - (b))
#define MC_MUL(a, b) ((a) * (b))
#define MC_DIV(a, b) ((a) / (b))
#endif
MC_HD inline void mc_vertex(const double origin[3], const double spacing[3], long long i, long long j, long long k, int ax, float va, float vb, float iso,
                            float out[3]) {
  const double t = MC_DIV(MC_SUB((double)iso, (double)va), MC_SUB((double)vb, (double)va));
  const long long p[3] = {i, j, k};
  for (int d = 0; d < 3; d++) {
    const double q = d == ax ? MC_ADD((double)p[d], t) : (double)p[d];
    out[d] = (float)MC_ADD(origin[d], MC_MUL(spacing[d], q));
  }
}
