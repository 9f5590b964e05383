// r2s_band.cuh -- which blocks of a lattice can hold the surface {f = iso} of the continuous field (r2s_isosurface_band, r2s_surf.cu),
// shared by the classification kernel and the host build (tests/host/band_host.cpp, g++ -ffp-contract=off).
//
// f(p) = fl(acc + th), acc = the fmaf chain of w_c phi_c over the taps of p (r2s_sample.cuh), phi_c >= 0.  A block is a closed box of lattice
// points [lo_d, hi_d] per axis; its Float32 box [a_d, b_d] comes from the two end indices (float(o) + float(i) * float(h) is monotone in i).
//   reach set R: the coarse points c in the candidate windows of both box ends ([floor(a) - 2, floor(b) + 3]) whose distance to the box,
//     in double, is within the cut radius after a relative margin of 2^-20 (it covers the Float32 roundings of e_d, e_d^2 and d2) -- every
//     tap of every point of the box is in R;
//   certain set S: the c of R in the window of every point ([floor(b) - 2, floor(a) + 3]) whose largest distance to the box passes the
//     cut test with the same margin the other way -- every point of the box includes every c of S;
//   inside (1): every w_c >= 0 over R (-0 counts).  Then every fma adds a term >= 0 to an accumulator >= 0, rounding is monotone, and
//     f >= fl(0 + th) = th.  Decided if th >= iso; otherwise if fl(L + th) >= iso for a Float32 L <= acc:
//       phi_c >= exp(-kappa D_c^2 (1 + 2^-20)) (1 - 2^-20)   (D_c the largest distance of c to the box; exp_f32 error <= 1.5 2^-24,
//                                                              the roundings of e, e^2, kappa e^2 and the two products)
//       acc >= sum_S w_c phi_c (1 - 2^-16) - 2^-120          (at most 124 fma roundings; the taps outside S add terms >= 0)
//     with L rounded down to Float32; fl(acc + th) >= fl(L + th) since rounding is monotone.
//   outside (2): the mirror, every w_c <= 0 over R (+0 counts), f <= th; decided if th < iso, or if fl(U + th) < iso for U >= acc.
//   anything else (0) is sampled: a NaN weight fails both tests; a weight above 2^100 in magnitude, or |th| > 2^126, is never skipped,
//   so a skipped value is finite (as the value the dense path would compute).
// The margins are parameters so that the host tests can run the classifier without them and show that the boundary cases catch it.
#pragma once
#include <math.h>
#include <stdint.h>
#include "r2s_sample.cuh"

#define R2S_BAND_B 8      // lattice cells per block edge: a block is the closed box of (B + 1)^3 lattice points

struct BandMargin { double d2_lo, d2_hi, phi, acc, tiny; };
R2S_HD BandMargin band_margin() { return BandMargin{1.0 - 0x1p-20, 1.0 + 0x1p-20, 1.0 - 0x1p-20, 1.0 - 0x1p-16, 0x1p-120}; }

R2S_HD float band_down(double x) {      // the largest float <= x
  float f = (float)x;
  if ((double)f > x) f = nextafterf(f, -INFINITY);
  return f;
}
R2S_HD float band_up(double x) {        // the smallest float >= x
  float f = (float)x;
  if ((double)f < x) f = nextafterf(f, INFINITY);
  return f;
}

// 0: sample, 1: every value of the Float32 box [a_d, b_d] (a_d <= b_d) is >= iso, 2: every value is < iso.  G: the weights every point of
// the box reads (one slab's).  The box form serves any set of points known to lie in the box (r2s_elemfrac.cuh: an element's Gauss points).
R2S_HD int band_classify_box(const SampleGrid &G, const float a[3], const float b[3], float iso, BandMargin M) {
  if (!(fabsf(G.th) <= 0x1p126f)) return 0;
  int rl[3], rh[3], sl[3], sh[3];
  for (int d = 0; d < 3; d++) {
    const int fa = smp_floor(G.C[d], G.n[d], G.c0[d], G.inv[d], a[d]), fb = smp_floor(G.C[d], G.n[d], G.c0[d], G.inv[d], b[d]);
    rl[d] = fa - 2 < 0 ? 0 : fa - 2; rh[d] = fb + 3 > G.n[d] - 1 ? G.n[d] - 1 : fb + 3;
    sl[d] = fb - 2; sh[d] = fa + 3;
  }
  const double t2 = (double)G.t2, kappa = (double)G.kappa;
  bool pos = false, neg = false;
  double sum = 0.0;      // sum over S of |w| times the phi lower bound
  for (int k = rl[2]; k <= rh[2]; k++) {
    const double cz = (double)G.C[2][k], nz = cz < a[2] ? a[2] - cz : cz > b[2] ? cz - b[2] : 0.0, fz = fmax(fabs(cz - a[2]), fabs(cz - b[2]));
    if (nz * nz * M.d2_lo - M.tiny > t2) continue;
    for (int j = rl[1]; j <= rh[1]; j++) {
      const double cy = (double)G.C[1][j], ny = cy < a[1] ? a[1] - cy : cy > b[1] ? cy - b[1] : 0.0, fy = fmax(fabs(cy - a[1]), fabs(cy - b[1]));
      if ((ny * ny + nz * nz) * M.d2_lo - M.tiny > t2) continue;
      const float *row = G.w + ((long long)k * G.ny + j) * G.px;
      for (int i = rl[0]; i <= rh[0]; i++) {
        const double cx = (double)G.C[0][i], nx = cx < a[0] ? a[0] - cx : cx > b[0] ? cx - b[0] : 0.0;
        if ((nx * nx + ny * ny + nz * nz) * M.d2_lo - M.tiny > t2) continue;
        const float w = smp_load(row + i);
        if (!(fabsf(w) <= 0x1p100f)) return 0;
        pos |= w > 0.0f; neg |= w < 0.0f;
        if (pos && neg) return 0;
        const double fx = fmax(fabs(cx - a[0]), fabs(cx - b[0])), D2 = (fx * fx + fy * fy) + fz * fz;
        if (i >= sl[0] && i <= sh[0] && j >= sl[1] && j <= sh[1] && k >= sl[2] && k <= sh[2] && D2 * M.d2_hi + M.tiny <= t2)
          sum += fabs((double)w) * (exp(-kappa * D2 * M.d2_hi) * M.phi);
      }
    }
  }
  const double s = sum * M.acc - M.tiny;
  if (!neg && (G.th >= iso || smp_add(band_down(s), G.th) >= iso)) return 1;
  if (!pos && (G.th < iso || smp_add(band_up(-s), G.th) < iso)) return 2;
  return 0;
}

// the lattice form: lo / hi are the box's end lattice indices per axis (lo <= hi) of the lattice o + float(i) h
R2S_HD int band_classify(const SampleGrid &G, const float o[3], const float h[3], const long long lo[3], const long long hi[3], float iso, BandMargin M) {
  float a[3], b[3];
  for (int d = 0; d < 3; d++) {
    const float pa = smp_add(o[d], smp_mul((float)lo[d], h[d])), pb = smp_add(o[d], smp_mul((float)hi[d], h[d]));
    a[d] = pa < pb ? pa : pb; b[d] = pa < pb ? pb : pa;
  }
  return band_classify_box(G, a, b, iso, M);
}
