// Host build of the cut-cell quadrature (rho2sdf.jl_b200/csrc/r2s_volq.cuh) next to a literal restatement of the loop it replaced, for
// tests/test_vol_host.py.  Built with -ffp-contract=off, so every product and sum below rounds where it is written.
#include <math.h>
#include "../../rho2sdf.jl_b200/csrc/r2s_volq.cuh"

// The earlier k_vol_cut / k_vl_eval loop.  nvcc contracted it (cuobjdump -sass of that build): c000 * xm + c100 * xi became
// fma(c100, xi, c000 * xm), c00 * em + c10 * eta became fma(c10, eta, c00 * em), part += wij * w[kq] became fma(wij, w[kq], part).
static float old_loop(const float cv[8], const GaussF &G, float iso, float *mabs) {
  const float c000 = cv[0], c100 = cv[1], c010 = cv[2], c110 = cv[3], c001 = cv[4], c101 = cv[5], c011 = cv[6], c111 = cv[7];
  float part = 0.0f, m = INFINITY;
  for (int iq = 0; iq < 9; iq++) {
    const float xi = (G.x[iq] + 1) / 2, xm = 1.0f - xi;
    const float c00 = fmaf(c100, xi, c000 * xm), c01 = fmaf(c101, xi, c001 * xm);
    const float c10 = fmaf(c110, xi, c010 * xm), c11 = fmaf(c111, xi, c011 * xm);
    for (int jq = 0; jq < 9; jq++) {
      const float eta = (G.x[jq] + 1) / 2, em = 1.0f - eta;
      const float c0 = fmaf(c10, eta, c00 * em), c1 = fmaf(c11, eta, c01 * em);
      const float wij = G.w[iq] * G.w[jq], dc = c1 - c0;
      for (int kq = 0; kq < 9; kq++) {
        const float ps = fmaf(dc, (G.x[kq] + 1) / 2, c0);
        if (ps >= iso) part = fmaf(wij, G.w[kq], part);
        m = fminf(m, fabsf(ps));
      }
    }
  }
  *mabs = m;
  return part;
}

extern "C" void vol_host_quad9(const float *cells, long n, const float *gx, const float *gw, float iso, float *part_new, float *m_new, float *part_old, float *m_old) {
  GaussF G;
  for (int q = 0; q < 9; q++) { G.x[q] = gx[q]; G.w[q] = gw[q]; }
  for (long i = 0; i < n; i++) {
    part_new[i] = cut_cell_quad9<true>(cells + 8 * i, G, iso, &m_new[i]);
    part_old[i] = old_loop(cells + 8 * i, G, iso, &m_old[i]);
    float unused;
    if (cut_cell_quad9<false>(cells + 8 * i, G, iso, &unused) != part_new[i]) part_new[i] = NAN;      // the two instantiations agree
  }
}

// ---- whole-grid reference of calculate_volume_from_sdf at order 9 ---------------------------------------------------------------------
// The library's rules restated: a cell's corner values c = v - th (th = 0 for calculate_volume_from_sdf; the threshold search classifies
// v against th, which is the same test because IEEE subtraction is sign-exact); the cell is empty iff max(c) < iso, full iff min(c) >= iso,
// otherwise cut_cell_quad9(c) against iso with the library's Gauss table.  Each cut cell adds llrint(part * 2^37) to an exact 128-bit sum
// S; the volume is nfull * ev + (S / 2^37) * jac with ev = edge * edge * edge and jac = ev / 8 in float, S rounded to double once.
// memo != 0: each thread keeps the last quadratures in a small direct-mapped table keyed by the eight corner bit patterns (the result is a
// function of those bits alone, so this is exact); fields that repeat along x then cost one quadrature per distinct cell.
#define __constant__
#include "../../rho2sdf.jl_b200/csrc/r2s_tables.cuh"
#undef __constant__
#include <stdlib.h>
#include <string.h>

typedef unsigned __int128 u128;

static GaussF library_gauss9() {
  const GaussTab t = gauss_legendre_host(9);
  GaussF g;
  for (int q = 0; q < 9; q++) { g.x[q] = (float)t.x[q]; g.w[q] = (float)t.w[q]; }
  return g;
}

extern "C" void vol_host_gauss9(float *x, float *w) {
  const GaussF g = library_gauss9();
  for (int q = 0; q < 9; q++) { x[q] = g.x[q]; w[q] = g.w[q]; }
}

extern "C" void vol_host_grid(const float *sdf, long nx, long ny, long nz, long px, float iso, float th, float edge, int memo, long long *nfull_out,
                              unsigned long long *s_lo, unsigned long long *s_hi, double *vol) {
  const GaussF G = library_gauss9();
  const long ncx = nx - 1, ncy = ny - 1, ncz = nz - 1, nrows = ncy * ncz, sxy = px * ny;
  long long nfull = 0;
  u128 S = 0;
#pragma omp parallel
  {
    enum { NM = 256 };
    struct Memo { unsigned key[8]; unsigned long long q; int valid; };
    Memo *tab = memo ? (Memo *)calloc(NM, sizeof(Memo)) : nullptr;
    long long my_full = 0;
    u128 my_s = 0;
#pragma omp for schedule(dynamic, 16)
    for (long r = 0; r < nrows; r++) {
      const long j = r % ncy, k = r / ncy;
      for (long i = 0; i < ncx; i++) {
        const long b = (k * ny + j) * px + i;
        const float v[8] = {sdf[b], sdf[b + 1], sdf[b + px], sdf[b + px + 1], sdf[b + sxy], sdf[b + sxy + 1], sdf[b + sxy + px], sdf[b + sxy + px + 1]};
        float c[8], mn, mx;
        for (int a = 0; a < 8; a++) c[a] = v[a] - th;
        mn = mx = c[0];
        for (int a = 1; a < 8; a++) { if (c[a] < mn) mn = c[a]; if (c[a] > mx) mx = c[a]; }
        if (mx < iso) continue;
        if (mn >= iso) { my_full++; continue; }
        unsigned key[8]; memcpy(key, c, sizeof(key));
        unsigned h = 2166136261u;
        for (int a = 0; a < 8; a++) h = (h ^ key[a]) * 16777619u;
        Memo *m = tab ? &tab[h % NM] : nullptr;
        unsigned long long q;
        if (m && m->valid && memcmp(m->key, key, sizeof(key)) == 0) q = m->q;
        else {
          q = (unsigned long long)llrint((double)cut_cell_quad9<false>(c, G, iso, nullptr) * 137438953472.0);
          if (m) { memcpy(m->key, key, sizeof(key)); m->q = q; m->valid = 1; }
        }
        my_s += q;
      }
    }
#pragma omp critical
    { nfull += my_full; S += my_s; }
    free(tab);
  }
  const float ev = edge * edge * edge, jac = ev / 8.0f;
  *nfull_out = nfull; *s_lo = (unsigned long long)S; *s_hi = (unsigned long long)(S >> 64);
  *vol = (double)nfull * (double)ev + ((double)S / 137438953472.0) * (double)jac;
}

// the library's two-word fixed-point sum (vol_sum_flush's words s0, s1) -> double, against the 128-bit integer converted by the compiler
extern "C" void vol_host_fixed_value(const unsigned long long *s0, const unsigned long long *s1, long n, double *lib, double *ref) {
  for (long i = 0; i < n; i++) {
    lib[i] = vol_fixed_value(s0[i], s1[i]);
    ref[i] = (double)(((u128)s1[i] << 32) + s0[i]) / 137438953472.0;
  }
}
