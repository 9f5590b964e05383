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
