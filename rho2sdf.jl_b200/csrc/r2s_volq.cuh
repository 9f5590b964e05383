// r2s_volq.cuh -- the 9 x 9 x 9 Gauss quadrature of one cut cell (CalcVolumeFromSDF.jl:88-103), shared by the whole-grid volume
// (k_vol_cut) and the threshold search (k_vl_eval), and compiled for the host by tests/host/vol_host.cpp.
//
// The arithmetic is spelled out operation by operation so that the device and a host build (-ffp-contract=off) give the same bits:
// it is what nvcc made of the earlier loop (c000 * (1 - xi) + c100 * xi contracted to fma(c100, xi, c000 * xm), the same for eta;
// the zeta lerp as fma(c1 - c0, zeta, c0); the weight sum as fma(w_i w_j, w_k, part)).  Pairs of independent operations are packed
// into one f32x2 instruction on the device (FFMA2 / FMUL2: IEEE per half, the same bits as two scalar operations, one issue slot;
// tools/probes/ffma2_probe.cu): the lerps of the z = 0 and z = 1 faces, and the zeta lerps of Gauss points kq, kq + 1.
// The inside test stays a predicated add per lane: the 32 lanes hold 32 different cells, so no branch on the column's sign pattern.
#pragma once
#include <math.h>

#if defined(__CUDACC__)
#define R2S_HD __host__ __device__ __forceinline__
#else
#define R2S_HD inline
#endif

struct GaussF { float x[9]; float w[9]; };
struct F2 { float x, y; };

R2S_HD float q_mul(float a, float b) {
#if defined(__CUDA_ARCH__)
  return __fmul_rn(a, b);      // never contracted with a following add
#else
  return a * b;
#endif
}
R2S_HD float q_sub(float a, float b) {
#if defined(__CUDA_ARCH__)
  return __fsub_rn(a, b);
#else
  return a - b;
#endif
}
R2S_HD F2 q_mul2(F2 a, F2 b) {
#if defined(__CUDA_ARCH__)
  unsigned long long xa = *reinterpret_cast<unsigned long long *>(&a), xb = *reinterpret_cast<unsigned long long *>(&b), r;
  asm("mul.rn.f32x2 %0, %1, %2;" : "=l"(r) : "l"(xa), "l"(xb));
  return *reinterpret_cast<F2 *>(&r);
#else
  return F2{a.x * b.x, a.y * b.y};
#endif
}
R2S_HD F2 q_fma2(F2 a, F2 b, F2 c) {
#if defined(__CUDA_ARCH__)
  unsigned long long xa = *reinterpret_cast<unsigned long long *>(&a), xb = *reinterpret_cast<unsigned long long *>(&b), xc = *reinterpret_cast<unsigned long long *>(&c), r;
  asm("fma.rn.f32x2 %0, %1, %2, %3;" : "=l"(r) : "l"(xa), "l"(xb), "l"(xc));
  return *reinterpret_cast<F2 *>(&r);
#else
  return F2{fmaf(a.x, b.x, c.x), fmaf(a.y, b.y, c.y)};
#endif
}
// Gauss abscissa mapped to [0, 1]: (x + 1) / 2 (the halving is exact)
R2S_HD float q_unit(float x) { return q_mul(x + 1.0f, 0.5f); }

// c: the cell's corner values minus the threshold, c[a + 2 b + 4 d] at corner (x = a, y = b, z = d).  Returns the Float32 sum of
// w_i w_j w_k over the Gauss points whose value is >= iso, added in the order iq, then jq, then kq.  MARGIN: *mabs = the smallest
// |value| over the 729 points.
template <bool MARGIN>
R2S_HD float cut_cell_quad9(const float c[8], const GaussF &G, float iso, float *mabs) {
  const F2 f00 = {c[0], c[4]}, f10 = {c[1], c[5]}, f01 = {c[2], c[6]}, f11 = {c[3], c[7]};      // {z = 0, z = 1} pairs
  float part = 0.0f, m = INFINITY;
#if defined(__CUDA_ARCH__)
#pragma unroll 1      // the 81-point inner body stays unrolled; unrolling all 729 points (60 KB of code) thrashed the instruction cache
#endif
  for (int iq = 0; iq < 9; iq++) {
    const float xi = q_unit(G.x[iq]), xm = 1.0f - xi;
    const F2 vxi = {xi, xi}, vxm = {xm, xm};
    const F2 a = q_fma2(f10, vxi, q_mul2(f00, vxm));      // {c00, c01}: the y = 0 edge lerped in x, faces z = 0 and z = 1
    const F2 b = q_fma2(f11, vxi, q_mul2(f01, vxm));      // {c10, c11}: the y = 1 edge
#if defined(__CUDA_ARCH__)
#pragma unroll
#endif
    for (int jq = 0; jq < 9; jq++) {
      const float eta = q_unit(G.x[jq]), em = 1.0f - eta;
      const F2 cc = q_fma2(b, F2{eta, eta}, q_mul2(a, F2{em, em}));      // {c0, c1}: the column's values at z = 0 and z = 1
      const float c0 = cc.x, dc = q_sub(cc.y, cc.x), wij = q_mul(G.w[iq], G.w[jq]);
#if defined(__CUDA_ARCH__)
#pragma unroll
#endif
      for (int kq = 0; kq < 9; kq += 2) {
        float ps[2];
        if (kq + 1 < 9) {
          const F2 p = q_fma2(F2{dc, dc}, F2{q_unit(G.x[kq]), q_unit(G.x[kq + 1])}, F2{c0, c0});
          ps[0] = p.x; ps[1] = p.y;
        } else {
          ps[0] = fmaf(dc, q_unit(G.x[kq]), c0); ps[1] = 0.0f;
        }
#if defined(__CUDA_ARCH__)
#pragma unroll
#endif
        for (int h = 0; h < 2; h++) {
          if (kq + h >= 9) break;
          if (ps[h] >= iso) part = fmaf(wij, G.w[kq + h], part);
          if (MARGIN) m = fminf(m, fabsf(ps[h]));
        }
      }
    }
  }
  if (MARGIN) *mabs = m;
  return part;
}

// The cut-cell sum in fixed point.  A cell's Float32 sum part (in [0, 8]) enters the volume as q = llrint(part * 2^37) < 2^40 (exact for
// a sum of 9-point Gauss weight products).  A thread adds its cells' q into one 64-bit word (vol_cell_add: fewer than 2^24 cells per
// thread in every kernel, so it cannot wrap); the kernels then add the low 32 bits and the rest of the thread sums into two separate
// 64-bit words s0, s1 (vol_sum_flush in r2s_rbf.cu), neither of which wraps below 2^31 cells (s0 < 2^63, s1 < 2^39).  A single word
// wrapped once the parts added up to 2^27.  The integer sum S = s1 * 2^32 + s0 does not depend on the order of the cells.
R2S_HD void vol_cell_add(unsigned long long &local, float part) {
  local += (unsigned long long)llrint((double)part * 137438953472.0 /* 2^37 */);
}
// S / 2^37 as a double, rounded once (to nearest, ties to even).  Below 2^64 this is (double)S / 2^37, the value of the single-word sum.
R2S_HD double vol_fixed_value(unsigned long long s0w, unsigned long long s1w) {
  const unsigned long long lo = s0w + (s1w << 32), hi = (s1w >> 32) + (lo < s0w ? 1ull : 0ull);      // S = hi * 2^64 + lo
  if (hi == 0) return (double)lo / 137438953472.0;
  int sh = 0;
  while (sh < 64 && (hi >> sh) != 0) sh++;      // S < 2^(64 + sh): keep its top 64 bits, the bits shifted out as a sticky bit
  const unsigned long long t = (lo >> sh) | (hi << (64 - sh)) | ((lo & ((1ull << sh) - 1)) != 0 ? 1ull : 0ull);
  return ldexp((double)t, sh - 37);
}
