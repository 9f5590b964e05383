// r2s_sample.cuh -- the continuous smoothed SDF of rbf_interpolation_kdtree (SdfSmoothing/RBFs4Smoothing.jl:219-248) at one point,
// shared by the sampling kernels (r2s_sample.cu) and compiled for the host by tests/host/sample_host.cpp.
//
//   fine_sdf(x) = th + sum_c w_c exp(-|x - c|^2 / cell^2)   over the coarse points c with |x - c| <= maxd
//
// Every operation is spelled out (device: __fmul_rn / __fadd_rn, never contracted; host: built with -ffp-contract=off), so a host build
// gives the same bits as the device.  For a point p (Float32 coordinates, rounded once from double):
//   e_d = C_d[i] - p_d                       C_d = the Float32 coordinate table range(amin_d, amax_d, length = N_d + 1)
//   d2  = (e_x e_x + e_y e_y) + e_z e_z      coarse point included iff d2 <= t2 (smp_t2: the same test as sqrtf(d2) <= maxd)
//   phi = (a_x a_y) a_z,  a_d = exp_f32(-(kappa (e_d e_d))),  kappa = float(1 / cell^2)
//   value    = (sum fmaf(w, phi, acc) in ascending (k, j, i), from 0) + th
//   gradient = (kappa + kappa) * sum fmaf(w phi, e_d, g_d), same order       (d/dx of w exp(-kappa |x - c|^2) = 2 kappa w phi (c - x))
// The factorised phi is within Float32 round-off of exp(-kappa d2), as in the stencil CG (r2s_rbf.cu): 18 exponentials per point
// instead of one per tap.
//
// exp_f32 accuracy (tests/test_sample_host.py checks every float argument in [-16, 0]): |exp_f32(x) - exp(x)| <= 1.5 * 2^-24 * exp(x).
// The kernel evaluates it on [-kappa t2, 0], i.e. at most about ln(1/rbf_cut) < 8 in magnitude.
#pragma once
#include <math.h>
#include <stdint.h>
#include <string.h>

#ifndef R2S_HD
#if defined(__CUDACC__)
#define R2S_HD __host__ __device__ __forceinline__
#else
#define R2S_HD inline
#endif
#endif

R2S_HD float smp_mul(float a, float b) {
#if defined(__CUDA_ARCH__)
  return __fmul_rn(a, b);
#else
  return a * b;
#endif
}
R2S_HD float smp_add(float a, float b) {
#if defined(__CUDA_ARCH__)
  return __fadd_rn(a, b);
#else
  return a + b;
#endif
}
R2S_HD float smp_sub(float a, float b) {
#if defined(__CUDA_ARCH__)
  return __fsub_rn(a, b);
#else
  return a - b;
#endif
}
R2S_HD float smp_pow2i(int n) {      // 2^n for -126 <= n <= 127
  const uint32_t bits = (uint32_t)(n + 127) << 23;
#if defined(__CUDA_ARCH__)
  return __uint_as_float(bits);
#else
  float f; memcpy(&f, &bits, 4); return f;
#endif
}
R2S_HD float smp_load(const float *p) {
#if defined(__CUDA_ARCH__)
  return __ldg(p);
#else
  return *p;
#endif
}

// exp(x) for x <= 0: n = round(x / ln 2) (the 1.5 * 2^23 shift rounds it inside one fma), r = x - n ln 2 in two fma steps (Cody-Waite),
// exp(r) by its degree-7 Taylor polynomial (truncation below 0.1 ulp for |r| <= ln(2) / 2), times 2^n.  0 below -87.
R2S_HD float exp_f32(float x) {
  if (!(x > -87.0f)) return 0.0f;
  const float t = fmaf(x, 1.44269504f, 12582912.0f);
  const float n = smp_sub(t, 12582912.0f);
  float r = fmaf(n, -0.693145751953125f, x);
  r = fmaf(n, -1.428606765330187e-06f, r);
  float p = 1.98412698e-4f;
  p = fmaf(p, r, 1.38888889e-3f);
  p = fmaf(p, r, 8.33333333e-3f);
  p = fmaf(p, r, 4.16666667e-2f);
  p = fmaf(p, r, 1.66666667e-1f);
  p = fmaf(p, r, 0.5f);
  p = fmaf(p, r, 1.0f);
  p = fmaf(p, r, 1.0f);
  return smp_mul(p, smp_pow2i((int)n));
}

// the coarse grid and weights a point is evaluated on; w of coarse point (i, j, k) at w[(k * ny + j) * px + i]
struct SampleGrid {
  const float *w;
  long long px, ny;
  const float *C[3];        // Float32 coordinate tables
  int n[3];                 // points per axis
  float c0[3], inv[3];      // floor estimate (p - c0) * inv, then fixed up against the table
  float kappa, t2, th;
};

// floor plane of p on one axis: the largest c with C[c] <= p, clamped to [0, n - 1].  The estimate only picks the start of the search.
R2S_HD int smp_floor(const float *C, int n, float c0, float inv, float p) {
  float q = smp_mul(smp_sub(p, c0), inv);
  q = fminf(fmaxf(q, 0.0f), (float)(n - 1));
  int c = (int)q;
  while (c > 0 && C[c] > p) c--;
  while (c < n - 1 && C[c + 1] <= p) c++;
  return c;
}

// candidates of one axis: coarse indices lo .. lo + count - 1 = [c - 2, c + 3] within the grid (|e| <= maxd < 3 cells needs no more);
// e, e^2 and the axis factor a (0 where e^2 alone exceeds t2: no tap of that index can be included)
R2S_HD int smp_axis(const SampleGrid &G, int d, float p, int *lo, float e[6], float ee[6], float a[6]) {
  const int c = smp_floor(G.C[d], G.n[d], G.c0[d], G.inv[d], p);
  const int l = c - 2 < 0 ? 0 : c - 2, h = c + 3 > G.n[d] - 1 ? G.n[d] - 1 : c + 3;
#if defined(__CUDA_ARCH__)
#pragma unroll
#endif
  for (int q = 0; q < 6; q++) {
    e[q] = 0.0f; ee[q] = INFINITY; a[q] = 0.0f;
    if (l + q <= h) {
      const float eq = smp_sub(G.C[d][l + q], p), e2 = smp_mul(eq, eq);
      e[q] = eq; ee[q] = e2;
      if (e2 <= G.t2) a[q] = exp_f32(-smp_mul(G.kappa, e2));
    }
  }
  *lo = l;
  return h - l + 1;
}

// value at p (and the gradient into grad[3] when GRAD)
template <bool GRAD>
R2S_HD float sample_point(const SampleGrid &G, float px, float py, float pz, float *grad) {
  float ex[6], exx[6], ax[6], ey[6], eyy[6], ay[6], ez[6], ezz[6], az[6];
  int ix, iy, iz;
  const int nxq = smp_axis(G, 0, px, &ix, ex, exx, ax), nyq = smp_axis(G, 1, py, &iy, ey, eyy, ay), nzq = smp_axis(G, 2, pz, &iz, ez, ezz, az);
  float acc = 0.0f, gx = 0.0f, gy = 0.0f, gz = 0.0f;
  // fixed trip counts with guards: on the device the loops unroll and the per-axis arrays stay in registers
#if defined(__CUDA_ARCH__)
#pragma unroll
#endif
  for (int qk = 0; qk < 6; qk++) {
#if defined(__CUDA_ARCH__)
#pragma unroll
#endif
    for (int qj = 0; qj < 6; qj++) {
      // d2 >= fl(e_y^2 + e_z^2) for every i (rounding is monotone), so a row above t2 holds no tap: skipping it changes no bit
      if (qk >= nzq || qj >= nyq || smp_add(eyy[qj], ezz[qk]) > G.t2) continue;
      const float *row = G.w + ((long long)(iz + qk) * G.ny + (iy + qj)) * G.px + ix;
#if defined(__CUDA_ARCH__)
#pragma unroll
#endif
      for (int qi = 0; qi < 6; qi++) {
        if (qi < nxq && smp_add(smp_add(exx[qi], eyy[qj]), ezz[qk]) <= G.t2) {
          const float phi = smp_mul(smp_mul(ax[qi], ay[qj]), az[qk]);
          const float wv = smp_load(row + qi);
          acc = fmaf(wv, phi, acc);
          if (GRAD) {
            const float wp = smp_mul(wv, phi);
            gx = fmaf(wp, ex[qi], gx); gy = fmaf(wp, ey[qj], gy); gz = fmaf(wp, ez[qk], gz);
          }
        }
      }
    }
  }
  if (GRAD) {
    const float k2 = smp_add(G.kappa, G.kappa);
    grad[0] = smp_mul(k2, gx); grad[1] = smp_mul(k2, gy); grad[2] = smp_mul(k2, gz);
  }
  return smp_add(acc, G.th);
}

// ---- host set-up, shared by the library and the host build ----------------------------------------------------------------------------
// range(Float32(a), Float32(b), length = n) with a Float64 intermediate, the last point exactly b (RBFs4Smoothing.jl:41-43)
static inline void smp_range(double amin, double amax, int n, float *out) {
  const float a = (float)amin, b = (float)amax;
  for (int i = 0; i < n; i++) out[i] = (n > 1) ? (float)((double)a + (double)i * (((double)b - (double)a) / (double)(n - 1))) : a;
  if (n > 1) out[n - 1] = b;
}
// maxd = float(sqrt(-ln(cut) cell^2)) as the reference's kernel radius (RBFs4Smoothing.jl:221); t2 = the largest float whose correctly
// rounded square root is <= maxd, so that d2 <= t2 is the reference's sqrt(d2) <= maxd without a square root
static inline float smp_maxd(double rbf_cut, double cell) { return (float)sqrt(-log(rbf_cut) * cell * cell); }
static inline float smp_t2(float maxd) {
  float t = (float)((double)maxd * (double)maxd);
  while (t > 0.0f && sqrtf(t) > maxd) t = nextafterf(t, 0.0f);
  while (sqrtf(nextafterf(t, INFINITY)) <= maxd) t = nextafterf(t, INFINITY);
  return t;
}
// the state of one smoothing result: weights w (row pitch px), host coordinate tables C (they also give the floor estimate), cell, cut, th
static inline void smp_setup(SampleGrid *G, const float *w, long long px, const float *const C[3], const int n[3], double cell, double rbf_cut, float th) {
  G->w = w; G->px = px; G->ny = n[1];
  for (int d = 0; d < 3; d++) {
    G->C[d] = C[d]; G->n[d] = n[d]; G->c0[d] = C[d][0];
    G->inv[d] = n[d] > 1 ? (float)((double)(n[d] - 1) / ((double)C[d][n[d] - 1] - (double)C[d][0])) : 0.0f;
  }
  G->kappa = (float)(1.0 / (cell * cell));
  G->t2 = smp_t2(smp_maxd(rbf_cut, cell));
  G->th = th;
}
