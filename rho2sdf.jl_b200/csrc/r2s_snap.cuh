// r2s_snap.cuh -- the vertex of a lattice edge on the zero set of the continuous field (r2s_isosurface_lattice, r2s_surf.cu): a
// deterministic bracketing search over the Float32 values of the edge, shared by the snapping kernel and the host build
// (tests/host/snap_host.cpp, g++ -ffp-contract=off).  The rule, exactly (include/r2s.h states it too):
//
//   The edge runs from lattice point a (coordinate x_a on its axis, value va) to b (x_b, vb); s(x) = (f(x) >= iso), s(a) != s(b).
//   Bracket (lo, hi) = (x_a, x_b) with flo = va, fhi = vb (the lattice values: no re-evaluation), Illinois residuals
//   glo = double(va) - double(iso), ghi = double(vb) - double(iso), last = none.  Float x is mapped to an order-preserving 32-bit key
//   (snap_key: -inf < ... < -0 < +0 < ... < +inf).  Loop:
//     1. stop if |key(lo) - key(hi)| <= 1 (adjacent floats, or equal) or R2S_SNAP_MAX_EVALS evaluations have been made;
//     2. t = glo / (glo - ghi), xd = lo + (hi - lo) * t, every operation a rounded double operation (no contraction); x = float(xd);
//        if key(x) is not strictly between key(lo) and key(hi), x = the float of key m = kmin + (kmax - kmin) / 2 (unsigned, truncated);
//     3. fx = f(x) (one evaluation); r = double(fx) - double(iso);
//        s(x) == s(a): lo = x, flo = fx, glo = r, and ghi = ghi * 0.5 if the previous step also replaced lo; last = lo;
//        otherwise:    hi = x, fhi = fx, ghi = r, and glo = glo * 0.5 if the previous step also replaced hi; last = hi.
//   Result: hi if |double(fhi) - double(iso)| < |double(flo) - double(iso)|, else lo (ties go to lo).
// The result is lo or hi, so it lies in [x_a, x_b] (closed), on the vertex's own edge; the invariant s(lo) = s(a), s(hi) = s(b) holds
// at every step, so at a stop by adjacency lo and hi are neighbouring floats that straddle iso under the inside rule.
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

#define R2S_SNAP_MAX_EVALS 48      // evaluation cap of one edge: bisection alone needs at most 32 steps between any two floats

R2S_HD uint32_t snap_key(float x) {
  uint32_t u;
#if defined(__CUDA_ARCH__)
  u = __float_as_uint(x);
#else
  memcpy(&u, &x, 4);
#endif
  return (u & 0x80000000u) ? ~u : (u | 0x80000000u);
}
R2S_HD float snap_unkey(uint32_t k) {
  const uint32_t u = (k & 0x80000000u) ? (k & 0x7fffffffu) : ~k;
#if defined(__CUDA_ARCH__)
  return __uint_as_float(u);
#else
  float x; memcpy(&x, &u, 4); return x;
#endif
}
R2S_HD double snap_dadd(double a, double b) {
#if defined(__CUDA_ARCH__)
  return __dadd_rn(a, b);
#else
  return a + b;
#endif
}
R2S_HD double snap_dsub(double a, double b) {
#if defined(__CUDA_ARCH__)
  return __dsub_rn(a, b);
#else
  return a - b;
#endif
}
R2S_HD double snap_dmul(double a, double b) {
#if defined(__CUDA_ARCH__)
  return __dmul_rn(a, b);
#else
  return a * b;
#endif
}
R2S_HD double snap_ddiv(double a, double b) {
#if defined(__CUDA_ARCH__)
  return __ddiv_rn(a, b);
#else
  return a / b;
#endif
}

// the final bracket of one search (for the host tests; the kernel ignores it)
struct SnapTrace { float lo, hi, flo, fhi; int evals; };

// the search above; f(x) evaluates the field at axis coordinate x (the other two coordinates are the edge's)
template <class F>
R2S_HD float snap_search(const F &f, float xa, float xb, float va, float vb, float iso, SnapTrace *tr) {
  const bool sa = va >= iso;
  float lo = xa, hi = xb, flo = va, fhi = vb;
  double glo = snap_dsub((double)va, (double)iso), ghi = snap_dsub((double)vb, (double)iso);
  uint32_t klo = snap_key(lo), khi = snap_key(hi);
  int last = 0, n = 0;      // last: 1 = the previous step replaced lo, 2 = it replaced hi
  while (n < R2S_SNAP_MAX_EVALS) {
    const uint32_t kmin = klo < khi ? klo : khi, kmax = klo < khi ? khi : klo;
    if (kmax - kmin <= 1u) break;
    const double t = snap_ddiv(glo, snap_dsub(glo, ghi));
    float x = (float)snap_dadd((double)lo, snap_dmul(snap_dsub((double)hi, (double)lo), t));
    uint32_t kx = snap_key(x);
    if (!(kx > kmin && kx < kmax)) { kx = kmin + (kmax - kmin) / 2u; x = snap_unkey(kx); }
    const float fx = f(x);
    const double r = snap_dsub((double)fx, (double)iso);
    n++;
    if ((fx >= iso) == sa) {
      lo = x; flo = fx; glo = r; klo = kx;
      if (last == 1) ghi = snap_dmul(ghi, 0.5);
      last = 1;
    } else {
      hi = x; fhi = fx; ghi = r; khi = kx;
      if (last == 2) glo = snap_dmul(glo, 0.5);
      last = 2;
    }
  }
  if (tr) { tr->lo = lo; tr->hi = hi; tr->flo = flo; tr->fhi = fhi; tr->evals = n; }
  return fabs(snap_dsub((double)fhi, (double)iso)) < fabs(snap_dsub((double)flo, (double)iso)) ? hi : lo;
}
