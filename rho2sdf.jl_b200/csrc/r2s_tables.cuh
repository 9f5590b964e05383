// r2s_tables.cuh -- element topology (ElementTypes/ElementTypes.jl:15-78, 0-based), Gauss-Legendre tables and the HEX8 shape functions.
// The device tables are CUDA-only; the rest also compiles for the host (tests/host/elemfrac_host.cpp).
#pragma once
#include <math.h>

#ifndef R2S_HD
#if defined(__CUDACC__)
#define R2S_HD __host__ __device__ __forceinline__
#else
#define R2S_HD inline
#endif
#endif

#if defined(__CUDACC__)
// face -> local nodes (ISN)
static __constant__ int c_hex_isn[6][4] = {{0, 3, 2, 1}, {0, 1, 5, 4}, {1, 2, 6, 5}, {2, 3, 7, 6}, {3, 0, 4, 7}, {4, 5, 6, 7}};
static __constant__ int c_tet_isn[4][3] = {{0, 2, 1}, {0, 1, 3}, {1, 2, 3}, {0, 3, 2}};
// natural coordinates of the HEX8 nodes (hex8_shape.jl:27-34)
static __constant__ double c_hex_sg[8][3] = {{-1, -1, -1}, {1, -1, -1}, {1, 1, -1}, {-1, 1, -1}, {-1, -1, 1}, {1, -1, 1}, {1, 1, 1}, {-1, 1, 1}};
static __constant__ int c_hex_edges[12][2] = {{0, 1}, {1, 2}, {2, 3}, {3, 0}, {4, 5}, {5, 6}, {6, 7}, {7, 4}, {0, 4}, {1, 5}, {2, 6}, {3, 7}};
#endif

// Gauss-Legendre rule of order n (what FastGaussQuadrature.gausslegendre(n) returns): Newton on P_n in long double,
// nodes ascending, symmetrised.  Host side; the tables travel to kernels by value.
struct GaussTab { double x[32]; double w[32]; int n; };      // orders up to 32 (the reference uses 3, 9, 15 and, in its convergence tests, 20)
static inline GaussTab gauss_legendre_host(int n) {
  GaussTab t; t.n = n;
  for (int i = 0; i < n; i++) {
    long double z = cosl(3.14159265358979323846264338327950288L * (i + 0.75L) / (n + 0.5L)), pp = 0;
    for (int it = 0; it < 100; it++) {
      long double p1 = 1, p2 = 0;
      for (int j = 0; j < n; j++) { long double p3 = p2; p2 = p1; p1 = ((2 * j + 1) * z * p2 - j * p3) / (j + 1); }
      pp = n * (z * p1 - p2) / (z * z - 1);
      long double dz = p1 / pp; z -= dz;
      if (fabsl(dz) < 1e-19L) break;
    }
    long double p1 = 1, p2 = 0;
    for (int j = 0; j < n; j++) { long double p3 = p2; p2 = p1; p1 = ((2 * j + 1) * z * p2 - j * p3) / (j + 1); }
    pp = n * (z * p1 - p2) / (z * z - 1);
    t.x[n - 1 - i] = (double)z; t.w[n - 1 - i] = (double)(2 / ((1 - z * z) * pp * pp));
  }
  for (int i = 0; i < n / 2; i++) {
    double a = 0.5 * (t.x[n - 1 - i] - t.x[i]); t.x[i] = -a; t.x[n - 1 - i] = a;
    double b = 0.5 * (t.w[i] + t.w[n - 1 - i]); t.w[i] = b; t.w[n - 1 - i] = b;
  }
  if (n & 1) t.x[n / 2] = 0.0;
  return t;
}

// shape functions in the reference's form (ShapeFunctions/hex8_shape.jl:2-70).  Callers compile them without contraction (-fmad=false,
// host -ffp-contract=off): calculate_mesh_volume (r2s_mesh.cu) and the element volume fractions (r2s_elemfrac.cuh) share their bits.
R2S_HD void hex8_shape_d(const double xi[3], double N[8], double dN[8][3]) {
  double m1 = xi[0] - 1, p1 = xi[0] + 1, m2 = xi[1] - 1, p2 = xi[1] + 1, m3 = xi[2] - 1, p3 = xi[2] + 1;
  double t1 = m1 * m2, t2 = p1 * m2, t3 = p1 * p2, t4 = m1 * p2, c = 0.125;
  N[0] = -c * t1 * m3; N[1] = c * t2 * m3; N[2] = -c * t3 * m3; N[3] = c * t4 * m3;
  N[4] = c * t1 * p3;  N[5] = -c * t2 * p3; N[6] = c * t3 * p3; N[7] = -c * t4 * p3;
  double d = c * m3, dp = c * p3;
  dN[0][0] = -d * m2; dN[1][0] = d * m2; dN[2][0] = -d * p2; dN[3][0] = d * p2;
  dN[4][0] = dp * m2; dN[5][0] = -dp * m2; dN[6][0] = dp * p2; dN[7][0] = -dp * p2;
  dN[0][1] = -d * m1; dN[1][1] = d * p1; dN[2][1] = -d * p1; dN[3][1] = d * m1;
  dN[4][1] = dp * m1; dN[5][1] = -dp * p1; dN[6][1] = dp * p1; dN[7][1] = -dp * m1;
  dN[0][2] = -c * t1; dN[1][2] = c * t2; dN[2][2] = -c * t3; dN[3][2] = c * t4;
  dN[4][2] = c * t1;  dN[5][2] = -c * t2; dN[6][2] = c * t3;  dN[7][2] = -c * t4;
}
R2S_HD double det3(const double J[3][3]) {
  return J[0][0] * (J[1][1] * J[2][2] - J[1][2] * J[2][1]) - J[0][1] * (J[1][0] * J[2][2] - J[1][2] * J[2][0]) +
         J[0][2] * (J[1][0] * J[2][1] - J[1][1] * J[2][0]);
}
