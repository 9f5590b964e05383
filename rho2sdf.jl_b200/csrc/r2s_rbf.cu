// r2s_rbf.cu -- RBFs_smoothing (SdfSmoothing/RBFs4Smoothing.jl:321-377) and calculate_volume_from_sdf
// (SdfSmoothing/CalcVolumeFromSDF.jl:26-125) on the GPU, Float32 like the reference.
//
// On the regular SDF grid the truncated Gaussian kernel matrix K (:142-176, sigma = cell, cut 1e-3) is an 81-point
// stencil (offsets with |d|^2 <= 6, weights exp(-|d|^2)); the KD-tree / sparse-matrix machinery of the reference becomes
//   * a shared-memory tiled stencil mat-vec fused with the CG vector updates and dot products (HBM-bound),
//   * an 8-phase polyphase stencil for the evaluation on the :fine grid (taps with |d|^2 <= ln(1000) in half cells),
//   * a two-pass cut-cell quadrature for the volume-matching bisection (LS_Threshold, :265-300).
// Sums are deterministic: block partials in fixed slots (double) or fixed-point integer atomics (vol_cell_add, r2s_volq.cuh).
#include <float.h>
#include <stdlib.h>
#include <algorithm>
#include <cuda.h>
#include "r2s_common.cuh"
#include "r2s_tables.cuh"
#include "r2s_p2p.cuh"
#include "r2s_volq.cuh"

// ------------------------------------------------------------------------------------------------ process_vector (:15-22)
__global__ void __launch_bounds__(256) k_to_f32(i64 n, i64 v0, int nx, int px, const double *__restrict__ sdf, float *__restrict__ s, unsigned *__restrict__ maxbits) {
  // sdf: rows of nx doubles; s: rows of px >= nx floats (the pad stays zero).  n values starting at the unpadded offset v0 (a multiple of nx).
  __shared__ float red[8];
  float a = -1.0f;
  const i64 row0 = v0 / nx;
  for (i64 v = blockIdx.x * (i64)blockDim.x + threadIdx.x; v < n; v += (i64)gridDim.x * blockDim.x) {
    const i64 row = v / nx; const int i = (int)(v - row * nx);
    float f = (float)sdf[v0 + v]; s[(row0 + row) * px + i] = f; float af = fabsf(f); if (af < 1.0e9f) a = fmaxf(a, af);
  }
  for (int o = 16; o > 0; o >>= 1) a = fmaxf(a, __shfl_down_sync(0xffffffffu, a, o));
  if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = a;
  __syncthreads();
  if (threadIdx.x == 0) {
    for (int i = 1; i < 8; i++) a = fmaxf(a, red[i]);
    if (a >= 0.0f) atomicMax(maxbits, __float_as_uint(a) + 1u);   // +1 so that "found 0.0" differs from "none"; one atomic per CTA
  }
}
__global__ void k_replace_far(i64 n, float *__restrict__ s, const unsigned *__restrict__ maxbits) {
  i64 v = blockIdx.x * (i64)blockDim.x + threadIdx.x;
  if (v >= n) return;
  float maxv = __uint_as_float(*maxbits - 1u);
  float f = s[v], a = fabsf(f); const float big = 1.0e10f, rt = sqrtf(FLT_EPSILON);
  if (fabsf(a - big) <= rt * fmaxf(a, big)) s[v] = (f > 0 ? 1.0f : (f < 0 ? -1.0f : 0.0f)) * maxv;    // isapprox(|v|, 1f10), default rtol
}

// ------------------------------------------------------------------------------------------------ 81-point stencil
// weights by squared offset m = di^2+dj^2+dk^2 <= 6
struct StencilW { float w[8]; };
// The CTA that finishes LAST adds up the per-CTA partial sums (fixed order: 256 strided sums, then slot 0..255 sequentially -- the same
// order whatever CTA happens to be last, so the result is deterministic) and stores the total: no separate reduction launch.
// Call with all threads of the CTA after thread 0 has written partial[this CTA].
// F.enabled (several GPUs, peer-memory transport): the CTAs have also stored halo values into the neighbours' arrays, so the fence before
// the ticket is system-wide, and the last CTA all-reduces the total over the ranks through the mailbox itself (p2p_allreduce_cta).
__device__ __forceinline__ bool cta_sum_last(const double *partial, int nblocks, unsigned *ticket, double *dst, const P2PFuse &F) {
  __shared__ bool s_last; __shared__ double s_sum[256];
  const int tid = threadIdx.x;
  if (F.enabled) { __threadfence_system(); __syncthreads(); }
  if (tid == 0) { __threadfence(); s_last = atomicAdd(ticket, 1u) == (unsigned)nblocks - 1u; }
  __syncthreads();
  if (!s_last) return false;
  __threadfence();
  for (int v = tid; v < 256; v += (int)blockDim.x) {      // 256 strided sums whatever the block size
    double a = 0; for (int i = v; i < nblocks; i += 256) a += __ldcg(&partial[i]);
    s_sum[v] = a;
  }
  __syncthreads();
  __shared__ double s_tot;
  if (tid == 0) { double t = 0; for (int i = 0; i < 256; i++) t += s_sum[i]; s_tot = t; *ticket = 0; }
  __syncthreads();
  double t = s_tot;                                          // every thread holds the local total: thread p sends it to rank p
  if (F.enabled) t = p2p_allreduce_cta(F, F.seq_ar, t);
  if (tid == 0) { *dst = t; __threadfence(); }
  __syncthreads();
  return true;
}
// ---- plane marching (2.5-D blocking) with TMA-staged planes, two outputs per thread ------------------------------------------------
// A CTA owns a 32 x 16 column of the grid and marches along z over zc output planes.  Each input plane tile (40 x 20 floats with its
// x-y halo) is brought into shared memory by ONE bulk tensor copy (cp.async.bulk.tensor.3d, TMA) issued by one thread NST - 1 planes
// ahead and signalled through an mbarrier: no per-thread address arithmetic, no bounds tests (coordinates outside the grid are
// zero-filled by the TMA unit -- K has no entries there), loads in flight for several planes.  The fields are stored with a row pitch
// that is a multiple of 4 floats (TMA needs 16-byte global strides); the tensor map carries the logical extent nx.
// CG form (BETA): the stencil input is u_new = r + beta * u_old; the r and u_old tiles arrive by TMA, the threads combine them into a
// second shared buffer and write the interior back to u_new (separate array: other CTAs still read u_old for their halos).
// A thread owns two x-adjacent columns: the six row values it needs come in as three 8-byte shared-memory loads and serve both
// outputs.  The tap weight depends on the squared distance only and w[m] = exp(-m), so w[m2 + dz^2] = w[m2] * w[dz^2]: the in-plane
// sums S9 (taps with m2 <= 2) and S21 = S9 + S12 (all 21 in-plane taps) are formed once per input plane and enter the five output
// planes (rotating register queue) as a2 += S21, a1/a3 += w[1] S21, a0/a4 += w[4] S9 -- 27 FMA-pipe operations per column and plane
// instead of 81.  The products w[m2] * w[dz^2] differ from float(exp(-(m2 + dz^2))) by Float32 round-off (mat-vec 4e-7 relative; CG
// iteration counts and weights equal to the oracle's, tests/test_gpu_parity.py).
#define S3_X 32            // outputs per CTA in x (16 threads x 2)
#define S3_Y 16
#define S3_HX 4            // x halo of the TILE: the stencil needs 2, but the innermost TMA coordinate must be a multiple of 16 bytes (4 floats):
                           // a box starting at bx - 2 raises "illegal instruction" on B200 (tools/probes/tma_probe.cu), bx - 4 is fine
#define S3_TX (S3_X + 2 * S3_HX)   // 40 x 20 tile; 40 floats = 160 B per row (a multiple of 16 B, as the TMA box requires)
#define S3_TY (S3_Y + 4)
#ifndef S3_NST
#define S3_NST 4           // TMA stages: loads run 3 planes ahead of the compute
#endif
#define S3_TILE_BYTES (S3_TX * S3_TY * 4)
#define S3_SLOT 3200       // stage stride in shared memory (= tile bytes, a multiple of 128: destinations are 128-byte aligned)
__device__ __forceinline__ unsigned smem_u32(const void *p) { return (unsigned)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void mbar_init(unsigned long long *bar, unsigned count) { asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count)); }
// bar / dst are shared-window addresses (smem_u32), taken once per kernel: the generic -> shared conversion per use was 5 % of the stencil kernel's instructions
__device__ __forceinline__ void mbar_expect_tx(unsigned bar, unsigned bytes) { asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(bytes) : "memory"); }
__device__ __forceinline__ void mbar_wait(unsigned bar, unsigned parity) {
  asm volatile("{\n .reg .pred p;\n WAIT_%=:\n mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n @p bra DONE_%=;\n bra WAIT_%=;\n DONE_%=:\n}" ::"r"(bar), "r"(parity) : "memory");
}
__device__ __forceinline__ void tma_load_3d(unsigned dst, const CUtensorMap *map, int c0, int c1, int c2, unsigned bar) {
  asm volatile("cp.async.bulk.tensor.3d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%2, %3, %4}], [%5];" ::"r"(dst), "l"(map), "r"(c0), "r"(c1),
               "r"(c2), "r"(bar)
               : "memory");
}
// packed FP32 FMA (FFMA2 on sm_100a): IEEE fma per half, i.e. the same bits as two scalar FMAs, in ONE issue slot.  tools/probes/ffma2_probe.cu:
// the same flop rate as FFMA (72.9 vs 71.7 TFLOP/s) -- it helps kernels that are bound by instruction issue (k_fine_eval2: 6.97 -> 5.73 ms),
// not the stencil (LDS / barrier bound: no change measured)
#ifndef R2S_F32X2
#define R2S_F32X2 1
#endif
__device__ __forceinline__ float2 ffma2(float2 a, float2 b, float2 c) {
  unsigned long long xa = *reinterpret_cast<unsigned long long *>(&a), xb = *reinterpret_cast<unsigned long long *>(&b), xc = *reinterpret_cast<unsigned long long *>(&c), r;
  asm("fma.rn.f32x2 %0, %1, %2, %3;" : "=l"(r) : "l"(xa), "l"(xb), "l"(xc));
  return *reinterpret_cast<float2 *>(&r);
}
#ifndef R2S_ST_NO
#define R2S_ST_NO 4        // x-adjacent outputs per thread of the stencil kernel (2 or 4): 4 = 128 threads per CTA, 40 B of shared-memory loads per output instead of 60
#endif
template <bool BETA, int NO>
__global__ void __launch_bounds__(16 * S3_X / NO) k_stencil81_tma(const __grid_constant__ CUtensorMap mapA, const __grid_constant__ CUtensorMap mapB, int nx, int ny, int nz, int px,
                                                                   int kz0, int kz1, int zc, float *__restrict__ unew, const float *__restrict__ scal, float *__restrict__ out,
                                                                   double *__restrict__ partial, StencilW W, unsigned *__restrict__ ticket, double *__restrict__ dot_out, const P2PFuse F) {
  static_assert(NO == 2 || NO == 4, "outputs per thread");
  constexpr int TX = S3_TX, TY = S3_TY, NT = TX * TY, NARR = BETA ? 2 : 1, NTHR = 16 * S3_X / NO, NV = NO + 4;
  if (BETA && scal[5] != 0.0f) return;      // CG has converged: the iterations launched ahead of the host's check are no-ops
  __shared__ __align__(128) unsigned char stage[S3_NST * NARR * S3_SLOT];
  __shared__ __align__(16) float comb[BETA ? 2 : 1][BETA ? NT : 4];      // combined plane r + beta * u (double buffered), CG form only
  __shared__ __align__(8) unsigned long long full[S3_NST];
  __shared__ double red[8];
  const int tid = threadIdx.x, tx = tid % (S3_X / NO), ty = tid / (S3_X / NO);
  const int bx = blockIdx.x * S3_X, by = blockIdx.y * S3_Y;
  const int zc0 = kz0 + blockIdx.z * zc, zc1 = min(zc0 + zc, kz1);      // zc output planes per CTA (chosen by the host so that the chunks are even)
  const int np = zc1 - zc0 + 4;                                           // input planes zc0 - 2 .. zc1 + 1
  // NO == 4: the CTA's outputs are the columns [bx - 2, bx + 30), so that the eight values a thread needs per row (x0 - 2 .. x0 + 5) are two
  // ALIGNED 16-byte shared-memory loads (tile column 4 tx .. 4 tx + 7) -- the kernel is bound by shared-memory wavefronts (ncu: l1tex 87 %),
  // and an unaligned 8 + 16 + 8 byte split costs 12 wavefronts per warp and row instead of 8.  The grid has cdiv(nx + 2, 32) columns.
  constexpr int XS = NO == 4 ? 2 : 0;
  const int gx = bx - XS + NO * tx, gy = by + ty;
  bool in[NO];
#pragma unroll
  for (int o = 0; o < NO; o++) in[o] = gx + o >= 0 && gx + o < nx && gy < ny;
  float beta = 0.0f;
  if (BETA) beta = scal[0];
  if (tid == 0) {
#pragma unroll
    for (int q = 0; q < S3_NST; q++) mbar_init(&full[q], 1);
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  __syncthreads();
  const unsigned stage_a = smem_u32(stage), full_a = smem_u32(full);
  auto issue = [&](int p) {      // thread 0: plane p of this CTA's march into stage p % NST
    const int st = p % S3_NST;
    mbar_expect_tx(full_a + 8 * st, S3_TILE_BYTES * NARR);
    tma_load_3d(stage_a + (st * NARR) * S3_SLOT, &mapA, bx - S3_HX, by - 2, zc0 - 2 + p, full_a + 8 * st);
    if (BETA) tma_load_3d(stage_a + (st * NARR + 1) * S3_SLOT, &mapB, bx - S3_HX, by - 2, zc0 - 2 + p, full_a + 8 * st);
  };
  if (tid == 0) for (int p = 0; p < S3_NST - 1 && p < np; p++) issue(p);
  // CG form: the threads combine the tile float4 by float4 (16-byte shared loads / stores); a float4 of the tile interior is also written
  // back to u_new with one 16-byte store (x is a multiple of 4, the row pitch too; values beyond nx are the TMA's zero fill and land in
  // the zero pad columns)
  static_assert(NT % 4 == 0 && S3_TX % 4 == 0 && S3_HX % 4 == 0, "float4 combine");
  constexpr int NC = (NT / 4 + NTHR - 1) / NTHR;
  bool c_act[NC], c_int[NC]; i64 c_off[NC];
#pragma unroll
  for (int q = 0; q < NC; q++) {
    c_act[q] = false; c_int[q] = false; c_off[q] = 0;
    if (BETA) {
      const int t4 = tid + q * NTHR, t = 4 * t4, ly = t / TX, lx = t % TX, x = bx + lx - S3_HX, y = by + ly - 2;
      c_act[q] = t4 < NT / 4;
      c_int[q] = c_act[q] && lx >= S3_HX && lx < TX - S3_HX && ly >= 2 && ly < TY - 2 && x < nx && y < ny;
      c_off[q] = (i64)y * px + x;
    }
  }
  const i64 pl = (i64)px * ny;
  float acc[5][NO], ctr0[NO], ctr1[NO];      // acc[q][o]: output plane (current input plane - 2 + q) of column o; ctr: centre values (= u) of the two planes before
#pragma unroll
  for (int o = 0; o < NO; o++) { ctr0[o] = ctr1[o] = 0.f; for (int q = 0; q < 5; q++) acc[q][o] = 0.f; }
  double dsum = 0.0;
  for (int p = 0; p < np; p++) {
    const int st = p % S3_NST, zin = zc0 - 2 + p;
    // the stage that plane p + NST - 1 goes into was read during iteration p - 1; everybody has passed that iteration's barrier
    if (tid == 0 && p + S3_NST - 1 < np) issue(p + S3_NST - 1);
    mbar_wait(full_a + 8 * st, (unsigned)((p / S3_NST) & 1));
    const float *tile;
    if (BETA) {
      const float *tr = reinterpret_cast<const float *>(stage + (st * NARR) * S3_SLOT), *tu = reinterpret_cast<const float *>(stage + (st * NARR + 1) * S3_SLOT);
      float *cb = comb[p & 1];
#pragma unroll
      for (int q = 0; q < NC; q++)
        if (c_act[q]) {
          const int t4 = tid + q * NTHR;
          const float4 a = reinterpret_cast<const float4 *>(tr)[t4], b = reinterpret_cast<const float4 *>(tu)[t4];
          float4 v; v.x = a.x + beta * b.x; v.y = a.y + beta * b.y; v.z = a.z + beta * b.z; v.w = a.w + beta * b.w;
          reinterpret_cast<float4 *>(cb)[t4] = v;
          if (c_int[q] && zin >= zc0 && zin < zc1) *reinterpret_cast<float4 *>(unew + (i64)zin * pl + c_off[q]) = v;
        }
      __syncthreads();      // comb[p & 1] complete; also: every thread is done with the raw stage of plane p and with comb[(p + 1) & 1] of plane p - 1
      tile = cb;
    } else {
      tile = reinterpret_cast<const float *>(stage + st * S3_SLOT);
    }
    float ctr[NO], s9[NO], s12[NO];
#pragma unroll
    for (int o = 0; o < NO; o++) { ctr[o] = 0.f; s9[o] = 0.f; s12[o] = 0.f; }
#pragma unroll
    for (int dj = -2; dj <= 2; dj++) {
      const float *rowp = tile + (ty + 2 + dj) * TX + NO * tx + (S3_HX - 2 - XS);      // x0 - 2 .. x0 + NO + 1
      float v[NV];
      if (NO == 2) {
        const float2 *row = reinterpret_cast<const float2 *>(rowp);
        const float2 p0 = row[0], p1 = row[1], p2 = row[2];
        v[0] = p0.x; v[1] = p0.y; v[2] = p1.x; v[3] = p1.y; v[4] = p2.x; v[5] = p2.y;
      } else {
        const float4 p0 = *reinterpret_cast<const float4 *>(rowp), p1 = *reinterpret_cast<const float4 *>(rowp + 4);
        v[0] = p0.x; v[1] = p0.y; v[2] = p0.z; v[3] = p0.w; v[NV - 4] = p1.x; v[NV - 3] = p1.y; v[NV - 2] = p1.z; v[NV - 1] = p1.w;
      }
      if (dj == 0) {
#pragma unroll
        for (int o = 0; o < NO; o++) ctr[o] = v[2 + o];
      }
#pragma unroll
      for (int di = -2; di <= 2; di++) {
        const int m2 = di * di + dj * dj;
        if (m2 > 6) continue;
#pragma unroll
        for (int o = 0; o < NO; o++) {
          if (m2 <= 2) s9[o] = fmaf(W.w[m2], v[di + 2 + o], s9[o]); else s12[o] = fmaf(W.w[m2], v[di + 2 + o], s12[o]);
        }
      }
    }
    {
      const float e1 = W.w[1], e4 = W.w[4];
#pragma unroll
      for (int o = 0; o < NO; o++) {
        const float s21 = s9[o] + s12[o];
        acc[2][o] += s21; acc[1][o] = fmaf(e1, s21, acc[1][o]); acc[3][o] = fmaf(e1, s21, acc[3][o]); acc[0][o] = fmaf(e4, s9[o], acc[0][o]); acc[4][o] = fmaf(e4, s9[o], acc[4][o]);
      }
    }
    const int zo = zin - 2;
    if (zo >= zc0) {
      const i64 gi = (i64)zo * pl + (i64)gy * px + gx;
      const bool vec = NO == 4 && in[0] && in[NO - 1];      // gx is even and the row pitch a multiple of 4: 8-byte stores
      if (vec) { *reinterpret_cast<float2 *>(out + gi) = make_float2(acc[0][0], acc[0][1]); *reinterpret_cast<float2 *>(out + gi + 2) = make_float2(acc[0][2], acc[0][NO - 1]); }
#pragma unroll
      for (int o = 0; o < NO; o++)
        if (in[o]) { if (!vec) out[gi + o] = acc[0][o]; dsum += (double)ctr0[o] * (double)acc[0][o]; }
      if (BETA && F.enabled) {      // fused halo exchange: my boundary planes of c go straight into the neighbours' arrays over NVLink
#pragma unroll
        for (int o = 0; o < NO; o++) {      // per OUTPUT: gi itself may lie two columns left of the row (gx = -2 in the first CTA column)
          if (gi + o >= F.lo0 && gi + o < F.lo1 && in[o]) F.c_lower[gi + o] = acc[0][o];
          if (gi + o >= F.hi0 && gi + o < F.hi1 && in[o]) F.c_upper[gi + o] = acc[0][o];
        }
      }
    }
#pragma unroll
    for (int o = 0; o < NO; o++) {
      acc[0][o] = acc[1][o]; acc[1][o] = acc[2][o]; acc[2][o] = acc[3][o]; acc[3][o] = acc[4][o]; acc[4][o] = 0.f;
      ctr0[o] = ctr1[o]; ctr1[o] = ctr[o];
    }
    if (!BETA) __syncthreads();      // the stage of plane p may be overwritten by the load issued at the top of the next iteration
  }
  for (int o = 16; o > 0; o >>= 1) dsum += __shfl_down_sync(0xffffffffu, dsum, o);
  if ((tid & 31) == 0) red[tid >> 5] = dsum;
  __syncthreads();
  if (tid == 0) {
    double a = 0; for (int i = 0; i < NTHR / 32; i++) a += red[i];
    partial[(blockIdx.z * gridDim.y + blockIdx.y) * gridDim.x + blockIdx.x] = a;
  }
  if (ticket && cta_sum_last(partial, (int)(gridDim.x * gridDim.y * gridDim.z), ticket, dot_out, F) && F.enabled && tid == 0)
    p2p_raise_halo_flags(F);      // every CTA fenced its remote stores before its ticket: the neighbours may read their halos now
}
// tensor map of a coarse Float32 field (nx x ny x nz values, row pitch px floats) with the 40 x 20 x 1 box of the stencil tiles
typedef CUresult (*tmap_encode_fn)(CUtensorMap *, CUtensorMapDataType, cuuint32_t, void *, const cuuint64_t *, const cuuint64_t *, const cuuint32_t *, const cuuint32_t *,
                                   CUtensorMapInterleave, CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);
static int stencil_tensor_map(r2s_ctx *ctx, CUtensorMap *map, const float *base, int nx, int ny, int nz, int px) {
  static tmap_encode_fn encode = nullptr;
  if (!encode) {
    void *fn = nullptr; cudaDriverEntryPointQueryResult qres;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &fn, cudaEnableDefault, &qres) != cudaSuccess || qres != cudaDriverEntryPointSuccess || !fn)
      FAIL("cuTensorMapEncodeTiled is not available in this driver (TMA-staged stencil needs CUDA 12 on sm_90+)");
    encode = (tmap_encode_fn)fn;
  }
  const cuuint64_t gdim[3] = {(cuuint64_t)nx, (cuuint64_t)ny, (cuuint64_t)nz}, gstr[2] = {(cuuint64_t)px * 4, (cuuint64_t)px * ny * 4};
  const cuuint32_t box[3] = {S3_TX, S3_TY, 1}, estr[3] = {1, 1, 1};
  const CUresult rc = encode(map, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 3, (void *)base, gdim, gstr, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_NONE,
                             CU_TENSOR_MAP_L2_PROMOTION_L2_128B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (rc != CUDA_SUCCESS) { char b[96]; snprintf(b, sizeof(b), "cuTensorMapEncodeTiled failed (CUresult %d)", (int)rc); FAIL(b); }
  return 0;
}
// CG scalar bookkeeping (IterativeSolvers.cg, CGIterable): scal = {beta, alpha, residual, prev_residual, tol, converged flag, iterations, initial residual}
__global__ void k_sum_to(const double *__restrict__ part, int n, double *__restrict__ dst) {
  __shared__ double sh[256];
  double a = 0; for (int i = threadIdx.x; i < n; i += 256) a += part[i];
  sh[threadIdx.x] = a; __syncthreads();
  if (threadIdx.x == 0) { double s = 0; for (int i = 0; i < 256; i++) s += sh[i]; *dst = s; }
}
// elementwise over [0, n) (owned planes plus halo); the residual norm is summed over the owned part [o_lo, o_hi) only.
// Grid-stride with a fixed grid (CG_BLOCKS CTAs): few, fat CTAs keep the loads in flight and leave only CG_BLOCKS partial sums.
// alpha = residual^2 / dot(u, c) is formed by every thread from the (all-reduced) dot product; the last CTA adds up the partial sums of
// |r|^2 and, on a single rank (finalize), closes the iteration: residual, beta, iteration count, convergence flag.
#define CG_BLOCKS (148 * 8)
__device__ __forceinline__ void cg_close_iteration(float *scal, double rr) {      // prev = residual; residual = norm(r); beta for the next iteration (IterativeSolvers CGIterable)
  const float prev = scal[2], res = (float)sqrt(rr);
  scal[3] = prev; scal[2] = res; scal[0] = res * res / (prev * prev);
  scal[6] += 1.0f;
  if (res <= scal[4]) scal[5] = 1.0f;
  else if (!(res < 1.0e8f * scal[7])) scal[5] = 2.0f;      // NaN / Inf residual, or one that has grown by 10^8 (bad input or a failed exchange -- CG on an SPD system does not do that): stop instead of iterating to maxiter = n
}
__global__ void __launch_bounds__(256) k_cg_update(i64 n, i64 o_lo, i64 o_hi, float *__restrict__ scal, const double *__restrict__ uc, const float *__restrict__ u,
                                                   const float *__restrict__ c, float *__restrict__ x, float *__restrict__ r, double *__restrict__ partial, unsigned *__restrict__ ticket,
                                                   double *__restrict__ rr_out, int finalize, const P2PFuse F) {
  __shared__ double red[8];
  if (scal[5] != 0.0f) return;
  if (F.enabled) {      // the halo planes of c are written by the neighbours' mat-vec kernels: wait for their flags of this iteration
    if (threadIdx.x == 0) p2p_wait_halo_flags(F);
    __syncthreads();
  }
  const float res0 = scal[2], alpha = res0 * res0 / (float)(*uc); double rr = 0.0;
  const i64 stride = (i64)gridDim.x * blockDim.x;
  for (i64 v = blockIdx.x * (i64)blockDim.x + threadIdx.x; v < n; v += 4 * stride) {       // 4 independent elements per trip: 16 loads in flight
    float xv[4], uv[4], rv[4], cv[4];
#pragma unroll
    for (int q = 0; q < 4; q++) { i64 w = v + q * stride; if (w < n) { xv[q] = x[w]; uv[q] = u[w]; rv[q] = r[w]; cv[q] = c[w]; } }
#pragma unroll
    for (int q = 0; q < 4; q++) {
      i64 w = v + q * stride;
      if (w < n) { x[w] = xv[q] + alpha * uv[q]; float t = rv[q] - alpha * cv[q]; r[w] = t; if (w >= o_lo && w < o_hi) rr += (double)t * (double)t; }
    }
  }
  for (int o = 16; o > 0; o >>= 1) rr += __shfl_down_sync(0xffffffffu, rr, o);
  if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = rr;
  __syncthreads();
  if (threadIdx.x == 0) { double a = 0; for (int i = 0; i < (int)(blockDim.x >> 5); i++) a += red[i]; partial[blockIdx.x] = a; }
  if (cta_sum_last(partial, (int)gridDim.x, ticket, rr_out, F) && finalize && threadIdx.x == 0) { scal[1] = alpha; cg_close_iteration(scal, *rr_out); }
}
__global__ void k_cg_residual(float *scal, const double *rr) {      // several ranks: the same closing step after the all-reduce of |r|^2
  if (scal[5] != 0.0f) return;
  cg_close_iteration(scal, *rr);
}
__global__ void k_cg_init(float *scal, const double *rr) {
  float res = (float)sqrt(*rr);
  scal[2] = res; scal[3] = 1.0f; scal[4] = sqrtf(FLT_EPSILON) * res; scal[0] = res * res / (1.0f * 1.0f); scal[1] = 0.0f;
  scal[6] = 0.0f; scal[5] = (res <= scal[4]) ? 1.0f : 0.0f; scal[7] = res;      // [7]: the initial residual (divergence guard)
}
__global__ void __launch_bounds__(256) k_dot_self(i64 n, const float *__restrict__ a, double *__restrict__ partial) {
  __shared__ double red[8];
  double s = 0.0;
  for (i64 v = blockIdx.x * (i64)blockDim.x + threadIdx.x; v < n; v += (i64)gridDim.x * blockDim.x) s += (double)a[v] * (double)a[v];
  for (int o = 16; o > 0; o >>= 1) s += __shfl_down_sync(0xffffffffu, s, o);
  if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = s;
  __syncthreads();
  if (threadIdx.x == 0) { double t = 0; for (int i = 0; i < (int)(blockDim.x >> 5); i++) t += red[i]; partial[blockIdx.x] = t; }
}

// ------------------------------------------------------------------------------------------------ min / max of a float field
__global__ void __launch_bounds__(256) k_minmax(i64 n, int nx, int px, const float *__restrict__ a, unsigned *__restrict__ mm) {   // mm[0] = ordered-min, mm[1] = ordered-max
  // a: rows of px floats of which the first nx count (n = padded length, a multiple of px)
  __shared__ float rlo[8], rhi[8];
  float lo = INFINITY, hi = -INFINITY;
  for (i64 v = blockIdx.x * (i64)blockDim.x + threadIdx.x; v < n; v += (i64)gridDim.x * blockDim.x) { if ((int)(v % px) < nx) { float x = a[v]; lo = fminf(lo, x); hi = fmaxf(hi, x); } }
  for (int o = 16; o > 0; o >>= 1) { lo = fminf(lo, __shfl_down_sync(0xffffffffu, lo, o)); hi = fmaxf(hi, __shfl_down_sync(0xffffffffu, hi, o)); }
  if ((threadIdx.x & 31) == 0) { rlo[threadIdx.x >> 5] = lo; rhi[threadIdx.x >> 5] = hi; }
  __syncthreads();
  if (threadIdx.x == 0) {
    for (int i = 1; i < 8; i++) { lo = fminf(lo, rlo[i]); hi = fmaxf(hi, rhi[i]); }
    // order-preserving map float -> uint; one pair of atomics per CTA
    unsigned bl = __float_as_uint(lo), bh = __float_as_uint(hi);
    bl = (bl & 0x80000000u) ? ~bl : (bl | 0x80000000u); bh = (bh & 0x80000000u) ? ~bh : (bh | 0x80000000u);
    atomicMin(&mm[0], bl); atomicMax(&mm[1], bh);
  }
}
static inline float ordered_to_float(unsigned b) { b = (b & 0x80000000u) ? (b & 0x7fffffffu) : ~b; float f; memcpy(&f, &b, 4); return f; }

// ------------------------------------------------------------------------------------------------ volume (CalcVolumeFromSDF.jl:26-125)
// pass 2: ONE THREAD per cut cell (grid-stride over the list; the count is read from device memory so that no host round
// trip separates the two passes); cut_cell_quad9 (r2s_volq.cuh) does the 729 points.  The cell's Float32 sum is accumulated across
// cells as a 2^-37 fixed-point integer (vol_cell_add; deterministic); vol_sum_flush adds the low 32 bits and the rest of the thread sums
// into acc[2] and acc[7].  One pair of atomics per CTA, not per warp: same-address atomics retire about one per clock, and a second
// per-warp atomic cost ~10 us per launch of k_vl_step / k_vl_eval (B200).  Called by every thread of the CTA (at most 8 warps).
__device__ __forceinline__ void vol_sum_flush(u64 local, u64 *__restrict__ acc) {
  __shared__ u64 s_w[2][8];
  u64 s[2] = {local & 0xffffffffull, local >> 32};
  for (int o = 16; o > 0; o >>= 1) { s[0] += __shfl_down_sync(0xffffffffu, s[0], o); s[1] += __shfl_down_sync(0xffffffffu, s[1], o); }
  if ((threadIdx.x & 31) == 0) { s_w[0][threadIdx.x >> 5] = s[0]; s_w[1][threadIdx.x >> 5] = s[1]; }
  __syncthreads();
  if (threadIdx.x == 0) {
    u64 a = 0, b = 0;
    for (int w = 0; w < (int)(blockDim.x >> 5); w++) { a += s_w[0][w]; b += s_w[1][w]; }
    if (a) atomicAdd(&acc[2], a);
    if (b) atomicAdd(&acc[7], b);
  }
}
__global__ void __launch_bounds__(128) k_vol_cut(int nx, int ny, int px, const float *__restrict__ sdf, float th, float iso, const int *__restrict__ cutlist, int cutcap,
                                                 GaussF G, u64 *__restrict__ acc) {
  const int ncut = (int)min((u64)cutcap, acc[1]);
  const int nthr = gridDim.x * blockDim.x;
  const i64 sxy = (i64)px * ny;
  u64 local = 0;
  for (int base = blockIdx.x * blockDim.x; base < ncut; base += nthr) {      // warp-uniform trip count
    const int idx = base + threadIdx.x;
    if (idx < ncut) {
      const i64 c = cutlist[idx];
      const int i = (int)(c % (nx - 1)), j = (int)((c / (nx - 1)) % (ny - 1)), k = (int)(c / ((i64)(nx - 1) * (ny - 1)));
      const i64 b = ((i64)k * ny + j) * px + i;
      const float cv[8] = {sdf[b] - th, sdf[b + 1] - th, sdf[b + px] - th, sdf[b + px + 1] - th,
                           sdf[b + sxy] - th, sdf[b + sxy + 1] - th, sdf[b + sxy + px] - th, sdf[b + sxy + px + 1] - th};
      vol_cell_add(local, cut_cell_quad9<false>(cv, G, iso, nullptr));
    }
  }
  vol_sum_flush(local, acc);
}
// ---- LS_Threshold bisection (RBFs4Smoothing.jl:265-300): volume of {lsf - th >= 0} for a SEQUENCE of thresholds ----------
// V(th) is a sum over cells; a cell's class depends only on (cmin, cmax) = (min, max) of its 8 corner values: full iff
// cmin >= th, empty iff cmax < th (IEEE subtraction is sign-exact, so min_i(v_i - th) >= 0  <=>  cmin >= th).  Every later
// threshold of the bisection lies inside the current bracket [lo, hi], so a cell with cmin >= hi stays full and a cell with
// cmax < lo stays empty for the rest of the search: such cells are retired (full ones into a permanent counter) and only the
// remaining "active" cells are carried to the next step in a compacted list.  The sum is accumulated in integers, so the
// result is bit-identical to re-classifying every cell at every step, at ~3 full passes instead of 40.
// acc: [0] full cells of this step  [1] cut count  [2], [7] cut fixed-point sum (vol_sum_flush's two words)  [3] permanently full
//      [4],[5] list sizes (ping-pong)  [6] records handed out
// any quadrature order 1..32 (calculate_volume_from_sdf's detailed_quad_order; the convergence tests of the reference use 20): same
// organisation as k_vol_cut, loops not unrolled, abscissae / weights read from the kernel-parameter bank with uniform indices
struct GaussNF { float x[32]; float w[32]; int n; };
__global__ void __launch_bounds__(128) k_vol_cut_n(int nx, int ny, int px, const float *__restrict__ sdf, float th, float iso, const int *__restrict__ cutlist, int cutcap,
                                                   GaussNF G, u64 *__restrict__ acc) {
  const int ncut = (int)min((u64)cutcap, acc[1]);
  const int nthr = gridDim.x * blockDim.x;
  const i64 sxy = (i64)px * ny;
  u64 local = 0;
  for (int base = blockIdx.x * blockDim.x; base < ncut; base += nthr) {
    const int idx = base + threadIdx.x;
    if (idx < ncut) {
      const i64 c = cutlist[idx];
      const int i = (int)(c % (nx - 1)), j = (int)((c / (nx - 1)) % (ny - 1)), k = (int)(c / ((i64)(nx - 1) * (ny - 1)));
      const i64 b = ((i64)k * ny + j) * px + i;
      const float c000 = sdf[b] - th, c100 = sdf[b + 1] - th, c010 = sdf[b + px] - th, c110 = sdf[b + px + 1] - th;
      const float c001 = sdf[b + sxy] - th, c101 = sdf[b + sxy + 1] - th, c011 = sdf[b + sxy + px] - th, c111 = sdf[b + sxy + px + 1] - th;
      float part = 0.0f;
      for (int iq = 0; iq < G.n; iq++) {
        const float xi = (G.x[iq] + 1) / 2, xm = 1.0f - xi;
        const float c00 = c000 * xm + c100 * xi, c01 = c001 * xm + c101 * xi;
        const float c10 = c010 * xm + c110 * xi, c11 = c011 * xm + c111 * xi;
        for (int jq = 0; jq < G.n; jq++) {
          const float eta = (G.x[jq] + 1) / 2, em = 1.0f - eta;
          const float c0 = c00 * em + c10 * eta, c1 = c01 * em + c11 * eta;
          const float wij = G.w[iq] * G.w[jq], dc = c1 - c0;
          for (int kq = 0; kq < G.n; kq++) {
            const float ps = fmaf(dc, (G.x[kq] + 1) / 2, c0);
            if (ps >= iso) part += wij * G.w[kq];
          }
        }
      }
      vol_cell_add(local, part);
    }
  }
  vol_sum_flush(local, acc);
}
static GaussF gauss9f() { GaussTab t = gauss_legendre_host(9); GaussF g; for (int i = 0; i < 9; i++) { g.x[i] = (float)t.x[i]; g.w[i] = (float)t.w[i]; } return g; }

// active cell of the threshold search: id, min / max of its corner values, index of its quadrature record (-1: none yet)
struct VAct { int id; float mn, mx; int rec; };
// Whole-grid classification (bisection steps 1-3, the final fine-grid volume, r2s_dev_volume_from_sdf) by PLANE MARCHING: a warp owns a
// tile of VM_R cell rows x (32 VM_V - 1) cells and marches through VM_Z cell planes.  Lane l holds the values of columns
// x0 + VM_V l .. x0 + VM_V l + VM_V - 1 of the VM_R + 1 rows; per plane it forms the y-pair min / max of each column, and a cell's
// min / max over its 8 corners is that of its two columns (the right one of the lane's last cell comes from lane + 1 by shuffle) in
// planes k and k + 1.  Plane k + 1 of one layer is plane k of the next, so every value is loaded once per tile (rows shared by two
// tiles twice) and the next plane is loaded while the current one is classified.  The last lane's last cell has no right column: tiles
// overlap by one column.  Cell ids, counts and lists are those of a cell-by-cell pass; only the order of the lists differs.
// Cells of planes [kc0, kc1) are classified (values of plane kc1 are read: the halo plane of a slab).  Cut cells go to cutlist, (EMIT) cells
// the remaining bracket [lo, hi] can still cut go to the active list; cells that are full for every threshold still to come are counted in
// acc[3].
#define VM_V 2
#define VM_R 4
#define VM_Z 32
template <bool EMIT>
__global__ void __launch_bounds__(256) k_vol_march(int nx, int ny, int px, int kc0, int kc1, const float *__restrict__ sdf, float lo, float hi, float th, VAct *__restrict__ list_out,
                                                   u64 *__restrict__ n_out_ptr, i64 list_cap, u64 *__restrict__ acc, int *__restrict__ cutlist, int cutcap) {
  __shared__ int s_cut[8][WS_CAP];
  __shared__ VAct s_keep[EMIT ? 8 : 1][EMIT ? WS_CAP : 1];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  constexpr int TXC = 32 * VM_V - 1;
  const int ntx = (nx - 2 + TXC) / TXC, nty = (ny - 2 + VM_R) / VM_R, ntz = (kc1 - kc0 + VM_Z - 1) / VM_Z;
  const i64 ntile = (i64)ntx * nty * ntz, pl = (i64)px * ny;
  int nfull = 0, nperm = 0, ncq = 0, nkq = 0;
  for (i64 tile = (i64)blockIdx.x * 8 + warp; tile < ntile; tile += (i64)gridDim.x * 8) {      // warp-uniform
    const int tx = (int)(tile % ntx), ty = (int)((tile / ntx) % nty), tz = (int)(tile / ((i64)ntx * nty));
    const int x0 = tx * TXC, xl = x0 + VM_V * lane, j0 = ty * VM_R, k0 = kc0 + tz * VM_Z, k1 = min(k0 + VM_Z, kc1);
    bool vin[VM_R + 1][VM_V];
    int off[VM_R + 1][VM_V];
#pragma unroll
    for (int r = 0; r <= VM_R; r++)
#pragma unroll
      for (int u = 0; u < VM_V; u++) { vin[r][u] = xl + u < nx && j0 + r < ny; off[r][u] = (j0 + r) * px + xl + u; }
    auto load = [&](int k, float (&v)[VM_R + 1][VM_V]) {
      const float *p = sdf + (i64)k * pl;
#pragma unroll
      for (int r = 0; r <= VM_R; r++)
#pragma unroll
        for (int u = 0; u < VM_V; u++) v[r][u] = vin[r][u] ? p[off[r][u]] : 0.0f;
    };
    float v[VM_R + 1][VM_V], amn[VM_R][VM_V], amx[VM_R][VM_V];
    load(k0, v);
#pragma unroll
    for (int r = 0; r < VM_R; r++)
#pragma unroll
      for (int u = 0; u < VM_V; u++) { amn[r][u] = fminf(v[r][u], v[r + 1][u]); amx[r][u] = fmaxf(v[r][u], v[r + 1][u]); }
    load(k0 + 1, v);
    for (int k = k0; k < k1; k++) {
      float bmn[VM_R][VM_V], bmx[VM_R][VM_V];
#pragma unroll
      for (int r = 0; r < VM_R; r++)
#pragma unroll
        for (int u = 0; u < VM_V; u++) { bmn[r][u] = fminf(v[r][u], v[r + 1][u]); bmx[r][u] = fmaxf(v[r][u], v[r + 1][u]); }
      if (k + 2 <= k1) load(k + 2, v);      // plane k + 2 is in flight while plane k's cells are classified
#pragma unroll
      for (int r = 0; r < VM_R; r++) {
        const int j = j0 + r;
        float cmn[VM_V + 1], cmx[VM_V + 1];      // column min / max over the cell layer's 4 values; [VM_V] = lane + 1's first column
#pragma unroll
        for (int u = 0; u < VM_V; u++) { cmn[u] = fminf(amn[r][u], bmn[r][u]); cmx[u] = fmaxf(amx[r][u], bmx[r][u]); }
        cmn[VM_V] = __shfl_down_sync(0xffffffffu, cmn[0], 1); cmx[VM_V] = __shfl_down_sync(0xffffffffu, cmx[0], 1);
        const int cbase = (k * (ny - 1) + j) * (nx - 1);
#pragma unroll
        for (int u = 0; u < VM_V; u++) {
          const int i = xl + u;
          bool cut = false, keep = false;
          const float mn = fminf(cmn[u], cmn[u + 1]), mx = fmaxf(cmx[u], cmx[u + 1]);
          if (i < nx - 1 && j < ny - 1 && (lane < 31 || u < VM_V - 1)) {
            if (EMIT && mn >= hi) nperm++;
            else if (EMIT && mx < lo) {}
            else {
              keep = EMIT;
              if (!(mx < th)) { if (mn >= th) nfull++; else cut = true; }
            }
          }
          ws_push<int>(s_cut[warp], ncq, cut, cbase + i, cutlist, &acc[1], (i64)cutcap, lane);
          if (EMIT) { VAct e; e.id = cbase + i; e.mn = mn; e.mx = mx; e.rec = -1; ws_push<VAct>(s_keep[warp], nkq, keep, e, list_out, n_out_ptr, list_cap, lane); }
        }
#pragma unroll
        for (int u = 0; u < VM_V; u++) { amn[r][u] = bmn[r][u]; amx[r][u] = bmx[r][u]; }
      }
    }
  }
  ws_flush<int>(s_cut[warp], ncq, cutlist, &acc[1], (i64)cutcap, lane);
  if (EMIT) ws_flush<VAct>(s_keep[warp], nkq, list_out, n_out_ptr, list_cap, lane);
  for (int o = 16; o > 0; o >>= 1) { nfull += __shfl_down_sync(0xffffffffu, nfull, o); nperm += __shfl_down_sync(0xffffffffu, nperm, o); }
  if (lane == 0) { if (nfull) atomicAdd(&acc[0], (u64)nfull); if (nperm) atomicAdd(&acc[3], (u64)nperm); }
}
template <bool EMIT>
static void vol_march(cudaStream_t st, int nx, int ny, int px, int kc0, int kc1, const float *sdf, float lo, float hi, float th, VAct *list_out, u64 *n_out_ptr, i64 list_cap, u64 *acc,
                      int *cutlist, int cutcap) {
  const i64 ntile = (i64)((nx - 2 + 32 * VM_V - 1) / (32 * VM_V - 1)) * ((ny - 2 + VM_R) / VM_R) * ((kc1 - kc0 + VM_Z - 1) / VM_Z);
  const int grid = (int)std::min<i64>(std::max<i64>(cdiv(ntile, 8), 1), 148 * 16);
  k_vol_march<EMIT><<<grid, 256, 0, st>>>(nx, ny, px, kc0, kc1, sdf, lo, hi, th, list_out, n_out_ptr, list_cap, acc, cutlist, cutcap);
}
// volume of {sdf >= iso}; edge = cell edge length (Float32 like the reference)
static int volume_dev(r2s_ctx *ctx, const float *sdf, int nx, int ny, int nz, int px, float edge, float iso, int order, double *vol) {
  cudaStream_t st = ctx->stream;
  i64 ncell = (i64)(nx - 1) * (ny - 1) * (nz - 1);
  if (ncell >= (1ll << 31)) FAIL("calculate_volume_from_sdf: grid too large for 32-bit cell ids");
  CK(ctx->f_scal.reserve(256));
  u64 *acc = (u64 *)((char *)ctx->f_scal.p + 128);
  static const GaussF G9 = gauss9f();
  for (int attempt = 0; attempt < 2; attempt++) {
    int cutcap = (int)(ctx->cutlist.cap / sizeof(int));
    CK(cudaMemsetAsync(acc, 0, sizeof(u64) * 8, st));
    vol_march<false>(st, nx, ny, px, 0, nz - 1, sdf, iso, iso, iso, nullptr, nullptr, 0, acc, ctx->cutlist.as<int>(), cutcap); LAUNCH_CHECK();
    if (order == 9) k_vol_cut<<<148 * 16, 128, 0, st>>>(nx, ny, px, sdf, 0.0f, iso, ctx->cutlist.as<int>(), cutcap, G9, acc);
    else {
      GaussTab t = gauss_legendre_host(order); GaussNF G; G.n = order;
      for (int q = 0; q < 32; q++) { G.x[q] = q < order ? (float)t.x[q] : 0.0f; G.w[q] = q < order ? (float)t.w[q] : 0.0f; }
      k_vol_cut_n<<<148 * 16, 128, 0, st>>>(nx, ny, px, sdf, 0.0f, iso, ctx->cutlist.as<int>(), cutcap, G, acc);
    }
    LAUNCH_CHECK();
    u64 h[8];
    if (r2s_readback(ctx, h, acc, sizeof(h))) return 1;
    if ((i64)h[1] > cutcap) {     // the cut list was too small: grow it and redo both passes
      CK(ctx->cutlist.reserve(sizeof(int) * (size_t)(h[1] + h[1] / 2 + 1024)));
      continue;
    }
    float ev = edge * edge * edge, jac = ev / 8.0f;
    *vol = (double)h[0] * (double)ev + vol_fixed_value(h[2], h[7]) * (double)jac;
    return 0;
  }
  FAIL("calculate_volume_from_sdf: cut-cell list overflow");
}
// ---- bisection steps >= 4: the ACTIVE list carries everything a cell needs ------------------------------------------------------
// After three whole-grid steps only the cells that the remaining bracket [lo, hi] can still cut are active (a thin shell around the
// level set).  The active list holds 16 bytes per cell (id, min / max of its corners, record index); a cell that is cut for the first time
// gets a RECORD: its eight corner values (32 bytes, gathered once, read only by k_vl_eval) and, in a separate 16-byte array with the same
// index, a CACHE of its last quadrature: part (the Float32 sum of w_i w_j w_k over the inside Gauss points), the threshold it was
// computed at and a margin = the smallest |value| over the 729 Gauss points minus a bound on the Float32
// round-off of those values.  While |th - th_cached| stays below the margin no Gauss value can change sign, the inside set -- and
// with it the cell's Float32 sum, bit for bit -- is the same, and the cached sum is added without re-evaluating the cell.  As the
// bracket halves, almost every cell freezes: the 40 bisections cost about a dozen full quadratures instead of 40.  The total is an
// exact integer sum, so the result is bit-identical to re-evaluating every cut cell at every step (R2S_VOL_CACHE=0 does that).
struct VRec { float c[8]; };
struct VCache { float part, th_e, margin; int pad; };      // one 16-byte load in k_vl_step
// State of the bisection on the DEVICE (steps >= 4): the bracket update is a one-thread kernel, so the host enqueues all remaining steps
// without waiting for any of them and reads the result once.  A step whose threshold repeats the previous one (lo and hi adjacent floats)
// and every step after the stopping rule has fired are skipped by all kernels of the step (skip / skipf).
struct BisState {
  float lo, hi, th, th_prev; int nb, have_prev, done, skip; float skipf; int cur; double v, eps, target; float ev, jac; unsigned long long n_eval;
};
__device__ __forceinline__ void bis_begin(BisState *S, u64 *acc) {
  if (S->done) { S->skip = 1; S->skipf = 1.0f; return; }
  const float th = (S->lo + S->hi) / 2;
  S->th = th;
  const int skip = (S->have_prev && th == S->th_prev) ? 1 : 0;      // the volume of an identical threshold is not recomputed
  S->skip = skip; S->skipf = skip ? 1.0f : 0.0f;
  if (!skip) { acc[0] = 0; acc[1] = 0; acc[2] = 0; acc[7] = 0; acc[4 + (1 - S->cur)] = 0; }
}
__device__ __forceinline__ void bis_end(BisState *S, const u64 *acc, const u64 *red) {      // LS_Threshold's loop body after the volume (RBFs4Smoothing.jl:286-296)
  if (S->done) return;
  if (!S->skip) {
    // the contraction nvcc chose for the plain expression (full * ev + sum * jac), written out
    S->v = fma((double)red[0], (double)S->ev, __dmul_rn(vol_fixed_value(red[2], red[3]), (double)S->jac));
    S->cur = 1 - S->cur; S->n_eval += acc[1];
  }
  const float cur = (float)S->v;
  S->eps = fabs(S->target - (double)cur);
  if ((double)cur > S->target) S->lo = S->th; else S->hi = S->th;
  S->nb++; S->have_prev = 1; S->th_prev = S->th;
  if (!(S->nb < 40 && S->eps > 1.0e-4)) S->done = 1;
}
// active cells: retire / keep (compaction into `out`), classify at th from (mn, mx), use the cached quadrature of the cell's record or queue
// the cell for k_vl_eval.  acc[6] = records handed out so far.  The kernel moves little data per cell and is bound by the latency of its
// two dependent loads (list entry, then cache): a warp takes VL_U x 32 consecutive entries per trip and issues all list loads, then all
// cache loads, then the appends.
#define VL_U 4
__global__ void __launch_bounds__(256) k_vl_step(const BisState *__restrict__ S, VAct *l0, VAct *l1, i64 out_cap, int use_cache, u64 *__restrict__ acc, const VCache *__restrict__ cache,
                                                 int2 *__restrict__ evlist, i64 ev_cap) {
  if (S->skip) return;
  const int icur = S->cur;
  const VAct *__restrict__ in = icur ? l1 : l0; VAct *__restrict__ out = icur ? l0 : l1;
  const u64 *n_in_ptr = acc + 4 + icur; u64 *n_out_ptr = acc + 4 + (1 - icur);
  const float lo = S->lo, hi = S->hi, th = S->th;
  __shared__ VAct s_keep[8][WS_CAP];
  __shared__ int2 s_ev[8][WS_CAP];
  const i64 n_in = (i64)*n_in_ptr;
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  int nfull = 0, nperm = 0, nkq = 0, neq = 0; u64 local = 0;
  for (i64 t0 = ((i64)blockIdx.x * blockDim.x + (threadIdx.x & ~31)) * VL_U; t0 < n_in; t0 += (i64)gridDim.x * blockDim.x * VL_U) {      // warp-uniform
    VAct e[VL_U];
#pragma unroll
    for (int u = 0; u < VL_U; u++) {
      const i64 t = t0 + u * 32 + lane;
      if (t < n_in) { const int4 q = __ldcs(reinterpret_cast<const int4 *>(in) + t); e[u].id = q.x; e[u].mn = __int_as_float(q.y); e[u].mx = __int_as_float(q.z); e[u].rec = q.w; }
      else { e[u].id = 0; e[u].mn = INFINITY; e[u].mx = INFINITY; e[u].rec = -1; }      // beyond the list: counted as permanently full below, then masked
    }
    float4 r[VL_U];
#pragma unroll
    for (int u = 0; u < VL_U; u++) {
      r[u] = make_float4(0.f, 0.f, 0.f, 0.f);
      const bool cached = use_cache && e[u].rec >= 0 && !(e[u].mn >= hi) && !(e[u].mx < lo) && !(e[u].mx < th) && !(e[u].mn >= th);      // the tests below, in the same form
      if (cached) r[u] = __ldg(reinterpret_cast<const float4 *>(cache) + e[u].rec);
    }
#pragma unroll
    for (int u = 0; u < VL_U; u++) {
      const bool valid = t0 + u * 32 + lane < n_in;
      bool keep = false, miss = false, fresh = false;
      if (valid) {
        if (e[u].mn >= hi) nperm++;                     // full for every threshold still to come
        else if (e[u].mx < lo) {}                       // empty for every threshold still to come
        else {
          keep = true;
          if (!(e[u].mx < th)) {
            if (e[u].mn >= th) nfull++;
            else if (e[u].rec < 0) { miss = true; fresh = true; }
            else if (use_cache && fabsf(th - r[u].y) * 1.00001f < r[u].z) vol_cell_add(local, r[u].x);
            else miss = true;
          }
        }
      }
      // new records: one claim per warp round (only cells that are cut for the first time)
      const unsigned mf = __ballot_sync(0xffffffffu, fresh);
      if (mf) {
        int base = 0;
        if (lane == 0) base = (int)atomicAdd(&acc[6], (u64)__popc(mf));
        base = __shfl_sync(0xffffffffu, base, 0);
        if (fresh) e[u].rec = base + __popc(mf & ((1u << lane) - 1));
      }
      ws_push<VAct>(s_keep[warp], nkq, keep, e[u], out, n_out_ptr, out_cap, lane);
      ws_push<int2>(s_ev[warp], neq, miss, make_int2(e[u].rec | (fresh ? (int)0x80000000 : 0), e[u].id), evlist, &acc[1], ev_cap, lane);
    }
  }
  ws_flush<VAct>(s_keep[warp], nkq, out, n_out_ptr, out_cap, lane);
  ws_flush<int2>(s_ev[warp], neq, evlist, &acc[1], ev_cap, lane);
  for (int o = 16; o > 0; o >>= 1) { nfull += __shfl_down_sync(0xffffffffu, nfull, o); nperm += __shfl_down_sync(0xffffffffu, nperm, o); }
  if (lane == 0) { if (nfull) atomicAdd(&acc[0], (u64)nfull); if (nperm) atomicAdd(&acc[3], (u64)nperm); }
  vol_sum_flush(local, acc);
}
// quadrature of the queued cells at th (cut_cell_quad9, as k_vol_cut) + their new cache entries; a cell that is cut for the first time
// gathers its corner values into its record
__global__ void __launch_bounds__(128) k_vl_eval(const BisState *__restrict__ S, VRec *__restrict__ recs, VCache *__restrict__ cache, const int2 *__restrict__ evlist, int nx, int ny,
                                                 int px, const float *__restrict__ sdf, GaussF G, u64 *__restrict__ acc) {
  if (S->skip) return;
  const float th = S->th;
  const int nev = (int)acc[1];
  const int nthr = gridDim.x * blockDim.x;
  u64 local = 0;
  for (int base = blockIdx.x * blockDim.x; base < nev; base += nthr) {      // warp-uniform trip count
    const int idx = base + threadIdx.x;
    if (idx < nev) {
      const int2 q = evlist[idx];
      VRec &e = recs[q.x & 0x7fffffff];
      float c[8];
      if (q.x < 0) {
        const i64 cpl = (i64)(nx - 1) * (ny - 1), sxy = (i64)px * ny;
        const int i = q.y % (nx - 1), j = (q.y / (nx - 1)) % (ny - 1), k = (int)(q.y / cpl);
        const i64 b = ((i64)k * ny + j) * px + i;
        c[0] = sdf[b]; c[1] = sdf[b + 1]; c[2] = sdf[b + px]; c[3] = sdf[b + px + 1];
        c[4] = sdf[b + sxy]; c[5] = sdf[b + sxy + 1]; c[6] = sdf[b + sxy + px]; c[7] = sdf[b + sxy + px + 1];
        float4 *d = reinterpret_cast<float4 *>(e.c);
        d[0] = make_float4(c[0], c[1], c[2], c[3]); d[1] = make_float4(c[4], c[5], c[6], c[7]);
      } else {
        const float4 *d = reinterpret_cast<const float4 *>(e.c), a = d[0], b = d[1];
        c[0] = a.x; c[1] = a.y; c[2] = a.z; c[3] = a.w; c[4] = b.x; c[5] = b.y; c[6] = b.z; c[7] = b.w;
      }
#pragma unroll
      for (int a = 0; a < 8; a++) c[a] = c[a] - th;
      const float amax = fmaxf(fmaxf(fmaxf(fabsf(c[0]), fabsf(c[1])), fmaxf(fabsf(c[2]), fabsf(c[3]))), fmaxf(fmaxf(fabsf(c[4]), fabsf(c[5])), fmaxf(fabsf(c[6]), fabsf(c[7]))));
      float m;
      const float part = cut_cell_quad9<true>(c, G, 0.0f, &m);
      // a Gauss value moves by (th_cached - th) plus Float32 round-off of the corner subtractions and the three lerps: a few ulp of the
      // corner magnitude, bounded generously by 1e-5 * amax (the step test applies the same factor to the threshold difference)
      VCache w; w.part = part; w.th_e = th; w.margin = m - 1.0e-5f * amax; w.pad = 0;
      cache[q.x & 0x7fffffff] = w;
      vol_cell_add(local, part);
    }
  }
  vol_sum_flush(local, acc);
}
// acc -> red for the cross-rank sum: [0] full + permanently full, [1] 1 if this rank's cut list overflowed, [2], [3] cut sum (two words)
__device__ __forceinline__ void vol_pack(const u64 *__restrict__ acc, int cutcap, u64 *__restrict__ red, const BisState *S) {
  if (S && S->skip) return;
  red[0] = acc[0] + acc[3]; red[1] = acc[1] > (u64)cutcap ? 1 : 0; red[2] = acc[2]; red[3] = acc[7];
}
__global__ void k_vol_pack(const u64 *__restrict__ acc, int cutcap, u64 *__restrict__ red, const BisState *S) { vol_pack(acc, cutcap, red, S); }
// the one-thread kernels between two bisection steps, fused: what = 1 begin, 2 end, 4 pack (pack -> [all-reduce] -> end -> begin of the next step)
__global__ void k_bis_turn(BisState *S, u64 *acc, u64 *red, int what) {
  if (what & 4) vol_pack(acc, 0x7fffffff, red, S);
  if (what & 2) bis_end(S, acc, red);
  if (what & 1) bis_begin(S, acc);
}
// state of one LS_Threshold search (see k_vol_step)
struct VolBisect {
  const float *sdf; int nx, ny, px, kc0, kc1; float edge; int step, cur; i64 n_cur, n_eval; u64 *acc;
};
static int vol_bisect_begin(r2s_ctx *ctx, VolBisect &vb, const float *sdf, int nx, int ny, int nz, int px, int kc0, int kc1, float edge) {
  i64 ncell = (i64)(nx - 1) * (ny - 1) * (nz - 1);
  if (ncell >= (1ll << 31)) FAIL("LS_Threshold: grid too large for 32-bit cell ids");
  CK(ctx->f_scal.reserve(512));
  vb.sdf = sdf; vb.nx = nx; vb.ny = ny; vb.px = px; vb.kc0 = kc0; vb.kc1 = kc1; vb.edge = edge; vb.step = 0; vb.cur = 0; vb.n_eval = 0;
  vb.n_cur = (i64)(nx - 1) * (ny - 1) * (i64)(kc1 - kc0);
  vb.acc = (u64 *)((char *)ctx->f_scal.p + 128);       // acc[0..7], red[0..3] behind it
  CK(cudaMemsetAsync(vb.acc, 0, sizeof(u64) * 12, ctx->stream));
  return 0;
}
// volume of {sdf - th >= 0} over the cells of planes [kc0, kc1); [lo, hi] = the bracket th was taken from
static int vol_bisect_step(r2s_ctx *ctx, VolBisect &vb, float lo, float hi, float th, double *vol) {
  cudaStream_t st = ctx->stream;
  static const GaussF G9 = gauss9f();
  const i64 n_all = (i64)(vb.nx - 1) * (vb.ny - 1) * (i64)(vb.kc1 - vb.kc0);
  vb.step++;
  const bool emit = vb.step == 3;      // steps 1-3 classify the whole grid (k_vol_march); step 3 also emits the active list (into list 0)
  if (emit) CK(ctx->vent[0].reserve(sizeof(VAct) * (size_t)(n_all + 1)));
  u64 h[6];
  for (int attempt = 0; attempt < 2; attempt++) {
    int cutcap = (int)(ctx->cutlist.cap / sizeof(int));
    // acc[3..6] only come into use at step 3 (it is the first step that retires cells and emits the active list) and after it, in
    // vol_bisect_finish: all eight words start from zero at every step.  (A second attempt follows a cut-list overflow: the list has been
    // grown, the step is repeated from scratch.)
    CK(cudaMemsetAsync(vb.acc, 0, sizeof(u64) * 8, st));
    u64 *nout = vb.acc + 4;
    if (!emit) vol_march<false>(st, vb.nx, vb.ny, vb.px, vb.kc0, vb.kc1, vb.sdf, lo, hi, th, nullptr, nullptr, 0, vb.acc, ctx->cutlist.as<int>(), cutcap);
    else vol_march<true>(st, vb.nx, vb.ny, vb.px, vb.kc0, vb.kc1, vb.sdf, lo, hi, th, ctx->vent[0].as<VAct>(), nout, n_all + 1, vb.acc, ctx->cutlist.as<int>(), cutcap);
    LAUNCH_CHECK();
    k_vol_cut<<<148 * 16, 128, 0, st>>>(vb.nx, vb.ny, vb.px, vb.sdf, th, 0.0f, ctx->cutlist.as<int>(), cutcap, G9, vb.acc); LAUNCH_CHECK();
    // cross-rank sum of (full cells, overflow flag, the two words of the cut sum); integers, so the total does not depend on the slab count
    u64 *red = vb.acc + 8, hr[4];
    k_vol_pack<<<1, 1, 0, st>>>(vb.acc, cutcap, red, nullptr); LAUNCH_CHECK();
    if (r2s_allreduce(ctx, red, 4, 1)) return 1;
    {      // acc[0..5] and red[0..3] are contiguous (red = acc + 8): one read-back of 12 words
      u64 hall[12];
      if (r2s_readback(ctx, hall, vb.acc, sizeof(hall))) return 1;
      for (int q = 0; q < 6; q++) h[q] = hall[q];
      for (int q = 0; q < 4; q++) hr[q] = hall[8 + q];
    }
    if (hr[1] != 0) {      // some rank's cut list overflowed: every rank repeats the step (collectives stay matched)
      if ((i64)h[1] > cutcap) CK(ctx->cutlist.reserve(sizeof(int) * (size_t)(h[1] + h[1] / 2 + 1024)));
      continue;
    }
    if (emit) {      // step 3: list 0 holds the active cells; room for one record per active cell (only cells that get cut use one)
      vb.cur = 0; vb.n_cur = (i64)h[4];
      CK(ctx->vrec.reserve((sizeof(VRec) + sizeof(VCache)) * (size_t)(vb.n_cur + 1)));      // corner records, then the caches
    }
    vb.n_eval += (i64)h[1];
    float ev = vb.edge * vb.edge * vb.edge, jac = ev / 8.0f;
    *vol = (double)hr[0] * (double)ev + vol_fixed_value(hr[2], hr[3]) * (double)jac;
    return 0;
  }
  FAIL("LS_Threshold: cut-cell list overflow");
}
// Steps 4 .. 40 on the device: 16-byte active entries, records with cached quadratures for the cells that get cut (k_vl_step / k_vl_eval), the
// bracket update in k_bis_turn.  Everything is enqueued at once; the host reads the final state back.  h = state after step 3.
static int vol_bisect_finish(r2s_ctx *ctx, VolBisect &vb, float &lo, float &hi, float &th, double &v, double &eps, int &nb, float th_prev, double target) {
  cudaStream_t st = ctx->stream;
  static const GaussF G9 = gauss9f();
  CK(ctx->vent[1].reserve(sizeof(VAct) * (size_t)(vb.n_cur + 1)));
  CK(ctx->vlist[1].reserve(sizeof(int2) * (size_t)(vb.n_cur + 1)));      // queue of cells to evaluate
  CK(ctx->bis_state.reserve(256));
  BisState h; memset(&h, 0, sizeof(h));
  h.lo = lo; h.hi = hi; h.th = th; h.th_prev = th_prev; h.nb = nb; h.have_prev = 1; h.done = 0; h.cur = 0; h.v = v; h.eps = eps; h.target = target;
  h.ev = vb.edge * vb.edge * vb.edge; h.jac = h.ev / 8.0f;
  BisState *S = ctx->bis_state.as<BisState>();
  CK(cudaMemcpyAsync(S, &h, sizeof(h), cudaMemcpyHostToDevice, st));
  const int grid = (int)std::min<i64>(std::max<i64>(cdiv(vb.n_cur, 256 * VL_U), 1), 148 * 8);
  VRec *recs = ctx->vrec.as<VRec>(); VCache *cache = reinterpret_cast<VCache *>(recs + (vb.n_cur + 1));
  u64 *red = vb.acc + 8;
  ctx->skip_flag = &S->skipf;      // the peer-memory all-reduce of a skipped step skips itself (same flag value on every rank)
  const bool single = ctx->nranks == 1;
  k_bis_turn<<<1, 1, 0, st>>>(S, vb.acc, red, 1); LAUNCH_CHECK();
  for (int step = nb; step < 40; step++) {
    const int next = step + 1 < 40 ? 1 : 0;
    k_vl_step<<<grid, 256, 0, st>>>(S, ctx->vent[0].as<VAct>(), ctx->vent[1].as<VAct>(), vb.n_cur + 1, ctx->knobs.vol_cache, vb.acc, cache, ctx->vlist[1].as<int2>(), vb.n_cur + 1); LAUNCH_CHECK();
    k_vl_eval<<<148 * 16, 128, 0, st>>>(S, recs, cache, ctx->vlist[1].as<int2>(), vb.nx, vb.ny, vb.px, vb.sdf, G9, vb.acc); LAUNCH_CHECK();
    if (single) { k_bis_turn<<<1, 1, 0, st>>>(S, vb.acc, red, 4 | 2 | next); LAUNCH_CHECK(); }
    else {
      k_bis_turn<<<1, 1, 0, st>>>(S, vb.acc, red, 4); LAUNCH_CHECK();
      if (r2s_allreduce(ctx, red, 4, 1)) { ctx->skip_flag = nullptr; return 1; }
      k_bis_turn<<<1, 1, 0, st>>>(S, vb.acc, red, 2 | next); LAUNCH_CHECK();
    }
  }
  ctx->skip_flag = nullptr;
  if (r2s_readback(ctx, &h, S, sizeof(h))) return 1;
  lo = h.lo; hi = h.hi; th = h.th; v = h.v; eps = h.eps; nb = h.nb; vb.n_eval += (i64)h.n_eval;
  return 0;
}
int r2s_dev_volume_from_sdf(r2s_ctx *ctx, const float *sdf_dev, i64 nx, i64 ny, i64 nz, float edge, float iso, int order, double *vol) {
  if (order < 1 || order > 32) FAIL("calculate_volume_from_sdf: detailed_quad_order must be between 1 and 32");
  CK(ctx->cutlist.reserve(sizeof(int) * 1024));
  return volume_dev(ctx, sdf_dev, (int)nx, (int)ny, (int)nz, (int)nx, edge, iso, order, vol);
}

// ------------------------------------------------------------------------------------------------ fine-grid evaluation (:363)
// phase tables: for each of the smooth^3 sub-cell positions the taps (coarse offset, weight) with |d|^2 <= ln(1/cut)
struct TapTable { int n[8]; int off[8][96]; };     // off packs (di+4) | (dj+4)<<4 | (dk+4)<<8
__constant__ float c_tapw[8][96];
__constant__ TapTable c_taps;
#define FN_X 32
#define FN_Y 4
#define FN_Z 4
template <int SM>
__global__ void __launch_bounds__(FN_X *FN_Y *FN_Z) k_fine_eval(int nx, int ny, int nz, int px, int fx, int fy, int fz, int kf0, const float *__restrict__ w, float th, float *__restrict__ out) {
  // coarse tile covering this block's fine outputs, with halo 3 on each side (taps reach -2..+3)
  constexpr int CX = FN_X / SM + 6, CY = FN_Y / SM + 6 + 1, CZ = FN_Z / SM + 6 + 1;
  __shared__ float sm[CZ][CY][CX + 1];
  const int fbx = blockIdx.x * FN_X, fby = blockIdx.y * FN_Y, fbz = kf0 + blockIdx.z * FN_Z;        // fz = one past the last fine plane of this launch
  const int cbx = fbx / SM - 3, cby = fby / SM - 3, cbz = fbz / SM - 3;
  for (int t = threadIdx.x; t < CX * CY * CZ; t += blockDim.x) {
    int lx = t % CX, ly = (t / CX) % CY, lz = t / (CX * CY);
    int gx = cbx + lx, gy = cby + ly, gz = cbz + lz;
    float v = 0.0f;
    if (gx >= 0 && gx < nx && gy >= 0 && gy < ny && gz >= 0 && gz < nz) v = w[((i64)gz * ny + gy) * px + gx];
    sm[lz][ly][lx] = v;
  }
  __syncthreads();
  int i = fbx + threadIdx.x % FN_X, j = fby + (threadIdx.x / FN_X) % FN_Y, k = fbz + threadIdx.x / (FN_X * FN_Y);
  if (i >= fx || j >= fy || k >= fz) return;
  int ph = (i % SM) + SM * ((j % SM) + SM * (k % SM));
  int lx = i / SM - cbx, ly = j / SM - cby, lz = k / SM - cbz;
  float acc = 0.0f;
  int nt = c_taps.n[ph];
  for (int t = 0; t < nt; t++) {
    int o = c_taps.off[ph][t];
    acc = fmaf(c_tapw[ph][t], sm[lz + ((o >> 8) & 15) - 4][ly + ((o >> 4) & 15) - 4][lx + (o & 15) - 4], acc);
  }
  out[((i64)k * fy + j) * fx + i] = acc + th;
}
// :fine grid (smooth = 2): one thread per coarse cell (a, b, c) -> its 2x2x2 fine outputs.  The taps of fine point
// (2a+px, 2b+py, 2c+pz) are the coarse points (a+di, b+dj, c+dk), di,dj,dk in -2..3, with weight
// exp(-((di-px/2)^2 + (dj-py/2)^2 + (dk-pz/2)^2)) when inside the cut radius, else 0.  The weight table lives in constant
// memory and is indexed with COMPILE-TIME offsets (the loops are fully unrolled), so every FMA takes its weight as a
// constant-bank operand; taps that are outside the largest supported radius (|d|^2 > 8) are pruned at compile time.
// Per 6-value x-row loaded from shared memory up to 48 FMAs are issued (FMA-bound, not LDS-bound).  Accumulation order per
// output is dk, dj, di ascending -- the same as k_fine_eval<2> -- so both kernels give bit-identical results.
__constant__ float c_w2[2][2][6][6][6][2];          // [pz][py][dk+2][dj+2][di+2][px]: the two x-phases of a tap are adjacent (one 8-byte constant operand of FFMA2)
#define F2_X 32
#define F2_Y 4
#define F2_Z 8            // coarse cells per block along z (2 per thread)
#define F2_ZT 4           // threads along z
__device__ __forceinline__ constexpr bool f2_tap_possible(int px, int py, int pz, int di, int dj, int dk) {
  // 4*|d|^2 <= 32  (|d|^2 <= 8)
  return (2 * di - px) * (2 * di - px) + (2 * dj - py) * (2 * dj - py) + (2 * dk - pz) * (2 * dk - pz) <= 32;
}
template <int PZ, int PY, int DK, int DJ>
__device__ __forceinline__ void f2_row(const float row[6], float &acc0, float &acc1) {
#pragma unroll
  for (int di = -2; di <= 3; di++) {
#if R2S_F32X2
    if (f2_tap_possible(0, PY, PZ, di, DJ, DK) && f2_tap_possible(1, PY, PZ, di, DJ, DK)) {      // both x-phases take this value: one packed FMA (same bits as two scalar ones)
      const float2 t = ffma2(make_float2(c_w2[PZ][PY][DK + 2][DJ + 2][di + 2][0], c_w2[PZ][PY][DK + 2][DJ + 2][di + 2][1]), make_float2(row[di + 2], row[di + 2]), make_float2(acc0, acc1));
      acc0 = t.x; acc1 = t.y;
      continue;
    }
#endif
    if (f2_tap_possible(0, PY, PZ, di, DJ, DK)) acc0 = fmaf(c_w2[PZ][PY][DK + 2][DJ + 2][di + 2][0], row[di + 2], acc0);
    if (f2_tap_possible(1, PY, PZ, di, DJ, DK)) acc1 = fmaf(c_w2[PZ][PY][DK + 2][DJ + 2][di + 2][1], row[di + 2], acc1);
  }
}
template <int DK, int DJ>
__device__ __forceinline__ void f2_rows(const float row[6], float acc[8]) {
  // acc index = px + 2*py + 4*pz
  if (f2_tap_possible(0, 0, 0, 0, DJ, DK) || f2_tap_possible(1, 0, 0, 0, DJ, DK) || f2_tap_possible(1, 0, 0, 1, DJ, DK)) f2_row<0, 0, DK, DJ>(row, acc[0], acc[1]);
  if (f2_tap_possible(0, 1, 0, 0, DJ, DK) || f2_tap_possible(1, 1, 0, 0, DJ, DK) || f2_tap_possible(1, 1, 0, 1, DJ, DK)) f2_row<0, 1, DK, DJ>(row, acc[2], acc[3]);
  if (f2_tap_possible(0, 0, 1, 0, DJ, DK) || f2_tap_possible(1, 0, 1, 0, DJ, DK) || f2_tap_possible(1, 0, 1, 1, DJ, DK)) f2_row<1, 0, DK, DJ>(row, acc[4], acc[5]);
  if (f2_tap_possible(0, 1, 1, 0, DJ, DK) || f2_tap_possible(1, 1, 1, 0, DJ, DK) || f2_tap_possible(1, 1, 1, 1, DJ, DK)) f2_row<1, 1, DK, DJ>(row, acc[6], acc[7]);
}
template <int DK>
__device__ __forceinline__ void f2_plane(const float (*sm)[F2_Y + 5][F2_X + 5], int lz, int ly, int lx, float acc[8]) {
#pragma unroll
  for (int dj = -2; dj <= 3; dj++) {
    float row[6];
#pragma unroll
    for (int di = 0; di < 6; di++) row[di] = sm[lz + DK + 2][ly + dj + 2][lx + di];
    switch (dj) {     // dj is a compile-time constant after unrolling
      case -2: f2_rows<DK, -2>(row, acc); break;
      case -1: f2_rows<DK, -1>(row, acc); break;
      case 0: f2_rows<DK, 0>(row, acc); break;
      case 1: f2_rows<DK, 1>(row, acc); break;
      case 2: f2_rows<DK, 2>(row, acc); break;
      default: f2_rows<DK, 3>(row, acc); break;
    }
  }
}
// kc0/kc1: coarse planes whose fine outputs this launch produces (z-slab); fine planes 2c and 2c+1 (the latter if < fz)
__global__ void __launch_bounds__(F2_X *F2_Y *F2_ZT) k_fine_eval2(int nx, int ny, int nz, int px, int fx, int fy, int fz, int kc0, int kc1, const float *__restrict__ w, float th,
                                                                  float *__restrict__ out) {
  __shared__ float sm[F2_Z + 5][F2_Y + 5][F2_X + 5];
  const int cbx = blockIdx.x * F2_X, cby = blockIdx.y * F2_Y, cbz = kc0 + blockIdx.z * F2_Z;
  constexpr int TX = F2_X + 5, TY = F2_Y + 5, TZ = F2_Z + 5;
  for (int t = threadIdx.x; t < TX * TY * TZ; t += blockDim.x) {
    int lx = t % TX, ly = (t / TX) % TY, lz = t / (TX * TY);
    int gx = cbx + lx - 2, gy = cby + ly - 2, gz = cbz + lz - 2;
    float v = 0.0f;
    if (gx >= 0 && gx < nx && gy >= 0 && gy < ny && gz >= 0 && gz < nz) v = w[((i64)gz * ny + gy) * px + gx];
    sm[lz][ly][lx] = v;
  }
  __syncthreads();
  const int lx = threadIdx.x % F2_X, ly = (threadIdx.x / F2_X) % F2_Y, lzt = threadIdx.x / (F2_X * F2_Y);
  const int a = cbx + lx, b = cby + ly;
  if (a >= nx || b >= ny) return;
#pragma unroll 1
  for (int q = 0; q < F2_Z / F2_ZT; q++) {
    const int lz = lzt + q * F2_ZT, c = cbz + lz;
    if (c >= kc1 || c >= nz) continue;
    float acc[8];
#pragma unroll
    for (int i = 0; i < 8; i++) acc[i] = 0.0f;
    f2_plane<-2>(sm, lz, ly, lx, acc); f2_plane<-1>(sm, lz, ly, lx, acc); f2_plane<0>(sm, lz, ly, lx, acc);
    f2_plane<1>(sm, lz, ly, lx, acc); f2_plane<2>(sm, lz, ly, lx, acc); f2_plane<3>(sm, lz, ly, lx, acc);
#pragma unroll
    for (int pz = 0; pz < 2; pz++)
#pragma unroll
      for (int py = 0; py < 2; py++) {
        int i = 2 * a, j = 2 * b + py, k = 2 * c + pz;
        if (j < fy && k < fz) {
          i64 o = ((i64)k * fy + j) * fx + i;
          out[o] = acc[2 * py + 4 * pz] + th;
          if (i + 1 < fx) out[o + 1] = acc[1 + 2 * py + 4 * pz] + th;
        }
      }
  }
}
// u_new = r + beta * u_old on the halo planes of a slab (the fused stencil kernel writes u_new on the owned planes only)
__global__ void k_unew_halo(i64 n1, i64 off2, i64 n2, const float *__restrict__ scal, const float *__restrict__ r, const float *__restrict__ u, float *__restrict__ unew) {
  i64 v = blockIdx.x * (i64)blockDim.x + threadIdx.x;
  if (v >= n1 + n2 || scal[5] != 0.0f) return;
  i64 i = v < n1 ? v : off2 + (v - n1);
  unew[i] = r[i] + scal[0] * u[i];
}

static int upload_taps(r2s_ctx *ctx, int sm, double rbf_cut, double cell) {
  TapTable T; static float W[8][96];
  memset(&T, 0, sizeof(T)); memset(W, 0, sizeof(W));
  float maxd = (float)sqrt(-log(rbf_cut) * cell * cell);            // :221
  for (int ph = 0; ph < sm * sm * sm; ph++) {
    int px = ph % sm, py = (ph / sm) % sm, pz = ph / (sm * sm), n = 0;
    for (int dk = -4; dk <= 4; dk++) for (int dj = -4; dj <= 4; dj++) for (int di = -4; di <= 4; di++) {
      double ox = di - (double)px / sm, oy = dj - (double)py / sm, oz = dk - (double)pz / sm, m = ox * ox + oy * oy + oz * oz;
      float dist = (float)(sqrt(m) * cell);
      if (dist <= maxd) {
        if (n >= 96) FAIL("rbf: tap table overflow (rbf_cut too small)");
        if (di < -3 || di > 3 || dj < -3 || dj > 3 || dk < -3 || dk > 3) FAIL("rbf: kernel support too wide for the tile halo");
        T.off[ph][n] = (di + 4) | ((dj + 4) << 4) | ((dk + 4) << 8); W[ph][n] = (float)exp(-m); n++;
      }
    }
    T.n[ph] = n;
  }
  if (sm == 2) {      // dense per-phase weight table of k_fine_eval2 (same inclusion test, zero = excluded)
    static float W2[2][2][6][6][6][2];
    for (int pz = 0; pz < 2; pz++) for (int py = 0; py < 2; py++) for (int dk = -2; dk <= 3; dk++) for (int dj = -2; dj <= 3; dj++)
      for (int px = 0; px < 2; px++) for (int di = -2; di <= 3; di++) {
        double ox = di - 0.5 * px, oy = dj - 0.5 * py, oz = dk - 0.5 * pz, m = ox * ox + oy * oy + oz * oz;
        float dist = (float)(sqrt(m) * cell);
        W2[pz][py][dk + 2][dj + 2][di + 2][px] = (dist <= maxd) ? (float)exp(-m) : 0.0f;
      }
    CK(cudaMemcpyToSymbolAsync(c_w2, W2, sizeof(W2), 0, cudaMemcpyHostToDevice, ctx->stream));
  }
  CK(cudaMemcpyToSymbolAsync(c_taps, &T, sizeof(T), 0, cudaMemcpyHostToDevice, ctx->stream));
  CK(cudaMemcpyToSymbolAsync(c_tapw, W, sizeof(W), 0, cudaMemcpyHostToDevice, ctx->stream));
  CK(cudaStreamSynchronize(ctx->stream));
  return 0;
}

// ------------------------------------------------------------------------------------------------ driver
// Slab layout: every field is indexed globally (plane k at offset k * nx * ny); a rank owns the coarse planes [k0, k1) and
// keeps up to 3 halo planes on each side valid.  With one rank [k0, k1) is the whole grid and every exchange is a no-op.
int r2s_dev_rbf(r2s_ctx *ctx, int is_interp, int smooth, double rbf_cut, double target, bool final_volume, float *th_out, float *vol_out) {
  const GridDev &g = ctx->g; cudaStream_t st = ctx->stream;
  // every coarse Float32 field (s, weights, r, u, c, lsf) is stored with a row pitch px = nx rounded up to 4 floats: the TMA tensor maps
  // of the stencil need 16-byte global strides.  The pad columns are kept at zero (they take part in the element-wise CG kernels).
  const int nx = g.np[0], ny = g.np[1], nz = g.np[2], px = (nx + 3) & ~3; const i64 upl = (i64)nx * ny, pl = (i64)px * ny, n = pl * nz;
  const int k0 = (int)ctx->k0, k1 = (int)ctx->k1;
  if (ctx->nranks == 1 && (k0 != 0 || k1 != nz)) FAIL("rbf smoothing on a z-slab needs the slab communicator (r2s_comm_init on every rank)");
  const int e0 = std::max(0, k0 - 2), e1 = std::min(nz, k1 + 2);        // owned planes + CG halo
  const i64 o_lo = (i64)k0 * pl, nown = (i64)(k1 - k0) * pl, x_lo = (i64)e0 * pl, next = (i64)(e1 - e0) * pl;
  const int fx = g.N[0] * smooth + 1, fy = g.N[1] * smooth + 1, fz = g.N[2] * smooth + 1; const i64 nf = (i64)fx * fy * fz, fpl = (i64)fx * fy;
  const int kf0 = smooth * k0, kf1 = (k1 < nz) ? smooth * k1 : fz;       // fine planes of this slab
  // the stencil form needs the reference's cut to sit strictly between lattice shells (true for the default 1e-3)
  StencilW W; { double L = -log(rbf_cut); if (!(L > 6.0 && L < 8.0)) FAIL("rbf: only kernel cut-offs with 6 < ln(1/cut) < 8 (81-point stencil) are supported"); for (int m = 0; m < 8; m++) W.w[m] = (float)exp(-(double)m); }
  ctx->have_rbf = false;      // f_s / f_w are rewritten below
  CK(cudaEventRecord(ctx->ev[4], st));
  CK(ctx->f_s.reserve(sizeof(float) * (size_t)n)); CK(ctx->f_lsf.reserve(sizeof(float) * (size_t)n));
  CK(ctx->f_fine.reserve(sizeof(float) * (size_t)nf));
  CK(ctx->f_scal.reserve(512));
  CK(ctx->cutlist.reserve(sizeof(int) * 4096));
  float *scal = ctx->f_scal.as<float>(); unsigned *ubits = (unsigned *)((char *)ctx->f_scal.p + 64); double *dsc = (double *)((char *)ctx->f_scal.p + 96);
  CK(cudaMemsetAsync(ctx->f_scal.p, 0, 256, st));
  float *s = ctx->f_s.as<float>();
  CK(cudaMemsetAsync(s + o_lo, 0, sizeof(float) * (size_t)nown, st));      // pad columns
  k_to_f32<<<(int)std::min<i64>(cdiv((i64)(k1 - k0) * upl, 256), CG_BLOCKS), 256, 0, st>>>((i64)(k1 - k0) * upl, (i64)k0 * upl, nx, px, ctx->sdf.as<double>(), s, ubits); LAUNCH_CHECK();
  if (r2s_allreduce(ctx, ubits, 1, 2)) return 1;                          // global max finite |v| (RBFs4Smoothing.jl:17)
  unsigned hb = 0;
  if (r2s_readback(ctx, &hb, ubits, sizeof(unsigned))) return 1;
  if (hb == 0) FAIL("RBFs_smoothing: the SDF holds no finite value (maximum over an empty collection, RBFs4Smoothing.jl:17)");
  k_replace_far<<<cdiv(nown, 256), 256, 0, st>>>(nown, s + o_lo, ubits); LAUNCH_CHECK();
  if (r2s_halo_exchange_f32(ctx, s, pl, k0, k1, nz, 2, 3)) return 1;
  CK(cudaEventRecord(ctx->ev[5], st));
  // mat-vec kernel: plane marching, two outputs per thread, factorised weights; even z-chunks of about 64 planes (a 65-plane slab is one chunk, not 64 + 1)
  const int nchunk = std::max(1, (k1 - k0 + 32) / 64), zc = cdiv(k1 - k0, nchunk);
  dim3 sgrid(cdiv(nx + (R2S_ST_NO == 4 ? 2 : 0), S3_X), cdiv(ny, S3_Y), cdiv(k1 - k0, zc));
  const int sthreads = 16 * S3_X / R2S_ST_NO;
  int nsb = (int)(sgrid.x * sgrid.y * sgrid.z), nub = (int)std::min<i64>(cdiv(next, 256), CG_BLOCKS);
  CK(ctx->f_part.reserve(sizeof(double) * (size_t)(nsb > nub ? nsb : nub)));
  double *part = ctx->f_part.as<double>();
  float *wgt = s; int iters = 0;
  if (is_interp) {
    // cg(K, s) with IterativeSolvers defaults (:199): x0 = 0, reltol = sqrt(eps(Float32)), maxiter = n
    CK(ctx->f_w.reserve(sizeof(float) * (size_t)n)); CK(ctx->f_r.reserve(sizeof(float) * (size_t)n));
    CK(ctx->f_u.reserve(sizeof(float) * 2 * (size_t)n));
    if (r2s_p2p_prepare_c(ctx, ctx->f_c.cap, sizeof(float) * (size_t)n)) return 1;      // peers must drop their mappings of c before it is re-allocated
    CK(ctx->f_c.reserve(sizeof(float) * (size_t)n));
    float *x = ctx->f_w.as<float>(), *r = ctx->f_r.as<float>(), *u = ctx->f_u.as<float>(), *c = ctx->f_c.as<float>();
    CK(cudaMemsetAsync(x + x_lo, 0, sizeof(float) * (size_t)next, st));
    CK(cudaMemsetAsync(u + x_lo, 0, sizeof(float) * (size_t)next, st));
    CK(cudaMemsetAsync(u + n + x_lo, 0, sizeof(float) * (size_t)next, st));
    CK(cudaMemsetAsync(c + x_lo, 0, sizeof(float) * (size_t)next, st));      // pad columns of c enter r through the element-wise update
    CUtensorMap tm_r, tm_u[2];
    if (stencil_tensor_map(ctx, &tm_r, r, nx, ny, nz, px) || stencil_tensor_map(ctx, &tm_u[0], u, nx, ny, nz, px) || stencil_tensor_map(ctx, &tm_u[1], u + n, nx, ny, nz, px)) return 1;
    int upar = 0;      // which half of u holds u_old
    CK(cudaMemcpyAsync(r + x_lo, s + x_lo, sizeof(float) * (size_t)next, cudaMemcpyDeviceToDevice, st));
    int nob = (int)std::min<i64>(cdiv(nown, 256), CG_BLOCKS);
    k_dot_self<<<nob, 256, 0, st>>>(nown, r + o_lo, part); LAUNCH_CHECK();
    k_sum_to<<<1, 256, 0, st>>>(part, nob, dsc); LAUNCH_CHECK();
    if (r2s_allreduce(ctx, dsc, 1, 0)) return 1;
    k_cg_init<<<1, 1, 0, st>>>(scal, dsc); LAUNCH_CHECK();
    float hs[8];
    if (r2s_readback(ctx, hs, scal, sizeof(hs))) return 1;
    float *u_old = u, *u_new = u + n;      // ping-pong halves of the u buffer
    if (r2s_p2p_map_c(ctx, c, sizeof(float) * (size_t)n)) return 1;
    const i64 nh_lo = (i64)(k0 - e0) * pl, nh_hi = (i64)(e1 - k1) * pl;      // halo sizes below / above
    unsigned *tick = (unsigned *)((char *)ctx->f_scal.p + 80);               // tickets of the two fused reductions
    // The convergence test lives on the device (scal[5]); the host launches CG_CHUNK iterations at a time and then reads the flag and the
    // iteration count back.  Iterations launched after convergence return at their first instruction (and the peer-memory exchanges skip
    // themselves through ctx->skip_flag), so the result is that of IterativeSolvers' loop: while iters < maxiter && residual > tol.
    constexpr int CG_CHUNK = 4;
    ctx->skip_flag = scal + 5;
    int launched = 0; bool probed = false;
    const int single = ctx->nranks == 1 ? 1 : 0;
    while (hs[5] == 0.0f && launched < n) {
      for (int q = 0; q < CG_CHUNK; q++, launched++) {
        const bool probe = launched == 3;      // one iteration is split by events for the report (cg_probe)
        if (probe) CK(cudaEventRecord(ctx->ev_probe[0], st));
        // u_new = r + beta*u_old ; c = K u_new ; uc = dot(u_new, c)  (partial sums added up by the last CTA)
        // Peer-memory transport: the two kernels of an iteration do their exchanges themselves -- the mat-vec stores its boundary planes of
        // c into the neighbours' arrays while it computes, its last CTA all-reduces the dot product through the mailbox and raises the
        // halo flags; the update waits for the neighbours' flags, its last CTA all-reduces |r|^2 and closes the iteration.
        P2PFuse fs, fu;
        if (r2s_p2p_fuse_params(ctx, &fs, &fu, pl, k0, k1, 2)) return 1;
        k_stencil81_tma<true, R2S_ST_NO><<<sgrid, sthreads, 0, st>>>(tm_r, tm_u[upar], nx, ny, nz, px, k0, k1, zc, u_new, scal, c, part, W, tick, dsc + 1, fs);
        LAUNCH_CHECK();
        if (nh_lo + nh_hi > 0) { k_unew_halo<<<cdiv(nh_lo + nh_hi, 256), 256, 0, st>>>(nh_lo, (i64)(k1 - e0) * pl, nh_hi, scal, r + x_lo, u_old + x_lo, u_new + x_lo); LAUNCH_CHECK(); }
        if (probe) CK(cudaEventRecord(ctx->ev_probe[1], st));
        if (!fs.enabled && !single) {
          if (r2s_group_start(ctx)) return 1;          // NCCL / event transport: scalar all-reduce + halo planes of c
          if (r2s_allreduce(ctx, dsc + 1, 1, 0)) return 1;
          if (r2s_halo_exchange_f32(ctx, c, pl, k0, k1, nz, 2, 2)) return 1;
          if (r2s_group_end(ctx)) return 1;
        }
        if (probe) CK(cudaEventRecord(ctx->ev_probe[2], st));
        const int closes = (single || fs.enabled) ? 1 : 0;      // the update's last CTA closes the iteration unless |r|^2 still needs a separate all-reduce
        k_cg_update<<<nub, 256, 0, st>>>(next, o_lo - x_lo, o_lo - x_lo + nown, scal, dsc + 1, u_new + x_lo, c + x_lo, x + x_lo, r + x_lo, part, tick + 1, dsc + 2, closes, fu); LAUNCH_CHECK();
        if (probe) CK(cudaEventRecord(ctx->ev_probe[3], st));
        if (!closes) {
          if (r2s_allreduce(ctx, dsc + 2, 1, 0)) return 1;
          k_cg_residual<<<1, 1, 0, st>>>(scal, dsc + 2); LAUNCH_CHECK();
        }
        if (probe) CK(cudaEventRecord(ctx->ev_probe[4], st));
        { float *t = u_old; u_old = u_new; u_new = t; upar ^= 1; }
      }
      if (r2s_readback(ctx, hs, scal, sizeof(hs))) { ctx->skip_flag = nullptr; return 1; }
      if (!probed && launched > 3) { probed = true; for (int q = 0; q < 4; q++) CK(cudaEventElapsedTime(&ctx->rep.cg_probe[q], ctx->ev_probe[q], ctx->ev_probe[q + 1])); }
    }
    ctx->skip_flag = nullptr;
    if (hs[5] == 2.0f) FAIL("RBFs_smoothing: the CG residual is not finite or diverges (non-finite SDF input, or a peer-memory exchange failed)");
    iters = (int)hs[6];
    wgt = x;
    if (r2s_halo_exchange_f32(ctx, x, pl, k0, k1, nz, 2, 3)) return 1;      // the fine evaluation reaches 3 planes up
  }
  ctx->rep.cg_iters = iters;
  CK(cudaEventRecord(ctx->ev[6], st));
  // LSF on the coarse grid (:357) = K * weights
  float *lsf = ctx->f_lsf.as<float>();
  {
    CUtensorMap tm_w;
    if (stencil_tensor_map(ctx, &tm_w, wgt, nx, ny, nz, px)) return 1;
    { P2PFuse f0; memset(&f0, 0, sizeof(f0)); k_stencil81_tma<false, R2S_ST_NO><<<sgrid, sthreads, 0, st>>>(tm_w, tm_w, nx, ny, nz, px, k0, k1, zc, nullptr, nullptr, lsf, part, W, nullptr, nullptr, f0); }
  }
  LAUNCH_CHECK();
  if (r2s_halo_exchange_f32(ctx, lsf, pl, k0, k1, nz, 0, 1)) return 1;      // cells of my top plane need plane k1
  // LS_Threshold (:265-300)
  unsigned init_mm[2] = {0xffffffffu, 0u};
  CK(cudaMemcpyAsync(ubits + 2, init_mm, sizeof(init_mm), cudaMemcpyHostToDevice, st));
  k_minmax<<<(int)std::min<i64>(cdiv(nown, 256), CG_BLOCKS), 256, 0, st>>>(nown, nx, px, lsf + o_lo, ubits + 2); LAUNCH_CHECK();
  if (r2s_group_start(ctx)) return 1;
  if (r2s_allreduce(ctx, ubits + 2, 1, 3)) return 1;
  if (r2s_allreduce(ctx, ubits + 3, 1, 2)) return 1;
  if (r2s_group_end(ctx)) return 1;
  unsigned hmm[2];
  if (r2s_readback(ctx, hmm, ubits + 2, sizeof(hmm))) return 1;
  CK(cudaEventRecord(ctx->ev[7], st));
  float lo = ordered_to_float(hmm[0]), hi = ordered_to_float(hmm[1]);
  // coarse cell edge as the reference measures it: norm(grid[2,1,1] - grid[1,1,1]) with Float32 range() coordinates (:41-43)
  float edge;
  {
    float a = (float)g.amin[0], b = (float)g.amax[0];
    float x0 = a, x1 = (nx > 1) ? (float)((double)a + 1.0 * (((double)b - (double)a) / (double)(nx - 1))) : a;
    if (nx == 2) x1 = b;
    float ex = x1 - x0; edge = sqrtf(ex * ex);
  }
  double eps = 1.0; int nb = 0; float th = 0.0f; double v = 0.0; bool have_prev = false; float th_prev = 0.0f;
  VolBisect vb;
  if (vol_bisect_begin(ctx, vb, lsf, nx, ny, nz, px, k0, std::min(k1, nz - 1), edge)) return 1;
  while (nb < 40 && eps > 1.0e-4) {
    th = (lo + hi) / 2;
    // once lo and hi are adjacent floats the midpoint repeats: the volume of an identical threshold is not recomputed
    if (!(have_prev && th == th_prev)) { if (vol_bisect_step(ctx, vb, lo, hi, th, &v)) return 1; }
    have_prev = true; th_prev = th;
    float cur = (float)v;
    eps = fabs(target - (double)cur);
    if ((double)cur > target) lo = th; else hi = th;
    nb++;
    // three whole-grid steps driven from the host (they size the lists); the rest of the search runs on the device without host round trips
    if (vb.step == 3 && nb < 40 && eps > 1.0e-4) { if (vol_bisect_finish(ctx, vb, lo, hi, th, v, eps, nb, th_prev, target)) return 1; break; }
  }
  ctx->rep.bisections = nb;
  float tho = -th;
  CK(cudaEventRecord(ctx->ev[13], st));
  // fine grid (:363-366): the fine planes of my coarse planes
  if (upload_taps(ctx, smooth, rbf_cut, g.cell)) return 1;
  {
    // evaluated in chunks of coarse planes; when a host buffer is attached (r2s_pipeline_slab) each finished chunk is
    // downloaded on the copy stream while the next chunks and the final volume are computed
    const int chunk = ctx->async_fine_host ? 32 : (k1 - k0);
    for (int c0 = k0; c0 < k1; c0 += chunk) {
      const int c1 = std::min(c0 + chunk, k1);
      const int f0 = smooth * c0, f1 = (c1 < nz) ? smooth * c1 : fz;
      if (smooth == 1) {
        dim3 fgrid(cdiv(fx, FN_X), cdiv(fy, FN_Y), cdiv(f1 - f0, FN_Z));
        k_fine_eval<1><<<fgrid, FN_X * FN_Y * FN_Z, 0, st>>>(nx, ny, nz, px, fx, fy, f1, f0, wgt, tho, ctx->f_fine.as<float>());
      } else {
        dim3 g2(cdiv(nx, F2_X), cdiv(ny, F2_Y), cdiv(c1 - c0, F2_Z));
        k_fine_eval2<<<g2, F2_X * F2_Y * F2_ZT, 0, st>>>(nx, ny, nz, px, fx, fy, fz, c0, c1, wgt, tho, ctx->f_fine.as<float>());
      }
      LAUNCH_CHECK();
      if (ctx->async_fine_host) {
        cudaEvent_t e = ctx->ev_copy[ctx->n_ev_copy++ % 64];
        CK(cudaEventRecord(e, st));
        CK(cudaStreamWaitEvent(ctx->copy_stream, e, 0));
        CK(cudaMemcpyAsync(ctx->async_fine_host + (size_t)(f0 - kf0) * fpl, ctx->f_fine.as<float>() + (size_t)f0 * fpl, sizeof(float) * (size_t)(f1 - f0) * fpl, cudaMemcpyDeviceToHost,
                           ctx->copy_stream));
      }
    }
  }
  CK(cudaEventRecord(ctx->ev[14], st));
  float volf = 0.0f;
  if (final_volume) {      // calculate_volume_from_sdf on the fine grid (:373), iso = 0
    float a = (float)g.amin[0], b = (float)g.amax[0];
    float dxf = (b - a) / (float)(fx - 1); float x0 = a, x1 = a + 1.0f * dxf; float e = sqrtf((x1 - x0) * (x1 - x0));
    if (r2s_halo_exchange_f32(ctx, ctx->f_fine.as<float>(), fpl, kf0, kf1, fz, 0, 1)) return 1;
    VolBisect vf; double vv;
    if (vol_bisect_begin(ctx, vf, ctx->f_fine.as<float>(), fx, fy, fz, fx, kf0, std::min(kf1, fz - 1), e)) return 1;
    if (vol_bisect_step(ctx, vf, 0.0f, 0.0f, 0.0f, &vv)) return 1;
    volf = (float)vv;
  }
  CK(cudaEventRecord(ctx->ev[15], st));
  CK(cudaStreamSynchronize(st));
  ctx->smooth_last = smooth; ctx->have_fine = true;
  if (r2s_sample_record(ctx, wgt, px, tho, rbf_cut)) return 1;
  *th_out = tho; *vol_out = volf;
  CK(cudaEventElapsedTime(&ctx->rep.ms_rbf_prep, ctx->ev[4], ctx->ev[5]));
  CK(cudaEventElapsedTime(&ctx->rep.ms_cg, ctx->ev[5], ctx->ev[6]));
  CK(cudaEventElapsedTime(&ctx->rep.ms_lsf, ctx->ev[6], ctx->ev[7]));
  CK(cudaEventElapsedTime(&ctx->rep.ms_threshold, ctx->ev[7], ctx->ev[13]));
  CK(cudaEventElapsedTime(&ctx->rep.ms_fine, ctx->ev[13], ctx->ev[14]));
  CK(cudaEventElapsedTime(&ctx->rep.ms_volume, ctx->ev[14], ctx->ev[15]));
  return 0;
}
