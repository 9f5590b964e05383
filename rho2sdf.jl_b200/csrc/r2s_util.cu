// r2s_util.cu -- device-wide scan / radix sort plumbing (CUB from the CUDA toolkit) used by the binning steps
#include <cub/cub.cuh>
#include <string.h>
#include "r2s_common.cuh"

int r2s_scan_exclusive_i64(r2s_ctx *ctx, const i64 *in, i64 *out, i64 n) {
  size_t tmp = 0;
  CK(cub::DeviceScan::ExclusiveSum(nullptr, tmp, in, out, (int)n, ctx->stream));
  CK(ctx->cubtmp.reserve(tmp));
  CK(cub::DeviceScan::ExclusiveSum(ctx->cubtmp.p, tmp, in, out, (int)n, ctx->stream));
  ctx->launches += 2;
  return 0;
}
int r2s_scan_exclusive_i32(r2s_ctx *ctx, const int *in, int *out, i64 n) {
  size_t tmp = 0;
  CK(cub::DeviceScan::ExclusiveSum(nullptr, tmp, in, out, (int)n, ctx->stream));
  CK(ctx->cubtmp.reserve(tmp));
  CK(cub::DeviceScan::ExclusiveSum(ctx->cubtmp.p, tmp, in, out, (int)n, ctx->stream));
  ctx->launches += 2;
  return 0;
}
// sorts n 64-bit keys on bits [0,end_bit); *sorted points at whichever of keys/alt holds the result
int r2s_sort_keys_u64(r2s_ctx *ctx, u64 *keys, u64 *alt, i64 n, int end_bit, u64 **sorted) {
  cub::DoubleBuffer<u64> db(keys, alt);
  size_t tmp = 0;
  CK(cub::DeviceRadixSort::SortKeys(nullptr, tmp, db, (int)n, 0, end_bit, ctx->stream));
  CK(ctx->cubtmp.reserve(tmp));
  CK(cub::DeviceRadixSort::SortKeys(ctx->cubtmp.p, tmp, db, (int)n, 0, end_bit, ctx->stream));
  ctx->launches += (end_bit + 7) / 8 + 1;
  *sorted = db.Current();
  return 0;
}
int r2s_tile_lists(r2s_ctx *ctx, u64 *keys, u64 *alt, i64 nkeys, int *tile_ptr, u64 **sorted) {
  const i64 ntiles = ctx->g.ntiles;
  int tbits = 1; while ((1ll << tbits) < ntiles) tbits++;
  *sorted = keys;
  if (nkeys > 0 && r2s_sort_keys_u64(ctx, keys, alt, nkeys, 32 + tbits, sorted)) return 1;
  CK(ctx->s_cnt.reserve(sizeof(int) * (size_t)(ntiles + 2)));
  if (r2s_scan_exclusive_i32(ctx, tile_ptr + 1, ctx->s_cnt.as<int>(), ntiles + 1)) return 1;
  CK(cudaMemcpyAsync(tile_ptr, ctx->s_cnt.as<int>(), sizeof(int) * (size_t)(ntiles + 1), cudaMemcpyDeviceToDevice, ctx->stream));
  return 0;
}

// sorts n doubles ascending (used by the edge-length median of the grid set-up)
int r2s_sort_f64(r2s_ctx *ctx, double *keys, double *alt, i64 n, double **sorted) {
  cub::DoubleBuffer<double> db(keys, alt);
  size_t tmp = 0;
  CK(cub::DeviceRadixSort::SortKeys(nullptr, tmp, db, (int)n, 0, 64, ctx->stream));
  CK(ctx->cubtmp.reserve(tmp));
  CK(cub::DeviceRadixSort::SortKeys(ctx->cubtmp.p, tmp, db, (int)n, 0, 64, ctx->stream));
  ctx->launches += 9;
  *sorted = db.Current();
  return 0;
}

int r2s_unique_f64(r2s_ctx *ctx, const double *sorted, double *out, i64 n, i64 *count) {
  size_t tmp = 0;
  CK(ctx->counters.reserve(64));
  i64 *dn = ctx->counters.as<i64>();
  CK(cub::DeviceSelect::Unique(nullptr, tmp, sorted, out, dn, (int)n, ctx->stream));
  CK(ctx->cubtmp.reserve(tmp));
  CK(cub::DeviceSelect::Unique(ctx->cubtmp.p, tmp, sorted, out, dn, (int)n, ctx->stream));
  ctx->launches += 2;
  return r2s_readback(ctx, count, dn, sizeof(i64));
}

// ------------------------------------------------------------------------------------------------ small read-backs
__global__ void k_readback(const unsigned *__restrict__ src, unsigned *__restrict__ dst, int nwords) {
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < nwords; i += gridDim.x * blockDim.x) dst[i] = src[i];
}
size_t r2s_rb_put(r2s_ctx *ctx, const void *src_dev, size_t bytes) {
  const size_t words = (bytes + 3) / 4, off = ctx->rb_off;
  if (!ctx->rb_host || off + words * 4 > R2S_RB_BYTES || ((size_t)src_dev & 3)) { ctx->err = "read-back buffer overflow / misaligned source"; return (size_t)-1; }
  const int nb = words > 4096 ? 8 : 1;
  k_readback<<<nb, 256, 0, ctx->stream>>>((const unsigned *)src_dev, (unsigned *)((char *)ctx->rb_dev + off), (int)words);
  if (cudaGetLastError() != cudaSuccess) { ctx->err = "read-back kernel launch failed"; return (size_t)-1; }
  ctx->rb_off = (off + words * 4 + 7) & ~(size_t)7;
  return off;
}
int r2s_rb_sync(r2s_ctx *ctx) {
  ctx->rb_off = 0;
  CK(cudaStreamSynchronize(ctx->stream));
  return 0;
}
int r2s_readback(r2s_ctx *ctx, void *dst_host, const void *src_dev, size_t bytes) {
  const size_t off = r2s_rb_put(ctx, src_dev, bytes);
  if (off == (size_t)-1) return 1;
  if (r2s_rb_sync(ctx)) return 1;
  memcpy(dst_host, r2s_rb_at(ctx, off), bytes);
  return 0;
}

// ------------------------------------------------------------------------------------------------ roofline denominators
// FMA-pipe peak measured on the device the context drives: 8 independent FMA chains per thread, enough CTAs to fill
// every SM.  MEASURED_PEAKS.json holds HBM and bf16-tensor peaks only; the iso-projection kernel is FP64-FMA bound
// and the fine-grid RBF evaluation FP32-FMA bound (SURVEY.md 8d), so bench.py measures those two denominators here.
template <typename T>
__global__ void __launch_bounds__(256) k_fma_peak(T *out, int iters, T a, T b) {
  T x0 = (T)threadIdx.x, x1 = x0 + (T)1, x2 = x0 + (T)2, x3 = x0 + (T)3, x4 = x0 + (T)4, x5 = x0 + (T)5, x6 = x0 + (T)6, x7 = x0 + (T)7;
  for (int i = 0; i < iters; i++) {
    x0 = x0 * a + b; x1 = x1 * a + b; x2 = x2 * a + b; x3 = x3 * a + b;
    x4 = x4 * a + b; x5 = x5 * a + b; x6 = x6 * a + b; x7 = x7 * a + b;
  }
  T s = ((x0 + x1) + (x2 + x3)) + ((x4 + x5) + (x6 + x7));
  if (s == (T)123456789) out[0] = s;          // never true; keeps the chains alive
}
template <typename T>
static int fma_peak(r2s_ctx *ctx, double *tflops) {
  CK(cudaSetDevice(ctx->device));
  CK(ctx->cubtmp.reserve(256));
  cudaDeviceProp prop; CK(cudaGetDeviceProperties(&prop, ctx->device));
  int blocks = prop.multiProcessorCount * 8, iters = 1 << 14;
  double best = 0.0;
  for (int rep = 0; rep < 5; rep++) {
    CK(cudaEventRecord(ctx->ev[0], ctx->stream));
    k_fma_peak<T><<<blocks, 256, 0, ctx->stream>>>((T *)ctx->cubtmp.p, iters, (T)0.999999, (T)1e-7);
    CK(cudaGetLastError());
    CK(cudaEventRecord(ctx->ev[1], ctx->stream));
    CK(cudaStreamSynchronize(ctx->stream));
    float ms = 0; CK(cudaEventElapsedTime(&ms, ctx->ev[0], ctx->ev[1]));
    double fl = 2.0 * 8.0 * (double)iters * 256.0 * (double)blocks;
    if (rep > 0 && ms > 0) { double t = fl / (ms * 1e-3) / 1e12; if (t > best) best = t; }
  }
  *tflops = best;
  return 0;
}
extern "C" int r2s_measure_fma_peak(r2s_ctx *ctx, int fp64, double *tflops) {
  if (!ctx || !tflops) return 1;
  return fp64 ? fma_peak<double>(ctx, tflops) : fma_peak<float>(ctx, tflops);
}
