// r2s_sample.cu -- the continuous smoothed SDF of the last smoothing call (rbf_interpolation_kdtree, SdfSmoothing/RBFs4Smoothing.jl:219-248)
// at arbitrary points and on any lattice, with an optional analytic gradient.  The per-point arithmetic is r2s_sample.cuh.
//
// The weights and the offset th stay where r2s_dev_rbf left them (r2s_sample_record); nothing here writes them.  Host arrays pass through
// a bounded device staging buffer in chunks of SMP_CHUNK points, so the point count is limited by host memory only.
#include <math.h>
#include <algorithm>
#include "r2s_common.cuh"
#include "r2s_sample.cuh"

#define SMP_CHUNK (1ll << 22)      // points per staging chunk: 96 MB of coordinates, 64 MB of values + gradients
#define SL_X 16                    // lattice tile of one CTA: 16 x 4 x 4 points, a compact box whose weight rows are shared through L1
#define SL_Y 4
#define SL_Z 4

// one thread per point; pts: x y z per point (double); err: set to 1 when a coordinate is not finite
template <bool GRAD>
__global__ void __launch_bounds__(256) k_sample_points(SampleGrid G, i64 n, const double *__restrict__ pts, float *__restrict__ val, float *__restrict__ grad,
                                                       int *__restrict__ err) {
  const i64 t = blockIdx.x * (i64)blockDim.x + threadIdx.x;
  if (t >= n) return;
  const double X = pts[3 * t], Y = pts[3 * t + 1], Z = pts[3 * t + 2];
  if (!isfinite(X) || !isfinite(Y) || !isfinite(Z)) { *err = 1; return; }
  float g[3];
  const float v = sample_point<GRAD>(G, __double2float_rn(X), __double2float_rn(Y), __double2float_rn(Z), g);
  val[t] = v;
  if (GRAD) { grad[3 * t] = g[0]; grad[3 * t + 1] = g[1]; grad[3 * t + 2] = g[2]; }
}

// the box [i0, i0 + bx) x [j0, j0 + by) x [k0, k0 + bz) of the lattice o + float(i) h, written x fastest into out
struct LatBox { float o[3], h[3]; int i0, j0, k0, bx, by, bz, tx, ty; };
__global__ void __launch_bounds__(SL_X *SL_Y *SL_Z) k_sample_lattice(SampleGrid G, LatBox B, float *__restrict__ out) {
  const i64 b = blockIdx.x;
  const int tx = (int)(b % B.tx), ty = (int)((b / B.tx) % B.ty), tz = (int)(b / ((i64)B.tx * B.ty));
  const int bi = tx * SL_X + threadIdx.x % SL_X, bj = ty * SL_Y + (threadIdx.x / SL_X) % SL_Y, bk = tz * SL_Z + threadIdx.x / (SL_X * SL_Y);
  if (bi >= B.bx || bj >= B.by || bk >= B.bz) return;
  const float x = smp_add(B.o[0], smp_mul((float)(B.i0 + bi), B.h[0]));
  const float y = smp_add(B.o[1], smp_mul((float)(B.j0 + bj), B.h[1]));
  const float z = smp_add(B.o[2], smp_mul((float)(B.k0 + bk), B.h[2]));
  out[((i64)bk * B.by + bj) * B.bx + bi] = sample_point<false>(G, x, y, z, nullptr);
}

// called at the end of r2s_dev_rbf: w (row pitch px, whole-grid plane indexing) and th define the field until the next smoothing call
int r2s_sample_record(r2s_ctx *ctx, const float *w, int px, float th, double rbf_cut) {
  const GridDev &g = ctx->g;
  i64 tot = 0;
  for (int d = 0; d < 3; d++) {
    ctx->rbf_c[d].resize((size_t)g.np[d]);
    smp_range(g.amin[d], g.amax[d], g.np[d], ctx->rbf_c[d].data());
    // candidates are looked for within [c - 2, c + 3] of the floor plane c: that holds every point within maxd < sqrt(8) cells only if
    // no step of the Float32 table is below maxd / 3
    const float md = smp_maxd(rbf_cut, g.cell);
    for (int i = 0; i + 1 < g.np[d]; i++)
      if (!((double)ctx->rbf_c[d][(size_t)i + 1] - ctx->rbf_c[d][(size_t)i] > (double)md / 3.0)) FAIL("sampling: the grid's coordinate steps do not match cell_size");
    tot += g.np[d];
  }
  CK(ctx->rbf_tab.reserve(sizeof(float) * (size_t)tot));
  i64 off = 0;
  for (int d = 0; d < 3; d++) {
    CK(cudaMemcpyAsync(ctx->rbf_tab.as<float>() + off, ctx->rbf_c[d].data(), sizeof(float) * (size_t)g.np[d], cudaMemcpyHostToDevice, ctx->stream));
    off += g.np[d];
  }
  CK(cudaStreamSynchronize(ctx->stream));
  ctx->rbf_w = w; ctx->rbf_px = px; ctx->rbf_th = th; ctx->rbf_cut = rbf_cut; ctx->have_rbf = true;
  return 0;
}

// the sampler state of this context; dev = true: coordinate tables on the device (kernels), else on the host (routing)
int r2s_sample_grid(r2s_ctx *ctx, SampleGrid *G, bool dev) {
  if (!ctx->has_grid) FAIL("r2s_set_grid has not been called");
  if (!ctx->have_rbf) FAIL("sampling: no smoothed field for the current grid on the device yet (run the pipeline or the smoothing first)");
  const GridDev &g = ctx->g;
  const float *C[3] = {ctx->rbf_c[0].data(), ctx->rbf_c[1].data(), ctx->rbf_c[2].data()};
  smp_setup(G, ctx->rbf_w, ctx->rbf_px, C, g.np, g.cell, ctx->rbf_cut, ctx->rbf_th);
  if (dev) { G->C[0] = ctx->rbf_tab.as<float>(); G->C[1] = G->C[0] + g.np[0]; G->C[2] = G->C[1] + g.np[1]; }
  return 0;
}

static int rank_check(r2s_ctx *ctx, const char *who) {
  if (ctx->nranks > 1) {
    ctx->err = std::string(who) + (ctx->lg ? ": this context is one slab of an r2s_multi group; use the r2s_multi_ variant"
                                           : ": not available on a slab rank of the NCCL communicator (one process per GPU); sample on one context or with r2s_multi");
    return 1;
  }
  return 0;
}

// points of this context (the caller checked the rank): values and, if grad, gradients
int r2s_sample_points_ctx(r2s_ctx *ctx, const double *pts, i64 n, float *val, float *grad) {
  if (n < 0) FAIL("sampling: negative point count");
  if (n > 0 && (!pts || !val)) FAIL("sampling: points and values are required when n > 0");
  SampleGrid G;
  if (r2s_sample_grid(ctx, &G, true)) return 1;
  if (n == 0) return 0;
  CK(cudaSetDevice(ctx->device));
  const i64 ch = std::min<i64>(n, SMP_CHUNK);
  CK(ctx->smp_in.reserve(sizeof(double) * 3 * (size_t)ch));
  CK(ctx->smp_out.reserve(sizeof(float) * 4 * (size_t)ch + 64));
  int *err = (int *)(ctx->smp_out.as<char>() + sizeof(float) * 4 * (size_t)ch);
  CK(cudaMemsetAsync(err, 0, sizeof(int), ctx->stream));
  float *dv = ctx->smp_out.as<float>(), *dg = dv + ch;
  for (i64 s = 0; s < n; s += ch) {
    const i64 m = std::min(ch, n - s);
    CK(cudaMemcpyAsync(ctx->smp_in.p, pts + 3 * s, sizeof(double) * 3 * (size_t)m, cudaMemcpyHostToDevice, ctx->stream));
    if (grad) k_sample_points<true><<<cdiv(m, 256), 256, 0, ctx->stream>>>(G, m, ctx->smp_in.as<double>(), dv, dg, err);
    else k_sample_points<false><<<cdiv(m, 256), 256, 0, ctx->stream>>>(G, m, ctx->smp_in.as<double>(), dv, nullptr, err);
    LAUNCH_CHECK();
    CK(cudaMemcpyAsync(val + s, dv, sizeof(float) * (size_t)m, cudaMemcpyDeviceToHost, ctx->stream));
    if (grad) CK(cudaMemcpyAsync(grad + 3 * s, dg, sizeof(float) * 3 * (size_t)m, cudaMemcpyDeviceToHost, ctx->stream));
    int herr = 0;
    CK(cudaMemcpyAsync(&herr, err, sizeof(int), cudaMemcpyDeviceToHost, ctx->stream));
    CK(cudaStreamSynchronize(ctx->stream));
    if (herr) FAIL("sampling: a point coordinate is NaN or infinite");
  }
  return 0;
}

// lattice origin / spacing as Float32, with the finiteness and dims checks every entry point shares
int r2s_sample_lattice_check(r2s_ctx *ctx, const double origin[3], const double spacing[3], const int64_t dims[3], float o[3], float h[3]) {
  if (!origin || !spacing || !dims) FAIL("sampling: origin, spacing and dims are required");
  for (int d = 0; d < 3; d++) {
    if (dims[d] < 1) FAIL("sampling: lattice dims must be >= 1");
    if (dims[d] > (1ll << 31) - 1) FAIL("sampling: lattice dims must be < 2^31");
    o[d] = (float)origin[d]; h[d] = (float)spacing[d];
    const float last = smp_add(o[d], smp_mul((float)(dims[d] - 1), h[d]));
    if (!std::isfinite(origin[d]) || !std::isfinite(spacing[d]) || !std::isfinite(o[d]) || !std::isfinite(h[d]) || !std::isfinite(last))
      FAIL("sampling: a lattice coordinate is NaN or infinite");
  }
  return 0;
}

// the lattice planes [ka, kb) of a dims lattice into out (x fastest, plane ka first), in boxes of at most SMP_CHUNK points
int r2s_sample_lattice_planes(r2s_ctx *ctx, const float o[3], const float h[3], const int64_t dims[3], i64 ka, i64 kb, float *out) {
  SampleGrid G;
  if (r2s_sample_grid(ctx, &G, true)) return 1;
  if (!out) FAIL("sampling: values are required");
  CK(cudaSetDevice(ctx->device));
  CK(ctx->smp_out.reserve(sizeof(float) * (size_t)SMP_CHUNK));
  const i64 nx = dims[0], ny = dims[1], pl = nx * ny;
  // a box is several whole planes, or several whole rows of one plane, or a piece of one row: its values are contiguous in out
  i64 bz = 1, by = 1, bx = nx;
  if (pl <= SMP_CHUNK) { bz = SMP_CHUNK / pl; by = ny; }
  else if (nx <= SMP_CHUNK) by = SMP_CHUNK / nx;
  else bx = SMP_CHUNK;
  for (i64 k = ka; k < kb; k += bz)
    for (i64 j = 0; j < ny; j += by)
      for (i64 i = 0; i < nx; i += bx) {
        LatBox B;
        for (int d = 0; d < 3; d++) { B.o[d] = o[d]; B.h[d] = h[d]; }
        B.i0 = (int)i; B.j0 = (int)j; B.k0 = (int)k;
        B.bx = (int)std::min(bx, nx - i); B.by = (int)std::min(by, ny - j); B.bz = (int)std::min(bz, kb - k);
        B.tx = cdiv(B.bx, SL_X); B.ty = cdiv(B.by, SL_Y);
        const i64 nb = (i64)B.tx * B.ty * cdiv(B.bz, SL_Z), m = (i64)B.bx * B.by * B.bz;
        k_sample_lattice<<<(unsigned)nb, SL_X * SL_Y * SL_Z, 0, ctx->stream>>>(G, B, ctx->smp_out.as<float>());
        LAUNCH_CHECK();
        CK(cudaMemcpyAsync(out + (k - ka) * pl + j * nx + i, ctx->smp_out.p, sizeof(float) * (size_t)m, cudaMemcpyDeviceToHost, ctx->stream));
        CK(cudaStreamSynchronize(ctx->stream));
      }
  return 0;
}

// this context's weight planes [k0, k1) into the whole-grid array w (unpitched, x fastest)
int r2s_sample_download_weights(r2s_ctx *ctx, float *w, float *th, i64 k0, i64 k1) {
  SampleGrid G;
  if (r2s_sample_grid(ctx, &G, true)) return 1;
  CK(cudaSetDevice(ctx->device));
  const GridDev &g = ctx->g;
  const size_t nx = (size_t)g.np[0], ny = (size_t)g.np[1];
  if (w && k1 > k0)
    CK(cudaMemcpy2DAsync(w + (size_t)k0 * ny * nx, nx * sizeof(float), ctx->rbf_w + (size_t)k0 * ny * (size_t)ctx->rbf_px, (size_t)ctx->rbf_px * sizeof(float),
                         nx * sizeof(float), (size_t)(k1 - k0) * ny, cudaMemcpyDeviceToHost, ctx->stream));
  CK(cudaStreamSynchronize(ctx->stream));
  if (th) *th = ctx->rbf_th;
  return 0;
}

extern "C" {

int r2s_sample_sdf(r2s_ctx *ctx, const double *points, int64_t n, float *values, float *gradients) {
  if (!ctx) return 1;
  if (rank_check(ctx, "r2s_sample_sdf")) return 1;
  return r2s_sample_points_ctx(ctx, points, n, values, gradients);
}

int r2s_sample_sdf_lattice(r2s_ctx *ctx, const double origin[3], const double spacing[3], const int64_t dims[3], float *values) {
  if (!ctx) return 1;
  if (rank_check(ctx, "r2s_sample_sdf_lattice")) return 1;
  float o[3], h[3];
  if (r2s_sample_lattice_check(ctx, origin, spacing, dims, o, h)) return 1;
  return r2s_sample_lattice_planes(ctx, o, h, dims, 0, dims[2], values);
}

int r2s_download_rbf_weights(r2s_ctx *ctx, float *weights, float *th) {
  if (!ctx) return 1;
  if (rank_check(ctx, "r2s_download_rbf_weights")) return 1;
  if (!weights && !th) FAIL("r2s_download_rbf_weights: weights or th is required");
  return r2s_sample_download_weights(ctx, weights, th, 0, ctx->has_grid ? ctx->g.np[2] : 0);
}

}  // extern "C"
