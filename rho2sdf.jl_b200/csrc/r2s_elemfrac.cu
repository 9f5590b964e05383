// r2s_elemfrac.cu -- per-element solid volume fractions of the continuous smoothed SDF on the FE mesh (r2s_element_volume_fractions):
// calculate_isocontour_volume's rule (Isocontour_volume.jl:1-75) -- a Heaviside at the Gauss points of every element, weighted by |det J|
// -- applied to the field r2s_sample_sdf evaluates.  The point rule, the ordered sums and the element box are r2s_elemfrac.cuh.  Built with
// -fmad=false (the geometry is r2s_mesh.cu's arithmetic; the sampler spells out its own operations).
//
// Two passes over the elements [e0, e1) of a context:
//   k_ef_classify  one thread per element: its box, the block classifier of the band surface on it (r2s_band.cuh); the elements to sample
//                  go to a list through the warp-staged ws_push / ws_flush, and each warp then computes V for its skipped elements (lanes
//                  over the Gauss points, no sampler) -- their fraction is exactly 1 or 0, the bits full evaluation would give
//   k_ef_eval      one warp per listed element, lanes over its Gauss points: V and S in the fixed order of the header; the points of one
//                  element share their sampler window, so the weight gathers hit L1
// Several slabs: every point reads the weights of the slab owning its floor plane (SurfSlabW, peer memory), as r2s_multi_sample_sdf routes
// it; an element whose box reaches two slabs' floor planes is always sampled.
#include <algorithm>
#include "r2s_common.cuh"
#include "r2s_elemfrac.cuh"

struct EfArgs {
  i64 e0, n;                 // elements [e0, e0 + n) of the mesh; outputs and the list are indexed by e - e0
  const double *X;
  const int *IEN;
  int nen, npts, nslab;      // npts = q^3
  float iso;
  GaussTab G;
  const SurfSlabW *tab;
  double *frac, *vol;
  int *list;
  u64 *cnt;                  // cnt[0]: listed elements
};

__device__ __forceinline__ void ef_load(const EfArgs &A, i64 e, EfElem &E) {
  E.nen = A.nen;
  for (int a = 0; a < A.nen; a++) {
    const i64 nd = A.IEN[(i64)A.nen * e + a];
    for (int d = 0; d < 3; d++) E.xe[d][a] = A.X[3 * nd + d];
  }
}

// the slab whose weights serve a point (or a box end) at Float32 z
__device__ __forceinline__ int ef_slab(const SampleGrid &G, const EfArgs &A, float z) {
  if (A.nslab == 1) return 0;
  const int c = smp_floor(G.C[2], G.n[2], G.c0[2], G.inv[2], z);
  int r = 0;
  while (r + 1 < A.nslab && c >= A.tab[r].k1) r++;
  return r;
}

// V and S of element E into lane 0 (SAMPLE = false: V only, S = 0): lane l sums the points t = l mod 32, then the tree of the header
template <bool SAMPLE>
__device__ __forceinline__ void ef_warp_sums(const SampleGrid &G, const EfArgs &A, const EfElem &E, int lane, double *V, double *S) {
  double v = 0.0, s = 0.0;
  for (int t = lane; t < A.npts; t += R2S_EF_LANES) {
    double x[3], W;
    if (!ef_point(E, A.G, t, x, &W)) continue;
    v += W;
    if (SAMPLE) {
      SampleGrid g = G;
      if (A.nslab > 1) { const int r = ef_slab(G, A, (float)x[2]); g.w = A.tab[r].w; g.px = A.tab[r].px; }
      s += ef_inside(g, x, A.iso) ? W : 0.0;
    }
  }
#pragma unroll
  for (int o = R2S_EF_LANES / 2; o > 0; o >>= 1) {
    v += __shfl_down_sync(0xffffffffu, v, o);
    if (SAMPLE) s += __shfl_down_sync(0xffffffffu, s, o);
  }
  *V = v; *S = s;
}

#define EF_THREADS 256
__global__ void __launch_bounds__(EF_THREADS) k_ef_classify(SampleGrid G, EfArgs A) {
  __shared__ int s_list[EF_THREADS / 32][WS_CAP];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const i64 t = blockIdx.x * (i64)blockDim.x + threadIdx.x;
  const bool valid = t < A.n;
  int c = 0;
  if (valid) {
    EfElem E;
    ef_load(A, A.e0 + t, E);
    float a[3], b[3];
    ef_box(E, a, b);
    const int r = ef_slab(G, A, a[2]);
    if (r == ef_slab(G, A, b[2])) {
      SampleGrid g = G;
      g.w = A.tab[r].w; g.px = A.tab[r].px;
      c = band_classify_box(g, a, b, A.iso, band_margin());
    }
  }
  int n = 0;
  ws_push<int>(s_list[warp], n, valid && c == 0, (int)t, A.list, A.cnt, A.n, lane);
  ws_flush<int>(s_list[warp], n, A.list, A.cnt, A.n, lane);
  // the warp's skipped elements, one after the other: V from the geometry; S is V (every point inside) or +0 (none)
  unsigned m = __ballot_sync(0xffffffffu, valid && c != 0);
  while (m) {
    const int src = __ffs(m) - 1;
    m &= m - 1;
    const i64 ts = t - lane + src;
    const int cs = __shfl_sync(0xffffffffu, c, src);
    EfElem E;
    ef_load(A, A.e0 + ts, E);
    double V, S;
    ef_warp_sums<false>(G, A, E, lane, &V, &S);
    if (lane == 0) {
      S = cs == 1 ? V : 0.0;
      A.vol[ts] = V; A.frac[ts] = ef_fraction(S, V);
    }
  }
}

__global__ void __launch_bounds__(EF_THREADS) k_ef_eval(SampleGrid G, EfArgs A, i64 nlist) {
  const i64 w = (blockIdx.x * (i64)blockDim.x + threadIdx.x) >> 5;
  const int lane = threadIdx.x & 31;
  if (w >= nlist) return;      // warp-uniform
  const i64 t = A.list[w];
  EfElem E;
  ef_load(A, A.e0 + t, E);
  double V, S;
  ef_warp_sums<true>(G, A, E, lane, &V, &S);
  if (lane == 0) { A.vol[t] = V; A.frac[t] = ef_fraction(S, V); }
}

// the argument checks of both entry points, on the context that serves them (slab 0 of r2s_multi)
int r2s_ef_check(r2s_ctx *ctx, float iso, int quad_order, const double *fractions) {
  if (quad_order < 1 || quad_order > 32) FAIL("element volume fractions: quad_order must be in 1..32");
  if (!isfinite(iso)) FAIL("element volume fractions: iso must be finite");
  if (!fractions) FAIL("element volume fractions: fractions is required");
  if (ctx->nel == 0) FAIL("r2s_set_mesh has not been called");
  SampleGrid G;
  return r2s_sample_grid(ctx, &G, false);
}

// the elements [e0, e1) of this context's mesh: fractions and (if vol) volumes into frac[0 .. e1 - e0), the elements sampled into *nev
int r2s_ef_range(r2s_ctx *ctx, const std::vector<SurfSlabW> &slabs, i64 e0, i64 e1, float iso, int quad_order, double *frac, double *vol, i64 *nev) {
  *nev = 0;
  SampleGrid G;
  if (r2s_sample_grid(ctx, &G, true)) return 1;
  const i64 n = e1 - e0;
  if (n <= 0) return 0;
  CK(cudaSetDevice(ctx->device));
  const size_t nb = sizeof(double) * 2 * (size_t)n, wb = sizeof(SurfSlabW) * slabs.size();
  struct Scratch : DevBuf { ~Scratch() { release(); } } buf;      // freed on every return
  CK(buf.reserve(nb + 16 + wb + sizeof(int) * (size_t)n));
  EfArgs A;
  A.e0 = e0; A.n = n; A.X = ctx->X.as<double>(); A.IEN = ctx->IEN32.as<int>(); A.nen = ctx->nen;
  A.G = gauss_legendre_host(quad_order); A.npts = quad_order * quad_order * quad_order;
  A.iso = iso; A.nslab = (int)slabs.size();
  A.frac = buf.as<double>(); A.vol = A.frac + n;
  A.cnt = (u64 *)(A.vol + n);
  A.tab = (const SurfSlabW *)(A.cnt + 2);
  A.list = (int *)((char *)A.tab + wb);
  CK(cudaMemsetAsync(A.cnt, 0, 16, ctx->stream));
  CK(cudaMemcpyAsync((void *)A.tab, slabs.data(), wb, cudaMemcpyHostToDevice, ctx->stream));
  k_ef_classify<<<cdiv(n, EF_THREADS), EF_THREADS, 0, ctx->stream>>>(G, A);
  LAUNCH_CHECK();
  u64 nlist = 0;
  if (r2s_readback(ctx, &nlist, A.cnt, sizeof(u64))) return 1;
  if (nlist > 0) {
    k_ef_eval<<<cdiv((i64)nlist * 32, EF_THREADS), EF_THREADS, 0, ctx->stream>>>(G, A, (i64)nlist);
    LAUNCH_CHECK();
  }
  CK(cudaMemcpyAsync(frac, A.frac, sizeof(double) * (size_t)n, cudaMemcpyDeviceToHost, ctx->stream));
  if (vol) CK(cudaMemcpyAsync(vol, A.vol, sizeof(double) * (size_t)n, cudaMemcpyDeviceToHost, ctx->stream));
  CK(cudaStreamSynchronize(ctx->stream));
  *nev = (i64)nlist;
  return 0;
}

extern "C" int r2s_element_volume_fractions(r2s_ctx *ctx, float iso, int quad_order, double *fractions, double *volumes, int64_t *n_evaluated) {
  if (!ctx) return 1;
  if (ctx->nranks > 1)
    FAIL(ctx->lg ? "r2s_element_volume_fractions: this context is one slab of an r2s_multi group; use r2s_multi_element_volume_fractions"
                 : "r2s_element_volume_fractions: not available on a slab rank of the NCCL communicator (one process per GPU); use one context or r2s_multi");
  if (r2s_ef_check(ctx, iso, quad_order, fractions)) return 1;
  i64 nev = 0;
  if (r2s_ef_range(ctx, std::vector<SurfSlabW>(1, SurfSlabW{INT64_MAX, ctx->rbf_w, (long long)ctx->rbf_px}), 0, ctx->nel, iso, quad_order, fractions, volumes, &nev))
    return 1;
  if (n_evaluated) *n_evaluated = nev;
  return 0;
}
