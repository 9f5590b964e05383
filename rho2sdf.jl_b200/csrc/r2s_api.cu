// r2s_api.cu -- the C ABI of libr2s.so (include/r2s.h): context, mesh/grid upload, per-stage entry points, pipeline
#include <math.h>
#include <stdlib.h>
#include <string.h>
#include <new>
#include "r2s_common.cuh"


extern "C" {

int r2s_create(r2s_ctx **out, int device, void *stream) {
  if (!out) return 1;
  *out = nullptr;
  int ndev = 0;
  if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0 || device < 0 || device >= ndev) return 2;   // no CPU fallback
  r2s_ctx *ctx = new (std::nothrow) r2s_ctx();
  if (!ctx) return 3;
  ctx->device = device;
  memset(&ctx->rep, 0, sizeof(ctx->rep));
  if (cudaSetDevice(device) != cudaSuccess) { delete ctx; return 4; }
  if (stream) { ctx->stream = (cudaStream_t)stream; ctx->own_stream = false; }
  else { if (cudaStreamCreateWithFlags(&ctx->stream, cudaStreamNonBlocking) != cudaSuccess) { delete ctx; return 5; } ctx->own_stream = true; }
  for (int i = 0; i < 16; i++) cudaEventCreate(&ctx->ev[i]);
  for (int i = 0; i < 5; i++) { cudaEventCreate(&ctx->ev_probe[i]); cudaEventCreate(&ctx->ev_k[i]); }
  cudaStreamCreateWithFlags(&ctx->copy_stream, cudaStreamNonBlocking);
  for (int i = 0; i < 64; i++) cudaEventCreateWithFlags(&ctx->ev_copy[i], cudaEventDisableTiming);
  for (int i = 0; i < 2; i++) cudaEventCreateWithFlags(&ctx->ev_done[i], cudaEventDisableTiming);
  if (cudaHostAlloc(&ctx->rb_host, R2S_RB_BYTES, cudaHostAllocMapped) != cudaSuccess || cudaHostGetDevicePointer(&ctx->rb_dev, ctx->rb_host, 0) != cudaSuccess) { r2s_destroy(ctx); return 6; }
  auto knob = [](const char *name, int dflt) { const char *e = getenv(name); return e ? atoi(e) : dflt; };
  ctx->knobs.p2p = knob("R2S_P2P", 1); ctx->knobs.sign_lattice = knob("R2S_SIGN_LATTICE", 1);
  ctx->knobs.proj_box = knob("R2S_PROJ_BOX", 1); ctx->knobs.proj_prune = knob("R2S_PROJ_PRUNE", 1); ctx->knobs.vol_cache = knob("R2S_VOL_CACHE", 1); ctx->knobs.debug_sync = knob("R2S_DEBUG_SYNC", 0);
  *out = ctx;
  return 0;
}
void r2s_destroy(r2s_ctx *ctx) {
  if (!ctx) return;
  cudaSetDevice(ctx->device);
  cudaStreamSynchronize(ctx->stream);
  r2s_comm_destroy(ctx);
  DevBuf *all[] = {&ctx->X, &ctx->IEN32, &ctx->ine_ptr, &ctx->ine_el, &ctx->fbnd, &ctx->ezr, &ctx->ebox, &ctx->rho_e, &ctx->rho_n, &ctx->gtab_d, &ctx->gtab_i, &ctx->cls, &ctx->act_flag,
                   &ctx->act_idx, &ctx->act_rec, &ctx->cnt_a, &ctx->cnt_b, &ctx->keys, &ctx->keys_alt, &ctx->tile_ptr, &ctx->tile_faces, &ctx->face_tiles, &ctx->fc_list, &ctx->tri_cnt, &ctx->tri_rec, &ctx->pairbuf, &ctx->pairxp, &ctx->cubtmp,
                   &ctx->counters, &ctx->box_rec, &ctx->plist, &ctx->dist, &ctx->xp, &ctx->sdf, &ctx->signs, &ctx->s_rng, &ctx->s_el, &ctx->s_cnt, &ctx->s_keys, &ctx->s_keys_alt, &ctx->s_tile_ptr,
                   &ctx->cc_label, &ctx->cc_size, &ctx->cc_scal, &ctx->cc_bits, &ctx->cc_bits_all, &ctx->cc_gsz, &ctx->cc_seen, &ctx->f_s, &ctx->f_w, &ctx->f_r, &ctx->f_u, &ctx->f_c, &ctx->f_lsf, &ctx->f_fine, &ctx->f_part,
                   &ctx->f_scal, &ctx->cutlist, &ctx->slablist, &ctx->v_part, &ctx->vlist[0], &ctx->vlist[1], &ctx->vent[0], &ctx->vent[1], &ctx->vrec, &ctx->bis_state, &ctx->lat_xs, &ctx->lat_cell, &ctx->lat_map, &ctx->lat_info, &ctx->lat_pt,
                   &ctx->surf_rows, &ctx->surf_V, &ctx->surf_T, &ctx->rbf_tab, &ctx->smp_in, &ctx->smp_out, &ctx->pt_rn, &ctx->pt_cls, &ctx->pt_flag, &ctx->pt_idx,
                   &ctx->pt_rec, &ctx->pt_hex, &ctx->pt_cnt, &ctx->pt_off, &ctx->pt_tkeys, &ctx->pt_tkeys_alt, &ctx->pt_tile_ptr, &ctx->pt_tri, &ctx->pt_in, &ctx->pt_keys, &ctx->pt_keys_alt,
                   &ctx->pt_out, &ctx->pt_ctr};
  for (DevBuf *b : all) b->release();
  for (int i = 0; i < 16; i++) cudaEventDestroy(ctx->ev[i]);
  for (int i = 0; i < 5; i++) { cudaEventDestroy(ctx->ev_probe[i]); cudaEventDestroy(ctx->ev_k[i]); }
  for (int i = 0; i < 64; i++) cudaEventDestroy(ctx->ev_copy[i]);
  for (int i = 0; i < 2; i++) cudaEventDestroy(ctx->ev_done[i]);
  if (ctx->copy_stream) cudaStreamDestroy(ctx->copy_stream);
  if (ctx->rb_host) cudaFreeHost(ctx->rb_host);
  if (ctx->own_stream) cudaStreamDestroy(ctx->stream);
  delete ctx;
}
const char *r2s_last_error(r2s_ctx *ctx) { return ctx ? ctx->err.c_str() : "r2s: no context (no CUDA device?)"; }

void r2s_default_params(r2s_params *p) {
  p->rho_t = 0.5; p->delta_factor = 1.1; p->remove_artifacts = 1; p->artifact_threshold = 0.0; p->artifact_min_ratio = 0.01;
  p->rbf_interp = 1; p->smooth = 1; p->rbf_cut = 1e-3; p->target_volume = 0.0; p->final_volume = 1;
}
int r2s_last_report(r2s_ctx *ctx, r2s_report *rep) { if (!ctx || !rep) return 1; *rep = ctx->rep; return 0; }

int r2s_set_mesh(r2s_ctx *ctx, int nen, int64_t nnp, const double *X, int64_t nel, const int64_t *IEN) {
  if (!ctx) return 1;
  if (nen != 8 && nen != 4) FAIL("r2s_set_mesh: nen must be 8 (HEX8) or 4 (TET4)");
  if (nnp <= 0 || nel <= 0 || !X || !IEN) FAIL("r2s_set_mesh: empty mesh");
  if (nel * nen >= (1ll << 31) || nnp >= (1ll << 31)) FAIL("r2s_set_mesh: mesh too large for 32-bit connectivity");
  CK(cudaSetDevice(ctx->device));
  for (i64 t = 0; t < nel * nen; t++) if (IEN[t] < 1 || IEN[t] > nnp) FAIL("r2s_set_mesh: IEN entry out of range (expected 1-based node ids)");
  ctx->have_sdf = ctx->have_fine = ctx->have_rbf = ctx->have_surface = false;
  ctx->nen = nen; ctx->nes = nen == 8 ? 6 : 4; ctx->nsn = nen == 8 ? 4 : 3; ctx->nnp = nnp; ctx->nel = nel;
  CK(ctx->X.reserve(sizeof(double) * 3 * (size_t)nnp));
  CK(ctx->IEN32.reserve(sizeof(int) * (size_t)(nel * nen)));
  CK(cudaMemcpyAsync(ctx->X.p, X, sizeof(double) * 3 * (size_t)nnp, cudaMemcpyHostToDevice, ctx->stream));
  if (r2s_mesh_upload_ien(ctx, IEN)) return 1;
  CK(ctx->rho_e.reserve(sizeof(double) * (size_t)nel));
  CK(ctx->rho_n.reserve(sizeof(double) * (size_t)nnp));
  if (r2s_mesh_build_tables(ctx)) return 1;
  return r2s_mesh_build_lattice(ctx);
}

int r2s_set_grid(r2s_ctx *ctx, const double amin[3], const double amax[3], const int64_t N[3], double cell) {
  if (!ctx) return 1;
  CK(cudaSetDevice(ctx->device));
  GridDev &g = ctx->g;
  i64 ngp = 1, tot_p = 0, tot_c = 0;
  for (int d = 0; d < 3; d++) {
    if (N[d] < 1 || N[d] > 100000 || !(amax[d] > amin[d])) FAIL("r2s_set_grid: invalid grid");
    g.amin[d] = amin[d]; g.amax[d] = amax[d]; g.N[d] = (int)N[d]; g.np[d] = (int)N[d] + 1; ngp *= (N[d] + 1);
    g.pc_off[d] = (int)tot_p; g.cs_off[d] = (int)tot_c; tot_p += N[d] + 1; tot_c += N[d] + 3;
  }
  g.cell = cell; g.ngp = ngp;
  g.nt[0] = cdiv(g.np[0], TILE_X); g.nt[1] = cdiv(g.np[1], TILE_Y); g.nt[2] = cdiv(g.np[2], TILE_Z);
  g.ntiles = (i64)g.nt[0] * g.nt[1] * g.nt[2];
  if (g.ntiles >= (1ll << 31)) FAIL("r2s_set_grid: too many tiles");
  // per-axis tables in the reference's operation order (Grid.jl:58,87); host code is built with -ffp-contract=off
  std::vector<double> pc((size_t)tot_p);
  std::vector<int> it((size_t)(tot_p + tot_c));
  for (int d = 0; d < 3; d++) {
    ctx->h_pc[d].resize((size_t)g.np[d]);
    for (int i = 0; i < g.np[d]; i++) {
      volatile double prod = cell * (double)i;
      volatile double x = amin[d] + prod;
      volatile double diff = x - amin[d];
      volatile double num = (double)g.N[d] * diff;
      volatile double den = amax[d] - amin[d];
      double q = num / den;
      pc[(size_t)g.pc_off[d] + i] = x; ctx->h_pc[d][(size_t)i] = x;
      it[(size_t)g.pc_off[d] + i] = (int)floor(q);
    }
    int p = 0;
    for (int c = 0; c <= g.N[d] + 1; c++) {
      while (p <= g.N[d] && it[(size_t)g.pc_off[d] + p] < c) p++;
      it[(size_t)tot_p + g.cs_off[d] + c] = p;
    }
  }
  CK(ctx->gtab_d.reserve(sizeof(double) * (size_t)tot_p));
  CK(ctx->gtab_i.reserve(sizeof(int) * (size_t)(tot_p + tot_c)));
  CK(cudaMemcpyAsync(ctx->gtab_d.p, pc.data(), sizeof(double) * (size_t)tot_p, cudaMemcpyHostToDevice, ctx->stream));
  CK(cudaMemcpyAsync(ctx->gtab_i.p, it.data(), sizeof(int) * (size_t)(tot_p + tot_c), cudaMemcpyHostToDevice, ctx->stream));
  CK(cudaStreamSynchronize(ctx->stream));
  g.pc = ctx->gtab_d.as<double>(); g.cellof = ctx->gtab_i.as<int>(); g.cstart = ctx->gtab_i.as<int>() + tot_p;
  ctx->has_grid = true; ctx->k0 = 0; ctx->k1 = g.np[2];
  ctx->have_sdf = ctx->have_fine = ctx->have_rbf = ctx->have_surface = false; ctx->slab_k0.clear();
  return 0;
}
int r2s_set_slab(r2s_ctx *ctx, int64_t k0, int64_t k1) {
  if (!ctx) return 1;
  if (!ctx->has_grid) FAIL("r2s_set_slab: call r2s_set_grid first");
  if (k0 < 0 || k1 > ctx->g.np[2] || k0 >= k1) FAIL("r2s_set_slab: invalid plane range");
  if (ctx->nranks > 1 && k1 - k0 < 3) FAIL("r2s_set_slab: a slab needs at least 3 planes (smoothing halo)");
  ctx->k0 = k0; ctx->k1 = k1;
  ctx->slab_k0.clear(); ctx->have_sdf = ctx->have_fine = ctx->have_rbf = ctx->have_surface = false;
  if (ctx->nranks > 1) {
    // every rank learns the whole partition (collective: all ranks call r2s_set_slab); slabs must tile [0, N3+1) in rank order
    CK(cudaSetDevice(ctx->device));
    CK(ctx->cc_scal.reserve(sizeof(unsigned) * 2 * 64 + 64));
    if (ctx->nranks > 64) FAIL("r2s_set_slab: more than 64 slabs");
    unsigned mine[2] = {(unsigned)k0, (unsigned)k1}, all[128];
    unsigned *d = ctx->cc_scal.as<unsigned>();
    CK(cudaMemcpyAsync(d + 2 * ctx->rank, mine, sizeof(mine), cudaMemcpyHostToDevice, ctx->stream));
    if (r2s_allgather_u32(ctx, d + 2 * ctx->rank, d, 2)) return 1;
    CK(cudaMemcpyAsync(all, d, sizeof(unsigned) * 2 * (size_t)ctx->nranks, cudaMemcpyDeviceToHost, ctx->stream));
    CK(cudaStreamSynchronize(ctx->stream));
    for (int r = 0; r < ctx->nranks; r++) {
      if ((r == 0 && all[0] != 0) || (r > 0 && all[2 * r] != all[2 * r - 1]) || all[2 * r + 1] - all[2 * r] < 3)
        FAIL("r2s_set_slab: slabs must tile the planes contiguously in rank order, at least 3 planes each");
      ctx->slab_k0.push_back((int)all[2 * r]);
    }
    if ((int)all[2 * ctx->nranks - 1] != ctx->g.np[2]) FAIL("r2s_set_slab: slabs do not cover the grid");
    ctx->slab_k0.push_back(ctx->g.np[2]);
  }
  return 0;
}

static int upload_rho_n(r2s_ctx *ctx, const double *rho_n) {
  if (ctx->nnp == 0) FAIL("r2s_set_mesh has not been called");
  CK(cudaSetDevice(ctx->device));
  CK(cudaMemcpyAsync(ctx->rho_n.p, rho_n, sizeof(double) * (size_t)ctx->nnp, cudaMemcpyHostToDevice, ctx->stream));
  return 0;
}
static int upload_rho_e(r2s_ctx *ctx, const double *rho_e) {
  if (ctx->nel == 0) FAIL("r2s_set_mesh has not been called");
  CK(cudaSetDevice(ctx->device));
  CK(cudaMemcpyAsync(ctx->rho_e.p, rho_e, sizeof(double) * (size_t)ctx->nel, cudaMemcpyHostToDevice, ctx->stream));
  return 0;
}

int r2s_mesh_volume(r2s_ctx *ctx, const double *rho_e, double *V_domain, double *V_frac) {
  if (!ctx) return 1;
  ctx->launches = 0;
  if (upload_rho_e(ctx, rho_e)) return 1;
  return r2s_dev_mesh_volume(ctx, V_domain, V_frac);
}
int r2s_nodal_densities(r2s_ctx *ctx, const double *rho_e, double *rho_n) {
  if (!ctx) return 1;
  ctx->launches = 0;
  if (upload_rho_e(ctx, rho_e)) return 1;
  if (r2s_dev_nodal_densities(ctx)) return 1;
  CK(cudaMemcpyAsync(rho_n, ctx->rho_n.p, sizeof(double) * (size_t)ctx->nnp, cudaMemcpyDeviceToHost, ctx->stream));
  CK(cudaStreamSynchronize(ctx->stream));
  return 0;
}
int r2s_isocontour_volume(r2s_ctx *ctx, const double *rho_n, double threshold, double *volume) {
  if (!ctx) return 1;
  ctx->launches = 0;
  if (upload_rho_n(ctx, rho_n)) return 1;
  return r2s_dev_isocontour_volume(ctx, threshold, volume);
}
// find_threshold_for_volume (MeshGrid/Isocontour_volume.jl:77-154)
int r2s_find_threshold(r2s_ctx *ctx, const double *rho_n, double target, double rtol, int maxit, double *rho_t) {
  if (!ctx) return 1;
  ctx->launches = 0;
  if (upload_rho_n(ctx, rho_n)) return 1;
  double lo = 0.0, hi = 1.0, vmin, vmax;
  if (r2s_dev_isocontour_volume(ctx, hi, &vmin)) return 1;
  if (r2s_dev_isocontour_volume(ctx, lo, &vmax)) return 1;
  if (target > vmax || target < vmin) {
    char b[256]; snprintf(b, sizeof(b), "Requested volume %.17g is outside the possible range [%.17g, %.17g]", target, vmin, vmax);
    FAIL(b);
  }
  int it = 0; double best = 0.0, best_err = INFINITY;
  while (it < maxit) {
    double th = (lo + hi) / 2, v;
    if (r2s_dev_isocontour_volume(ctx, th, &v)) return 1;
    double err = fabs(v - target) / target;
    if (err < best_err) { best = th; best_err = err; }
    if (err < rtol) break;
    if (v > target) lo = th; else hi = th;
    it++;
  }
  *rho_t = best;
  return 0;
}

int r2s_eval_distances(r2s_ctx *ctx, const double *rho_n, double rho_t, double delta_factor, double *dist, double *xp) {
  if (!ctx) return 1;
  ctx->launches = 0;
  if (upload_rho_n(ctx, rho_n)) return 1;
  if (r2s_dev_eval_distances(ctx, rho_t, delta_factor, xp != nullptr)) return 1;
  CK(cudaMemcpyAsync(dist, ctx->dist.p, sizeof(double) * (size_t)ctx->g.ngp, cudaMemcpyDeviceToHost, ctx->stream));
  if (xp) CK(cudaMemcpyAsync(xp, ctx->xp.p, sizeof(double) * 3 * (size_t)ctx->g.ngp, cudaMemcpyDeviceToHost, ctx->stream));
  CK(cudaStreamSynchronize(ctx->stream));
  ctx->rep.launches = ctx->launches;
  return 0;
}
int r2s_sign_detection(r2s_ctx *ctx, const double *rho_n, double rho_t, double *signs) {
  if (!ctx) return 1;
  ctx->launches = 0;
  if (upload_rho_n(ctx, rho_n)) return 1;
  if (r2s_dev_sign(ctx, rho_t, true, false)) return 1;
  CK(cudaMemcpyAsync(signs, ctx->signs.p, sizeof(double) * (size_t)ctx->g.ngp, cudaMemcpyDeviceToHost, ctx->stream));
  CK(cudaStreamSynchronize(ctx->stream));
  ctx->rep.launches = ctx->launches;
  return 0;
}
int r2s_remove_artifacts(r2s_ctx *ctx, double *sdf, double threshold, double min_ratio, int64_t *flipped) {
  if (!ctx) return 1;
  if (!ctx->has_grid) FAIL("r2s_set_grid has not been called");
  if (ctx->k0 != 0 || ctx->k1 != ctx->g.np[2]) FAIL("r2s_remove_artifacts works on the whole grid: a z-slab is set (use the pipeline calls on slab contexts)");
  ctx->launches = 0;
  CK(cudaSetDevice(ctx->device));
  CK(ctx->sdf.reserve(sizeof(double) * (size_t)ctx->g.ngp));
  CK(cudaMemcpyAsync(ctx->sdf.p, sdf, sizeof(double) * (size_t)ctx->g.ngp, cudaMemcpyHostToDevice, ctx->stream));
  ctx->have_sdf = true;
  i64 fl = 0;
  if (r2s_dev_remove_artifacts(ctx, threshold, min_ratio, &fl)) return 1;
  CK(cudaMemcpyAsync(sdf, ctx->sdf.p, sizeof(double) * (size_t)ctx->g.ngp, cudaMemcpyDeviceToHost, ctx->stream));
  CK(cudaStreamSynchronize(ctx->stream));
  if (flipped) *flipped = fl;
  ctx->rep.n_flipped = fl; ctx->rep.launches = ctx->launches;
  return 0;
}
int r2s_rbf_smoothing(r2s_ctx *ctx, const double *sdf, int is_interp, int smooth, double rbf_cut, double target_volume, float *fine_sdf, float *th, float *volume) {
  if (!ctx) return 1;
  if (!ctx->has_grid) FAIL("r2s_set_grid has not been called");
  if (smooth < 1 || smooth > 2) FAIL("r2s_rbf_smoothing: smooth must be 1 (:same) or 2 (:fine)");
  if (ctx->k0 != 0 || ctx->k1 != ctx->g.np[2]) FAIL("r2s_rbf_smoothing works on the whole grid: a z-slab is set (use the pipeline calls on slab contexts)");
  ctx->launches = 0;
  CK(cudaSetDevice(ctx->device));
  CK(ctx->sdf.reserve(sizeof(double) * (size_t)ctx->g.ngp));
  CK(cudaMemcpyAsync(ctx->sdf.p, sdf, sizeof(double) * (size_t)ctx->g.ngp, cudaMemcpyHostToDevice, ctx->stream));
  ctx->have_sdf = true;
  float t = 0, v = 0;
  if (r2s_dev_rbf(ctx, is_interp, smooth, rbf_cut, target_volume, volume != nullptr, &t, &v)) return 1;
  size_t nf = (size_t)(ctx->g.N[0] * (i64)smooth + 1) * (size_t)(ctx->g.N[1] * (i64)smooth + 1) * (size_t)(ctx->g.N[2] * (i64)smooth + 1);
  CK(cudaMemcpyAsync(fine_sdf, ctx->f_fine.p, sizeof(float) * nf, cudaMemcpyDeviceToHost, ctx->stream));
  CK(cudaStreamSynchronize(ctx->stream));
  if (th) *th = t;
  if (volume) *volume = v;
  ctx->rep.launches = ctx->launches;
  return 0;
}
int r2s_volume_from_sdf(r2s_ctx *ctx, const float *sdf, int64_t nx, int64_t ny, int64_t nz, float edge, float iso, int quad_order, double *volume) {
  if (!ctx) return 1;
  if (nx < 2 || ny < 2 || nz < 2) FAIL("r2s_volume_from_sdf: grid must have at least 2 points per axis");
  ctx->launches = 0;
  CK(cudaSetDevice(ctx->device));
  DevBuf tmp;
  CK(tmp.reserve(sizeof(float) * (size_t)(nx * ny * nz)));
  CK(cudaMemcpyAsync(tmp.p, sdf, sizeof(float) * (size_t)(nx * ny * nz), cudaMemcpyHostToDevice, ctx->stream));
  int rc = r2s_dev_volume_from_sdf(ctx, tmp.as<float>(), nx, ny, nz, edge, iso, quad_order, volume);
  cudaStreamSynchronize(ctx->stream);
  tmp.release();
  return rc;
}

// ---- the timed region of rho2sdf() (RhoToSDF.jl:164-227) ------------------------------------------------------
int r2s_upload_nodal_densities(r2s_ctx *ctx, const double *rho_n) {
  if (!ctx) return 1;
  if (upload_rho_n(ctx, rho_n)) return 1;
  CK(cudaStreamSynchronize(ctx->stream));
  return 0;
}
int r2s_pipeline_resident(r2s_ctx *ctx, const r2s_params *p, r2s_report *rep) {
  if (!ctx || !p) return 1;
  if (!ctx->has_grid) FAIL("r2s_set_grid has not been called");
  if (p->smooth < 1 || p->smooth > 2) FAIL("r2s_pipeline: smooth must be 1 (:same) or 2 (:fine)");
  if (ctx->nranks > 1 && (int)ctx->slab_k0.size() != ctx->nranks + 1) FAIL("r2s_pipeline: r2s_set_grid resets the slab of a multi-rank context: call r2s_set_slab (collective) before the pipeline");
  CK(cudaSetDevice(ctx->device));
  ctx->launches = 0; ctx->collectives = 0;
  memset(&ctx->rep, 0, sizeof(ctx->rep));
  CK(cudaEventRecord(ctx->ev[8], ctx->stream));
  if (r2s_dev_eval_distances(ctx, p->rho_t, p->delta_factor, false)) return 1;
  CK(cudaEventRecord(ctx->ev[9], ctx->stream));
  // pipelined calls: the previous call's downloads read ctx->sdf / ctx->f_fine, which are first overwritten from here on
  if (ctx->done_pending >= 0) { CK(cudaStreamWaitEvent(ctx->stream, ctx->ev_done[ctx->done_pending], 0)); ctx->done_pending = -1; }
  if (r2s_dev_sign(ctx, p->rho_t, false, true)) return 1;                 // sdf = dist .* signs (RhoToSDF.jl:171)
  CK(cudaEventRecord(ctx->ev[10], ctx->stream));
  if (p->remove_artifacts) { i64 fl = 0; if (r2s_dev_remove_artifacts(ctx, p->artifact_threshold, p->artifact_min_ratio, &fl)) return 1; ctx->rep.n_flipped = fl; }
  CK(cudaEventRecord(ctx->ev[11], ctx->stream));
  if (ctx->async_sdf_host) {      // sdf_dists is final here: its download overlaps the smoothing stage
    const size_t pl = (size_t)ctx->g.np[0] * ctx->g.np[1];
    cudaEvent_t e = ctx->ev_copy[ctx->n_ev_copy++ % 64];
    CK(cudaEventRecord(e, ctx->stream));
    CK(cudaStreamWaitEvent(ctx->copy_stream, e, 0));
    CK(cudaMemcpyAsync(ctx->async_sdf_host, ctx->sdf.as<double>() + pl * (size_t)ctx->k0, sizeof(double) * pl * (size_t)(ctx->k1 - ctx->k0), cudaMemcpyDeviceToHost, ctx->copy_stream));
  }
  float th = 0, vol = 0;
  if (r2s_dev_rbf(ctx, p->rbf_interp, p->smooth, p->rbf_cut, p->target_volume, p->final_volume != 0, &th, &vol)) return 1;
  CK(cudaEventRecord(ctx->ev[12], ctx->stream));
  CK(cudaStreamSynchronize(ctx->stream));
  if (r2s_p2p_check(ctx)) return 1;
  ctx->rep.th = th; ctx->rep.volume = vol;
  CK(cudaEventElapsedTime(&ctx->rep.ms_sign, ctx->ev[9], ctx->ev[10]));
  CK(cudaEventElapsedTime(&ctx->rep.ms_cc, ctx->ev[10], ctx->ev[11]));
  CK(cudaEventElapsedTime(&ctx->rep.ms_total, ctx->ev[8], ctx->ev[12]));
  ctx->rep.launches = ctx->launches; ctx->rep.collectives = ctx->collectives;
  if (rep) *rep = ctx->rep;
  return 0;
}
int r2s_download_sdf(r2s_ctx *ctx, double *sdf) {
  if (!ctx) return 1;
  CK(cudaMemcpyAsync(sdf, ctx->sdf.p, sizeof(double) * (size_t)ctx->g.ngp, cudaMemcpyDeviceToHost, ctx->stream));
  CK(cudaStreamSynchronize(ctx->stream));
  return 0;
}
int r2s_download_fine_sdf(r2s_ctx *ctx, float *fine) {
  if (!ctx) return 1;
  int s = ctx->smooth_last;
  size_t nf = (size_t)(ctx->g.N[0] * (i64)s + 1) * (size_t)(ctx->g.N[1] * (i64)s + 1) * (size_t)(ctx->g.N[2] * (i64)s + 1);
  CK(cudaMemcpyAsync(fine, ctx->f_fine.p, sizeof(float) * nf, cudaMemcpyDeviceToHost, ctx->stream));
  CK(cudaStreamSynchronize(ctx->stream));
  return 0;
}
int r2s_result_ptrs_dev(r2s_ctx *ctx, void **sdf_dev, void **fine_dev) {
  if (!ctx) return 1;
  if (sdf_dev) *sdf_dev = ctx->sdf.p;
  if (fine_dev) *fine_dev = ctx->f_fine.p;
  return 0;
}
int r2s_pipeline_slab(r2s_ctx *ctx, const r2s_params *p, const double *rho_n, double *sdf_slab, float *fine_slab, r2s_report *rep);
int r2s_pipeline(r2s_ctx *ctx, const r2s_params *p, const double *rho_n, double *sdf_dists, float *fine_sdf, r2s_report *rep) {
  if (!ctx || !p) return 1;
  if (ctx->has_grid && (ctx->k0 != 0 || ctx->k1 != ctx->g.np[2])) FAIL("r2s_pipeline: a z-slab is set; use r2s_pipeline_slab");
  return r2s_pipeline_slab(ctx, p, rho_n, sdf_dists, fine_sdf, rep);      // whole grid = one slab; downloads overlap the compute
}
// Host-buffer entry point for one z-slab (== r2s_pipeline when the slab is the whole grid): uploads rho_n, runs the timed
// region, returns ONLY this rank's planes: sdf_slab[(k1-k0) * np0 * np1] (coarse planes [k0,k1)) and
// fine_slab[(kf1-kf0) * f0 * f1] with kf0 = smooth*k0, kf1 = smooth*k1 (the last slab also owns the final fine plane).
int r2s_pipeline_slab(r2s_ctx *ctx, const r2s_params *p, const double *rho_n, double *sdf_slab, float *fine_slab, r2s_report *rep) {
  if (!ctx || !p) return 1;
  if (upload_rho_n(ctx, rho_n)) return 1;
  // the downloads are enqueued by the stages themselves as soon as a result is final (sdf_dists after the artifact removal,
  // fine_sdf chunk by chunk behind the fine-grid evaluation) and run on a second stream while the remaining kernels execute
  ctx->async_sdf_host = sdf_slab; ctx->async_fine_host = fine_slab; ctx->n_ev_copy = 0;
  int rc = r2s_pipeline_resident(ctx, p, rep);
  ctx->async_sdf_host = nullptr; ctx->async_fine_host = nullptr;
  cudaError_t e = cudaStreamSynchronize(ctx->copy_stream);
  if (rc) return 1;
  CK(e);
  CK(cudaStreamSynchronize(ctx->stream));
  return 0;
}
// Pipelined form of r2s_pipeline_slab for a sequence of density fields on the same mesh and grid: _begin returns when the device
// work of this call is finished and its result downloads are ENQUEUED (copy stream); they drain while the next _begin computes.
// The host buffers of a call belong to the library until r2s_pipeline_slab_wait(ticket) returns; alternate between two sets.
int r2s_pipeline_slab_begin(r2s_ctx *ctx, const r2s_params *p, const double *rho_n, double *sdf_slab, float *fine_slab, r2s_report *rep, int *ticket) {
  if (!ctx || !p || !ticket) return 1;
  if (upload_rho_n(ctx, rho_n)) return 1;
  ctx->async_sdf_host = sdf_slab; ctx->async_fine_host = fine_slab; ctx->n_ev_copy = 0;
  int rc = r2s_pipeline_resident(ctx, p, rep);
  ctx->async_sdf_host = nullptr; ctx->async_fine_host = nullptr;
  if (rc) { cudaStreamSynchronize(ctx->copy_stream); ctx->done_pending = -1; return 1; }
  const int t = ctx->done_next; ctx->done_next ^= 1;
  CK(cudaEventRecord(ctx->ev_done[t], ctx->copy_stream));
  ctx->done_pending = t;
  *ticket = t;
  return 0;
}
int r2s_pipeline_slab_wait(r2s_ctx *ctx, int ticket) {
  if (!ctx || ticket < 0 || ticket > 1) return 1;
  CK(cudaEventSynchronize(ctx->ev_done[ticket]));
  return 0;
}
}  // extern "C"
