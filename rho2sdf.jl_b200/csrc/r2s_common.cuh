// r2s_common.cuh -- context, device buffers, launch bookkeeping shared by the kernels of libr2s.so
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>
#include <string>
#include <vector>
#include "../../include/r2s.h"

typedef long long i64;
typedef unsigned long long u64;

#define R2S_BIG 1.0e10

// tile of grid points handled by one CTA of the per-voxel (gather) kernels
#define TILE_X 8
#define TILE_Y 8
#define TILE_Z 4
#define TILE_VOX (TILE_X * TILE_Y * TILE_Z)

struct DevBuf {
  void *p = nullptr;
  size_t cap = 0;
  // grow-only; contents are NOT preserved
  cudaError_t reserve(size_t bytes) {
    if (bytes <= cap) return cudaSuccess;
    if (p) cudaFree(p);
    p = nullptr; cap = 0;
    size_t want = bytes + bytes / 8 + 256;
    cudaError_t e = cudaMalloc(&p, want);
    if (e == cudaSuccess) cap = want;
    return e;
  }
  void release() { if (p) cudaFree(p); p = nullptr; cap = 0; }
  template <typename T> T *as() const { return (T *)p; }
};

// per-active-element record produced by the binning step (elements that can change the distance field)
struct ActRec {
  int ps[3];      // first grid-point index per axis inside the element's (AABB +- delta) cell range
  int pe[3];      // one past the last
  int el;         // element id (0-based)
  int cls;        // 1 solid (only boundary faces), 2 crossing
  int fmask;      // bit sg set <=> face sg is a boundary face
  int tri_off;    // first record of this element's boundary-face triangles in the triangle table (fmask != 0)
  i64 pair_off;   // offset of this element's (element, point) block in the pair buffer (crossing only)
};

struct GridDev {
  double amin[3], amax[3], cell;
  int N[3];        // cells per axis
  int np[3];       // points per axis = N+1
  i64 ngp;
  int nt[3];       // tiles per axis
  i64 ntiles;
  // device tables, concatenated per axis: offsets ax_off[d]
  const double *pc;      // point coordinate
  const int *cellof;     // cell of point
  const int *cstart;     // first point of cell c (length N+3 per axis)
  int pc_off[3], cs_off[3];
};

// tuning / A-B knobs, read from the environment ONCE by r2s_create (every one of them is exercised by a GPU test)
struct Knobs {
  int p2p = 1;            // R2S_P2P=0: NCCL only, no peer-memory mailbox (tests/slab_parity_ranks.py)
  int sign_lattice = 1;   // R2S_SIGN_LATTICE=0: tensor-product lattice meshes take the general (sorted candidate list) sign kernel
  int proj_box = 1;       // R2S_PROJ_BOX=0: axis-aligned box elements take the general trilinear projection
  int proj_prune = 1;     // R2S_PROJ_PRUNE=0: the box projection evaluates every (element, point) pair (no lower-bound pruning)
  int debug_sync = 0;     // R2S_DEBUG_SYNC=1: synchronise after every kernel launch, so that a device fault is reported at the launch that caused it
  int vol_cache = 1;      // R2S_VOL_CACHE=0: LS_Threshold re-evaluates every cut cell at every bisection (no cached quadratures)
};

struct LocalGroup;      // in-process slab group (r2s_multi_*): r2s_comm.cu

struct r2s_ctx {
  int device = 0;
  Knobs knobs;
  // small device -> host read-backs go through a MAPPED pinned buffer written by a tiny kernel (no DMA engine involved, so they never
  // queue behind the multi-GB result downloads of the copy stream); r2s_util.cu
  void *rb_host = nullptr, *rb_dev = nullptr; size_t rb_off = 0;
  cudaStream_t stream = nullptr;
  bool own_stream = false;
  std::string err;
  r2s_report rep;
  i64 launches = 0;
  cudaEvent_t ev[16]; cudaEvent_t ev_probe[5]; cudaEvent_t ev_k[5];      // ev_k: per-kernel timing of the pair-list projection (report: ms_solve / ms_scan)
  // overlap of the result download with compute (r2s_pipeline_slab): copies run on copy_stream behind events of the main stream
  cudaStream_t copy_stream = nullptr; cudaEvent_t ev_copy[64]; int n_ev_copy = 0;
  double *async_sdf_host = nullptr; float *async_fine_host = nullptr;
  // pipelined host-buffer calls (r2s_pipeline_slab_begin / _wait): the downloads of call k drain while call k+1 computes
  cudaEvent_t ev_done[2] = {nullptr, nullptr}; int done_next = 0; int done_pending = -1;

  // mesh
  int nen = 0, nes = 0, nsn = 0;
  i64 nnp = 0, nel = 0;
  DevBuf X, IEN32, ine_ptr, ine_el, fbnd, ezr;   // X double[3*nnp]; IEN32 int[nen*nel] 0-based; INE CSR; fbnd uint8[nel]
  DevBuf ebox; i64 n_box = 0;                    // HEX8: uint8[nel] 1 = axis-aligned box in canonical node order (iso::HexBox), and their count
  // tensor-product lattice meshes (every element a box whose corners are neighbouring values of three per-axis coordinate tables):
  // lat_xs = the tables (concatenated, offsets lat_off), lat_cell[e] = lattice cell of element e, lat_map[cell] = element or -1
  bool lattice = false; int lat_nd[3] = {0, 0, 0}, lat_off[3] = {0, 0, 0}; i64 lat_ncell = 0;
  DevBuf lat_xs, lat_cell, lat_map, lat_info, lat_pt;
  DevBuf rho_e, rho_n;

  // grid
  bool has_grid = false;
  GridDev g;
  i64 k0 = 0, k1 = 0;                       // slab of coarse planes handled by this context
  const float *skip_flag = nullptr;          // device flag: while set and non-zero, the peer-memory exchange kernels return at once (CG iterations launched ahead of the convergence check)
  LocalGroup *lg = nullptr;                  // set when this context is one slab of an in-process group (threads instead of processes, no NCCL)
  void *comm = nullptr; int rank = 0, nranks = 1; i64 collectives = 0; std::vector<int> slab_k0;
  // peer-memory fast path for the latency-critical exchanges (scalar all-reduces, CG halo planes): every rank maps every
  // peer's mailbox (and the CG vector c) through CUDA IPC and writes into it directly over NVLink (r2s_comm.cu)
  bool p2p = false; void *p2p_box = nullptr; void *p2p_peer_box[64]; void **p2p_peer_box_dev = nullptr; unsigned p2p_seq = 0;
  void *p2p_c_local = nullptr; void *p2p_c_peer[2] = {nullptr, nullptr}; unsigned p2p_halo_seq = 0; i64 p2p_ops = 0;    // NCCL communicator of the slab decomposition (r2s_comm.cu)
  DevBuf gtab_d, gtab_i;
  std::vector<double> h_pc[3];

  // distance / sign work buffers
  DevBuf cls, act_flag, act_idx, act_rec, cnt_a, cnt_b, keys, keys_alt, tile_ptr, tile_faces, face_tiles, fc_list, tri_cnt, tri_rec, pairbuf, pairxp, cubtmp, counters, box_rec, plist, pseed;
  DevBuf dist, xp, sdf, signs;
  // evalDistances / Sign_Detection at arbitrary points (r2s_points.cu): own nodal densities and scratch, so a points call leaves every
  // resident result (sdf, fine_sdf, smoothing weights, isosurface, the uploaded rho_n) as it found it
  DevBuf pt_rn, pt_cls, pt_flag, pt_idx, pt_rec, pt_hex, pt_cnt, pt_off, pt_tkeys, pt_tkeys_alt, pt_tile_ptr, pt_tri, pt_in, pt_keys, pt_keys_alt, pt_out, pt_ctr;
  DevBuf s_rng, s_el, s_cnt, s_keys, s_keys_alt, s_tile_ptr;
  // connected components
  DevBuf cc_label, cc_size, cc_scal, cc_bits, cc_bits_all, cc_gsz, cc_seen;
  // smoothing
  DevBuf f_s, f_w, f_r, f_u, f_c, f_lsf, f_fine, f_part, f_scal, cutlist, slablist, vlist[2], vent[2], vrec, bis_state;
  int smooth_last = 1;
  bool have_sdf = false, have_fine = false;      // ctx->sdf / ctx->f_fine hold a result of the CURRENT grid (cleared by r2s_set_grid / r2s_set_mesh)
  // the continuous field of the last smoothing call (r2s_sample.cu): weights rbf_w (f_w after the CG, f_s in approximation mode; row
  // pitch rbf_px, whole-grid plane indexing, owned planes + 2 below / 3 above valid), offset rbf_th, the Float32 coordinate tables (host
  // rbf_c, device rbf_tab).  have_rbf is cleared with have_fine; nothing but r2s_dev_rbf writes f_w / f_s.
  bool have_rbf = false; const float *rbf_w = nullptr; int rbf_px = 0; float rbf_th = 0.0f; double rbf_cut = 0.0;
  std::vector<float> rbf_c[3]; DevBuf rbf_tab, smp_in, smp_out;

  // volumes
  DevBuf v_part;

  // isosurface (r2s_surf.cu): per-row counts / bases, the mesh part of this context (vertices from global id surf_vglob on); have_surface is
  // cleared by r2s_set_grid / r2s_set_mesh / r2s_set_slab; surf_part = the mesh is one slab's part of an r2s_multi mesh
  DevBuf surf_rows, surf_V, surf_T;
  bool have_surface = false, surf_part = false;
  const float *surf_f = nullptr; i64 surf_nx = 0, surf_ny = 0, surf_nz = 0, surf_z0 = 0, surf_z1 = 0; float surf_iso = 0.0f;
  double surf_origin[3] = {0, 0, 0}, surf_spacing[3] = {0, 0, 0};
  i64 surf_nv = 0, surf_nt = 0, surf_vglob = 0, surf_nv_all = 0, surf_nt_all = 0;
};

#define CK(call)                                                                                   \
  do {                                                                                             \
    cudaError_t _e = (call);                                                                       \
    if (_e != cudaSuccess) {                                                                       \
      char _b[512];                                                                                \
      snprintf(_b, sizeof(_b), "%s:%d: %s -> %s", __FILE__, __LINE__, #call, cudaGetErrorString(_e)); \
      ctx->err = _b;                                                                               \
      return 1;                                                                                    \
    }                                                                                              \
  } while (0)

#define FAIL(msg)           \
  do {                      \
    ctx->err = (msg);       \
    return 1;               \
  } while (0)

#define LAUNCH_CHECK()                                                          \
  do {                                                                          \
    ctx->launches++;                                                            \
    CK(cudaGetLastError());                                                     \
    if (ctx->knobs.debug_sync) CK(cudaStreamSynchronize(ctx->stream));          \
  } while (0)

static inline int cdiv(i64 a, i64 b) { return (int)((a + b - 1) / b); }

// ---- implemented in the individual translation units --------------------------------------------------
int r2s_mesh_upload_ien(r2s_ctx *ctx, const int64_t *IEN);                 // r2s_mesh.cu: int64 1-based -> int32 0-based on device
int r2s_mesh_build_tables(r2s_ctx *ctx);                                   // r2s_mesh.cu: INE + boundary faces
int r2s_dev_mesh_volume(r2s_ctx *ctx, double *vd, double *vf);             // r2s_mesh.cu
int r2s_dev_nodal_densities(r2s_ctx *ctx);                                 // r2s_mesh.cu (rho_e -> rho_n, device)
int r2s_dev_isocontour_volume(r2s_ctx *ctx, double thr, double *vol);      // r2s_mesh.cu
int r2s_dev_eval_distances(r2s_ctx *ctx, double rho_t, double delta_factor, bool want_xp);   // r2s_dist.cu -> ctx->dist (,xp)
int r2s_dev_sign(r2s_ctx *ctx, double rho_t, bool write_signs, bool write_sdf);              // r2s_sign.cu -> ctx->signs / ctx->sdf
int r2s_dev_remove_artifacts(r2s_ctx *ctx, double thr, double ratio, i64 *flipped);          // r2s_cc.cu on ctx->sdf
int r2s_dev_rbf(r2s_ctx *ctx, int is_interp, int smooth, double rbf_cut, double target, bool final_volume, float *th, float *vol);   // r2s_rbf.cu: ctx->sdf -> ctx->f_fine
int r2s_dev_volume_from_sdf(r2s_ctx *ctx, const float *sdf_dev, i64 nx, i64 ny, i64 nz, float edge, float iso, int order, double *vol);        // r2s_rbf.cu
int r2s_scan_exclusive_i64(r2s_ctx *ctx, const i64 *in, i64 *out, i64 n);  // r2s_util.cu (cub)
int r2s_scan_exclusive_i32(r2s_ctx *ctx, const int *in, int *out, i64 n);
int r2s_sort_keys_u64(r2s_ctx *ctx, u64 *keys, u64 *alt, i64 n, int end_bit, u64 **sorted);
int r2s_sort_f64(r2s_ctx *ctx, double *keys, double *alt, i64 n, double **sorted);
int r2s_unique_f64(r2s_ctx *ctx, const double *sorted, double *out, i64 n, i64 *count);      // distinct values of a sorted array
// read-backs through the mapped buffer: rb_put enqueues a copy of `bytes` at src_dev and returns its offset (or (size_t)-1), rb_sync
// waits for the stream; rb_at(off) is then valid until the next rb_put after a sync.  r2s_readback = put + sync + memcpy.
#define R2S_RB_BYTES (192 * 1024)
size_t r2s_rb_put(r2s_ctx *ctx, const void *src_dev, size_t bytes);
int r2s_rb_sync(r2s_ctx *ctx);
static inline const void *r2s_rb_at(r2s_ctx *ctx, size_t off) { return (const char *)ctx->rb_host + off; }
int r2s_readback(r2s_ctx *ctx, void *dst_host, const void *src_dev, size_t bytes);
int r2s_mesh_build_lattice(r2s_ctx *ctx);                                  // r2s_mesh.cu: tensor-product lattice detection + tables
// r2s_comm.cu: collectives over the slab communicator (no-ops for a single rank)
int r2s_allreduce(r2s_ctx *ctx, void *buf, size_t count, int kind /*0 f64 sum, 1 u64 sum, 2 u32 max, 3 u32 min, 4 u64 max*/);
int r2s_p2p_prepare_c(r2s_ctx *ctx, size_t have_bytes, size_t need_bytes);                  // collective; before c may be re-allocated
int r2s_p2p_map_c(r2s_ctx *ctx, float *c, size_t bytes);                                     // (re)map the neighbours' CG vector c
struct P2PFuse;
int r2s_p2p_fuse_params(r2s_ctx *ctx, P2PFuse *stencil, P2PFuse *update, i64 plane_elems, int k0, int k1, int H);      // r2s_p2p.cuh
int r2s_p2p_check(r2s_ctx *ctx);
int r2s_group_start(r2s_ctx *ctx);
int r2s_group_end(r2s_ctx *ctx);
int r2s_allgather_u32(r2s_ctx *ctx, const unsigned *send, unsigned *recv, size_t count);
int r2s_halo_exchange_f32(r2s_ctx *ctx, float *a, i64 plane_elems, int k0, int k1, int nz, int below, int above);
extern "C" int r2s_comm_destroy(r2s_ctx *ctx);
extern "C" int r2s_export_vti(r2s_ctx *ctx, const char *path, const char *label, int which);
extern "C" int r2s_export_pvti(r2s_ctx *ctx, const char *path, const char *label, int which, const char *piece_base);
// r2s_surf.cu: isosurface passes of one slab, for r2s_multi.cu
int r2s_surf_count_slab(r2s_ctx *ctx, float iso, i64 *nv, i64 *nt);       // pass 1 + scans on the resident fine field (collective: halo planes)
int r2s_surf_emit(r2s_ctx *ctx, i64 vglob, i64 nv_total);                  // pass 2 with this slab's first global vertex id
int r2s_surf_download_slab(r2s_ctx *ctx, float *V, int32_t *T, i64 tglob, bool staging);   // this slab's part into the whole arrays
int r2s_surf_write_file(const char *path, int format, const float *V, i64 nv, const int *T, i64 nt, std::string *err);
// r2s_sample.cu: the sampler of the continuous field, for r2s_rbf.cu (record) and r2s_multi.cu (one slab's share, no rank check)
struct SampleGrid;
int r2s_sample_record(r2s_ctx *ctx, const float *w, int px, float th, double rbf_cut);
int r2s_sample_grid(r2s_ctx *ctx, SampleGrid *G, bool dev);
int r2s_sample_points_ctx(r2s_ctx *ctx, const double *pts, i64 n, float *val, float *grad);
int r2s_sample_lattice_check(r2s_ctx *ctx, const double origin[3], const double spacing[3], const int64_t dims[3], float o[3], float h[3]);
int r2s_sample_lattice_planes(r2s_ctx *ctx, const float o[3], const float h[3], const int64_t dims[3], i64 ka, i64 kb, float *out);
int r2s_sample_download_weights(r2s_ctx *ctx, float *w, float *th, i64 k0, i64 k1);
// r2s_points.cu: evalDistances / Sign_Detection at n host points (rho_n on the host)
int r2s_points_distances(r2s_ctx *ctx, const double *rho_n, double rho_t, double delta_factor, const double *pts, i64 n, double *dist, double *xp);
int r2s_points_signs(r2s_ctx *ctx, const double *rho_n, double rho_t, const double *pts, i64 n, double *signs);
// in-process groups (r2s_multi.cu drives them): one context per slab, one host thread per context
LocalGroup *r2s_local_group_create(r2s_ctx **ctxs, int n, std::string *err);
void r2s_local_group_destroy(LocalGroup *g);
void r2s_local_group_abort(LocalGroup *g);      // a rank failed: wake everybody waiting at a host barrier

#ifdef __CUDACC__
// ---- warp-private staging of list entries in shared memory ------------------------------------------------------------------------
// Every device-built list (pairs, cut cells, active cells, cells to evaluate, hard sign points) is appended to through ONE global counter.  Same-address atomics
// retire at about one per clock, so a claim per 32-lane round makes a kernel atomic-bound (measured: k_vol_rows, k_vl_step, k_pair_scan).
// Each warp therefore collects its entries in a shared-memory buffer and claims slots for ~100 entries at a time.  n is warp-uniform.
#define WS_CAP 128
template <typename T>
__device__ __forceinline__ void ws_flush(T *buf, int &n, T *__restrict__ gout, u64 *__restrict__ gcount, i64 cap, int lane) {
  if (n == 0) return;
  u64 base = 0;
  if (lane == 0) base = atomicAdd(gcount, (u64)n);
  base = __shfl_sync(0xffffffffu, base, 0);
  for (int i = lane; i < n; i += 32) if ((i64)(base + i) < cap) gout[base + i] = buf[i];
  __syncwarp();
  n = 0;
}
template <typename T>
__device__ __forceinline__ void ws_push(T *buf, int &n, bool pred, const T &val, T *__restrict__ gout, u64 *__restrict__ gcount, i64 cap, int lane) {
  const unsigned m = __ballot_sync(0xffffffffu, pred);
  if (!m) return;
  if (pred) buf[n + __popc(m & ((1u << lane) - 1))] = val;
  n += __popc(m);
  __syncwarp();
  if (n > WS_CAP - 32) ws_flush(buf, n, gout, gcount, cap, lane);
}
#endif
