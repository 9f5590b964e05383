// r2s_multi.cu -- ONE host call drives ALL GPUs of the box: the single-call multi-GPU entry behind rho2sdf() (RhoToSDF.jl:116-242).
//
// The Julia drop-in is one process; `r2s_multi` gives it the whole node without mpiexec: one r2s_ctx per z-slab (normally one per GPU),
// one library-internal host thread per context, the in-process exchange layer of r2s_comm.cu (peer access over NVLink, no NCCL, no IPC).
// The mesh and the nodal densities are replicated, the coarse planes are cut into contiguous slabs (SURVEY.md 8e), every slab writes
// its planes straight into the caller's whole-grid host arrays.  Device ids may repeat: several slabs on one GPU run the same code
// path (that is how the multi-slab logic is tested on a one-GPU box).  After every call the slabs are re-cut by measured cost (the
// planes next to the mesh boundary carry the boundary-face work).
#include <math.h>
#include <cmath>
#include <string.h>
#include <algorithm>
#include <functional>
#include <new>
#include <thread>
#include <vector>
#include "r2s_common.cuh"
#include "r2s_sample.cuh"

struct r2s_multi {
  int n = 0;
  std::vector<r2s_ctx *> ctx;
  std::vector<int> dev;
  LocalGroup *lg = nullptr;
  std::string err;
  std::vector<i64> cut, next_cut;  // n + 1 plane boundaries in force / to be applied at the start of the next call
  std::vector<double> plane_cost;  // per coarse plane, from the last pipeline call (empty = even cut)
  bool has_grid = false, rebalance = true, recut_pending = false;      // a re-cut is applied at the START of the next pipeline call (the resident results stay valid for export)
  int nz = 0;
  bool have_surface = false;        // an r2s_multi_isosurface result is resident on the slabs
  std::vector<i64> surf_vb, surf_tb;  // n + 1 global vertex / triangle bases of the slabs' parts
};

// runs fn(rank) on one host thread per slab; a failing rank wakes the others out of their host barriers
static int run_all(r2s_multi *m, const std::function<int(int)> &fn) {
  if (m->n == 1) { int rc = fn(0); if (rc) m->err = m->ctx[0]->err; return rc; }
  std::vector<int> rc((size_t)m->n, 0);
  std::vector<std::thread> th;
  for (int r = 0; r < m->n; r++)
    th.emplace_back([&, r] {
      rc[(size_t)r] = fn(r);
      if (rc[(size_t)r]) r2s_local_group_abort(m->lg);
    });
  for (auto &t : th) t.join();
  int bad = 0;
  for (int r = 0; r < m->n; r++)
    if (rc[(size_t)r]) { if (!bad || m->ctx[(size_t)r]->err.find("another slab failed") == std::string::npos) m->err = "slab " + std::to_string(r) + ": " + m->ctx[(size_t)r]->err; bad = 1; }
  return bad;
}
static void even_cut(r2s_multi *m) {
  m->cut.assign((size_t)m->n + 1, 0);
  const i64 base = m->nz / m->n, rem = m->nz % m->n;
  for (int r = 0; r < m->n; r++) m->cut[(size_t)r + 1] = m->cut[(size_t)r] + base + (r < rem ? 1 : 0);
}
// cuts that equalise the cumulative plane cost, at least 3 planes per slab (smoothing halo)
static void cost_cut(r2s_multi *m) {
  const int n = m->n, nz = m->nz;
  std::vector<double> cum((size_t)nz + 1, 0.0);
  for (int k = 0; k < nz; k++) cum[(size_t)k + 1] = cum[(size_t)k] + std::max(m->plane_cost[(size_t)k], 1e-12);
  m->cut.assign((size_t)n + 1, 0);
  for (int r = 1; r < n; r++) {
    const double want = cum[(size_t)nz] * r / n;
    i64 k = std::lower_bound(cum.begin(), cum.end(), want) - cum.begin();
    k = std::max<i64>(k, m->cut[(size_t)r - 1] + 3);
    k = std::min<i64>(k, nz - (i64)(n - r) * 3);
    m->cut[(size_t)r] = k;
  }
  m->cut[(size_t)n] = nz;
}
static int apply_cut(r2s_multi *m) {
  return run_all(m, [&](int r) { return r2s_set_slab(m->ctx[(size_t)r], m->cut[(size_t)r], m->cut[(size_t)r + 1]); });
}

extern "C" {

int r2s_multi_create(r2s_multi **out, const int *device_ids, int ndev) {
  if (!out) return 1;
  *out = nullptr;
  if (!device_ids || ndev < 1 || ndev > 64) return 2;
  r2s_multi *m = new (std::nothrow) r2s_multi();
  if (!m) return 3;
  m->n = ndev;
  for (int r = 0; r < ndev; r++) {
    r2s_ctx *c = nullptr;
    if (r2s_create(&c, device_ids[r], nullptr) != 0) { for (r2s_ctx *q : m->ctx) r2s_destroy(q); delete m; return 4; }      // no CPU fallback
    m->ctx.push_back(c); m->dev.push_back(device_ids[r]);
  }
  if (ndev > 1) {
    std::string e;
    m->lg = r2s_local_group_create(m->ctx.data(), ndev, &e);
    if (!m->lg) { for (r2s_ctx *q : m->ctx) r2s_destroy(q); delete m; return 5; }
  }
  *out = m;
  return 0;
}
void r2s_multi_destroy(r2s_multi *m) {
  if (!m) return;
  if (m->lg) r2s_local_group_destroy(m->lg);
  for (r2s_ctx *c : m->ctx) r2s_destroy(c);
  delete m;
}
const char *r2s_multi_last_error(r2s_multi *m) { return m ? m->err.c_str() : "r2s_multi: no handle (no CUDA device?)"; }
int r2s_multi_size(r2s_multi *m) { return m ? m->n : 0; }
// context of one slab, e.g. slab 0 for the pre-timer stages (r2s_mesh_volume, r2s_nodal_densities, r2s_find_threshold work on the whole mesh)
r2s_ctx *r2s_multi_context(r2s_multi *m, int slab) { return (m && slab >= 0 && slab < m->n) ? m->ctx[(size_t)slab] : nullptr; }

int r2s_multi_set_mesh(r2s_multi *m, int nen, int64_t nnp, const double *X, int64_t nel, const int64_t *IEN) {
  if (!m) return 1;
  m->has_grid = false; m->have_surface = false;
  return run_all(m, [&](int r) { return r2s_set_mesh(m->ctx[(size_t)r], nen, nnp, X, nel, IEN); });
}
int r2s_multi_set_grid(r2s_multi *m, const double amin[3], const double amax[3], const int64_t N[3], double cell) {
  if (!m) return 1;
  if (N[2] + 1 < 3 * (int64_t)m->n) { m->err = "r2s_multi_set_grid: fewer than 3 coarse planes per slab"; return 1; }
  // r2s_set_grid resets a context to the whole grid; the slabs are set (collectively) right after
  for (int r = 0; r < m->n; r++) if (r2s_set_grid(m->ctx[(size_t)r], amin, amax, N, cell)) { m->err = m->ctx[(size_t)r]->err; return 1; }
  m->nz = (int)N[2] + 1; m->plane_cost.clear(); m->has_grid = true; m->recut_pending = false; m->have_surface = false;
  even_cut(m);
  return m->n > 1 ? apply_cut(m) : 0;
}
int r2s_multi_slab_planes(r2s_multi *m, int64_t *cuts /* n + 1 */) {
  if (!m || !cuts || !m->has_grid) return 1;
  for (int r = 0; r <= m->n; r++) cuts[r] = m->cut[(size_t)r];
  return 0;
}
int r2s_multi_set_rebalance(r2s_multi *m, int on) { if (!m) return 1; m->rebalance = on != 0; return 0; }

// The timed region of rho2sdf() on all slabs.  Host arrays are WHOLE-GRID: sdf_dists[ngp], fine_sdf[prod(N*smooth+1)], x fastest.
int r2s_multi_pipeline(r2s_multi *m, const r2s_params *p, const double *rho_n, double *sdf_dists, float *fine_sdf, r2s_report *rep) {
  if (!m || !p) return 1;
  if (!m->has_grid) { m->err = "r2s_multi_set_grid has not been called"; return 1; }
  if (m->n == 1) { m->have_surface = false; int rc = r2s_pipeline(m->ctx[0], p, rho_n, sdf_dists, fine_sdf, rep); if (rc) m->err = m->ctx[0]->err; return rc; }
  m->have_surface = false;
  if (m->recut_pending) { m->recut_pending = false; m->cut = m->next_cut; if (apply_cut(m)) return 1; }
  const GridDev &g = m->ctx[0]->g;
  const size_t pl = (size_t)g.np[0] * g.np[1];
  const int s = p->smooth;
  const size_t fpl = (size_t)(g.N[0] * (i64)s + 1) * (size_t)(g.N[1] * (i64)s + 1);
  std::vector<r2s_report> reps((size_t)m->n);
  int rc = run_all(m, [&](int r) {
    const i64 k0 = m->cut[(size_t)r];
    return r2s_pipeline_slab(m->ctx[(size_t)r], p, rho_n, sdf_dists ? sdf_dists + pl * (size_t)k0 : nullptr, fine_sdf ? fine_sdf + fpl * (size_t)(s * k0) : nullptr, &reps[(size_t)r]);
  });
  if (rc) return 1;
  if (rep) {
    r2s_report a = reps[0];
    for (int r = 1; r < m->n; r++) {
      const r2s_report &b = reps[(size_t)r];
      a.n_solid += b.n_solid; a.n_crossing += b.n_crossing; a.n_active += b.n_active; a.n_pairs += b.n_pairs; a.n_not_converged += b.n_not_converged;
      a.n_newton_iters += b.n_newton_iters; a.n_pairs_pruned += b.n_pairs_pruned; a.launches += b.launches; a.collectives += b.collectives;
      float *fa = &a.ms_bin; const float *fb = &b.ms_bin;
      for (int q = 0; q < 12; q++) fa[q] = std::max(fa[q], fb[q]);      // ms_bin .. ms_total are contiguous floats
      a.ms_solve = std::max(a.ms_solve, b.ms_solve); a.ms_scan = std::max(a.ms_scan, b.ms_scan);
    }
    *rep = a;
  }
  // re-cut the slabs for the next call by measured cost: collective-free stages per plane of the slab that ran them + the smoothing
  // cost per plane of the slab that waited least
  if (m->rebalance) {
    double cu = 1e300;
    std::vector<double> freec((size_t)m->n);
    for (int r = 0; r < m->n; r++) {
      const r2s_report &b = reps[(size_t)r]; const double planes = (double)(m->cut[(size_t)r + 1] - m->cut[(size_t)r]);
      freec[(size_t)r] = (b.ms_bin + b.ms_project + b.ms_assemble + b.ms_sign) / planes;
      cu = std::min(cu, (double)(b.ms_rbf_prep + b.ms_cg + b.ms_lsf + b.ms_threshold + b.ms_fine + b.ms_volume) / planes);
    }
    m->plane_cost.assign((size_t)m->nz, 0.0);
    for (int r = 0; r < m->n; r++) for (i64 k = m->cut[(size_t)r]; k < m->cut[(size_t)r + 1]; k++) m->plane_cost[(size_t)k] = freec[(size_t)r] + cu;
    std::vector<i64> old = m->cut;
    cost_cut(m);
    if (old != m->cut) {
      // the slabs in force (and the results resident on them) stay as they are until the next call; keep `cut` describing them
      m->next_cut = m->cut; m->cut = old; m->recut_pending = true;
    }
  }
  return 0;
}

// pinning the caller's result arrays once makes their downloads asynchronous and ~2x faster (plain cudaHostRegister / Unregister)
int r2s_pin_host(void *p, size_t bytes) { return cudaHostRegister(p, bytes, cudaHostRegisterPortable) == cudaSuccess ? 0 : 1; }
int r2s_unpin_host(void *p) { return cudaHostUnregister(p) == cudaSuccess ? 0 : 1; }

// Result export of all slabs: <base>_<slab>.vti pieces + <base>.pvti index (exportSdfToVTI, DataExport/ExportToVTI.jl:22-67, for a result
// that lives on several GPUs).  One slab: a plain <base>.vti.
int r2s_multi_export_vti(r2s_multi *m, const char *base, const char *label, int which) {
  if (!m || !base || !label) return 1;
  if (!m->has_grid) { m->err = "r2s_multi_set_grid has not been called"; return 1; }
  std::string b(base);
  if (b.size() > 4 && b.substr(b.size() - 4) == ".vti") b.resize(b.size() - 4);
  if (m->n == 1) { int rc = r2s_export_vti(m->ctx[0], (b + ".vti").c_str(), label, which); if (rc) m->err = m->ctx[0]->err; return rc; }
  int rc = run_all(m, [&](int r) { return r2s_export_vti(m->ctx[(size_t)r], (b + "_" + std::to_string(r) + ".vti").c_str(), label, which); });
  if (rc) return 1;
  rc = r2s_export_pvti(m->ctx[0], (b + ".pvti").c_str(), label, which, base);
  if (rc) m->err = m->ctx[0]->err;
  return rc;
}

// Zero surface of the fine field that lives on the slabs (r2s_surf.cu): every slab counts its planes, the host scans the slab counts,
// every slab emits its part with its global bases.  The concatenation of the parts in slab order equals one context's mesh of the field.
int r2s_multi_isosurface(r2s_multi *m, float iso, int64_t *n_vertices, int64_t *n_triangles) {
  if (!m) return 1;
  if (!m->has_grid) { m->err = "r2s_multi_set_grid has not been called"; return 1; }
  m->have_surface = false;
  std::vector<i64> nv((size_t)m->n, 0), nt((size_t)m->n, 0);
  if (m->n == 1) {
    int64_t a = 0, b = 0;
    if (r2s_isosurface(m->ctx[0], iso, &a, &b)) { m->err = m->ctx[0]->err; return 1; }
    nv[0] = a; nt[0] = b;
  } else {
    if (run_all(m, [&](int r) { return r2s_surf_count_slab(m->ctx[(size_t)r], iso, &nv[(size_t)r], &nt[(size_t)r]); })) return 1;
  }
  m->surf_vb.assign((size_t)m->n + 1, 0); m->surf_tb.assign((size_t)m->n + 1, 0);
  for (int r = 0; r < m->n; r++) { m->surf_vb[(size_t)r + 1] = m->surf_vb[(size_t)r] + nv[(size_t)r]; m->surf_tb[(size_t)r + 1] = m->surf_tb[(size_t)r] + nt[(size_t)r]; }
  if (m->n > 1 && run_all(m, [&](int r) { return r2s_surf_emit(m->ctx[(size_t)r], m->surf_vb[(size_t)r], m->surf_vb[(size_t)m->n]); })) return 1;
  m->have_surface = true;
  if (n_vertices) *n_vertices = m->surf_vb[(size_t)m->n];
  if (n_triangles) *n_triangles = m->surf_tb[(size_t)m->n];
  return 0;
}
// vertices[3 * nv], triangles[3 * nt]: the whole mesh, every slab writes its part
static int multi_download(r2s_multi *m, float *vertices, int32_t *triangles, bool staging) {
  if (!m->have_surface) { m->err = "isosurface: no surface on this handle (call r2s_multi_isosurface first)"; return 1; }
  return run_all(m, [&](int r) { return r2s_surf_download_slab(m->ctx[(size_t)r], vertices, triangles, m->surf_tb[(size_t)r], staging); });
}
int r2s_multi_download_isosurface(r2s_multi *m, float *vertices, int32_t *triangles) { return m ? multi_download(m, vertices, triangles, false) : 1; }
// one file for the whole mesh (format 0 binary STL, 1 binary little-endian PLY)
// ---- sampling the continuous field (r2s_sample.cu): a point whose floor plane in the Float32 z-table is c needs weight planes c - 2 .. c + 3;
// a slab keeps its owned planes [k0, k1) plus 2 below and 3 above valid (the fine evaluation reads the same), so the slab owning c has them
static int multi_sample_ready(r2s_multi *m, SampleGrid *G) {
  if (!m->has_grid) { m->err = "r2s_multi_set_grid has not been called"; return 1; }
  for (int r = 0; r < m->n; r++)
    if (r2s_sample_grid(m->ctx[(size_t)r], G, false)) { m->err = "slab " + std::to_string(r) + ": " + m->ctx[(size_t)r]->err; return 1; }
  return 0;
}
static int owner_of(const r2s_multi *m, const SampleGrid &G, float z) {
  const int c = smp_floor(G.C[2], G.n[2], G.c0[2], G.inv[2], z);
  return (int)(std::upper_bound(m->cut.begin() + 1, m->cut.end(), (i64)c) - m->cut.begin()) - 1;
}
int r2s_multi_sample_sdf(r2s_multi *m, const double *points, int64_t n, float *values, float *gradients) {
  if (!m) return 1;
  if (m->n == 1) { int rc = r2s_sample_sdf(m->ctx[0], points, n, values, gradients); if (rc) m->err = m->ctx[0]->err; return rc; }
  if (n < 0) { m->err = "sampling: negative point count"; return 1; }
  if (n > 0 && (!points || !values)) { m->err = "sampling: points and values are required when n > 0"; return 1; }
  SampleGrid G;
  if (multi_sample_ready(m, &G)) return 1;
  std::vector<std::vector<i64>> idx((size_t)m->n);
  for (i64 t = 0; t < n; t++) {
    const double *p = points + 3 * t;
    if (!std::isfinite(p[0]) || !std::isfinite(p[1]) || !std::isfinite(p[2])) { m->err = "sampling: a point coordinate is NaN or infinite"; return 1; }
    idx[(size_t)owner_of(m, G, (float)p[2])].push_back(t);
  }
  return run_all(m, [&](int r) {
    const std::vector<i64> &id = idx[(size_t)r];
    const size_t k = id.size();
    std::vector<double> p(3 * k);
    std::vector<float> v(k), g(gradients ? 3 * k : 0);
    for (size_t q = 0; q < k; q++) for (int d = 0; d < 3; d++) p[3 * q + d] = points[3 * id[q] + d];
    if (r2s_sample_points_ctx(m->ctx[(size_t)r], p.data(), (i64)k, v.data(), gradients ? g.data() : nullptr)) return 1;
    for (size_t q = 0; q < k; q++) {
      values[id[q]] = v[q];
      if (gradients) for (int d = 0; d < 3; d++) gradients[3 * id[q] + d] = g[3 * q + d];
    }
    return 0;
  });
}
int r2s_multi_sample_sdf_lattice(r2s_multi *m, const double origin[3], const double spacing[3], const int64_t dims[3], float *values) {
  if (!m) return 1;
  if (m->n == 1) { int rc = r2s_sample_sdf_lattice(m->ctx[0], origin, spacing, dims, values); if (rc) m->err = m->ctx[0]->err; return rc; }
  float o[3], h[3];
  if (r2s_sample_lattice_check(m->ctx[0], origin, spacing, dims, o, h)) { m->err = m->ctx[0]->err; return 1; }
  SampleGrid G;
  if (multi_sample_ready(m, &G)) return 1;
  if (!values) { m->err = "sampling: values are required"; return 1; }
  // runs of consecutive lattice planes with the same owner (a plane's z is o_z + float(k) h_z, the same formula as the kernel)
  std::vector<std::vector<std::pair<i64, i64>>> runs((size_t)m->n);
  int prev = -1;
  for (i64 k = 0; k < dims[2]; k++) {
    const int r = owner_of(m, G, smp_add(o[2], smp_mul((float)k, h[2])));
    if (r == prev) runs[(size_t)r].back().second = k + 1;
    else runs[(size_t)r].push_back({k, k + 1});
    prev = r;
  }
  const i64 pl = dims[0] * dims[1];
  return run_all(m, [&](int r) {
    for (const auto &ab : runs[(size_t)r])
      if (r2s_sample_lattice_planes(m->ctx[(size_t)r], o, h, dims, ab.first, ab.second, values + ab.first * pl)) return 1;
    return 0;
  });
}
// every slab writes its owned weight planes; th is the same on all slabs (the threshold search is collective)
int r2s_multi_download_rbf_weights(r2s_multi *m, float *weights, float *th) {
  if (!m) return 1;
  if (m->n == 1) { int rc = r2s_download_rbf_weights(m->ctx[0], weights, th); if (rc) m->err = m->ctx[0]->err; return rc; }
  if (!weights && !th) { m->err = "r2s_download_rbf_weights: weights or th is required"; return 1; }
  SampleGrid G;
  if (multi_sample_ready(m, &G)) return 1;
  return run_all(m, [&](int r) { return r2s_sample_download_weights(m->ctx[(size_t)r], weights, r == 0 ? th : nullptr, m->cut[(size_t)r], m->cut[(size_t)r + 1]); });
}

int r2s_multi_export_isosurface(r2s_multi *m, const char *path, int format) {
  if (!m) return 1;
  if (!path) { m->err = "r2s_multi_export_isosurface: path is required"; return 1; }
  if (!m->have_surface) { m->err = "isosurface: no surface on this handle (call r2s_multi_isosurface first)"; return 1; }
  const i64 nv = m->surf_vb[(size_t)m->n], nt = m->surf_tb[(size_t)m->n];
  std::vector<float> V((size_t)(3 * nv));
  std::vector<int32_t> T((size_t)(3 * nt));
  if (multi_download(m, V.data(), T.data(), true)) return 1;
  return r2s_surf_write_file(path, format, V.data(), nv, T.data(), nt, &m->err);
}
}  // extern "C"
