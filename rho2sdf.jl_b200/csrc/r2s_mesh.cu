// r2s_mesh.cu -- mesh tables and the pre-timer stages of rho2sdf(): node->element connectivity, boundary faces,
// calculate_mesh_volume, DenseInNodes, calculate_isocontour_volume.   Compiled with -fmad=false: these values feed
// threshold comparisons downstream, so they are evaluated in the reference's operation order without contraction.
#include "r2s_common.cuh"
#include "r2s_tables.cuh"
#include "r2s_iso.cuh"

// ---------------------------------------------------------------------------------------------------------------
// INE: node -> elements (MeshGrid/MeshInformations.jl:69-77), lists sorted ascending like the reference's push! order
// ---------------------------------------------------------------------------------------------------------------
__global__ void k_ine_count(const int *__restrict__ IEN, i64 n, int *__restrict__ cnt) {
  i64 t = blockIdx.x * (i64)blockDim.x + threadIdx.x;
  if (t < n) atomicAdd(&cnt[IEN[t]], 1);
}
__global__ void k_ine_fill(const int *__restrict__ IEN, i64 n, int nen, const int *__restrict__ ptr, int *__restrict__ cur, int *__restrict__ out) {
  i64 t = blockIdx.x * (i64)blockDim.x + threadIdx.x;
  if (t < n) { int nd = IEN[t]; int s = atomicAdd(&cur[nd], 1); out[ptr[nd] + s] = (int)(t / nen); }
}
__global__ void k_ine_sort(i64 nnp, const int *__restrict__ ptr, int *__restrict__ lst) {
  i64 n = blockIdx.x * (i64)blockDim.x + threadIdx.x;
  if (n >= nnp) return;
  int a = ptr[n], b = ptr[n + 1];
  for (int i = a + 1; i < b; i++) { int v = lst[i], j = i - 1; while (j >= a && lst[j] > v) { lst[j + 1] = lst[j]; j--; } lst[j + 1] = v; }
}
__global__ void k_ien_convert(const i64 *__restrict__ in, i64 n, int *__restrict__ out) {
  i64 t = blockIdx.x * (i64)blockDim.x + threadIdx.x;
  if (t < n) out[t] = (int)(in[t] - 1);
}
// boundary faces (SignedDistances/sdfOnDensityField.jl:511-519): the INE lists of the face's nodes share exactly one element
__global__ void k_face_boundary(i64 nel, int nen, int nes, int nsn, const int *__restrict__ IEN, const int *__restrict__ ptr, const int *__restrict__ lst,
                                unsigned char *__restrict__ fb) {
  i64 e = blockIdx.x * (i64)blockDim.x + threadIdx.x;
  if (e >= nel) return;
  int mask = 0;
  for (int sg = 0; sg < nes; sg++) {
    const int *fn = nen == 8 ? c_hex_isn[sg] : c_tet_isn[sg];
    int n0 = IEN[nen * e + fn[0]], count = 0;
    for (int p = ptr[n0]; p < ptr[n0 + 1]; p++) {
      int e2 = lst[p]; bool all = true;
      for (int a = 1; a < nsn && all; a++) {
        int na = IEN[nen * e + fn[a]]; bool found = false;
        for (int b = 0; b < nen; b++) found |= (IEN[nen * (i64)e2 + b] == na);
        all = found;
      }
      if (all) count++;
    }
    if (count == 1) mask |= 1 << sg;
  }
  fb[e] = (unsigned char)mask;
}

int r2s_mesh_upload_ien(r2s_ctx *ctx, const int64_t *IEN) {
  i64 n = ctx->nel * ctx->nen;
  DevBuf tmp;
  CK(tmp.reserve(sizeof(i64) * (size_t)n));
  CK(cudaMemcpyAsync(tmp.p, IEN, sizeof(i64) * (size_t)n, cudaMemcpyHostToDevice, ctx->stream));
  k_ien_convert<<<cdiv(n, 256), 256, 0, ctx->stream>>>(tmp.as<i64>(), n, ctx->IEN32.as<int>()); LAUNCH_CHECK();
  CK(cudaStreamSynchronize(ctx->stream));
  tmp.release();
  return 0;
}
// z-extent of every element (geometry only, built with the mesh): lets a z-slab rank discard the elements far from its planes
// with one 16-byte read instead of gathering their nodes
__global__ void k_elem_zrange(i64 nel, int nen, const int *__restrict__ IEN, const double *__restrict__ X, double2 *__restrict__ ezr) {
  i64 e = blockIdx.x * (i64)blockDim.x + threadIdx.x;
  if (e >= nel) return;
  double lo = 1e300, hi = -1e300;
  for (int a = 0; a < nen; a++) { double z = X[3 * (i64)IEN[nen * e + a] + 2]; lo = fmin(lo, z); hi = fmax(hi, z); }
  ezr[e] = make_double2(lo, hi);
}
// HEX8 elements that are axis-aligned boxes in canonical node order (every mixed monomial coefficient of the geometry exactly zero):
// the projection kernel has a variant for them (iso::HexBox, r2s_iso.cuh).  Geometry only, so the flag is built with the mesh.
__global__ void k_elem_box(i64 nel, const int *__restrict__ IEN, const double *__restrict__ X, unsigned char *__restrict__ ebox, unsigned long long *__restrict__ count) {
  i64 e = blockIdx.x * (i64)blockDim.x + threadIdx.x;
  bool box = false;
  if (e < nel) {
    double A[4][8];
    for (int d = 0; d < 3; d++) {
      double nv[8];
      for (int a = 0; a < 8; a++) nv[a] = X[3 * (i64)IEN[8 * e + a] + d];
      iso::monomial8(nv, A[d]);
    }
    box = iso::is_box(A) && A[0][1] != 0.0 && A[1][2] != 0.0 && A[2][3] != 0.0;
    ebox[e] = box ? 1 : 0;
  }
  unsigned m = __ballot_sync(0xffffffffu, box);
  if ((threadIdx.x & 31) == 0 && m) atomicAdd(count, (unsigned long long)__popc(m));
}
int r2s_mesh_build_tables(r2s_ctx *ctx) {
  i64 n = ctx->nel * ctx->nen;
  CK(ctx->ine_ptr.reserve(sizeof(int) * (size_t)(ctx->nnp + 1)));
  CK(ctx->ine_el.reserve(sizeof(int) * (size_t)n));
  CK(ctx->fbnd.reserve((size_t)ctx->nel));
  DevBuf cnt, cur;
  CK(cnt.reserve(sizeof(int) * (size_t)(ctx->nnp + 1)));
  CK(cur.reserve(sizeof(int) * (size_t)(ctx->nnp + 1)));
  CK(cudaMemsetAsync(cnt.p, 0, sizeof(int) * (size_t)(ctx->nnp + 1), ctx->stream));
  CK(cudaMemsetAsync(cur.p, 0, sizeof(int) * (size_t)(ctx->nnp + 1), ctx->stream));
  k_ine_count<<<cdiv(n, 256), 256, 0, ctx->stream>>>(ctx->IEN32.as<int>(), n, cnt.as<int>()); LAUNCH_CHECK();
  if (r2s_scan_exclusive_i32(ctx, cnt.as<int>(), ctx->ine_ptr.as<int>(), ctx->nnp + 1)) return 1;
  k_ine_fill<<<cdiv(n, 256), 256, 0, ctx->stream>>>(ctx->IEN32.as<int>(), n, ctx->nen, ctx->ine_ptr.as<int>(), cur.as<int>(), ctx->ine_el.as<int>()); LAUNCH_CHECK();
  k_ine_sort<<<cdiv(ctx->nnp, 256), 256, 0, ctx->stream>>>(ctx->nnp, ctx->ine_ptr.as<int>(), ctx->ine_el.as<int>()); LAUNCH_CHECK();
  k_face_boundary<<<cdiv(ctx->nel, 256), 256, 0, ctx->stream>>>(ctx->nel, ctx->nen, ctx->nes, ctx->nsn, ctx->IEN32.as<int>(), ctx->ine_ptr.as<int>(),
                                                                ctx->ine_el.as<int>(), ctx->fbnd.as<unsigned char>()); LAUNCH_CHECK();
  CK(ctx->ezr.reserve(sizeof(double2) * (size_t)ctx->nel));
  k_elem_zrange<<<cdiv(ctx->nel, 256), 256, 0, ctx->stream>>>(ctx->nel, ctx->nen, ctx->IEN32.as<int>(), ctx->X.as<double>(), ctx->ezr.as<double2>()); LAUNCH_CHECK();
  ctx->n_box = 0;
  if (ctx->nen == 8) {
    const size_t flag_bytes = ((size_t)ctx->nel + 7) & ~(size_t)7;      // the 8-byte counter sits behind the flags
    CK(ctx->ebox.reserve(flag_bytes + 8));
    unsigned long long *dcount = (unsigned long long *)(ctx->ebox.as<unsigned char>() + flag_bytes), hcount = 0;
    CK(cudaMemsetAsync(dcount, 0, 8, ctx->stream));
    k_elem_box<<<cdiv(ctx->nel, 256), 256, 0, ctx->stream>>>(ctx->nel, ctx->IEN32.as<int>(), ctx->X.as<double>(), ctx->ebox.as<unsigned char>(), dcount); LAUNCH_CHECK();
    if (r2s_readback(ctx, &hcount, dcount, 8)) return 1;
    ctx->n_box = (i64)hcount;
  }
  CK(cudaStreamSynchronize(ctx->stream));
  cnt.release(); cur.release();
  return 0;
}

// ---------------------------------------------------------------------------------------------------------------
// Tensor-product lattice meshes.  When every HEX8 element is an axis-aligned box in canonical node order whose two corner
// coordinates are NEIGHBOURING entries of three per-axis tables of distinct node coordinates (voxel-type SIMP meshes, also
// graded ones and ones with holes, any element numbering), the elements whose closed AABB contains a point -- the candidate set
// of Sign_Detection_HEX8 (SignDetection.jl:30) -- follow from the point's position in the three tables: no sort, no lists.
// Built with the mesh: lat_xs (tables), lat_cell[e] (cell of element e), lat_map[cell] (element of a cell or -1).
// ---------------------------------------------------------------------------------------------------------------
__global__ void k_gather_axis(i64 nnp, const double *__restrict__ X, int d, double *__restrict__ out) {
  i64 i = blockIdx.x * (i64)blockDim.x + threadIdx.x;
  if (i < nnp) out[i] = X[3 * i + d];
}
__device__ inline int lat_find(const double *xs, int n, double v) {      // index of v in the sorted table or -1
  int l = 0, h = n;
  while (l < h) { int m = (l + h) >> 1; if (xs[m] < v) l = m + 1; else h = m; }
  return (l < n && xs[l] == v) ? l : -1;
}
__global__ void k_lat_cells(i64 nel, const int *__restrict__ IEN, const double *__restrict__ X, const double *__restrict__ xs, int o0, int o1, int o2, int n0, int n1, int n2,
                            int *__restrict__ cell_of, int *__restrict__ map, int *__restrict__ fail) {
  i64 e = blockIdx.x * (i64)blockDim.x + threadIdx.x;
  if (e >= nel) return;
  const i64 na = IEN[8 * e], nb = IEN[8 * e + 6];      // opposite corners (-1,-1,-1) and (+1,+1,+1) of the canonical node order
  const int off[3] = {o0, o1, o2}, nd[3] = {n0, n1, n2};
  int a[3]; bool ok = true;
  for (int d = 0; d < 3; d++) {
    const double lo = X[3 * na + d], hi = X[3 * nb + d];
    a[d] = lat_find(xs + off[d], nd[d], lo);
    ok = ok && a[d] >= 0 && a[d] + 1 < nd[d] && xs[off[d] + a[d] + 1] == hi && lo < hi;
  }
  if (!ok) { atomicExch(fail, 1); cell_of[e] = -1; return; }
  const i64 c = ((i64)a[2] * (n1 - 1) + a[1]) * (n0 - 1) + a[0];
  cell_of[e] = (int)c;
  if (atomicCAS(&map[c], -1, (int)e) != -1) atomicExch(fail, 1);      // two elements in one cell: not a lattice mesh
}
int r2s_mesh_build_lattice(r2s_ctx *ctx) {
  ctx->lattice = false; ctx->lat_ncell = 0;
  if (ctx->nen != 8 || ctx->n_box != ctx->nel || ctx->nel >= (1ll << 28)) return 0;
  cudaStream_t st = ctx->stream;
  DevBuf a, b, u;
  CK(a.reserve(sizeof(double) * (size_t)ctx->nnp)); CK(b.reserve(sizeof(double) * (size_t)ctx->nnp)); CK(u.reserve(sizeof(double) * (size_t)ctx->nnp));
  std::vector<double> tabs; int nd[3], off[3];
  for (int d = 0; d < 3; d++) {
    k_gather_axis<<<cdiv(ctx->nnp, 256), 256, 0, st>>>(ctx->nnp, ctx->X.as<double>(), d, a.as<double>()); LAUNCH_CHECK();
    double *sorted = nullptr; i64 cnt = 0;
    if (r2s_sort_f64(ctx, a.as<double>(), b.as<double>(), ctx->nnp, &sorted)) return 1;
    if (r2s_unique_f64(ctx, sorted, u.as<double>(), ctx->nnp, &cnt)) return 1;
    if (cnt < 2 || cnt > 100000) { a.release(); b.release(); u.release(); return 0; }      // not a lattice worth tabulating
    off[d] = (int)tabs.size(); nd[d] = (int)cnt; tabs.resize(tabs.size() + (size_t)cnt);
    if (r2s_readback(ctx, tabs.data() + off[d], u.p, sizeof(double) * (size_t)cnt)) return 1;
  }
  a.release(); b.release(); u.release();
  const i64 ncell = (i64)(nd[0] - 1) * (nd[1] - 1) * (nd[2] - 1);
  if (ncell >= (1ll << 31) || ncell > 64 * ctx->nel + 4096) return 0;                       // a sparse point cloud of boxes: the cell map would not pay
  CK(ctx->lat_xs.reserve(sizeof(double) * tabs.size()));
  CK(cudaMemcpyAsync(ctx->lat_xs.p, tabs.data(), sizeof(double) * tabs.size(), cudaMemcpyHostToDevice, st));
  CK(ctx->lat_cell.reserve(sizeof(int) * (size_t)ctx->nel));
  CK(ctx->lat_map.reserve(sizeof(int) * (size_t)ncell + 8));
  CK(cudaMemsetAsync(ctx->lat_map.p, 0xff, sizeof(int) * (size_t)ncell + 8, st));
  int *fail = ctx->lat_map.as<int>() + ncell;      // one word behind the map
  CK(cudaMemsetAsync(fail, 0, sizeof(int), st));
  k_lat_cells<<<cdiv(ctx->nel, 256), 256, 0, st>>>(ctx->nel, ctx->IEN32.as<int>(), ctx->X.as<double>(), ctx->lat_xs.as<double>(), off[0], off[1], off[2], nd[0], nd[1], nd[2],
                                                   ctx->lat_cell.as<int>(), ctx->lat_map.as<int>(), fail); LAUNCH_CHECK();
  int hfail = 1;
  if (r2s_readback(ctx, &hfail, fail, sizeof(int))) return 1;
  if (hfail) return 0;
  for (int d = 0; d < 3; d++) { ctx->lat_nd[d] = nd[d]; ctx->lat_off[d] = off[d]; }
  ctx->lat_ncell = ncell; ctx->lattice = true;
  return 0;
}
extern "C" int r2s_mesh_is_lattice(r2s_ctx *ctx, int *is_lattice) {
  if (!ctx || !is_lattice) return 1;
  *is_lattice = ctx->lattice ? 1 : 0;
  return 0;
}

// deterministic sum: per-block partials in a fixed slot, summed in slot order by one thread
__global__ void k_sum_partials(const double *__restrict__ part, int n, int stride, double *__restrict__ out) {
  if (threadIdx.x == 0 && blockIdx.x == 0)
    for (int s = 0; s < stride; s++) { double acc = 0; for (int i = 0; i < n; i++) acc += part[(size_t)i * stride + s]; out[s] = acc; }
}
template <int NV>
__device__ inline void block_sum_store(double v[NV], double *part) {
  __shared__ double sh[NV][32];
  int lane = threadIdx.x & 31, w = threadIdx.x >> 5, nw = (blockDim.x + 31) >> 5;
#pragma unroll
  for (int q = 0; q < NV; q++) {
    double x = v[q];
    for (int o = 16; o > 0; o >>= 1) x += __shfl_down_sync(0xffffffffu, x, o);
    if (lane == 0) sh[q][w] = x;
  }
  __syncthreads();
  if (threadIdx.x == 0)
    for (int q = 0; q < NV; q++) { double acc = 0; for (int i = 0; i < nw; i++) acc += sh[q][i]; part[(size_t)blockIdx.x * NV + q] = acc; }
}

// calculate_mesh_volume (MeshGrid/MeshVolume.jl:4-117), 3x3x3 Gauss
__global__ void k_mesh_volume(i64 nel, int nen, const double *__restrict__ X, const int *__restrict__ IEN, const double *__restrict__ rho,
                              GaussTab G3, double *__restrict__ part) {
  i64 e = blockIdx.x * (i64)blockDim.x + threadIdx.x;
  double v2[2] = {0.0, 0.0};
  if (e < nel) {
    double vol = 0.0;
    if (nen == 8) {
      double xe[3][8];
      for (int a = 0; a < 8; a++) for (int d = 0; d < 3; d++) xe[d][a] = X[3 * (i64)IEN[8 * e + a] + d];
      double N[8], dN[8][3];
      for (int k = 0; k < 3; k++) for (int j = 0; j < 3; j++) for (int i = 0; i < 3; i++) {
        double xi[3] = {G3.x[i], G3.x[j], G3.x[k]}; hex8_shape_d(xi, N, dN);
        double J[3][3];
        for (int r = 0; r < 3; r++) for (int c = 0; c < 3; c++) { double s = 0; for (int a = 0; a < 8; a++) s += xe[r][a] * dN[a][c]; J[r][c] = s; }
        vol += G3.w[i] * G3.w[j] * G3.w[k] * fabs(det3(J));
      }
    } else {
      double xe[3][4];
      for (int a = 0; a < 4; a++) for (int d = 0; d < 3; d++) xe[d][a] = X[3 * (i64)IEN[4 * e + a] + d];
      double J[3][3];
      for (int r = 0; r < 3; r++) { J[r][0] = xe[r][0] - xe[r][3]; J[r][1] = xe[r][1] - xe[r][3]; J[r][2] = xe[r][2] - xe[r][3]; }
      double adet = fabs(det3(J));
      for (int k = 0; k < 3; k++) for (int j = 0; j < 3; j++) for (int i = 0; i < 3; i++) {
        double xi = (G3.x[i] + 1.0) / 2.0, eta = (G3.x[j] + 1.0) / 2.0 * (1.0 - xi), zeta = (G3.x[k] + 1.0) / 2.0 * (1.0 - xi - eta);
        if (xi < 0 || eta < 0 || zeta < 0 || xi + eta + zeta > 1.0) continue;
        double jt = (1.0 - xi) * (1.0 - xi) * (1.0 - xi - eta) / 8.0;
        vol += G3.w[i] * G3.w[j] * G3.w[k] * adet * jt;
      }
    }
    v2[0] = vol; v2[1] = vol * rho[e];
  }
  block_sum_store<2>(v2, part);
}
int r2s_dev_mesh_volume(r2s_ctx *ctx, double *vd, double *vf) {
  int nb = cdiv(ctx->nel, 128);
  CK(ctx->v_part.reserve(sizeof(double) * (size_t)(2 * nb + 2)));
  double *part = ctx->v_part.as<double>();
  k_mesh_volume<<<nb, 128, 0, ctx->stream>>>(ctx->nel, ctx->nen, ctx->X.as<double>(), ctx->IEN32.as<int>(), ctx->rho_e.as<double>(), gauss_legendre_host(3), part); LAUNCH_CHECK();
  k_sum_partials<<<1, 32, 0, ctx->stream>>>(part, nb, 2, part + 2 * (size_t)nb); LAUNCH_CHECK();
  double h[2];
  if (r2s_readback(ctx, h, part + 2 * (size_t)nb, sizeof(h))) return 1;
  *vd = h[0]; *vf = h[1] / h[0];
  return 0;
}

// ---------------------------------------------------------------------------------------------------------------
// DenseInNodes (MeshGrid/NodalDensities.jl:89-218)
// ---------------------------------------------------------------------------------------------------------------
__global__ void k_centroids(i64 nel, int nen, const double *__restrict__ X, const int *__restrict__ IEN, double *__restrict__ C) {
  i64 e = blockIdx.x * (i64)blockDim.x + threadIdx.x;
  if (e >= nel) return;
  for (int d = 0; d < 3; d++) { double s = 0; for (int a = 0; a < nen; a++) s += X[3 * (i64)IEN[nen * e + a] + d]; C[3 * e + d] = s / nen; }
}
__device__ inline void jacobi_eig4(double A[4][4], double lam[4], double V[4][4]) {
  for (int i = 0; i < 4; i++) for (int j = 0; j < 4; j++) V[i][j] = (i == j);
  for (int sweep = 0; sweep < 60; sweep++) {
    double off = 0; for (int p = 0; p < 4; p++) for (int q = p + 1; q < 4; q++) off += A[p][q] * A[p][q];
    if (off == 0.0) break;
    for (int p = 0; p < 4; p++) for (int q = p + 1; q < 4; q++) {
      if (A[p][q] == 0.0) continue;
      double theta = (A[q][q] - A[p][p]) / (2.0 * A[p][q]);
      double t = (theta >= 0 ? 1.0 : -1.0) / (fabs(theta) + sqrt(theta * theta + 1.0));
      double c = 1.0 / sqrt(t * t + 1.0), s = t * c;
      for (int k = 0; k < 4; k++) { double akp = A[k][p], akq = A[k][q]; A[k][p] = c * akp - s * akq; A[k][q] = s * akp + c * akq; }
      for (int k = 0; k < 4; k++) { double apk = A[p][k], aqk = A[q][k]; A[p][k] = c * apk - s * aqk; A[q][k] = s * apk + c * aqk; }
      for (int k = 0; k < 4; k++) { double vkp = V[k][p], vkq = V[k][q]; V[k][p] = c * vkp - s * vkq; V[k][q] = s * vkp + c * vkq; }
    }
  }
  for (int i = 0; i < 4; i++) lam[i] = A[i][i];
  for (int i = 0; i < 4; i++) for (int j = i + 1; j < 4; j++) if (lam[j] < lam[i]) {
    double t = lam[i]; lam[i] = lam[j]; lam[j] = t;
    for (int k = 0; k < 4; k++) { double u = V[k][i]; V[k][i] = V[k][j]; V[k][j] = u; }
  }
}
__global__ void k_nodal_densities(i64 nnp, const double *__restrict__ X, const double *__restrict__ C, const int *__restrict__ ptr, const int *__restrict__ lst,
                                  const double *__restrict__ rho, double *__restrict__ out) {
  i64 i = blockIdx.x * (i64)blockDim.x + threadIdx.x;
  if (i >= nnp) return;
  int a0 = ptr[i], n1 = ptr[i + 1] - a0; const int *els = lst + a0;
  if (n1 == 0) { out[i] = 0.0; return; }
  if (n1 == 1) { out[i] = rho[els[0]]; return; }
  if (n1 < 4) {
    double L[3], Lmax = 0;
    for (int j = 0; j < n1; j++) {
      double v0 = X[3 * i] - C[3 * (i64)els[j]], v1 = X[3 * i + 1] - C[3 * (i64)els[j] + 1], v2 = X[3 * i + 2] - C[3 * (i64)els[j] + 2];
      L[j] = sqrt((v0 * v0 + v1 * v1) + v2 * v2); if (L[j] > Lmax) Lmax = L[j];
    }
    Lmax *= 1.2; double dm = 0, de = 0;
    for (int j = 0; j < n1; j++) { dm += rho[els[j]] * (1 - L[j] / Lmax); de += (1 - L[j] / Lmax); }
    out[i] = dm / de; return;
  }
  double AtA[4][4] = {{0}}, Atb[4] = {0, 0, 0, 0}, bsum = 0;
  for (int j = 0; j < n1; j++) {
    double row[4] = {1.0, C[3 * (i64)els[j]], C[3 * (i64)els[j] + 1], C[3 * (i64)els[j] + 2]}, b = rho[els[j]];
    for (int r = 0; r < 4; r++) { for (int c = 0; c < 4; c++) AtA[r][c] += row[r] * row[c]; Atb[r] += row[r] * b; }
    bsum += b;
  }
  double lam[4], V[4][4]; jacobi_eig4(AtA, lam, V);
  double lmax = lam[0], lmin = lam[0];
  for (int k = 1; k < 4; k++) { if (lam[k] > lmax) lmax = lam[k]; if (lam[k] < lmin) lmin = lam[k]; }
  double e1 = fabs(lmax / lmin), e2 = fabs(lmax / lam[1]), e3 = fabs(lmax / lam[2]);
  int poz = -1;
  if (1e7 > e1 && 3e3 > e2) poz = 0;
  else if (1e7 < e1 && 3e3 > e2) poz = 1;
  else if (1e7 < e1 && 3e3 < e2) poz = (3e3 > e3) ? 2 : 3;
  if (poz < 0) { out[i] = bsum / (double)n1; return; }
  double b1[4], x2[4] = {0, 0, 0, 0}, xx[4];
  for (int k = 0; k < 4; k++) { double s = 0; for (int r = 0; r < 4; r++) s += V[r][k] * Atb[r]; b1[k] = s; }
  for (int k = poz; k < 4; k++) x2[k] = b1[k] / lam[k];
  for (int r = 0; r < 4; r++) { double s = 0; for (int k = 0; k < 4; k++) s += V[r][k] * x2[k]; xx[r] = s; }
  out[i] = 1.0 * xx[0] + X[3 * i] * xx[1] + X[3 * i + 1] * xx[2] + X[3 * i + 2] * xx[3];
}
int r2s_dev_nodal_densities(r2s_ctx *ctx) {
  DevBuf C;
  CK(C.reserve(sizeof(double) * 3 * (size_t)ctx->nel));
  CK(ctx->rho_n.reserve(sizeof(double) * (size_t)ctx->nnp));
  k_centroids<<<cdiv(ctx->nel, 256), 256, 0, ctx->stream>>>(ctx->nel, ctx->nen, ctx->X.as<double>(), ctx->IEN32.as<int>(), C.as<double>()); LAUNCH_CHECK();
  k_nodal_densities<<<cdiv(ctx->nnp, 128), 128, 0, ctx->stream>>>(ctx->nnp, ctx->X.as<double>(), C.as<double>(), ctx->ine_ptr.as<int>(), ctx->ine_el.as<int>(),
                                                                   ctx->rho_e.as<double>(), ctx->rho_n.as<double>()); LAUNCH_CHECK();
  CK(cudaStreamSynchronize(ctx->stream));
  C.release();
  return 0;
}

// ---------------------------------------------------------------------------------------------------------------
// calculate_isocontour_volume (MeshGrid/Isocontour_volume.jl:1-75): 15^3 Gauss in crossing elements, 3^3 in solid ones
// one warp per element; lanes stride over the quadrature points, fixed-order warp reduction
// ---------------------------------------------------------------------------------------------------------------
__global__ void k_iso_volume(i64 nel, const double *__restrict__ X, const int *__restrict__ IEN, const double *__restrict__ rn, double thr,
                             GaussTab G3, GaussTab G15, double *__restrict__ part) {
  i64 e = (blockIdx.x * (i64)blockDim.x + threadIdx.x) >> 5; int lane = threadIdx.x & 31;
  double v1[1] = {0.0};
  if (e < nel) {
    double ev[8], mn = 1e300, mx = -1e300, xe[3][8];
    for (int a = 0; a < 8; a++) { int n = IEN[8 * e + a]; ev[a] = rn[n]; mn = fmin(mn, ev[a]); mx = fmax(mx, ev[a]); for (int d = 0; d < 3; d++) xe[d][a] = X[3 * (i64)n + d]; }
    if (!(mx < thr)) {
      bool chk = !(mn >= thr); int n = chk ? 15 : 3; const double *gp = chk ? G15.x : G3.x, *w = chk ? G15.w : G3.w;
      double vol = 0.0, N[8], dN[8][3];
      for (int q = lane; q < n * n * n; q += 32) {
        int i = q % n, j = (q / n) % n, k = q / (n * n);
        double xi[3] = {gp[i], gp[j], gp[k]}; hex8_shape_d(xi, N, dN);
        if (chk) { double v = 0; for (int a = 0; a < 8; a++) v += N[a] * ev[a]; if (v < thr) continue; }
        double J[3][3];
        for (int r = 0; r < 3; r++) for (int c = 0; c < 3; c++) { double s = 0; for (int a = 0; a < 8; a++) s += xe[r][a] * dN[a][c]; J[r][c] = s; }
        vol += w[i] * w[j] * w[k] * fabs(det3(J));
      }
      v1[0] = vol;
    }
  }
  block_sum_store<1>(v1, part);
}
int r2s_dev_isocontour_volume(r2s_ctx *ctx, double thr, double *vol) {
  if (ctx->nen != 8) FAIL("calculate_isocontour_volume is implemented for HEX8 only (as in the reference, Isocontour_volume.jl:27-38)");
  int nb = cdiv(ctx->nel * 32, 256);
  CK(ctx->v_part.reserve(sizeof(double) * (size_t)(nb + 2)));
  double *part = ctx->v_part.as<double>();
  k_iso_volume<<<nb, 256, 0, ctx->stream>>>(ctx->nel, ctx->X.as<double>(), ctx->IEN32.as<int>(), ctx->rho_n.as<double>(), thr, gauss_legendre_host(3), gauss_legendre_host(15), part); LAUNCH_CHECK();
  k_sum_partials<<<1, 32, 0, ctx->stream>>>(part, nb, 1, part + nb); LAUNCH_CHECK();
  double h;
  if (r2s_readback(ctx, &h, part + nb, sizeof(h))) return 1;
  *vol = h;
  return 0;
}

// ------------------------------------------------------------------------------------------------ grid set-up statistics (SURVEY.md 8f-3)
// calculate_edge_distances + analyze_mesh (MeshGrid/Grid_setup.jl:28-92): the lengths of all element edges and their
// median, which is the grid step of the :automatic set-up (noninteractive_sdf_grid_setup, :94-109).  Edge tables:
// ElementTypes.jl:30-35 (HEX8) and :63-66 (TET4).  sqrt(dx^2 + dy^2 + dz^2) without contraction, like the Julia expression.
__constant__ int c_edges_hex[12][2] = {{0, 1}, {1, 2}, {2, 3}, {3, 0}, {4, 5}, {5, 6}, {6, 7}, {7, 4}, {0, 4}, {1, 5}, {2, 6}, {3, 7}};
__constant__ int c_edges_tet[6][2] = {{0, 1}, {1, 2}, {2, 0}, {0, 3}, {1, 3}, {2, 3}};
__global__ void k_edge_lengths(i64 nel, int nen, int noe, const int *__restrict__ IEN, const double *__restrict__ X, double *__restrict__ out) {
  i64 t = blockIdx.x * (i64)blockDim.x + threadIdx.x;
  if (t >= nel * noe) return;
  i64 e = t / noe; int q = (int)(t % noe);
  int a = nen == 8 ? c_edges_hex[q][0] : c_edges_tet[q][0], b = nen == 8 ? c_edges_hex[q][1] : c_edges_tet[q][1];
  i64 na = IEN[nen * e + a], nb = IEN[nen * e + b];
  double dx = __dsub_rn(X[3 * nb], X[3 * na]), dy = __dsub_rn(X[3 * nb + 1], X[3 * na + 1]), dz = __dsub_rn(X[3 * nb + 2], X[3 * na + 2]);
  out[t] = sqrt(__dadd_rn(__dadd_rn(__dmul_rn(dx, dx), __dmul_rn(dy, dy)), __dmul_rn(dz, dz)));
}
extern "C" int r2s_mesh_box_elements(r2s_ctx *ctx, int64_t *n_box) {
  if (!ctx || !n_box) return 1;
  if (ctx->nel == 0) FAIL("r2s_set_mesh has not been called");
  *n_box = ctx->n_box;
  return 0;
}
extern "C" int r2s_edge_length_stats(r2s_ctx *ctx, double *median, double *shortest, double *longest) {
  if (!ctx) return 1;
  if (ctx->nel == 0) FAIL("r2s_set_mesh has not been called");
  CK(cudaSetDevice(ctx->device));
  const int noe = ctx->nen == 8 ? 12 : 6; const i64 n = ctx->nel * noe;
  if (n >= (1ll << 31)) FAIL("r2s_edge_length_stats: too many edges for one sort");
  DevBuf a, b;
  CK(a.reserve(sizeof(double) * (size_t)n)); CK(b.reserve(sizeof(double) * (size_t)n));
  k_edge_lengths<<<cdiv(n, 256), 256, 0, ctx->stream>>>(ctx->nel, ctx->nen, noe, ctx->IEN32.as<int>(), ctx->X.as<double>(), a.as<double>()); LAUNCH_CHECK();
  double *sorted = nullptr;
  int rc = r2s_sort_f64(ctx, a.as<double>(), b.as<double>(), n, &sorted);
  double h[4] = {0, 0, 0, 0};
  if (!rc) {
    // Julia's median: middle element, or the mean of the two middle elements for an even count
    cudaMemcpyAsync(&h[0], sorted, sizeof(double), cudaMemcpyDeviceToHost, ctx->stream);
    cudaMemcpyAsync(&h[1], sorted + (n - 1), sizeof(double), cudaMemcpyDeviceToHost, ctx->stream);
    cudaMemcpyAsync(&h[2], sorted + (n - 1) / 2, sizeof(double), cudaMemcpyDeviceToHost, ctx->stream);
    cudaMemcpyAsync(&h[3], sorted + n / 2, sizeof(double), cudaMemcpyDeviceToHost, ctx->stream);
    if (cudaStreamSynchronize(ctx->stream) != cudaSuccess) rc = 1;
  }
  a.release(); b.release();
  if (rc) FAIL("r2s_edge_length_stats: sort failed");
  if (shortest) *shortest = h[0];
  if (longest) *longest = h[1];
  if (median) *median = (n % 2) ? h[2] : (h[2] + h[3]) / 2;
  return 0;
}
