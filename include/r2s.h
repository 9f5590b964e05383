/*
 * r2s.h -- C ABI of libr2s.so, the B200 (sm_100a) implementation of the rho2sdf grid-sampling hot path.
 *
 * The reference (kopacja/rho2sdf.jl) has no FFI seam of its own: the drop-in boundary is the Julia
 * function seam.  Each entry point below replaces the body of one reference function; the Julia wrapper
 * (rho2sdf.jl_b200/julia/Rho2sdfB200.jl, see INTEGRATION.md) keeps the reference signatures and `ccall`s these.
 *
 * Conventions
 *   - every function returns 0 on success, non-zero on failure; r2s_last_error() gives the message
 *     (the Julia wrapper turns it into error(msg), mirroring the reference's error(...) calls)
 *   - arrays are Julia's: column-major, X = 3 x nnp (double), IEN = nen x nel (int64, 1-BASED node ids),
 *     grid point linear id = k*(N1+1)*(N2+1) + j*(N1+1) + i with i fastest (src/MeshGrid/Grid.jl:84-90)
 *   - all pointer arguments are HOST pointers unless the name ends in _dev; the caller owns every buffer,
 *     the library never keeps a host pointer after the call returns; device memory belongs to the context
 *   - calls are synchronous; a context is not re-entrant; one r2s_ctx drives one GPU.  Several GPUs: either r2s_multi (ONE host call
 *     drives all GPUs of the box from one process -- what the Julia drop-in uses), or one process per GPU with r2s_comm_init
 *   - there is no CPU fallback: without a CUDA device every call fails with an error
 */
#ifndef R2S_H
#define R2S_H
#include <stddef.h>
#include <stdint.h>
#ifdef __cplusplus
extern "C" {
#endif

typedef struct r2s_ctx r2s_ctx;

/* hidden constants of the reference made explicit (SURVEY.md section 5); r2s_default_params() fills the reference values */
typedef struct r2s_params {
  double rho_t;                 /* threshold density (RhoToSDF.jl:151-156)                               */
  double delta_factor;          /* band half width in cells, 1.1 (sdfOnDensityField.jl:158)              */
  int32_t remove_artifacts;     /* RhoToSDF.jl:174                                                        */
  double artifact_threshold;    /* 0.0 (RhoToSDF.jl:195)                                                  */
  double artifact_min_ratio;    /* 0.01 (RhoToSDF.jl:27)                                                  */
  int32_t rbf_interp;           /* 1 = interpolation (CG solve), 0 = approximation (RhoToSDF.jl:25)       */
  int32_t smooth;               /* 1 = :same, 2 = :fine (RhoToSDF.jl:222)                                 */
  double rbf_cut;               /* 1e-3 (RBFs4Smoothing.jl:328)                                           */
  double target_volume;         /* V_frac * V_domain (RBFs4Smoothing.jl:267)                              */
  int32_t final_volume;         /* 1 = also evaluate calculate_volume_from_sdf on the fine grid (:373)    */
} r2s_params;

typedef struct r2s_report {
  int64_t n_solid, n_crossing, n_active, n_pairs, n_not_converged, n_newton_iters;
  int64_t n_flipped;            /* remove_sdf_artifacts! return value                                     */
  int32_t cg_iters, bisections;
  float th, volume;             /* LS_Threshold offset and final fine-grid volume                          */
  float ms_bin, ms_project, ms_assemble, ms_sign, ms_cc, ms_rbf_prep, ms_cg, ms_lsf, ms_threshold, ms_fine, ms_volume, ms_total;
  int64_t launches;             /* kernels launched by the last call                                       */
  int64_t collectives;          /* NCCL collectives / grouped halo exchanges issued by the last call       */
  float cg_probe[4];            /* one CG iteration split: mat-vec, exchange 1 (dot + halo), update, exchange 2 (ms) */
  int64_t n_pairs_pruned;       /* (element, point) pairs never projected: their lower bound was not below the point's minimum */
  float ms_solve, ms_scan;      /* pair-list projection: the two k_project_list launches / record building + the two k_pair_scan launches (ms) */
} r2s_report;

/* ---- context -------------------------------------------------------------------------------------------- */
/* stream: a cudaStream_t to launch on (e.g. torch's current stream) or NULL for a private stream */
int r2s_create(r2s_ctx **ctx, int device, void *stream);
void r2s_destroy(r2s_ctx *ctx);
const char *r2s_last_error(r2s_ctx *ctx);
void r2s_default_params(r2s_params *p);
int r2s_last_report(r2s_ctx *ctx, r2s_report *rep);

/* ---- Mesh{T} container: replaces MeshGrid.Mesh ctor data (src/MeshGrid/MeshInformations.jl:36-67) --------- */
/* nen = 8 (HEX8) or 4 (TET4).  Builds INE (MeshInformations.jl:69-77) and the boundary-face table on the device. */
int r2s_set_mesh(r2s_ctx *ctx, int nen, int64_t nnp, const double *X, int64_t nel, const int64_t *IEN);
/* Grid fields exactly as Julia's Grid ctor computed them (src/MeshGrid/Grid.jl:10-34) */
int r2s_set_grid(r2s_ctx *ctx, const double amin[3], const double amax[3], const int64_t N[3], double cell_size);

/* calculate_mesh_volume (src/MeshGrid/MeshVolume.jl:4-42) */
int r2s_mesh_volume(r2s_ctx *ctx, const double *rho_e, double *V_domain, double *V_frac);
/* DenseInNodes (src/MeshGrid/NodalDensities.jl:89-109) */
int r2s_nodal_densities(r2s_ctx *ctx, const double *rho_e, double *rho_n);
/* calculate_isocontour_volume / find_threshold_for_volume (src/MeshGrid/Isocontour_volume.jl:1-154), HEX8 only */
int r2s_isocontour_volume(r2s_ctx *ctx, const double *rho_n, double threshold, double *volume);
int r2s_find_threshold(r2s_ctx *ctx, const double *rho_n, double target_volume, double rtol, int maxit, double *rho_t);

/* evalDistances (src/SignedDistances/sdfOnDensityField.jl:139-486): dist[ngp]; xp[3*ngp] or NULL */
int r2s_eval_distances(r2s_ctx *ctx, const double *rho_n, double rho_t, double delta_factor, double *dist, double *xp);
/* Sign_Detection (src/SignedDistances/SignDetection.jl:275-283): signs[ngp] in {-1,+1} */
int r2s_sign_detection(r2s_ctx *ctx, const double *rho_n, double rho_t, double *signs);
/* evalDistances / Sign_Detection at arbitrary points (csrc/r2s_points.cu): the reference's `points` argument, which it bins with
 * LinkedList(grid, points) (Grid.jl:47-69).  r2s_set_mesh and r2s_set_grid must have been called: the grid is the frame of the binning.
 * Points are double, x y z per point (Julia's 3 x n; Python's (n, 3) like generateGridPoints).
 *   distances: a point's cell per axis is c_d = floor(N_d (x_d - amin_d) / (amax_d - amin_d)) (the reference's cell expression, every
 *     operation rounded, not clamped).  An element, and each of its boundary-face triangles, considers the point iff c lies in its
 *     clamped cell range (calculateMiniAABB_grid, Grid.jl:122-154, AABB +- delta_factor * cell_size) on all three axes.  The value is the
 *     reference's running minimum over the elements in ascending index -- boundary faces before the iso projection
 *     (process_isocontour_element!), the strict < of WriteValue, xp from the first writer -- and dist = |value|.  A point that no element
 *     considers gets 1e10 and xp = 0; in particular every point whose cell lies outside [0, N_d] on some axis (this library's rule for
 *     points outside the grid).  For the grid's own points the rule is the grid path's: their cells are the cells r2s_eval_distances uses.
 *   signs: SignDetection.jl per point.  HEX8: the candidates are the elements whose closed AABB contains the point, in ascending index;
 *     TET4: the elements of the padded per-cell lists of create_grid_tetrahedra_mapping_TET4 for the point's cell point_to_grid_index =
 *     clamp(floor((x - amin) / cell_size) + 1, 1, N + 1).  A point without a candidate gets -1.
 * The results are a function of the point alone: independent of the order of the points, of chunking, and of a slab set with
 * r2s_set_slab (element ranges are never clipped); any context works, a slab rank or r2s_multi_context(m, 0) too (the call is local to
 * it).  Host arrays pass through a bounded device buffer in chunks of 2^22 points.  The call leaves the resident results as it found them
 * (sdf_dists, fine_sdf, the smoothing weights and th, an isosurface, the nodal densities of r2s_upload_nodal_densities): it uploads rho_n
 * into buffers of its own.  Rejected with an error: non-finite coordinates, n < 0, n > 0 with a NULL array, no mesh, no grid.
 * Report (r2s_last_report): the distance call sets n_solid, n_crossing, n_active, n_pairs ((crossing element, point) pairs whose range
 * holds the point), n_pairs_pruned (those skipped by a lower bound), n_newton_iters, n_not_converged, ms_bin and ms_project (the whole
 * call); the sign call sets ms_bin and ms_sign (the whole call).  R2S_PROJ_PRUNE=0 turns the bound pruning off (same bits). */
int r2s_eval_distances_points(r2s_ctx *ctx, const double *rho_n, double rho_t, double delta_factor, const double *points, int64_t n, double *dist,
                              double *xp /* 3 * n or NULL */);
int r2s_sign_detection_points(r2s_ctx *ctx, const double *rho_n, double rho_t, const double *points, int64_t n, double *signs);
/* remove_sdf_artifacts! (src/SignedDistances/SdfArtifactRemoval.jl:134-245): sdf[ngp] in/out */
int r2s_remove_artifacts(r2s_ctx *ctx, double *sdf, double threshold, double min_component_ratio, int64_t *flipped);
/* RBFs_smoothing (src/SdfSmoothing/RBFs4Smoothing.jl:321-377): fine_sdf[prod(N*smooth+1)], x fastest */
int r2s_rbf_smoothing(r2s_ctx *ctx, const double *sdf, int is_interp, int smooth, double rbf_cut, double target_volume,
                      float *fine_sdf, float *th, float *volume);
/* calculate_volume_from_sdf (src/SdfSmoothing/CalcVolumeFromSDF.jl:26-125) on an nx x ny x nz Float32 grid; quad_order =
 * detailed_quad_order (:30, default 9; 1..32 -- test/ConvergenceTests/SphereConvergenceTest.jl:67 calls it with 20) */
int r2s_volume_from_sdf(r2s_ctx *ctx, const float *sdf, int64_t nx, int64_t ny, int64_t nz, float edge, float iso, int quad_order, double *volume);

/* ---- the timed region of rho2sdf() (src/RhoToSDF.jl:164-227) as one call ---------------------------------- */
/* host buffers in/out (H2D of rho_n, D2H of sdf_dists and fine_sdf inside the call) */
int r2s_pipeline(r2s_ctx *ctx, const r2s_params *p, const double *rho_n, double *sdf_dists, float *fine_sdf, r2s_report *rep);
/* device-resident variant: rho_n already uploaded, results stay on the device */
int r2s_upload_nodal_densities(r2s_ctx *ctx, const double *rho_n);
int r2s_pipeline_resident(r2s_ctx *ctx, const r2s_params *p, r2s_report *rep);
int r2s_download_sdf(r2s_ctx *ctx, double *sdf_dists);
int r2s_download_fine_sdf(r2s_ctx *ctx, float *fine_sdf);
/* device pointers of the results of the last pipeline (double[ngp], float[prod(N*smooth+1)]) */
int r2s_result_ptrs_dev(r2s_ctx *ctx, void **sdf_dev, void **fine_sdf_dev);

/* ---- z-slab sharding (one process per GPU; SURVEY.md section 8e) ------------------------------------------ */
/* restrict this context to coarse planes k in [k0,k1) of the grid set by r2s_set_grid (halo planes are handled
 * internally); k0 = 0, k1 = N3+1 restores the full grid.  While a slab is set, r2s_eval_distances / r2s_sign_detection fill only the
 * planes [k0,k1) of their whole-grid outputs, and the whole-grid stages r2s_remove_artifacts / r2s_rbf_smoothing refuse to run.
 * r2s_set_grid resets the slab; on a multi-rank context r2s_set_slab must be called again before the next pipeline call. */
int r2s_set_slab(r2s_ctx *ctx, int64_t k0, int64_t k1);
/* Slab communicator (NCCL, bound with dlopen; see csrc/r2s_comm.cu).  Rank 0 makes a 128-byte id with r2s_comm_unique_id,
 * the host program carries it to the other ranks (torch.distributed / MPI / a file), every rank calls r2s_comm_init and
 * then r2s_set_slab (collective: the ranks exchange their plane ranges, which must tile [0, N3+1) in rank order with at
 * least 3 planes each).  From then on r2s_pipeline_resident / r2s_pipeline_slab are collective calls: halo planes of the
 * smoothing fields travel by ncclSend/ncclRecv between z-neighbours, dot products / extrema / volume sums by all-reduce,
 * and the boundary planes (labels, sizes) of the artifact removal by one all-gather. */
int r2s_comm_unique_id(void *id128);
int r2s_comm_init(r2s_ctx *ctx, int rank, int nranks, const void *id128);
int r2s_comm_destroy(r2s_ctx *ctx);
/* r2s_pipeline for one slab with host buffers: returns only this rank's planes, sdf_slab[(k1-k0)*np0*np1] and
 * fine_slab[(kf1-kf0)*f0*f1], kf0 = smooth*k0, kf1 = smooth*k1 (the last slab also owns the final fine plane) */
int r2s_pipeline_slab(r2s_ctx *ctx, const r2s_params *p, const double *rho_n, double *sdf_slab, float *fine_slab, r2s_report *rep);

/* Pipelined form for a sequence of density fields on one mesh/grid (batch use of rho2sdf): _begin returns when the device work is
 * done and the result downloads are enqueued; they drain while the next _begin computes.  The host buffers of a call belong to
 * the library until _wait(ticket) returns -- alternate between two sets of buffers. */
int r2s_pipeline_slab_begin(r2s_ctx *ctx, const r2s_params *p, const double *rho_n, double *sdf_slab, float *fine_slab, r2s_report *rep, int *ticket);
int r2s_pipeline_slab_wait(r2s_ctx *ctx, int ticket);

/* ---- all GPUs of the box from ONE host call (csrc/r2s_multi.cu) ------------------------------------------------------------ */
/* The single-process counterpart of the slab communicator above, made for the Julia drop-in (rho2sdf() is one call in one process,
 * RhoToSDF.jl:116-242): one context and one library-internal host thread per entry of device_ids, the planes cut into z-slabs
 * (re-cut by measured cost after every call), exchanges over peer memory (NVLink) -- no NCCL, no mpiexec.  device_ids may repeat
 * (several slabs on one GPU; used by the tests on one-GPU boxes).  Host arrays are WHOLE-GRID arrays; every slab writes its planes. */
typedef struct r2s_multi r2s_multi;
int r2s_multi_create(r2s_multi **m, const int *device_ids, int ndev);
void r2s_multi_destroy(r2s_multi *m);
const char *r2s_multi_last_error(r2s_multi *m);
int r2s_multi_size(r2s_multi *m);
/* context of one slab; slab 0 serves the pre-timer stages that work on the whole mesh (r2s_mesh_volume, r2s_nodal_densities,
 * r2s_find_threshold, r2s_edge_length_stats) */
r2s_ctx *r2s_multi_context(r2s_multi *m, int slab);
int r2s_multi_set_mesh(r2s_multi *m, int nen, int64_t nnp, const double *X, int64_t nel, const int64_t *IEN);
int r2s_multi_set_grid(r2s_multi *m, const double amin[3], const double amax[3], const int64_t N[3], double cell_size);
int r2s_multi_slab_planes(r2s_multi *m, int64_t *cuts /* ndev + 1 plane boundaries */);
int r2s_multi_set_rebalance(r2s_multi *m, int on);      /* 1 (default): re-cut the slabs by measured cost after every pipeline call */
/* the timed region of rho2sdf() (RhoToSDF.jl:164-227): sdf_dists[ngp], fine_sdf[prod(N*smooth+1)]; rep: stage times = max over slabs */
int r2s_multi_pipeline(r2s_multi *m, const r2s_params *p, const double *rho_n, double *sdf_dists, float *fine_sdf, r2s_report *rep);
/* exportSdfToVTI for a result that lives on several GPUs: <base>_<slab>.vti pieces + <base>.pvti (one slab: <base>.vti) */
int r2s_multi_export_vti(r2s_multi *m, const char *base, const char *label, int which);
/* page-lock / release a caller-owned host array (cudaHostRegister): result arrays pinned once download asynchronously and faster */
int r2s_pin_host(void *p, size_t bytes);
int r2s_unpin_host(void *p);

/* ---- grid set-up statistics: calculate_edge_distances + analyze_mesh (src/MeshGrid/Grid_setup.jl:28-92) ---------------------- */
/* median / shortest / longest element edge; the median is the grid step of noninteractive_sdf_grid_setup (:94-109) */
int r2s_edge_length_stats(r2s_ctx *ctx, double *median, double *shortest, double *longest);

/* number of HEX8 elements that are axis-aligned boxes in canonical node order (geometry statistic built by r2s_set_mesh; such
 * elements take the box variant of the projection kernel that stands for compute_coords_on_iso, ComputeCoordsOnIso.jl:16-87) */
int r2s_mesh_box_elements(r2s_ctx *ctx, int64_t *n_box);
/* 1 when the mesh is a tensor-product lattice of such boxes (any numbering, holes allowed): Sign_Detection_HEX8's candidate search
 * (SignDetection.jl:27-36) then reads the <= 8 cells around a point from per-axis tables instead of sorted candidate lists */
int r2s_mesh_is_lattice(r2s_ctx *ctx, int *is_lattice);

/* ---- result export: exportSdfToVTI (src/DataExport/ExportToVTI.jl:22-67) ----------------------------------------------- */
/* VTK ImageData (.vti), one PointData scalar `label` ("distance" in rho2sdf, RhoToSDF.jl:267-273), raw appended block.
 * r2s_export_vti streams a device-resident result (which = 0: sdf_dists Float64 on the coarse grid, 1: fine_sdf Float32 on the
 * grid N*smooth+1) chunk by chunk; on a slab rank it is collective and writes that rank's piece (its planes + the shared boundary
 * plane), r2s_export_pvti (any rank) writes the PImageData index naming the pieces "<piece_base>_<rank>.vti".
 * r2s_write_vti_host writes a host array (x fastest) and needs no context or GPU. */
int r2s_export_vti(r2s_ctx *ctx, const char *path, const char *label, int which);
int r2s_export_pvti(r2s_ctx *ctx, const char *path, const char *label, int which, const char *piece_base);
int r2s_write_vti_host(const char *path, const char *label, const void *values, int is_f64, int64_t nx, int64_t ny, int64_t nz, const double origin[3],
                       const double spacing[3]);

/* ---- zero surface of the smoothed SDF (csrc/r2s_surf.cu; replaces the isosurface step the reference leaves to src/Visualizations) ------- */
/* Marching cubes with a face rule that separates the two inside corners of an ambiguous face: a closed, consistently oriented mesh of
 * {value = iso}, a corner inside iff value >= iso.  One vertex per grid edge that crosses iso, ordered by (linear id of the edge's lower
 * point, axis x < y < z); coordinate origin[d] + spacing[d] * (p_d [+ t on the edge's axis]), t = (iso - va) / (vb - va) in double, rounded
 * to float once.  Triangles (int32 vertex ids, 0-based) ordered by linear cell id, then by case-table order; counter-clockwise seen from
 * outside the solid {value >= iso}.  The result is a function of the field and iso alone (no atomics decide the order), the same on one
 * context and on several slabs.  Unpaired mesh edges can only lie in the grid's boundary faces.  Rejected with an error: a non-finite value
 * or iso, fewer than 2 points on an axis, 2^31 or more cells or vertices.  The mesh stays on the device until it is downloaded or exported;
 * r2s_set_grid / r2s_set_mesh / r2s_set_slab drop it. */
/* surface {fine_sdf = iso} of the device-resident fine_sdf of the last pipeline / smoothing call: kept on the device; frame of
 * r2s_export_vti (origin AABB_min, spacing cell_size / smooth).  Fails on a slab rank of the NCCL communicator (use r2s_multi). */
int r2s_isosurface(r2s_ctx *ctx, float iso, int64_t *n_vertices, int64_t *n_triangles);
/* the same for a host field sdf[nx*ny*nz] (x fastest) in the given frame; does not touch the pipeline's resident results */
int r2s_isosurface_from_sdf(r2s_ctx *ctx, const float *sdf, int64_t nx, int64_t ny, int64_t nz, const double origin[3],
                            const double spacing[3], float iso, int64_t *n_vertices, int64_t *n_triangles);
/* vertices[3*nv] (x y z per vertex), triangles[3*nt] */
int r2s_download_isosurface(r2s_ctx *ctx, float *vertices, int32_t *triangles);
/* format 0: binary STL (unit facet normals from a double cross product, 0 0 0 for a degenerate triangle); 1: binary little-endian PLY
 * (shared vertices).  The mesh is downloaded to host memory once and written from there. */
int r2s_export_isosurface(r2s_ctx *ctx, const char *path, int format);
/* the fine_sdf of the last r2s_multi_pipeline, on all slabs: the same mesh as one context on the same field */
int r2s_multi_isosurface(r2s_multi *m, float iso, int64_t *n_vertices, int64_t *n_triangles);
int r2s_multi_download_isosurface(r2s_multi *m, float *vertices, int32_t *triangles);
int r2s_multi_export_isosurface(r2s_multi *m, const char *path, int format);

/* ---- the smoothed SDF as a continuous function (csrc/r2s_sample.cu, r2s_sample.cuh; rbf_interpolation_kdtree, RBFs4Smoothing.jl:219-248) -- */
/* The last pipeline / smoothing call leaves the field
 *     fine_sdf(x) = th + sum_c w_c exp(-(|x - c| / sigma)^2)   over the coarse grid points c with |x - c| <= maxd
 * on the device: weights w (the CG solution, or the processed Float32 SDF in approximation mode), th (the offset added to fine_sdf),
 * sigma = cell_size, maxd = float(sqrt(-ln(rbf_cut) cell_size^2)).  It lives as long as fine_sdf does: r2s_set_grid / r2s_set_mesh /
 * r2s_set_slab drop it (and a failed smoothing call), and sampling without it fails with an error.  For one query point:
 *   1. p = float(x) per coordinate, rounded once; points are double, x y z per point (Julia's 3 x n column-major)
 *   2. C_d[i] = range(Float32(amin_d), Float32(amax_d), length = N_d + 1) with a Float64 intermediate (the reference's coarse coordinates)
 *   3. e_d = C_d[i] - p_d in Float32; d2 = (e_x e_x + e_y e_y) + e_z e_z, every operation rounded; coarse point included iff
 *      sqrtf(d2) <= maxd, tested as d2 <= t2 with t2 the largest float whose correctly rounded square root is <= maxd
 *   4. phi = (a_x[i] a_y[j]) a_z[k], a_d = exp_f32(-(kappa (e_d e_d))), kappa = float(1 / cell_size^2); exp_f32 is the library's own
 *      Float32 exponential (relative error <= 1.5 2^-24); phi is within Float32 round-off of exp(-kappa d2)
 *   5. value = (fmaf(w, phi, acc) over the included points in ascending (k, j, i), from 0) + th
 *   6. gradient (optional) = (kappa + kappa) * sum fmaf(w phi, e_d, g_d) per axis, same order (d/dx of th + sum w phi)
 *   7. lattice points: p_d = float(origin_d) + float(i_d) * float(spacing_d) in Float32 (origin = AABB_min, spacing = cell_size / k gives
 *      the points of the reference's create_smooth_grid for smooth = k)
 * The reference sums the 124 nearest coarse points within maxd; no ball of radius maxd (ln(1/cut) <= 8) holds more than 124 grid points
 * (tests/test_sample_host.py proves it), so the sets are equal and only the order of summation differs.  Points outside the grid are
 * legal: missing neighbours contribute nothing, far away the value is th.  The results are a function of the point alone: the same
 * for any order or chunking of the points, on one context and on several slabs (given the same weights).  Rejected with an error:
 * non-finite coordinates, n > 0 with a NULL array, lattice dims < 1; the single-context calls fail on a slab rank of the NCCL
 * communicator (use r2s_multi).  Host arrays pass through a bounded device buffer in chunks: n is limited by host memory only. */
/* values[n]; gradients: NULL or 3 * n (x y z per point) */
int r2s_sample_sdf(r2s_ctx *ctx, const double *points, int64_t n, float *values, float *gradients);
/* values[dims[0] * dims[1] * dims[2]], x fastest; the coordinates are generated on the device (none are stored) */
int r2s_sample_sdf_lattice(r2s_ctx *ctx, const double origin[3], const double spacing[3], const int64_t dims[3], float *values);
/* the field's definition: weights[(N1+1)(N2+1)(N3+1)] (x fastest, unpitched) and th; either may be NULL */
int r2s_download_rbf_weights(r2s_ctx *ctx, float *weights, float *th);
/* the field the last r2s_multi_pipeline left on the slabs: every point goes to the slab owning its floor plane (the largest z-table
 * entry <= p_z, clamped to the grid), results come back in input order */
int r2s_multi_sample_sdf(r2s_multi *m, const double *points, int64_t n, float *values, float *gradients);
int r2s_multi_sample_sdf_lattice(r2s_multi *m, const double origin[3], const double spacing[3], const int64_t dims[3], float *values);
int r2s_multi_download_rbf_weights(r2s_multi *m, float *weights, float *th);

/* ---- zero surface of the continuous field on any lattice (csrc/r2s_surf.cu, r2s_snap.cuh) ---------------------------------------- */
/* The surface {f = iso} of the continuous smoothed field f above (the field r2s_sample_sdf evaluates) on the lattice origin + i * spacing,
 * i < dims, streamed through the device: the lattice values are never held whole and never leave the device.
 *   lattice values: a lattice point's value is bit for bit what r2s_sample_sdf_lattice returns for it; its coordinates are
 *     float(origin_d) + float(i_d) * float(spacing_d) in Float32 (rule 7 above)
 *   topology and triangles: exactly those of r2s_isosurface_from_sdf applied to that lattice field with the same origin, spacing and iso
 *     -- the same corner rule (inside iff value >= iso), face rule and case table (r2s_mc.cuh), vertex numbering (the edge's lower point,
 *     then axis x < y < z), triangle order and orientation.  The triangle array is identical, so the mesh is closed and consistently
 *     oriented wherever that one is, and the vertex count is equal.
 *   vertex placement: a crossing edge runs from lattice point a to lattice point b along axis d (a the lower point).  The vertex's two
 *     other coordinates are the lattice's Float32 coordinates; its axis-d coordinate is a Float32 x in [x_a, x_b] found by a deterministic
 *     bracketing search over Float32 values, with f evaluated by the sampler's per-point arithmetic (rules 1-6; s(x) = f(x) >= iso):
 *       bracket (lo, hi) = (x_a, x_b), keeping s(lo) = s(a), s(hi) = s(b); it starts from the lattice values (no re-evaluation).
 *       step: the Illinois regula-falsi point lo + (hi - lo) * glo / (glo - ghi) in double (every operation rounded, glo / ghi the residuals
 *         f - iso of the two ends, the one kept twice in a row halved), rounded to float; if it is not strictly inside (lo, hi) the step
 *         takes the midpoint of lo and hi in the order-preserving integer image of the floats instead.  One evaluation per step.
 *       stop: lo and hi are adjacent floats, or R2S_SNAP_MAX_EVALS = 48 evaluations have been made.
 *       result: whichever of lo and hi has the smaller |f - iso| (in double), ties to lo.
 *     csrc/r2s_snap.cuh states every operation; a host build replays it bit for bit.  The vertex stays on its own edge, so connectivity
 *     and closedness are those of the triangle array.  These coordinates are in the sampler's Float32 lattice frame, which differs in the
 *     last bit from the double frame origin + spacing * (p + t) of r2s_isosurface / r2s_isosurface_from_sdf: a vertex that the search
 *     leaves at a lattice point can differ from that frame by one rounding.
 *   memory: planes stream through a device buffer of a bounded number of planes (R2S_SURF_PLANES per chunk, read by r2s_create; default
 *     as many as fit 1 GiB of values) plus the two planes above a chunk that marching cubes reads; every plane is sampled twice (a count
 *     sweep, then an emit sweep after a host scan of the chunk totals).  Device memory: O((chunk planes + 2) * nx * ny + per-row scratch
 *     of a chunk + the output mesh).  The mesh does not depend on the chunk size.
 *   determinism: the mesh is a function of (weights, th, lattice, iso) alone: the same for any chunk size, on one context and on any slab
 *     layout of r2s_multi (given the same weights).  Several slabs: each extracts the lattice planes r2s_multi_sample_sdf_lattice assigns
 *     it; it evaluates the two lattice planes above its last plane itself, and every evaluation (lattice points and the search) reads the
 *     weights of the slab that owns the point's floor plane, through peer memory -- the rule of r2s_multi_sample_sdf, so every value is the
 *     one that slab computes.  Global bases come from a host scan of the slab totals in plane order.
 * Rejected with an error: no smoothed field on the device, a non-finite origin, spacing or lattice coordinate, dims < 2 on an axis, 2^31
 * or more cells or vertices, a non-finite iso; the single-context call fails on a slab rank of the NCCL communicator (use r2s_multi).
 * sdf_dists, fine_sdf, the weights and th are untouched; the mesh replaces this context's (handle's) surface: download / export it with
 * r2s_download_isosurface / r2s_export_isosurface (r2s_multi_download_isosurface / r2s_multi_export_isosurface). */
int r2s_isosurface_lattice(r2s_ctx *ctx, const double origin[3], const double spacing[3], const int64_t dims[3], float iso,
                           int64_t *n_vertices, int64_t *n_triangles);
int r2s_multi_isosurface_lattice(r2s_multi *m, const double origin[3], const double spacing[3], const int64_t dims[3], float iso,
                                 int64_t *n_vertices, int64_t *n_triangles);

/* The same surface on lattices of any cell count, sampling only the lattice blocks that can hold it (csrc/r2s_band.cuh, r2s_surf.cu).
 *   same mesh: lattice values, vertex numbering, triangle order, orientation and the vertex search are those of r2s_isosurface_lattice,
 *     word for word: on every lattice that call accepts, the two meshes are bit for bit equal.
 *   limits: up to 2^31 - 1 points per axis and any cell count below 2^63; fewer than 2^31 vertices (triangles hold int32 ids).
 *   skipping: the lattice is cut into blocks of 8 x 8 x 8 cells (the closed box of their 9^3 points).  A block is skipped -- never
 *     sampled -- when every coarse weight that a tap of any of its points can reach has one sign and that sign puts every Float32 value
 *     of the box on one side of iso: weights >= 0 and th >= iso, or weights >= 0 and a rigorous lower bound of the sum reaching iso - th
 *     (mirror: weights <= 0, values < iso).  The bounds cover every Float32 rounding of the sampler (r2s_band.cuh states them), so a
 *     skipped cell has no crossing; every crossing edge lies in a sampled block, and every value marching cubes or the vertex search reads
 *     there is the sampler's.  A NaN weight, or a block whose points read two slabs' weights, is always sampled.  The mesh depends on
 *     neither the block size nor the chunk size.
 *   memory: planes stream through the chunk buffer of r2s_isosurface_lattice (R2S_SURF_PLANES); per chunk one byte and one int64 per block.
 *   n_sampled (NULL or): the lattice points evaluated by one of the two sweeps -- each point at most once; the share of the lattice skipped
 *     is 1 - n_sampled / (dims[0] dims[1] dims[2]).
 * Rejected with an error: no smoothed field, a non-finite origin, spacing, lattice coordinate or iso, dims < 2 or >= 2^31 on an axis, 2^31
 * or more vertices; the single-context call fails on a slab rank of the NCCL communicator (use r2s_multi).  The weights, th and fine_sdf
 * are untouched; the mesh replaces the context's (handle's) surface, for the download and export calls above. */
int r2s_isosurface_band(r2s_ctx *ctx, const double origin[3], const double spacing[3], const int64_t dims[3], float iso,
                        int64_t *n_vertices, int64_t *n_triangles, int64_t *n_sampled);
int r2s_multi_isosurface_band(r2s_multi *m, const double origin[3], const double spacing[3], const int64_t dims[3], float iso,
                              int64_t *n_vertices, int64_t *n_triangles, int64_t *n_sampled);

/* ---- the smoothed geometry on the FE mesh: per-element solid volume fractions (csrc/r2s_elemfrac.cu, r2s_elemfrac.cuh) -------------- */
/* calculate_isocontour_volume's rule (Isocontour_volume.jl:1-75) -- a Heaviside at the Gauss points of an element, weighted by |det J| --
 * applied to the continuous field f above (the field r2s_sample_sdf evaluates) on every element of the mesh of r2s_set_mesh.  Element e,
 * quadrature order q = quad_order (1..32; 15 is the reference's order for crossing elements), nodes g and weights w of
 * gauss_legendre(q), Gauss point t = (k q + j) q + i, i.e. ascending (k, j, i):
 *   HEX8 (any trilinear element): x = sum_a N_a(g_i, g_j, g_k) X_a in double, W = ((w_i w_j) w_k) |det J|, with the shape functions and the
 *     operation order of calculate_mesh_volume (r2s_mesh_volume), every operation rounded (no contraction).
 *   TET4: the collapsed cube of calculate_mesh_volume, xi = (g_i + 1) / 2, eta = (g_j + 1) / 2 (1 - xi), zeta = (g_k + 1) / 2 (1 - xi - eta),
 *     x = xi X_0 + eta X_1 + zeta X_2 + (1 - xi - eta - zeta) X_3, W = w_i w_j w_k |det J| (1 - xi) (1 - xi - eta) / 8 -- the geometrically
 *     correct Duffy factor (sum W = |det J| / 6), NOT the reference's (1 - xi)^2 (1 - xi - eta) / 8 (MeshVolume.jl:107, 3/4 of the volume),
 *     which would bias the ratio below.  So these V_e sum to the mesh volume, while r2s_mesh_volume's TET4 V_domain is 3/4 of it.
 *   each point: p = float(x) per coordinate (sampler rule 1), f(p) by rules 2-5; the point is inside iff f >= iso (the corner rule of the
 *     surface calls); a NaN value is outside.
 *   each element: V_e = sum W and S_e = sum (inside ? W : +0) in one fixed order: 32 partials, partial l summing the points t = l mod 32 in
 *     ascending t from +0, combined by p[l] += p[l + o] for o = 16, 8, 4, 2, 1 (l < o), the result p[0].  An element whose points are all
 *     inside has S_e == V_e bit for bit, fraction exactly 1.  fractions[e] = S_e / V_e, and 0 when V_e == 0.
 *   skipping: an element is never sampled when the block classifier of r2s_isosurface_band proves every Float32 value of its box on one
 *     side of iso.  The box holds every p of the element's Gauss points: per axis [down(min_a X_a - s), up(max_a X_a + s)], s = 2^-40
 *     max_a |X_a|, widened by one Float32 step (csrc/r2s_elemfrac.cuh gives the argument).  A skipped element's V_e is computed from the
 *     geometry in the same order, and its fraction is exactly 1 or 0 -- the bits full evaluation gives; the results do not depend on it.
 *   several slabs: the elements are split across the slabs; every Gauss point reads the weights of the slab owning its floor plane
 *     (peer memory), so any split gives the bits of one context with the same weights.  An element whose box reaches the floor planes of
 *     two slabs is always sampled.  Every slab writes its elements into the whole-mesh arrays.
 * volumes (NULL or nel): V_e; n_evaluated (NULL or): the elements sampled (the others were skipped).  Needs a mesh and a smoothed field on the
 * device; sdf_dists, fine_sdf, the weights, th and any surface are untouched.  Rejected with an error: quad_order outside 1..32, a non-finite
 * iso, a NULL fractions, no mesh, no smoothed field; the single-context call fails on a slab rank of the NCCL communicator (use r2s_multi). */
int r2s_element_volume_fractions(r2s_ctx *ctx, float iso, int quad_order, double *fractions, double *volumes, int64_t *n_evaluated);
int r2s_multi_element_volume_fractions(r2s_multi *m, float iso, int quad_order, double *fractions, double *volumes, int64_t *n_evaluated);

/* ---- measurement helper (bench.py): FMA-pipe peak of the device in TFLOP/s, fp64 != 0 -> double, else float -------- */
int r2s_measure_fma_peak(r2s_ctx *ctx, int fp64, double *tflops);

#ifdef __cplusplus
}
#endif
#endif
