"""rho2sdf.jl_b200 -- host-side mirror of the kopacja/rho2sdf.jl API for the grid-sampling hot path, bound to
libr2s.so (CUDA sm_100a, C ABI in include/r2s.h) with ctypes.

The production host is the Julia wrapper in julia/Rho2sdfB200.jl (same `ccall`s); Julia is not available in the build
image, so this module carries the same names, argument meaning and error behaviour for the tests and the benchmark:

    Rho2sdfOptions, rho2sdf, rho2sdf_hex8, rho2sdf_tet4                     (reference src/RhoToSDF.jl:9-77,116-304)
    Mesh, Grid, getMesh_AABB, generateGridPoints, noninteractive_sdf_grid_setup, DenseInNodes,
    find_threshold_for_volume, calculate_isocontour_volume                  (src/MeshGrid/*)
    evalDistances, Sign_Detection, remove_sdf_artifacts                     (src/SignedDistances/*)
    RBFs_smoothing, calculate_volume_from_sdf                               (src/SdfSmoothing/*)
    isosurface, isosurface_from_sdf, isosurface_lattice, isosurface_band, export_isosurface, read_stl, read_ply  (the surface {fine_sdf = iso}, or of the continuous field on any lattice; the reference leaves it to
                                                                             src/Visualizations / ParaView)
    sample_sdf, sample_sdf_lattice, rbf_weights                             (the smoothed SDF as a continuous function:
                                                                             rbf_interpolation_kdtree, RBFs4Smoothing.jl:219-248)

Array conventions: X is (nnp, 3) float64 (== Julia's 3 x nnp column-major), IEN is (nel, nen) int64 holding 1-BASED node
ids (== Julia's nen x nel), grid fields are indexed [k, j, i] (x fastest, == Julia's (i, j, k) column-major).

There is NO CPU fallback: every computational entry point raises if the CUDA library or a GPU is missing.
"""
import ctypes as C
import math
import os

import numpy as np

__all__ = ["HEX8", "TET4", "Rho2sdfOptions", "Mesh", "Grid", "getMesh_AABB", "generateGridPoints", "noninteractive_sdf_grid_setup",
           "DenseInNodes", "find_threshold_for_volume", "calculate_isocontour_volume", "evalDistances", "Sign_Detection",
           "remove_sdf_artifacts", "RBFs_smoothing", "calculate_volume_from_sdf", "rho2sdf", "rho2sdf_hex8", "rho2sdf_tet4",
           "exportSdfToVTI", "export_device_result_to_vti", "read_vti", "read_pvti",
           "isosurface", "isosurface_from_sdf", "isosurface_lattice", "isosurface_band", "export_isosurface", "read_stl", "read_ply",
           "sample_sdf", "sample_sdf_lattice", "rbf_weights", "element_volume_fractions", "MultiContext", "FineGrid", "R2SError", "slab_partition", "init_slab_comm", "broadcast_unique_id", "load_library", "library_path", "Params", "Report", "Context"]

_HERE = os.path.dirname(os.path.abspath(__file__))
_LIB = None


class R2SError(RuntimeError):
    pass


class HEX8:
    """ElementTypes.HEX8 (src/ElementTypes/ElementTypes.jl:11)."""
    nen = 8


class TET4:
    """ElementTypes.TET4 (src/ElementTypes/ElementTypes.jl:12)."""
    nen = 4


class Params(C.Structure):
    _fields_ = [("rho_t", C.c_double), ("delta_factor", C.c_double), ("remove_artifacts", C.c_int32), ("artifact_threshold", C.c_double),
                ("artifact_min_ratio", C.c_double), ("rbf_interp", C.c_int32), ("smooth", C.c_int32), ("rbf_cut", C.c_double),
                ("target_volume", C.c_double), ("final_volume", C.c_int32)]


class Report(C.Structure):
    _fields_ = [(n, C.c_int64) for n in ("n_solid", "n_crossing", "n_active", "n_pairs", "n_not_converged", "n_newton_iters", "n_flipped")] + \
               [("cg_iters", C.c_int32), ("bisections", C.c_int32), ("th", C.c_float), ("volume", C.c_float)] + \
               [(n, C.c_float) for n in ("ms_bin", "ms_project", "ms_assemble", "ms_sign", "ms_cc", "ms_rbf_prep", "ms_cg", "ms_lsf",
                                         "ms_threshold", "ms_fine", "ms_volume", "ms_total")] + [("launches", C.c_int64), ("collectives", C.c_int64), ("cg_probe", C.c_float * 4), ("n_pairs_pruned", C.c_int64), ("ms_solve", C.c_float), ("ms_scan", C.c_float)]

    def asdict(self):
        return {n: (list(getattr(self, n)) if n == "cg_probe" else getattr(self, n)) for n, _ in self._fields_}


def library_path():
    return os.path.join(_HERE, "libr2s.so")


def load_library():
    """Load libr2s.so (built in-tree by `make -C rho2sdf.jl_b200/csrc` / __graft_entry__.build()). Fails loudly if absent."""
    global _LIB
    if _LIB is not None:
        return _LIB
    path = library_path()
    if not os.path.exists(path):
        raise R2SError("libr2s.so is not built (%s); run __graft_entry__.build() -- there is no CPU fallback" % path)
    L = C.CDLL(path)
    vp, dp, ip, fp = C.c_void_p, C.POINTER(C.c_double), C.POINTER(C.c_int64), C.POINTER(C.c_float)
    L.r2s_create.argtypes = [C.POINTER(vp), C.c_int, vp]
    L.r2s_destroy.argtypes = [vp]
    L.r2s_destroy.restype = None
    L.r2s_last_error.argtypes = [vp]
    L.r2s_last_error.restype = C.c_char_p
    L.r2s_default_params.argtypes = [C.POINTER(Params)]
    L.r2s_default_params.restype = None
    L.r2s_last_report.argtypes = [vp, C.POINTER(Report)]
    L.r2s_set_mesh.argtypes = [vp, C.c_int, C.c_int64, vp, C.c_int64, vp]
    L.r2s_set_grid.argtypes = [vp, vp, vp, vp, C.c_double]
    L.r2s_set_slab.argtypes = [vp, C.c_int64, C.c_int64]
    L.r2s_mesh_volume.argtypes = [vp, vp, dp, dp]
    L.r2s_nodal_densities.argtypes = [vp, vp, vp]
    L.r2s_isocontour_volume.argtypes = [vp, vp, C.c_double, dp]
    L.r2s_find_threshold.argtypes = [vp, vp, C.c_double, C.c_double, C.c_int, dp]
    L.r2s_eval_distances.argtypes = [vp, vp, C.c_double, C.c_double, vp, vp]
    L.r2s_sign_detection.argtypes = [vp, vp, C.c_double, vp]
    L.r2s_eval_distances_points.argtypes = [vp, vp, C.c_double, C.c_double, vp, C.c_int64, vp, vp]
    L.r2s_sign_detection_points.argtypes = [vp, vp, C.c_double, vp, C.c_int64, vp]
    L.r2s_remove_artifacts.argtypes = [vp, vp, C.c_double, C.c_double, ip]
    L.r2s_rbf_smoothing.argtypes = [vp, vp, C.c_int, C.c_int, C.c_double, C.c_double, vp, fp, fp]
    L.r2s_volume_from_sdf.argtypes = [vp, vp, C.c_int64, C.c_int64, C.c_int64, C.c_float, C.c_float, C.c_int, dp]
    L.r2s_pipeline.argtypes = [vp, C.POINTER(Params), vp, vp, vp, C.POINTER(Report)]
    L.r2s_upload_nodal_densities.argtypes = [vp, vp]
    L.r2s_pipeline_resident.argtypes = [vp, C.POINTER(Params), C.POINTER(Report)]
    L.r2s_download_sdf.argtypes = [vp, vp]
    L.r2s_download_fine_sdf.argtypes = [vp, vp]
    L.r2s_result_ptrs_dev.argtypes = [vp, C.POINTER(vp), C.POINTER(vp)]
    L.r2s_pipeline_slab.argtypes = [vp, C.POINTER(Params), vp, vp, vp, C.POINTER(Report)]
    L.r2s_pipeline_slab_begin.argtypes = [vp, C.POINTER(Params), vp, vp, vp, C.POINTER(Report), C.POINTER(C.c_int)]
    L.r2s_pipeline_slab_wait.argtypes = [vp, C.c_int]
    L.r2s_comm_unique_id.argtypes = [vp]
    L.r2s_comm_init.argtypes = [vp, C.c_int, C.c_int, vp]
    L.r2s_comm_destroy.argtypes = [vp]
    L.r2s_edge_length_stats.argtypes = [vp, dp, dp, dp]
    L.r2s_mesh_box_elements.argtypes = [vp, C.POINTER(C.c_int64)]
    L.r2s_mesh_is_lattice.argtypes = [vp, C.POINTER(C.c_int)]
    L.r2s_export_vti.argtypes = [vp, C.c_char_p, C.c_char_p, C.c_int]
    L.r2s_export_pvti.argtypes = [vp, C.c_char_p, C.c_char_p, C.c_int, C.c_char_p]
    L.r2s_multi_create.argtypes = [C.POINTER(vp), C.POINTER(C.c_int), C.c_int]
    L.r2s_multi_destroy.argtypes = [vp]
    L.r2s_multi_destroy.restype = None
    L.r2s_multi_last_error.argtypes = [vp]
    L.r2s_multi_last_error.restype = C.c_char_p
    L.r2s_multi_size.argtypes = [vp]
    L.r2s_multi_context.argtypes = [vp, C.c_int]
    L.r2s_multi_context.restype = vp
    L.r2s_multi_set_mesh.argtypes = [vp, C.c_int, C.c_int64, vp, C.c_int64, vp]
    L.r2s_multi_set_grid.argtypes = [vp, vp, vp, vp, C.c_double]
    L.r2s_multi_slab_planes.argtypes = [vp, vp]
    L.r2s_multi_set_rebalance.argtypes = [vp, C.c_int]
    L.r2s_multi_pipeline.argtypes = [vp, C.POINTER(Params), vp, vp, vp, C.POINTER(Report)]
    L.r2s_multi_export_vti.argtypes = [vp, C.c_char_p, C.c_char_p, C.c_int]
    L.r2s_pin_host.argtypes = [vp, C.c_size_t]
    L.r2s_unpin_host.argtypes = [vp]
    L.r2s_write_vti_host.argtypes = [C.c_char_p, C.c_char_p, vp, C.c_int, C.c_int64, C.c_int64, C.c_int64, vp, vp]
    L.r2s_measure_fma_peak.argtypes = [vp, C.c_int, dp]
    L.r2s_isosurface.argtypes = [vp, C.c_float, ip, ip]
    L.r2s_isosurface_from_sdf.argtypes = [vp, vp, C.c_int64, C.c_int64, C.c_int64, vp, vp, C.c_float, ip, ip]
    L.r2s_download_isosurface.argtypes = [vp, vp, vp]
    L.r2s_export_isosurface.argtypes = [vp, C.c_char_p, C.c_int]
    L.r2s_multi_isosurface.argtypes = [vp, C.c_float, ip, ip]
    L.r2s_multi_download_isosurface.argtypes = [vp, vp, vp]
    L.r2s_multi_export_isosurface.argtypes = [vp, C.c_char_p, C.c_int]
    L.r2s_isosurface_lattice.argtypes = [vp, vp, vp, vp, C.c_float, ip, ip]
    L.r2s_multi_isosurface_lattice.argtypes = [vp, vp, vp, vp, C.c_float, ip, ip]
    L.r2s_isosurface_band.argtypes = [vp, vp, vp, vp, C.c_float, ip, ip, ip]
    L.r2s_multi_isosurface_band.argtypes = [vp, vp, vp, vp, C.c_float, ip, ip, ip]
    for pre in ("r2s_", "r2s_multi_"):
        getattr(L, pre + "element_volume_fractions").argtypes = [vp, C.c_float, C.c_int, vp, vp, ip]
        getattr(L, pre + "sample_sdf").argtypes = [vp, vp, C.c_int64, vp, vp]
        getattr(L, pre + "sample_sdf_lattice").argtypes = [vp, vp, vp, vp, vp]
        getattr(L, pre + "download_rbf_weights").argtypes = [vp, vp, fp]
    _LIB = L
    return L


def _f64(a):
    return np.ascontiguousarray(a, dtype=np.float64)


def _ptr(a):
    return a.ctypes.data_as(C.c_void_p)


class _BorrowedContext:
    """A slab context owned by a MultiContext (never destroyed from here)."""

    def __init__(self, lib, h):
        self.lib, self.h = lib, C.c_void_p(h)

    def check(self, rc):
        if rc != 0:
            raise R2SError(self.lib.r2s_last_error(self.h).decode())

    def close(self):
        pass

    def report(self):
        r = Report()
        self.lib.r2s_last_report(self.h, C.byref(r))
        return r


class MultiContext:
    """r2s_multi: ONE host call drives all listed GPUs (one z-slab and one library-internal thread per entry of `devices`; entries may
    repeat -- several slabs on one GPU).  This is what the Julia drop-in's rho2sdf() uses on a multi-GPU box."""

    def __init__(self, devices):
        self.lib = load_library()
        self.h = C.c_void_p()
        ids = (C.c_int * len(devices))(*[int(d) for d in devices])
        rc = self.lib.r2s_multi_create(C.byref(self.h), ids, len(devices))
        if rc != 0 or not self.h:
            raise R2SError("r2s_multi_create failed (rc=%d): no usable CUDA device / no peer access -- this library has no CPU fallback" % rc)
        self.n = len(devices)

    def check(self, rc):
        if rc != 0:
            raise R2SError(self.lib.r2s_multi_last_error(self.h).decode())

    def slab(self, r=0):
        return _BorrowedContext(self.lib, self.lib.r2s_multi_context(self.h, int(r)))

    def slab_planes(self):
        cuts = np.zeros(self.n + 1, dtype=np.int64)
        self.check(self.lib.r2s_multi_slab_planes(self.h, _ptr(cuts)))
        return [int(v) for v in cuts]

    def close(self):
        if self.h:
            self.lib.r2s_multi_destroy(self.h)
            self.h = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


class Context:
    """One r2s_ctx = one GPU.  `stream` may be a raw cudaStream_t (e.g. torch.cuda.current_stream().cuda_stream)."""

    def __init__(self, device=0, stream=None):
        self.lib = load_library()
        self.h = C.c_void_p()
        rc = self.lib.r2s_create(C.byref(self.h), int(device), C.c_void_p(stream) if stream else None)
        if rc != 0 or not self.h:
            raise R2SError("r2s_create failed (rc=%d): no usable CUDA device -- this library has no CPU fallback" % rc)
        self._keep = []

    def check(self, rc):
        if rc != 0:
            raise R2SError(self.lib.r2s_last_error(self.h).decode())

    def close(self):
        if self.h:
            self.lib.r2s_destroy(self.h)
            self.h = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def report(self):
        r = Report()
        self.lib.r2s_last_report(self.h, C.byref(r))
        return r


def slab_partition(nz_points, world, plane_cost=None, min_planes=3):
    """Contiguous z-slabs of coarse planes, one per rank (SURVEY.md section 8e): [(k0, k1), ...] covering [0, nz_points).
    Without `plane_cost` the planes are split evenly; with a per-plane cost estimate (any positive array of length nz_points)
    the cuts equalise the cumulative cost instead (load balancing: the mesh-boundary planes carry the boundary-face work)."""
    nz_points, world = int(nz_points), int(world)
    if world < 1 or nz_points < world * (min_planes if world > 1 else 1):
        raise R2SError("cannot cut %d planes into %d slabs" % (nz_points, world))
    if plane_cost is None:
        base, rem = divmod(nz_points, world)
        out, k = [], 0
        for r in range(world):
            n = base + (1 if r < rem else 0)
            out.append((k, k + n))
            k += n
        return out
    c = np.maximum(np.asarray(plane_cost, dtype=np.float64), 1e-12)
    if c.shape != (nz_points,):
        raise R2SError("plane_cost must have one entry per plane")
    cum = np.concatenate([[0.0], np.cumsum(c)])
    cuts = [0]
    for r in range(1, world):
        k = int(np.searchsorted(cum, cum[-1] * r / world))
        k = max(k, cuts[-1] + min_planes)
        k = min(k, nz_points - (world - r) * min_planes)
        cuts.append(k)
    cuts.append(nz_points)
    return [(cuts[r], cuts[r + 1]) for r in range(world)]


def broadcast_unique_id(make_id, rank, world, group=None):
    """Carry the 128-byte communicator id from rank 0 to every rank over torch.distributed (any backend: nccl or gloo).
    `make_id()` is called on rank 0 only and must return 128 bytes."""
    import torch
    import torch.distributed as dist
    dev = "cuda" if dist.get_backend(group) == "nccl" else "cpu"
    t = torch.zeros(128, dtype=torch.uint8, device=dev)
    if rank == 0:
        raw = make_id()
        if len(raw) != 128:
            raise R2SError("communicator id must be 128 bytes")
        t.copy_(torch.frombuffer(bytearray(raw), dtype=torch.uint8))
    dist.broadcast(t, src=0, group=group)
    return bytes(t.cpu().numpy().tobytes())


def init_slab_comm(ctx, rank, world, k0, k1, uid=None):
    """Make `ctx` one rank of a z-slab decomposition: NCCL communicator (id from rank 0, carried by torch.distributed unless
    `uid` is given) and the plane range [k0, k1) of this rank.  Collective: every rank must call it."""
    lib = ctx.lib
    if uid is None:
        def make():
            buf = C.create_string_buffer(128)
            if lib.r2s_comm_unique_id(buf) != 0:
                raise R2SError("r2s_comm_unique_id failed (is NCCL available?)")
            return buf.raw
        uid = broadcast_unique_id(make, rank, world)
    ctx.check(lib.r2s_comm_init(ctx.h, int(rank), int(world), C.c_char_p(uid)))
    ctx.check(lib.r2s_set_slab(ctx.h, int(k0), int(k1)))


# ---------------------------------------------------------------------------------------------------------------------
# MeshGrid
# ---------------------------------------------------------------------------------------------------------------------
class Grid:
    """MeshGrid.Grid (src/MeshGrid/Grid.jl:2-35): AABB grown by `margineCells` cells, N = ceil((max-min)/cell)."""

    def __init__(self, AABB_min, AABB_max, N_max, margineCells=3):
        amin = _f64(AABB_min).copy()
        amax = _f64(AABB_max).copy()
        cell = float(np.max(amax - amin) / N_max)
        amin = amin - margineCells * cell
        amax = amax + margineCells * cell
        N = np.ceil((amax - amin) / cell).astype(np.int64)
        amax = amin + N * cell
        self.AABB_min, self.AABB_max, self.N, self.cell_size = amin, amax, N, cell
        self.ngp = int(np.prod(N + 1))


def getMesh_AABB(X):
    """src/MeshGrid/Grid.jl:73-77."""
    X = _f64(X)
    return X.min(axis=0), X.max(axis=0)


def generateGridPoints(grid):
    """src/MeshGrid/Grid.jl:81-93; returns (ngp, 3) (== Julia's 3 x ngp)."""
    nx, ny, nz = (int(v) + 1 for v in grid.N)
    k, j, i = np.meshgrid(np.arange(nz), np.arange(ny), np.arange(nx), indexing="ij")
    P = np.empty((grid.ngp, 3))
    P[:, 0] = grid.AABB_min[0] + grid.cell_size * i.ravel()
    P[:, 1] = grid.AABB_min[1] + grid.cell_size * j.ravel()
    P[:, 2] = grid.AABB_min[2] + grid.cell_size * k.ravel()
    return P


_HEX_EDGES = [(0, 1), (1, 2), (2, 3), (3, 0), (4, 5), (5, 6), (6, 7), (7, 4), (0, 4), (1, 5), (2, 6), (3, 7)]
_TET_EDGES = [(0, 1), (1, 2), (2, 0), (0, 3), (1, 3), (2, 3)]


class Mesh:
    """MeshGrid.Mesh (src/MeshGrid/MeshInformations.jl:16-67).  Uploads the mesh to the GPU, builds INE and the
    boundary-face table there and computes V_domain / V_frac (calculate_mesh_volume)."""

    def __init__(self, X, IEN, rho, sfce=None, element_type=HEX8, device=0, stream=None, devices=None):
        """`devices` (list of GPU ids, may repeat): the mesh goes to every listed device and the pipeline runs as z-slabs through the
        single-call multi-GPU entry (r2s_multi_*); the per-stage functions (evalDistances, ...) then work on slab 0's whole-grid context."""
        self.element_type = element_type
        self.X = _f64(X)
        self.IEN = np.ascontiguousarray(IEN, dtype=np.int64)
        if self.X.ndim != 2 or self.X.shape[1] != 3:
            raise R2SError("X must be (nnp, 3)")
        self.nsd, self.nnp = 3, self.X.shape[0]
        self.nel, self.nen = self.IEN.shape
        if self.nen != element_type.nen:
            raise R2SError("Element connectivity size (%d) doesn't match element type nodes (%d)" % (self.nen, element_type.nen))  # MeshInformations.jl:59
        self.nes, self.nsn = (6, 4) if self.nen == 8 else (4, 3)
        self.edges = _HEX_EDGES if self.nen == 8 else _TET_EDGES
        self.rho = _f64(rho)
        self.multi = None
        if devices is not None and len(devices) > 1:
            self.multi = MultiContext(devices)
            self.multi.check(self.multi.lib.r2s_multi_set_mesh(self.multi.h, self.nen, self.nnp, _ptr(self.X), self.nel, _ptr(self.IEN)))
            self.ctx = self.multi.slab(0)
            c = self.ctx
        else:
            self.ctx = Context(devices[0] if devices else device, stream)
            c = self.ctx
            c.check(c.lib.r2s_set_mesh(c.h, self.nen, self.nnp, _ptr(self.X), self.nel, _ptr(self.IEN)))
        vd, vf = C.c_double(), C.c_double()
        c.check(c.lib.r2s_mesh_volume(c.h, _ptr(self.rho), C.byref(vd), C.byref(vf)))
        self.V_domain, self.V_frac = vd.value, vf.value
        self._grid_id = None

    @property
    def is_lattice(self):
        """True when the mesh is a tensor-product lattice of box elements (Sign_Detection then takes the list-free fast path)."""
        f = C.c_int(0)
        self.ctx.check(self.ctx.lib.r2s_mesh_is_lattice(self.ctx.h, C.byref(f)))
        return bool(f.value)

    def _use_grid(self, grid):
        key = (tuple(grid.AABB_min), tuple(grid.AABB_max), tuple(int(v) for v in grid.N), grid.cell_size)
        if self._grid_id != key:
            c = self.ctx
            amin, amax, N = _f64(grid.AABB_min), _f64(grid.AABB_max), np.ascontiguousarray(grid.N, dtype=np.int64)
            if self.multi is not None:
                self.multi.check(self.multi.lib.r2s_multi_set_grid(self.multi.h, _ptr(amin), _ptr(amax), _ptr(N), float(grid.cell_size)))
            else:
                c.check(c.lib.r2s_set_grid(c.h, _ptr(amin), _ptr(amax), _ptr(N), float(grid.cell_size)))
            self._grid_id = key

    def close(self):
        if self.multi is not None:
            self.multi.close()
        else:
            self.ctx.close()


def noninteractive_sdf_grid_setup(mesh):
    """src/MeshGrid/Grid_setup.jl:94-109: grid step = median element edge length (edge lengths, sort and median on the device)."""
    Xmin, Xmax = getMesh_AABB(mesh.X)
    c = mesh.ctx
    med, lo, hi = C.c_double(), C.c_double(), C.c_double()
    c.check(c.lib.r2s_edge_length_stats(c.h, C.byref(med), C.byref(lo), C.byref(hi)))
    mesh.edge_stats = {"median": med.value, "shortest": lo.value, "longest": hi.value}
    N_new = int(math.floor(np.max(Xmax - Xmin) / med.value))
    return Grid(Xmin, Xmax, N_new, 3)


def DenseInNodes(mesh, rho):
    """src/MeshGrid/NodalDensities.jl:89-109."""
    c = mesh.ctx
    rho = _f64(rho)
    out = np.empty(mesh.nnp)
    c.check(c.lib.r2s_nodal_densities(c.h, _ptr(rho), _ptr(out)))
    return out


def calculate_isocontour_volume(mesh, nodal_values, iso_threshold):
    """src/MeshGrid/Isocontour_volume.jl:1-75 (HEX8 only, like the reference)."""
    c = mesh.ctx
    v = C.c_double()
    rn = _f64(nodal_values)
    c.check(c.lib.r2s_isocontour_volume(c.h, _ptr(rn), float(iso_threshold), C.byref(v)))
    return v.value


def find_threshold_for_volume(mesh, nodal_values, tolerance=1e-4, max_iterations=60):
    """src/MeshGrid/Isocontour_volume.jl:77-154."""
    c = mesh.ctx
    out = C.c_double()
    rn = _f64(nodal_values)
    c.check(c.lib.r2s_find_threshold(c.h, _ptr(rn), mesh.V_domain * mesh.V_frac, float(tolerance), int(max_iterations), C.byref(out)))
    return out.value


# ---------------------------------------------------------------------------------------------------------------------
# SignedDistances
# ---------------------------------------------------------------------------------------------------------------------
def _points(points):
    p = np.ascontiguousarray(points, dtype=np.float64)
    if p.ndim != 2 or p.shape[1] != 3:
        raise R2SError("points must be an (n, 3) array")
    return p


def evalDistances(mesh, grid, points, rho_n, rho_t, delta_factor=1.1, want_xp=True):
    """src/SignedDistances/sdfOnDensityField.jl:139-486 -> (dists, xp).  `delta_factor` is the reference's hard-wired 1.1 (:158).
    points=None: at the grid's points (grid.ngp values).  points = (n, 3) float64: at those points, binned in the grid's frame like the
    reference's LinkedList(grid, points) -- (n,) and (n, 3); the rule (and what points outside the grid get) is stated in include/r2s.h."""
    mesh._use_grid(grid)
    c = mesh.ctx
    rn = _f64(rho_n)
    if points is not None:
        p = _points(points)
        n = p.shape[0]
        dist = np.empty(n)
        xp = np.zeros((n, 3)) if want_xp else None
        c.check(c.lib.r2s_eval_distances_points(c.h, _ptr(rn), float(rho_t), float(delta_factor), _ptr(p) if n else None, n, _ptr(dist) if n else None,
                                                _ptr(xp) if (want_xp and n) else None))
        return dist, xp
    dist = np.empty(grid.ngp)
    xp = np.zeros((grid.ngp, 3)) if want_xp else None
    c.check(c.lib.r2s_eval_distances(c.h, _ptr(rn), float(rho_t), float(delta_factor), _ptr(dist), _ptr(xp) if want_xp else None))
    return dist, xp


def Sign_Detection(mesh, grid, points, rho_n, rho_t):
    """src/SignedDistances/SignDetection.jl:275-283 -> signs in {-1, +1}.  points=None: at the grid's points; (n, 3) float64: at those
    points -> (n,)."""
    mesh._use_grid(grid)
    c = mesh.ctx
    rn = _f64(rho_n)
    if points is not None:
        p = _points(points)
        n = p.shape[0]
        s = np.empty(n)
        c.check(c.lib.r2s_sign_detection_points(c.h, _ptr(rn), float(rho_t), _ptr(p) if n else None, n, _ptr(s) if n else None))
        return s
    s = np.empty(grid.ngp)
    c.check(c.lib.r2s_sign_detection(c.h, _ptr(rn), float(rho_t), _ptr(s)))
    return s


def remove_sdf_artifacts(sdf_values, grid, threshold=0.0, min_component_ratio=0.01, mesh=None, ctx=None):
    """remove_sdf_artifacts! (src/SignedDistances/SdfArtifactRemoval.jl:134-245): modifies `sdf_values` in place, returns the
    number of flipped nodes.  Needs a context (pass the mesh, or a Context on which the grid gets set)."""
    if len(sdf_values) != grid.ngp:
        raise R2SError("SDF values length (%d) doesn't match grid points (%d)" % (len(sdf_values), grid.ngp))   # :142
    if not (isinstance(sdf_values, np.ndarray) and sdf_values.dtype == np.float64 and sdf_values.flags.c_contiguous):
        raise R2SError("sdf_values must be a contiguous float64 numpy array (modified in place)")
    if mesh is not None:
        mesh._use_grid(grid)
        c = mesh.ctx
    else:
        c = ctx or Context()
        amin, amax, N = _f64(grid.AABB_min), _f64(grid.AABB_max), np.ascontiguousarray(grid.N, dtype=np.int64)
        c.check(c.lib.r2s_set_grid(c.h, _ptr(amin), _ptr(amax), _ptr(N), float(grid.cell_size)))
    fl = C.c_int64()
    c.check(c.lib.r2s_remove_artifacts(c.h, _ptr(sdf_values), float(threshold), float(min_component_ratio), C.byref(fl)))
    return int(fl.value)


# ---------------------------------------------------------------------------------------------------------------------
# SdfSmoothing
# ---------------------------------------------------------------------------------------------------------------------
class FineGrid:
    """Lazy stand-in for the reference's `fine_grid::Array{Vector{Float32},3}` (create_smooth_grid, RBFs4Smoothing.jl:60-74):
    fine_grid[i, j, k] -> Float32 [x, y, z] with x = xmin + i*dx evaluated in Float32 (0-based indices here)."""

    def __init__(self, grid, smooth):
        self.shape = tuple(int(v) * smooth + 1 for v in grid.N)
        self.min = np.asarray(grid.AABB_min, dtype=np.float32)
        self.dx = np.float32((np.float32(grid.AABB_max[0]) - self.min[0]) / np.float32(self.shape[0] - 1))

    def axis(self, d):
        return (self.min[d] + np.arange(self.shape[d], dtype=np.float32) * self.dx).astype(np.float32)

    def __getitem__(self, ijk):
        i, j, k = ijk
        return np.array([self.min[0] + np.float32(i) * self.dx, self.min[1] + np.float32(j) * self.dx, self.min[2] + np.float32(k) * self.dx], dtype=np.float32)


def RBFs_smoothing(mesh, dist, my_grid, Is_interpolation, smooth, taskName="", threshold=1e-3, return_info=False):
    """src/SdfSmoothing/RBFs4Smoothing.jl:321-377 -> (fine_sdf[k, j, i] float32, fine_grid)."""
    mesh._use_grid(my_grid)
    c = mesh.ctx
    d = _f64(dist)
    dims = tuple(int(v) * smooth + 1 for v in my_grid.N)
    fine = np.empty(dims[2] * dims[1] * dims[0], dtype=np.float32)
    th, vol = C.c_float(), C.c_float()
    c.check(c.lib.r2s_rbf_smoothing(c.h, _ptr(d), int(bool(Is_interpolation)), int(smooth), float(threshold), mesh.V_frac * mesh.V_domain,
                                    _ptr(fine), C.byref(th), C.byref(vol)))
    fine = fine.reshape(dims[2], dims[1], dims[0])
    fg = FineGrid(my_grid, smooth)
    if return_info:
        rep = c.report()
        return fine, fg, {"th": th.value, "volume": vol.value, "cg_iters": rep.cg_iters, "bisections": rep.bisections}
    return fine, fg


def calculate_volume_from_sdf(fine_sdf, fine_grid, iso_threshold=0.0, detailed_quad_order=9, ctx=None):
    """src/SdfSmoothing/CalcVolumeFromSDF.jl:26-125.  fine_sdf[k, j, i] float32; fine_grid: FineGrid or an edge length."""
    a = np.ascontiguousarray(fine_sdf, dtype=np.float32)
    nz, ny, nx = a.shape
    if isinstance(fine_grid, FineGrid):
        p0, p1 = fine_grid[0, 0, 0], fine_grid[1, 0, 0]
        edge = np.float32(np.sqrt(np.float32(np.sum((p1 - p0) ** 2, dtype=np.float32))))
    else:
        edge = np.float32(fine_grid)
    c = ctx or Context()
    v = C.c_double()
    c.check(c.lib.r2s_volume_from_sdf(c.h, _ptr(a), nx, ny, nz, float(edge), float(iso_threshold), int(detailed_quad_order), C.byref(v)))
    return np.float32(v.value)


# ---------------------------------------------------------------------------------------------------------------------
# DataExport (SURVEY.md 8f-1)
# ---------------------------------------------------------------------------------------------------------------------
def exportSdfToVTI(filename, grid, values, value_label, smooth=None):
    """src/DataExport/ExportToVTI.jl:22-67: VTK ImageData with dims N*smooth+1, origin AABB_min, spacing cell_size/smooth and one
    point scalar `value_label`.  `values` is a host array (float32 or float64, x fastest); ".vti" is appended if missing."""
    sm = 1 if smooth is None else int(smooth)
    dims = [int(v) * sm + 1 for v in grid.N]
    a = np.ascontiguousarray(values)
    if a.dtype not in (np.float32, np.float64):
        a = a.astype(np.float64)
    if a.size != dims[0] * dims[1] * dims[2]:
        raise R2SError("Values vector length (%d) doesn't match grid dimensions (%d)." % (a.size, dims[0] * dims[1] * dims[2]))   # :44-46
    path = filename if filename.endswith(".vti") else filename + ".vti"
    origin = _f64(grid.AABB_min)
    spacing = _f64([grid.cell_size / sm] * 3)
    rc = load_library().r2s_write_vti_host(path.encode(), str(value_label).encode(), _ptr(a), int(a.dtype == np.float64), dims[0], dims[1], dims[2], _ptr(origin), _ptr(spacing))
    if rc != 0:
        raise R2SError("exportSdfToVTI: cannot write %s (code %d)" % (path, rc))
    return path


def export_device_result_to_vti(mesh, filename, value_label="distance", fine=True):
    """Stream the device-resident result of the last pipeline call (fine_sdf, or sdf_dists with fine=False) to a .vti file."""
    path = filename if filename.endswith(".vti") else filename + ".vti"
    c = mesh.ctx
    c.check(c.lib.r2s_export_vti(c.h, path.encode(), str(value_label).encode(), 1 if fine else 0))
    return path


def read_vti(path):
    """Minimal reader of the files written above (tests / round trips): returns (dims, origin, spacing, label, array[k, j, i])."""
    import re
    raw = open(path, "rb").read()
    cut = raw.index(b'<AppendedData encoding="raw">')
    head = raw[:cut].decode()
    ext = [int(v) for v in re.search(r'WholeExtent="([^"]+)"', head).group(1).split()]
    dims = (ext[1] - ext[0] + 1, ext[3] - ext[2] + 1, ext[5] - ext[4] + 1)      # a piece of a slab decomposition starts at z = ext[4]
    origin = [float(v) for v in re.search(r'Origin="([^"]+)"', head).group(1).split()]
    spacing = [float(v) for v in re.search(r'Spacing="([^"]+)"', head).group(1).split()]
    typ, label = re.search(r'<DataArray type="(\w+)" Name="([^"]+)"', head).groups()
    start = raw.index(b"_", cut) + 1
    nbytes = int(np.frombuffer(raw[start:start + 8], dtype="<u8")[0])
    dt = np.dtype("<f8" if typ == "Float64" else "<f4")
    data = np.frombuffer(raw[start + 8:start + 8 + nbytes], dtype=dt)
    return dims, origin, spacing, label, data.reshape(dims[2], dims[1], dims[0])


def read_pvti(path):
    """Assemble the pieces named by a .pvti index (r2s_multi_export_vti / r2s_export_pvti): returns (dims, origin, spacing, label, array[k, j, i])."""
    import re
    head = open(path).read()
    ext = [int(v) for v in re.search(r'WholeExtent="([^"]+)"', head).group(1).split()]
    dims = (ext[1] + 1, ext[3] + 1, ext[5] + 1)
    origin = [float(v) for v in re.search(r'Origin="([^"]+)"', head).group(1).split()]
    spacing = [float(v) for v in re.search(r'Spacing="([^"]+)"', head).group(1).split()]
    typ, label = re.search(r'<PDataArray type="(\w+)" Name="([^"]+)"', head).groups()
    out = np.full((dims[2], dims[1], dims[0]), np.nan, dtype=np.float64 if typ == "Float64" else np.float32)
    for pe, src in re.findall(r'<Piece Extent="([^"]+)" Source="([^"]+)"', head):
        e = [int(v) for v in pe.split()]
        _, _, _, _, arr = read_vti(os.path.join(os.path.dirname(os.path.abspath(path)), src))
        assert arr.shape == (e[5] - e[4] + 1, dims[1], dims[0])
        prev = out[e[4]:e[5] + 1]
        both = ~np.isnan(prev)
        assert np.array_equal(prev[both], arr[both])          # pieces agree on the boundary plane they share
        out[e[4]:e[5] + 1] = arr
    return dims, origin, spacing, label, out


# ---------------------------------------------------------------------------------------------------------------------
# Isosurface: the zero surface of the smoothed SDF (csrc/r2s_surf.cu)
# ---------------------------------------------------------------------------------------------------------------------
def _surface_format(path):
    low = str(path).lower()
    if low.endswith(".stl"):
        return 0
    if low.endswith(".ply"):
        return 1
    raise R2SError("export_isosurface: the file name must end in .stl (binary STL) or .ply (binary PLY): %s" % path)


def _download_surface(obj, download, nv, nt):
    V = np.empty((nv, 3), dtype=np.float32)
    T = np.empty((nt, 3), dtype=np.int32)
    obj.check(download(obj.h, _ptr(V), _ptr(T)))
    return V, T


def _lattice_args(origin, spacing, shape):
    o = _f64(np.broadcast_to(np.asarray(origin, dtype=np.float64), (3,)))
    h = _f64(np.broadcast_to(np.asarray(spacing, dtype=np.float64), (3,)))
    dims = np.ascontiguousarray(np.broadcast_to(np.asarray(shape, dtype=np.int64), (3,)))
    return o, h, dims


def _extract(mesh, iso, lattice=None, band=None):
    nv, nt = C.c_int64(), C.c_int64()
    if band is not None:
        o, h, dims = _lattice_args(*band)
        obj, pre = _sampler(mesh)
        ns = C.c_int64()
        obj.check(getattr(obj.lib, pre + "isosurface_band")(obj.h, _ptr(o), _ptr(h), _ptr(dims), float(iso), C.byref(nv), C.byref(nt), C.byref(ns)))
        return obj, getattr(obj.lib, pre + "download_isosurface"), nv.value, nt.value, ns.value
    if lattice is not None:
        o, h, dims = _lattice_args(*lattice)
        obj, pre = _sampler(mesh)
        obj.check(getattr(obj.lib, pre + "isosurface_lattice")(obj.h, _ptr(o), _ptr(h), _ptr(dims), float(iso), C.byref(nv), C.byref(nt)))
        return obj, getattr(obj.lib, pre + "download_isosurface"), nv.value, nt.value, None
    if mesh.multi is not None:
        m = mesh.multi
        m.check(m.lib.r2s_multi_isosurface(m.h, float(iso), C.byref(nv), C.byref(nt)))
        return m, m.lib.r2s_multi_download_isosurface, nv.value, nt.value, None
    c = mesh.ctx
    c.check(c.lib.r2s_isosurface(c.h, float(iso), C.byref(nv), C.byref(nt)))
    return c, c.lib.r2s_download_isosurface, nv.value, nt.value, None


def isosurface(mesh, iso=0.0):
    """Triangle mesh of {fine_sdf = iso} for the fine_sdf the last pipeline / smoothing call left on the device(s) of `mesh` (slab 0,
    or all slabs of a multi-GPU mesh).  Returns (V (nv, 3) float32, T (nt, 3) int32, 0-based): one vertex per grid edge that crosses
    iso (a point is inside iff value >= iso), triangles counter-clockwise seen from outside, in the frame of export_device_result_to_vti
    (origin AABB_min, spacing cell_size / smooth).  The mesh is closed wherever the field is below iso on the grid's border."""
    obj, dl, nv, nt, _ = _extract(mesh, iso)
    return _download_surface(obj, dl, nv, nt)


def isosurface_from_sdf(fine_sdf, origin, spacing, iso=0.0, ctx=None):
    """The same mesh for a host field fine_sdf[k, j, i] (float32, x fastest) with grid origin and spacing (3 values each)."""
    a = np.ascontiguousarray(fine_sdf, dtype=np.float32)
    if a.ndim != 3:
        raise R2SError("isosurface_from_sdf: fine_sdf must be a 3-D array [k, j, i]")
    nz, ny, nx = a.shape
    o = _f64(np.broadcast_to(np.asarray(origin, dtype=np.float64), (3,)))
    h = _f64(np.broadcast_to(np.asarray(spacing, dtype=np.float64), (3,)))
    c = ctx or Context()
    nv, nt = C.c_int64(), C.c_int64()
    c.check(c.lib.r2s_isosurface_from_sdf(c.h, _ptr(a), nx, ny, nz, _ptr(o), _ptr(h), float(iso), C.byref(nv), C.byref(nt)))
    return _download_surface(c, c.lib.r2s_download_isosurface, nv.value, nt.value)


def isosurface_lattice(mesh, origin, spacing, shape, iso=0.0):
    """Triangle mesh of {f = iso} for the continuous field f of the last pipeline / smoothing call on the device(s) of `mesh` (what
    sample_sdf evaluates), extracted on the lattice origin + i * spacing, i < shape (the arguments of sample_sdf_lattice) without holding
    the lattice field anywhere.  The triangles are those of isosurface_from_sdf(sample_sdf_lattice(mesh, origin, spacing, shape), origin,
    spacing, iso); each vertex lies on its lattice edge at the Float32 coordinate that a bracketing search on f finds closest to the zero
    set (include/r2s.h states the rule).  Returns (V (nv, 3) float32, T (nt, 3) int32, 0-based)."""
    obj, dl, nv, nt, _ = _extract(mesh, iso, (origin, spacing, shape))
    return _download_surface(obj, dl, nv, nt)


def isosurface_band(mesh, origin, spacing, shape, iso=0.0, stats=False):
    """The mesh of isosurface_lattice, bit for bit, sampling only the lattice blocks that can hold the surface: a block whose reachable
    coarse weights share one sign that provably keeps every value of the block on one side of iso is never evaluated.  Any cell count
    (fewer than 2^31 vertices).  Returns (V, T); with stats=True (V, T, n_sampled), n_sampled the lattice points evaluated per sweep."""
    obj, dl, nv, nt, ns = _extract(mesh, iso, band=(origin, spacing, shape))
    V, T = _download_surface(obj, dl, nv, nt)
    return (V, T, ns) if stats else (V, T)


def export_isosurface(mesh, path, iso=0.0, lattice=None, band=None):
    """Extract {fine_sdf = iso} on the device(s) of `mesh` and write it to `path`: binary STL (.stl) or binary little-endian PLY (.ply).
    lattice=(origin, spacing, shape): extract the continuous field's surface on that lattice instead, as isosurface_lattice does;
    band=(origin, spacing, shape): the same mesh through isosurface_band (any cell count)."""
    fmt = _surface_format(path)
    if lattice is not None and band is not None:
        raise R2SError("export_isosurface: give lattice= or band=, not both")
    obj, _, _, _, _ = _extract(mesh, iso, lattice, band)
    if mesh.multi is not None:
        obj.check(obj.lib.r2s_multi_export_isosurface(obj.h, str(path).encode(), fmt))
    else:
        obj.check(obj.lib.r2s_export_isosurface(obj.h, str(path).encode(), fmt))
    return str(path)


def read_stl(path):
    """Minimal reader of binary STL files: returns (normals (nt, 3), corners (nt, 3, 3)) float32."""
    raw = open(path, "rb").read()
    nt = int(np.frombuffer(raw[80:84], dtype="<u4")[0])
    if len(raw) != 84 + 50 * nt:
        raise R2SError("read_stl: %s is not a binary STL file of %d triangles" % (path, nt))
    rec = np.frombuffer(raw[84:], dtype=np.dtype([("n", "<f4", 3), ("v", "<f4", (3, 3)), ("attr", "<u2")]), count=nt)
    return rec["n"].copy(), rec["v"].copy()


def read_ply(path):
    """Minimal reader of the binary little-endian PLY files written above: returns (V (nv, 3) float32, T (nt, 3) int32)."""
    raw = open(path, "rb").read()
    end = raw.index(b"end_header\n") + len(b"end_header\n")
    head = raw[:end].decode()
    if "format binary_little_endian 1.0" not in head or "property list uchar int vertex_indices" not in head:
        raise R2SError("read_ply: unsupported PLY layout in %s" % path)
    nv = int(head.split("element vertex ")[1].split()[0])
    nt = int(head.split("element face ")[1].split()[0])
    V = np.frombuffer(raw, dtype="<f4", count=3 * nv, offset=end).reshape(nv, 3)
    F = np.frombuffer(raw, dtype=np.dtype([("n", "u1"), ("i", "<i4", 3)]), count=nt, offset=end + 12 * nv)
    if nt and not (F["n"] == 3).all():
        raise R2SError("read_ply: only triangles are supported")
    return V.astype(np.float32), F["i"].astype(np.int32)


# ---------------------------------------------------------------------------------------------------------------------
# The smoothed SDF as a continuous function (csrc/r2s_sample.cu)
# ---------------------------------------------------------------------------------------------------------------------
def _sampler(mesh):
    """(handle object, function prefix): all slabs of a multi-GPU mesh, else the mesh's context"""
    return (mesh.multi, "r2s_multi_") if mesh.multi is not None else (mesh.ctx, "r2s_")


def sample_sdf(mesh, points, gradient=False):
    """The reference's rbf_interpolation_kdtree(points, coarse_grid, weights, kernel) (RBFs4Smoothing.jl:219-248) for the field the last
    pipeline / smoothing call left on the device(s) of `mesh`: th + sum_c w_c exp(-(|x - c| / cell)^2) over the coarse points within the
    kernel's cut radius, evaluated on the GPU at arbitrary points (outside the grid too; far away the value is th).  points: (n, 3)
    float64.  Returns float32 values (n,), and with gradient=True also the analytic gradients (n, 3) float32.  The exact arithmetic is
    stated in include/r2s.h; a point's result does not depend on the other points or their order."""
    p = np.ascontiguousarray(points, dtype=np.float64)
    if p.ndim != 2 or p.shape[1] != 3:
        raise R2SError("sample_sdf: points must be an (n, 3) array")
    n = p.shape[0]
    val = np.empty(n, dtype=np.float32)
    g = np.empty((n, 3), dtype=np.float32) if gradient else None
    obj, pre = _sampler(mesh)
    obj.check(getattr(obj.lib, pre + "sample_sdf")(obj.h, _ptr(p) if n else None, n, _ptr(val) if n else None, _ptr(g) if (gradient and n) else None))
    return (val, g) if gradient else val


def sample_sdf_lattice(mesh, origin, spacing, shape):
    """rbf_interpolation_kdtree on the lattice origin + i * spacing (i = 0 .. shape - 1 per axis, Float32 arithmetic, no coordinates
    stored): returns float32 [k, j, i] of shape (shape[2], shape[1], shape[0]).  origin = AABB_min, spacing = cell_size / k gives the
    points of the reference's create_smooth_grid for smooth = k, i.e. resampling at any resolution."""
    o = _f64(np.broadcast_to(np.asarray(origin, dtype=np.float64), (3,)))
    h = _f64(np.broadcast_to(np.asarray(spacing, dtype=np.float64), (3,)))
    dims = np.ascontiguousarray(np.broadcast_to(np.asarray(shape, dtype=np.int64), (3,)))
    if (dims < 1).any():
        raise R2SError("sampling: lattice dims must be >= 1")
    out = np.empty((int(dims[2]), int(dims[1]), int(dims[0])), dtype=np.float32)
    obj, pre = _sampler(mesh)
    obj.check(getattr(obj.lib, pre + "sample_sdf_lattice")(obj.h, _ptr(o), _ptr(h), _ptr(dims), _ptr(out)))
    return out


def rbf_weights(mesh):
    """The definition of the continuous field: (w[k, j, i] float32 on the coarse grid, th float32), the weights and offset that
    rbf_interpolation_kdtree sums (the CG solution, or the processed SDF in approximation mode)."""
    obj, pre = _sampler(mesh)
    if mesh._grid_id is None:
        raise R2SError("r2s_set_grid has not been called")
    np_ = [v + 1 for v in mesh._grid_id[2]]
    w = np.empty((np_[2], np_[1], np_[0]), dtype=np.float32)
    th = C.c_float()
    obj.check(getattr(obj.lib, pre + "download_rbf_weights")(obj.h, _ptr(w), C.byref(th)))
    return w, np.float32(th.value)


def element_volume_fractions(mesh, iso=0.0, quad_order=15, return_volumes=False, stats=False):
    """The solid volume fraction of every element of `mesh` in the continuous field of the last pipeline / smoothing call (what sample_sdf
    evaluates): calculate_isocontour_volume's rule -- a Gauss point is solid iff f >= iso, weighted by |det J| -- at quad_order^3 points
    per element (1..32), on the GPU.  Elements whose box the band classifier proves one-sided are not sampled; their fractions are exactly
    1.0 or 0.0, the values full evaluation gives (include/r2s.h states the rule).  Returns fractions (nel,) float64; with return_volumes
    also V_e (nel,), the element volumes of the same quadrature; with stats also the number of elements sampled."""
    obj, pre = _sampler(mesh)
    frac = np.empty(mesh.nel, dtype=np.float64)
    vol = np.empty(mesh.nel, dtype=np.float64) if return_volumes else None
    ne = C.c_int64()
    obj.check(getattr(obj.lib, pre + "element_volume_fractions")(obj.h, float(iso), int(quad_order), _ptr(frac), _ptr(vol) if return_volumes else None,
                                                                  C.byref(ne)))
    out = (frac,) + ((vol,) if return_volumes else ()) + ((ne.value,) if stats else ())
    return out if len(out) > 1 else frac


# ---------------------------------------------------------------------------------------------------------------------
# RhoToSDF
# ---------------------------------------------------------------------------------------------------------------------
class Rho2sdfOptions:
    """src/RhoToSDF.jl:9-77 (same defaults, same warn-and-default validation)."""

    def __init__(self, threshold_density=None, sdf_grid_setup="manual", export_input_data=False, export_nodal_densities=False,
                 export_raw_sdf=False, rbf_interp=True, rbf_grid="same", remove_artifacts=True, artifact_min_component_ratio=0.01,
                 export_analysis=False, element_type=HEX8, grid_step=None):
        import warnings
        if threshold_density is not None:
            if not (0.0 <= threshold_density <= 1.0):
                warnings.warn("Threshold density %r is outside the valid range [0.0, 1.0]. Will use automatic calculation instead." % threshold_density)
                threshold_density = None
            elif threshold_density in (0.0, 1.0):
                warnings.warn("Using extreme threshold density value: %r" % threshold_density)
        sdf_grid_setup = str(sdf_grid_setup).lstrip(":")
        if sdf_grid_setup not in ("manual", "automatic"):
            warnings.warn("Invalid sdf_grid_setup: %s. Must be either :manual or :automatic. Using default :manual instead." % sdf_grid_setup)
            sdf_grid_setup = "manual"
        rbf_grid = str(rbf_grid).lstrip(":")
        if rbf_grid not in ("same", "fine"):
            warnings.warn("Invalid rbf_grid: %s. Must be either :same or :fine. Using default :same instead." % rbf_grid)
            rbf_grid = "same"
        if element_type not in (HEX8, TET4):
            warnings.warn("Invalid element_type. Must be subtype of AbstractElement. Using HEX8.")
            element_type = HEX8
        self.threshold_density, self.sdf_grid_setup = threshold_density, sdf_grid_setup
        self.export_input_data, self.export_nodal_densities, self.export_raw_sdf = export_input_data, export_nodal_densities, export_raw_sdf
        self.rbf_interp, self.rbf_grid, self.remove_artifacts = bool(rbf_interp), rbf_grid, bool(remove_artifacts)
        self.artifact_min_component_ratio, self.export_analysis, self.element_type = float(artifact_min_component_ratio), export_analysis, element_type
        self.grid_step = grid_step      # stands in for the stdin prompt of interactive_sdf_grid_setup (:manual)


def rho2sdf(taskName, X, IEN, rho, options=None, device=0, stream=None, return_report=False, devices=None, export_vti=None, export_surface=None):
    """src/RhoToSDF.jl:116-242 -> (fine_sdf, fine_grid, sdf_grid, sdf_dists).  `devices=[0, 1, ...]`: the timed region runs as z-slabs on
    all listed GPUs from this one call (r2s_multi_pipeline).  `export_vti=base`: the fine SDF is streamed from the device(s) to
    base.vti (one GPU) or base.pvti + pieces (RhoToSDF.jl:230-238, :267-273); VTU / JLD2 exports are out of scope.  `export_surface=path`:
    the zero surface of the fine SDF is extracted on the device(s) and written as one .stl or .ply file (export_isosurface)."""
    options = options or Rho2sdfOptions()
    mesh = Mesh(X, IEN, rho, None, element_type=options.element_type, device=device, stream=stream, devices=devices)
    if options.sdf_grid_setup == "manual":
        if options.grid_step is None:
            raise R2SError(":manual grid set-up prompts on stdin in the reference (Grid_setup.jl:111-154); pass Rho2sdfOptions(grid_step=B) here")
        Xmin, Xmax = getMesh_AABB(mesh.X)
        sdf_grid = Grid(Xmin, Xmax, int(math.floor(np.max(Xmax - Xmin) / options.grid_step)), 3)
    else:
        sdf_grid = noninteractive_sdf_grid_setup(mesh)
    rho_n = DenseInNodes(mesh, rho)
    rho_t = find_threshold_for_volume(mesh, rho_n) if options.threshold_density is None else options.threshold_density
    # ---- the reference's timed region (RhoToSDF.jl:164-227) as one device-resident call ----
    mesh._use_grid(sdf_grid)
    c = mesh.ctx
    p = Params()
    c.lib.r2s_default_params(C.byref(p))
    p.rho_t, p.remove_artifacts, p.artifact_min_ratio = float(rho_t), int(options.remove_artifacts), options.artifact_min_component_ratio
    p.rbf_interp, p.smooth, p.target_volume = int(options.rbf_interp), 1 if options.rbf_grid == "same" else 2, mesh.V_frac * mesh.V_domain
    dims = tuple(int(v) * p.smooth + 1 for v in sdf_grid.N)
    sdf_dists = np.empty(sdf_grid.ngp)
    fine = np.empty(dims[0] * dims[1] * dims[2], dtype=np.float32)
    rep = Report()
    rn = _f64(rho_n)
    if mesh.multi is not None:
        m = mesh.multi
        m.check(m.lib.r2s_multi_pipeline(m.h, C.byref(p), _ptr(rn), _ptr(sdf_dists), _ptr(fine), C.byref(rep)))
        if export_vti:
            m.check(m.lib.r2s_multi_export_vti(m.h, str(export_vti).encode(), b"distance", 1))
    else:
        c.check(c.lib.r2s_pipeline(c.h, C.byref(p), _ptr(rn), _ptr(sdf_dists), _ptr(fine), C.byref(rep)))
        if export_vti:
            export_device_result_to_vti(mesh, str(export_vti), "distance", fine=True)
    if export_surface:
        export_isosurface(mesh, export_surface, 0.0)
    out = (fine.reshape(dims[2], dims[1], dims[0]), FineGrid(sdf_grid, p.smooth), sdf_grid, sdf_dists)
    if return_report:
        return out + ({"rho_t": rho_t, "rho_n": rho_n, "V_domain": mesh.V_domain, "V_frac": mesh.V_frac, **rep.asdict()},)
    return out


def rho2sdf_hex8(taskName, X, IEN, rho, **kwargs):
    """src/RhoToSDF.jl:284-293."""
    extra = {k: kwargs.pop(k) for k in ("device", "stream", "return_report", "devices", "export_vti", "export_surface") if k in kwargs}
    return rho2sdf(taskName, X, IEN, rho, options=Rho2sdfOptions(element_type=HEX8, **kwargs), **extra)


def rho2sdf_tet4(taskName, X, IEN, rho, **kwargs):
    """src/RhoToSDF.jl:295-304."""
    extra = {k: kwargs.pop(k) for k in ("device", "stream", "return_report", "devices", "export_vti", "export_surface") if k in kwargs}
    return rho2sdf(taskName, X, IEN, rho, options=Rho2sdfOptions(element_type=TET4, **kwargs), **extra)
