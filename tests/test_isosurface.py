"""GPU tests of the isosurface stage (csrc/r2s_surf.cu): bit equality with the host reference (tests/host/mc_host.cpp) for host fields,
for the pipeline's resident fine_sdf and for several slabs; closedness and volume of the pipeline's surfaces; STL / PLY round trips; errors."""
import numpy as np
import pytest

import isosurface_ref as ref
from fixtures import load_mesh, simp_hex8

pytestmark = pytest.mark.gpu


def _field(kind, shape, seed=0):
    nz, ny, nx = shape
    z, y, x = np.meshgrid(np.arange(nz) - (nz - 1) / 2, np.arange(ny) - (ny - 1) / 2, np.arange(nx) - (nx - 1) / 2, indexing="ij")
    r = 0.4 * min(shape)
    if kind == "sphere":
        f = r - np.sqrt(x * x + y * y + z * z)
    elif kind == "torus":
        f = 0.15 * min(shape) - np.sqrt((np.sqrt(x * x + y * y) - r * 0.6) ** 2 + z * z)
    elif kind == "gyroid":
        w = 0.5
        f = np.sin(w * x) * np.cos(w * y) + np.sin(w * y) * np.cos(w * z) + np.sin(w * z) * np.cos(w * x)
    else:      # uniform noise: a crossing on about half of all edges, the largest output per point
        f = np.random.default_rng(seed).uniform(-2, 2, shape)
    return np.ascontiguousarray(f, dtype=np.float32)


SHAPES = [(2, 2, 2), (7, 5, 3), (34, 33, 65), (129, 4, 127)]


@pytest.fixture(scope="module")
def ctx(r2s):
    c = r2s.Context()
    yield c
    c.close()


@pytest.mark.parametrize("shape", SHAPES, ids=lambda s: "x".join(map(str, s[::-1])))
@pytest.mark.parametrize("kind", ["sphere", "torus", "gyroid", "noise"])
@pytest.mark.parametrize("iso", [0.0, 0.37, -1.5])
def test_host_field_equals_reference(r2s, ctx, shape, kind, iso):
    f = _field(kind, shape, seed=len(kind))
    origin, spacing = (0.25, -3.0, 1.5), (0.5, 0.25, 0.75)
    V, T = r2s.isosurface_from_sdf(f, origin, spacing, iso, ctx=ctx)
    Vr, Tr = ref.reference(f, origin, spacing, iso)
    assert np.array_equal(V, Vr) and np.array_equal(T, Tr)


def test_edge_values_equal_reference(r2s, ctx):
    rng = np.random.default_rng(7)
    shape = (9, 11, 37)
    # values exactly on iso, +-0 against iso = 0, magnitudes from 1e-30 to 1e30
    f = rng.choice(np.array([0.0, -0.0, 1e-30, -1e-30, 1e30, -1e30, 1.0, -1.0, 3e-8, -7e12], np.float32), size=shape)
    for iso in (0.0, 1.0, -1e-30):
        V, T = r2s.isosurface_from_sdf(f, (0, 0, 0), (1, 1, 1), iso, ctx=ctx)
        Vr, Tr = ref.reference(f, (0, 0, 0), (1, 1, 1), iso)
        assert np.array_equal(V, Vr) and np.array_equal(T, Tr)
        g = f.copy()
        g[[0, -1]] = g[:, [0, -1]] = g[:, :, [0, -1]] = -2.0      # a border below every iso used here
        V, T = r2s.isosurface_from_sdf(g, (0, 0, 0), (1, 1, 1), iso, ctx=ctx)
        assert np.array_equal(T, ref.reference(g, (0, 0, 0), (1, 1, 1), iso)[1]) and len(ref.unpaired_edges(T)) == 0      # exact-iso corners stay closed


def test_large_noise_grid_equals_reference(r2s, ctx):
    f = _field("gyroid", (401, 400, 403)) + np.float32(0.3) * _field("noise", (401, 400, 403), seed=3)
    V, T = r2s.isosurface_from_sdf(f, (0, 0, 0), (0.1, 0.1, 0.1), 0.0, ctx=ctx)
    Vr, Tr = ref.reference(f, (0, 0, 0), (0.1, 0.1, 0.1), 0.0)
    assert len(T) > 10 ** 6 and np.array_equal(V, Vr) and np.array_equal(T, Tr)


def _pipeline_case(r2s, case):
    if case.startswith("simp24"):
        X, IEN, rho = simp_hex8(24)
        opts = dict(threshold_density=0.5, sdf_grid_setup="manual", grid_step=0.5, rbf_interp=case == "simp24", rbf_grid="fine", remove_artifacts=True,
                    artifact_min_component_ratio=0.3)
    elif case == "sphere_same":
        X, IEN, rho = load_mesh("sphere")
        opts = dict(threshold_density=0.5, sdf_grid_setup="automatic", rbf_grid="same")
    else:
        X, IEN, rho = load_mesh({"sphere": "sphere", "cantilever": "cantilever_beam_vfrac_03"}[case])
        opts = dict(threshold_density=0.5 if case == "sphere" else None, sdf_grid_setup="automatic", rbf_grid="fine")
    return X, IEN, rho, r2s.Rho2sdfOptions(**opts)


def _grid_frame(grid, smooth):
    return tuple(grid.AABB_min), (grid.cell_size / smooth,) * 3


@pytest.mark.parametrize("case", ["sphere", "cantilever", "simp24", "sphere_same"])
def test_pipeline_surface(r2s, case, tmp_path):
    X, IEN, rho, opts = _pipeline_case(r2s, case)
    smooth = 2 if opts.rbf_grid == "fine" else 1
    mesh = r2s.Mesh(X, IEN, rho, element_type=opts.element_type)
    grid = r2s.noninteractive_sdf_grid_setup(mesh) if opts.sdf_grid_setup == "automatic" else r2s.Grid(X.min(0), X.max(0), int(np.floor(np.max(X.max(0) - X.min(0)) / opts.grid_step)), 3)
    rn = r2s.DenseInNodes(mesh, rho)
    rho_t = opts.threshold_density if opts.threshold_density is not None else r2s.find_threshold_for_volume(mesh, rn)
    d, _ = r2s.evalDistances(mesh, grid, None, rn, rho_t, want_xp=False)
    s = r2s.Sign_Detection(mesh, grid, None, rn, rho_t)
    sdf = d * s
    if opts.remove_artifacts:
        r2s.remove_sdf_artifacts(sdf, grid, 0.0, opts.artifact_min_component_ratio, mesh=mesh)
    fine, fg, info = r2s.RBFs_smoothing(mesh, sdf, grid, opts.rbf_interp, smooth, case, return_info=True)
    origin, spacing = _grid_frame(grid, smooth)
    V, T = r2s.isosurface(mesh)
    Vr, Tr = ref.reference(fine, origin, spacing, 0.0)
    assert len(T) > 100 and np.array_equal(V, Vr) and np.array_equal(T, Tr)
    border_negative = all((b < 0).all() for b in (fine[0], fine[-1], fine[:, 0], fine[:, -1], fine[:, :, 0], fine[:, :, -1]))
    print("%s: nv=%d nt=%d border negative: %s" % (case, len(V), len(T), border_negative))
    if border_negative:
        assert len(ref.unpaired_edges(T)) == 0
        # the divergence volume of the piecewise-linear surface against the quadrature volume of the same field: both converge to the
        # volume of {fine_sdf >= 0} at second order in the fine step h: each differs from it by about (surface area) * h^2 * curvature;
        # for these parts (a few fine cells across the thinnest member) that is a few per mille, and 5 % leaves room for thin members
        vol = ref.divergence_volume(V, T)
        print("%s: divergence volume %.6g, quadrature volume %.6g" % (case, vol, info["volume"]))
        assert abs(vol - info["volume"]) <= 0.05 * abs(info["volume"]), (vol, info["volume"])
    else:
        bad = ref.unpaired_edges(T)
        assert ref.on_boundary_face(V, T, bad, origin, spacing, fine.shape).all()
    # the resident results are untouched: the device fine field still streams out unchanged
    p = r2s.export_device_result_to_vti(mesh, str(tmp_path / "fine"), "distance", fine=True)
    assert np.array_equal(r2s.read_vti(p)[4], fine)
    mesh.close()


def _device_lists():
    import torch
    n = torch.cuda.device_count()
    lists = [[0, 0], [0, 0, 0]]
    if n >= 2:
        lists += [[0, 1], list(range(min(n, 4)))]
    return lists


@pytest.mark.parametrize("case", ["simp24", "simp24_approx"])
def test_multi_surface(r2s, case, tmp_path):
    X, IEN, rho, opts = _pipeline_case(r2s, case)
    fine1, fg1, grid1, sdf1 = r2s.rho2sdf(case, X, IEN, rho, options=opts, export_surface=str(tmp_path / "one.ply"))
    origin, spacing = _grid_frame(grid1, 2)
    V1, T1 = ref.reference(fine1, origin, spacing)
    assert np.array_equal(r2s.read_ply(str(tmp_path / "one.ply"))[0], V1) and np.array_equal(r2s.read_ply(str(tmp_path / "one.ply"))[1], T1)
    for devs in _device_lists():
        mesh = r2s.Mesh(X, IEN, rho, devices=devs)
        grid = grid1
        mesh._use_grid(grid)
        rn = r2s.DenseInNodes(mesh, rho)
        import ctypes as C
        m = mesh.multi
        p = r2s.Params(); m.lib.r2s_default_params(C.byref(p))
        p.rho_t, p.smooth, p.rbf_interp, p.remove_artifacts, p.artifact_min_ratio = 0.5, 2, int(opts.rbf_interp), 1, opts.artifact_min_component_ratio
        p.target_volume, p.final_volume = mesh.V_frac * mesh.V_domain, 1
        fine = np.empty(fine1.size, np.float32); sdf = np.empty(grid.ngp); rep = r2s.Report()
        m.check(m.lib.r2s_multi_pipeline(m.h, C.byref(p), rn.ctypes.data_as(C.c_void_p), sdf.ctypes.data_as(C.c_void_p), fine.ctypes.data_as(C.c_void_p), C.byref(rep)))
        fine = fine.reshape(fine1.shape)
        V, T = r2s.isosurface(mesh)
        Vr, Tr = ref.reference(fine, origin, spacing)
        assert np.array_equal(V, Vr) and np.array_equal(T, Tr), devs      # each layout's mesh is the reference mesh of its own field
        if not opts.rbf_interp:      # no CG: the fields are bit-identical across layouts, and so are the meshes
            assert np.array_equal(fine, fine1) and np.array_equal(V, V1) and np.array_equal(T, T1)
        # one file for the whole mesh, equal to the single-context file of the same arrays
        r2s.export_isosurface(mesh, str(tmp_path / "multi.stl"))
        c = r2s.Context()
        r2s.isosurface_from_sdf(fine, origin, spacing, 0.0, ctx=c)
        c.check(c.lib.r2s_export_isosurface(c.h, str(tmp_path / "single.stl").encode(), 0))
        c.close()
        assert open(tmp_path / "multi.stl", "rb").read() == open(tmp_path / "single.stl", "rb").read()
        mesh.close()


def test_stl_and_ply_round_trip(r2s, ctx, tmp_path):
    import ctypes as C
    f = _field("torus", (30, 41, 52))
    f[3, 4, 5:9] = 0.0      # corners on iso: zero-area triangles get 0 0 0 normals
    origin, spacing = (1.0, 2.0, -3.0), (0.2, 0.2, 0.2)
    V, T = r2s.isosurface_from_sdf(f, origin, spacing, 0.0, ctx=ctx)
    ctx.check(ctx.lib.r2s_export_isosurface(ctx.h, str(tmp_path / "s.stl").encode(), 0))
    ctx.check(ctx.lib.r2s_export_isosurface(ctx.h, str(tmp_path / "s.ply").encode(), 1))
    import os
    assert os.path.getsize(tmp_path / "s.stl") == 84 + 50 * len(T)
    N, P = r2s.read_stl(str(tmp_path / "s.stl"))
    assert np.array_equal(P, V[T])
    assert np.allclose(N, ref.stl_normals(V, T), atol=1e-6, rtol=0)
    ln = np.linalg.norm(N.astype(np.float64), axis=1)
    assert np.all((np.abs(ln - 1) < 1e-6) | (ln == 0))
    V2, T2 = r2s.read_ply(str(tmp_path / "s.ply"))
    assert np.array_equal(V2, V) and np.array_equal(T2, T)
    with pytest.raises(r2s.R2SError, match="format"):
        ctx.check(ctx.lib.r2s_export_isosurface(ctx.h, str(tmp_path / "s.obj").encode(), 2))


def test_errors(r2s, tmp_path):
    import ctypes as C
    c = r2s.Context()
    with pytest.raises(r2s.R2SError, match="no fine_sdf|r2s_set_grid"):
        c.check(c.lib.r2s_isosurface(c.h, 0.0, None, None))
    with pytest.raises(r2s.R2SError, match="no surface"):
        c.check(c.lib.r2s_download_isosurface(c.h, None, None))
    f = _field("sphere", (8, 9, 10))
    g = f.copy(); g[4, 4, 4] = np.nan
    with pytest.raises(r2s.R2SError, match="non-finite"):
        r2s.isosurface_from_sdf(g, (0, 0, 0), (1, 1, 1), ctx=c)
    g = f.copy(); g[7, 8, 9] = np.inf
    with pytest.raises(r2s.R2SError, match="non-finite"):
        r2s.isosurface_from_sdf(g, (0, 0, 0), (1, 1, 1), ctx=c)
    with pytest.raises(r2s.R2SError, match="iso must be finite"):
        r2s.isosurface_from_sdf(f, (0, 0, 0), (1, 1, 1), iso=float("nan"), ctx=c)
    with pytest.raises(r2s.R2SError, match="at least 2 points"):
        r2s.isosurface_from_sdf(f[:, :, :1], (0, 0, 0), (1, 1, 1), ctx=c)
    with pytest.raises(r2s.R2SError, match="no surface"):      # a failed extraction leaves no mesh behind
        c.check(c.lib.r2s_download_isosurface(c.h, None, None))
    with pytest.raises(r2s.R2SError, match=r"\.stl"):
        r2s.export_isosurface(None, str(tmp_path / "mesh.obj"))      # the format comes from the extension
    c.close()
