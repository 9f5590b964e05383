"""GPU parity tests: the CUDA path (through the C ABI of libr2s.so, via the host mirror) against the CPU oracle on the same
inputs, and against the reference's own golden values.  Run on a B200 with `pytest -m gpu`.

Tolerances (BASELINE.json north_star):
  * sign field and artifact-removal result: bit-exact
  * distances: |gpu - oracle| <= 1e-9 * h (FP64), far points (1e10) identical
  * nodal densities / iso-threshold (decision inputs): bit-exact
  * Float32 smoothing: |gpu - oracle| <= 1e-3 * h (the reference itself is only reproducible to Float32 round-off there:
    Float32 atomics and a reltol-3.45e-4 CG, SURVEY.md section 5), CG iteration count equal, volume within the bisection's 1e-4
"""
import os

import numpy as np
import pytest

import oracle
from fixtures import BLOCK_RHO_N, block_geometry, load_mesh, schlafli_tet4, simp_hex8

pytestmark = pytest.mark.gpu

DIST_TOL = 1e-9      # in units of the grid step h
RBF_TOL = 1e-3       # in units of h


def isapprox(a, b, rtol=0.0, atol=0.0):
    return abs(a - b) <= max(atol, rtol * max(abs(a), abs(b)))


def check_distances(r2s, mesh, X, IEN, grid, rn, rt, delta):
    d, xp = r2s.evalDistances(mesh, grid, None, rn, rt, delta_factor=delta)
    od, oxp, st = oracle.eval_distances(X, IEN, grid, rn, rt, delta)
    far = od > 1e9
    assert np.array_equal(d > 1e9, far), "band membership differs"
    assert np.array_equal(d[far], od[far])
    assert np.max(np.abs(d - od)) <= DIST_TOL * grid.cell_size
    rep = mesh.ctx.report()
    assert rep.n_pairs == st["pairs"] and rep.n_pairs_pruned == 0      # with xp every pair is projected
    # pairs whose iteration ran into its cap are still used (the reference uses NLopt's point even on :FAILURE,
    # ComputeCoordsOnIso.jl:82-86); they must be rare on both sides
    assert rep.n_not_converged <= 2 + 1e-5 * rep.n_pairs and st["not_converged"] <= 2 + 1e-5 * st["pairs"]
    # xp is tie-order dependent where two candidates are equidistant (SURVEY appendix A.2): compare through the distance it implies
    P = r2s.generateGridPoints(grid)
    near = ~far
    assert np.max(np.abs(np.linalg.norm(P[near] - xp[near], axis=1) - d[near])) <= 1e-9 * grid.cell_size
    # the pipeline's path (no xp: pair list with pruning, atomicMin, crossing-element faces folded into the pair buffer) must give the
    # same distances; the two paths are different kernels (FMA contraction may differ in the last bit), hence 1e-11 h instead of equality
    d2, _ = r2s.evalDistances(mesh, grid, None, rn, rt, delta_factor=delta, want_xp=False)
    assert np.array_equal(d > 1e9, d2 > 1e9) and np.max(np.abs(d - d2)) <= 1e-11 * grid.cell_size
    assert np.max(np.abs(d2 - od)) <= DIST_TOL * grid.cell_size
    return d, od


def check_sign_and_artifacts(r2s, mesh, X, IEN, grid, rn, rt, od):
    s = r2s.Sign_Detection(mesh, grid, None, rn, rt)
    os_ = oracle.sign_detection(X, IEN, grid, rn, rt)
    assert set(np.unique(s)) <= {-1.0, 1.0}
    assert np.array_equal(s, os_), "sign field differs at %d points" % int((s != os_).sum())
    sdf = od * os_
    g2 = sdf.copy()
    nf = r2s.remove_sdf_artifacts(g2, grid, mesh=mesh)
    o2, onf = oracle.remove_artifacts(sdf, grid)
    assert nf == onf and np.array_equal(g2, o2)
    # a noisy mask exercises many small components and the min-size rule
    rng = np.random.default_rng(1)
    noisy = sdf.copy()
    m = rng.random(sdf.size) < 0.03
    noisy[m] = np.abs(noisy[m]) * np.where(rng.random(int(m.sum())) < 0.5, 1, -1)
    for ratio in (0.01, 0.2):
        g3 = noisy.copy()
        nf = r2s.remove_sdf_artifacts(g3, grid, min_component_ratio=ratio, mesh=mesh)
        o3, onf = oracle.remove_artifacts(noisy, grid, 0.0, ratio)
        assert nf == onf and np.array_equal(g3, o3)
    return o2


def check_rbf(r2s, mesh, grid, sdf, target, combos=((True, 2), (True, 1), (False, 2), (False, 1))):
    for interp, sm in combos:
        fine, fg, info = r2s.RBFs_smoothing(mesh, sdf, grid, interp, sm, "t", return_info=True)
        ofine, oinfo = oracle.rbf_smoothing(sdf, grid, interp, sm, target, mode=0, nthreads=oracle.max_threads())
        assert fine.shape == ofine.shape == tuple(int(n) * sm + 1 for n in grid.N[::-1]) and fine.dtype == np.float32
        assert info["cg_iters"] == oinfo["cg_iters"]
        assert np.max(np.abs(fine - ofine)) <= RBF_TOL * grid.cell_size
        assert abs(info["th"] - oinfo["th"]) <= RBF_TOL * grid.cell_size
        if sm == 1:      # on the :same grid the returned field is the one the bisection matched
            assert abs(info["volume"] - target) <= max(2e-4, 2e-6 * target) or info["bisections"] == 40
        assert abs(info["volume"] - oinfo["volume"]) <= 1e-4 * max(1.0, abs(oinfo["volume"]))


# --------------------------------------------------------------------------------------------------------------------
def test_block_goldens_and_parity(r2s):
    """test/HexBlockSdfTest.jl: 2-element block, roof densities, Grid(20, 3), rho_t = 0.5."""
    X, IEN, rho = block_geometry([2, 1, 1])
    grid = r2s.Grid(X.min(0), X.max(0), 20, 3)
    mesh = r2s.Mesh(X, IEN, rho)
    vd, vf = oracle.mesh_volume(X, IEN, rho)
    assert isapprox(mesh.V_domain, vd, rtol=1e-12) and isapprox(mesh.V_frac, vf, rtol=1e-12)
    d25, od25 = check_distances(r2s, mesh, X, IEN, grid, BLOCK_RHO_N, 0.5, 2.5)
    s = r2s.Sign_Detection(mesh, grid, None, BLOCK_RHO_N, 0.5)
    sdf = d25 * s
    assert isapprox(sdf.max(), 0.4242640687119285, rtol=1e-10, atol=1e-12)        # HexBlockSdfTest.jl:25
    assert isapprox(sdf.mean(), -1.4699474563515213e9, atol=1e5)                   # :26
    assert (d25 >= 0).all() and not np.isnan(d25).any()                             # :84-90
    d11, od11 = check_distances(r2s, mesh, X, IEN, grid, BLOCK_RHO_N, 0.5, 1.1)
    clean = check_sign_and_artifacts(r2s, mesh, X, IEN, grid, BLOCK_RHO_N, 0.5, od11)
    check_rbf(r2s, mesh, grid, clean, vd * vf)
    mesh.ctx.close()


def test_sphere_goldens_and_parity(r2s):
    """test/HexSphereSdfTest.jl (BASELINE configs[0]): sphere.mat, DenseInNodes, Grid(10, 3), rho_t = 0.5."""
    X, IEN, rho = load_mesh("sphere")
    grid = r2s.Grid(*r2s.getMesh_AABB(X), 10, 3)
    mesh = r2s.Mesh(X, IEN, rho)
    rn = r2s.DenseInNodes(mesh, rho)
    assert np.array_equal(rn, oracle.nodal_densities(X, IEN, rho))
    assert isapprox(rn.max(), 1.0000000000000022, rtol=1e-10, atol=1e-12)          # HexSphereSdfTest.jl:26
    assert isapprox(rn.mean(), 0.29490556408887564, rtol=1e-10, atol=1e-12)        # :27
    d25, _ = check_distances(r2s, mesh, X, IEN, grid, rn, 0.5, 2.5)
    s = r2s.Sign_Detection(mesh, grid, None, rn, 0.5)
    sdf = d25 * s
    assert isapprox(sdf.max(), 0.8669785608800439, rtol=1e-10, atol=1e-12)         # :28
    assert isapprox(sdf.mean(), -3.7370242217627172e9, atol=1e5)                    # :29
    assert int((s > 0).sum()) < int((s < 0).sum())                                  # :123-125
    d11, od11 = check_distances(r2s, mesh, X, IEN, grid, rn, 0.5, 1.1)
    clean = check_sign_and_artifacts(r2s, mesh, X, IEN, grid, rn, 0.5, od11)
    check_rbf(r2s, mesh, grid, clean, mesh.V_domain * mesh.V_frac)
    # edge-case thresholds on a 5-cell grid (HexSphereSdfTest.jl:169-199)
    g5 = r2s.Grid(*r2s.getMesh_AABB(X), 5, 3)
    for thr in (0.1, 0.9):
        check_distances(r2s, mesh, X, IEN, g5, rn, thr, 1.1)
        s5 = r2s.Sign_Detection(mesh, g5, None, rn, thr)
        assert np.array_equal(s5, oracle.sign_detection(X, IEN, g5, rn, thr))
    mesh.ctx.close()


@pytest.mark.parametrize("name", ["cantilever_beam_vfrac_03", "chapadlo"])
def test_mat_fixtures_full_path(r2s, name):
    """BASELINE configs[1] and [2]: threshold auto, :automatic grid, rbf_interp, :fine grid, artifact removal."""
    X, IEN, rho = load_mesh(name)
    mesh = r2s.Mesh(X, IEN, rho)
    grid = r2s.noninteractive_sdf_grid_setup(mesh)
    assert list(grid.N) == ([66, 26, 10] if name.startswith("cant") else [25, 44, 64])     # SURVEY.md section 6
    # calculate_edge_distances / analyze_mesh (Grid_setup.jl:28-92): device median == numpy median of the same expression, bit for bit
    P = X[IEN - 1]
    d = np.stack([np.sqrt((P[:, b, 0] - P[:, a, 0]) ** 2 + (P[:, b, 1] - P[:, a, 1]) ** 2 + (P[:, b, 2] - P[:, a, 2]) ** 2) for a, b in mesh.edges])
    assert mesh.edge_stats["median"] == float(np.median(d)) and mesh.edge_stats["shortest"] == d.min() and mesh.edge_stats["longest"] == d.max()
    vd, vf = oracle.mesh_volume(X, IEN, rho)
    # the volumes are sums over elements: order of summation differs (the reference itself accumulates with atomics, MeshVolume.jl:24-40)
    assert isapprox(mesh.V_domain, vd, rtol=1e-12) and isapprox(mesh.V_frac, vf, rtol=1e-12)
    rn = r2s.DenseInNodes(mesh, rho)
    assert np.array_equal(rn, oracle.nodal_densities(X, IEN, rho))
    rt = r2s.find_threshold_for_volume(mesh, rn)
    assert rt == oracle.find_threshold(X, IEN, rn, vd * vf)
    assert isapprox(r2s.calculate_isocontour_volume(mesh, rn, rt), oracle.isocontour_volume(X, IEN, rn, rt), rtol=1e-12)
    d, od = check_distances(r2s, mesh, X, IEN, grid, rn, rt, 1.1)
    clean = check_sign_and_artifacts(r2s, mesh, X, IEN, grid, rn, rt, od)
    check_rbf(r2s, mesh, grid, clean, vd * vf, combos=((True, 2), (False, 1)))
    mesh.ctx.close()
    # the same through the public entry point, one device-resident pipeline call
    opts = r2s.Rho2sdfOptions(sdf_grid_setup="automatic", rbf_interp=True, rbf_grid="fine", remove_artifacts=True)
    fine, fg, g2, sdf, rep = r2s.rho2sdf(name, X, IEN, rho, options=opts, return_report=True)
    assert rep["rho_t"] == rt and list(g2.N) == list(grid.N)
    assert np.array_equal(np.sign(sdf), np.sign(clean)) and np.array_equal(np.abs(sdf) > 1e9, np.abs(clean) > 1e9)
    assert np.max(np.abs(sdf - clean)) <= DIST_TOL * grid.cell_size
    ofine, oinfo = oracle.rbf_smoothing(clean, grid, True, 2, vd * vf, mode=0, nthreads=oracle.max_threads())
    assert np.max(np.abs(fine - ofine)) <= RBF_TOL * grid.cell_size
    assert fg.shape == tuple(int(n) * 2 + 1 for n in grid.N) and rep["launches"] > 0


def test_threshold_out_of_range_raises(r2s):
    """Isocontour_volume.jl:93-95: a target volume outside [V(1), V(0)] is an error."""
    X, IEN, rho = load_mesh("sphere")
    mesh = r2s.Mesh(X, IEN, rho)
    rn = r2s.DenseInNodes(mesh, rho)
    mesh.V_frac = 5.0
    with pytest.raises(r2s.R2SError, match="outside the possible range"):
        r2s.find_threshold_for_volume(mesh, rn)
    mesh.ctx.close()


@pytest.mark.parametrize("n", [12, 24])
def test_synthetic_simp_hex8(r2s, n):
    """Reduced replicas of BASELINE configs[4] (synthetic SIMP field, grid step h_e / 2)."""
    X, IEN, rho = simp_hex8(n)
    mesh = r2s.Mesh(X, IEN, rho)
    grid = r2s.Grid(X.min(0), X.max(0), 2 * n, 3)
    rn = r2s.DenseInNodes(mesh, rho)
    assert np.array_equal(rn, oracle.nodal_densities(X, IEN, rho))
    d, od = check_distances(r2s, mesh, X, IEN, grid, rn, 0.5, 1.1)
    clean = check_sign_and_artifacts(r2s, mesh, X, IEN, grid, rn, 0.5, od)
    check_rbf(r2s, mesh, grid, clean, mesh.V_domain * mesh.V_frac, combos=((True, 2),))
    mesh.ctx.close()


@pytest.mark.parametrize("field", ["radial", "simp"])
def test_tet4_schlafli(r2s, field):
    """BASELINE configs[3] at reduced size: Schlaefli-split cube, explicit threshold (the reference's automatic threshold is
    HEX8-only, Isocontour_volume.jl:27-38), rho2sdf_tet4 path."""
    n = 8
    X, IEN, rn = schlafli_tet4(n, field)
    rho = rn[IEN - 1].mean(axis=1)
    mesh = r2s.Mesh(X, IEN, rho, element_type=r2s.TET4)
    vd, vf = oracle.mesh_volume(X, IEN, rho)
    # reference quirk kept for parity: the TET4 quadrature weights the cube->tet map with (1-xi)^2 (1-xi-eta)/8
    # (MeshVolume.jl:107) instead of (1-xi)(1-xi-eta)/8, so V_domain comes out as 3/4 of the geometric volume
    assert abs(mesh.V_domain - 0.75 * n ** 3) < 1e-9 and isapprox(mesh.V_domain, vd, rtol=1e-12) and isapprox(mesh.V_frac, vf, rtol=1e-12)
    grid = r2s.Grid(X.min(0), X.max(0), 2 * n, 3)
    d, od = check_distances(r2s, mesh, X, IEN, grid, rn, 0.5, 1.1)
    clean = check_sign_and_artifacts(r2s, mesh, X, IEN, grid, rn, 0.5, od)
    check_rbf(r2s, mesh, grid, clean, vd * vf, combos=((True, 2),))
    with pytest.raises(r2s.R2SError):
        r2s.Mesh(X, IEN, rho, element_type=r2s.HEX8)        # MeshInformations.jl:59
    mesh.ctx.close()


def test_volume_from_sdf_convergence(r2s):
    """test/ConvergenceTests/{Sphere,Cube}ConvergenceTest.jl: analytic volumes pi/6 and 1, error ladders; bit-equal to the oracle."""
    ctx = r2s.Context()
    errs = []
    for N, tol in ((16, 0.10), (32, 0.05), (64, 0.02)):
        ax = np.linspace(-1, 1, N + 1, dtype=np.float32)
        z, y, x = np.meshgrid(ax, ax, ax, indexing="ij")
        sph = (0.5 - np.sqrt(x * x + y * y + z * z)).astype(np.float32)
        v = float(r2s.calculate_volume_from_sdf(sph, np.float32(ax[1] - ax[0]), ctx=ctx))
        errs.append(abs(v - np.pi / 6) / (np.pi / 6))
        assert errs[-1] < tol
        assert abs(v - oracle.volume_from_sdf(sph, np.float32(ax[1] - ax[0]))) <= 2e-6 * v
        cube = (0.5 - np.maximum(np.maximum(np.abs(x), np.abs(y)), np.abs(z))).astype(np.float32)
        vc = float(r2s.calculate_volume_from_sdf(cube, np.float32(ax[1] - ax[0]), ctx=ctx))
        assert abs(vc - 1.0) < (0.05 if N < 32 else 0.02)
    assert errs[0] > errs[1] > errs[2]           # monotone decrease (SphereConvergenceTest.jl:400-410)
    # detailed_quad_order = 20, as the reference's acceptance suite calls it (SphereConvergenceTest.jl:67, CubeConvergenceTest.jl:67):
    # the ladders of :364-398 (sphere: < 10 % for N >= 16, < 5 % for N >= 32, < 2 % for N >= 64) and the oracle's value at the same order
    errs20 = []
    for N, tol in ((8, 0.5), (16, 0.10), (32, 0.05), (64, 0.02)):
        ax = np.linspace(-1, 1, N + 1, dtype=np.float32)
        z, y, x = np.meshgrid(ax, ax, ax, indexing="ij")
        sph = (0.5 - np.sqrt(x * x + y * y + z * z)).astype(np.float32)
        v = float(r2s.calculate_volume_from_sdf(sph, np.float32(ax[1] - ax[0]), detailed_quad_order=20, ctx=ctx))
        errs20.append(abs(v - np.pi / 6) / (np.pi / 6))
        assert errs20[-1] < tol
        assert abs(v - oracle.volume_from_sdf(sph, np.float32(ax[1] - ax[0]), order=20)) <= 2e-6 * v
        cube = (0.5 - np.maximum(np.maximum(np.abs(x), np.abs(y)), np.abs(z))).astype(np.float32)
        vc = float(r2s.calculate_volume_from_sdf(cube, np.float32(ax[1] - ax[0]), detailed_quad_order=20, ctx=ctx))
        assert abs(vc - oracle.volume_from_sdf(cube, np.float32(ax[1] - ax[0]), order=20)) <= 2e-6 * max(vc, 1e-3)
    assert errs20[1] > errs20[2] > errs20[3]
    for order in (1, 3, 15, 32):                 # every order the parameter admits; 0 and 33 are refused
        v = float(r2s.calculate_volume_from_sdf(sph, np.float32(ax[1] - ax[0]), detailed_quad_order=order, ctx=ctx))
        assert abs(v - oracle.volume_from_sdf(sph, np.float32(ax[1] - ax[0]), order=order)) <= 2e-6 * v
    for order in (0, 33):
        with pytest.raises(r2s.R2SError, match="detailed_quad_order"):
            r2s.calculate_volume_from_sdf(sph, np.float32(ax[1] - ax[0]), detailed_quad_order=order, ctx=ctx)
    ctx.close()


def test_empty_and_degenerate_inputs(r2s):
    """All-void and all-solid density fields, one-element meshes, invalid connectivity."""
    X, IEN, rho = block_geometry([2, 1, 1])
    grid = r2s.Grid(X.min(0), X.max(0), 8, 3)
    mesh = r2s.Mesh(X, IEN, rho)
    void = np.zeros(X.shape[0])
    d, _ = r2s.evalDistances(mesh, grid, None, void, 0.5)
    assert (d == 1e10).all()                                                       # nothing active: every point keeps |-1e10|
    assert (r2s.Sign_Detection(mesh, grid, None, void, 0.5) == -1).all()
    solid = np.ones(X.shape[0])
    d, _ = r2s.evalDistances(mesh, grid, None, solid, 0.5)
    od, _, _ = oracle.eval_distances(X, IEN, grid, solid, 0.5, 1.1)
    assert np.array_equal(d > 1e9, od > 1e9) and np.max(np.abs(d - od)) <= DIST_TOL * grid.cell_size
    s = r2s.Sign_Detection(mesh, grid, None, solid, 0.5)
    assert np.array_equal(s, oracle.sign_detection(X, IEN, grid, solid, 0.5))
    allneg = -np.ones(grid.ngp)
    assert r2s.remove_sdf_artifacts(allneg, grid, mesh=mesh) == 0
    with pytest.raises(r2s.R2SError):
        r2s.remove_sdf_artifacts(np.zeros(5), grid, mesh=mesh)                    # SdfArtifactRemoval.jl:142
    with pytest.raises(r2s.R2SError):
        r2s.RBFs_smoothing(mesh, np.full(grid.ngp, -1e10), grid, True, 1)         # no finite value (RBFs4Smoothing.jl:17)
    withnan = np.linspace(-1.0, 1.0, grid.ngp); withnan[grid.ngp // 2] = np.nan
    with pytest.raises(r2s.R2SError, match="not finite"):
        r2s.RBFs_smoothing(mesh, withnan, grid, True, 1)                          # CG stops on a NaN residual instead of running to maxiter = n
    mesh.ctx.close()
    bad = IEN.copy(); bad[0, 0] = 99
    with pytest.raises(r2s.R2SError):
        r2s.Mesh(X, bad, rho)


# --------------------------------------------------------------------------------------------------------------------
# size-independent properties at sizes the oracle cannot reach
# --------------------------------------------------------------------------------------------------------------------
def _run_pipeline(r2s, mesh, grid, rn, smooth=2, slab=None):
    import ctypes as C
    mesh._use_grid(grid)
    c = mesh.ctx
    if slab is not None:
        c.check(c.lib.r2s_set_slab(c.h, slab[0], slab[1]))
    p = r2s.Params(); c.lib.r2s_default_params(C.byref(p))
    p.rho_t, p.smooth, p.rbf_interp, p.target_volume = 0.5, smooth, 1, mesh.V_frac * mesh.V_domain
    c.check(c.lib.r2s_upload_nodal_densities(c.h, rn.ctypes.data_as(C.c_void_p)))
    rep = r2s.Report()
    c.check(c.lib.r2s_pipeline_resident(c.h, C.byref(p), C.byref(rep)))
    sdf = np.empty(grid.ngp); c.check(c.lib.r2s_download_sdf(c.h, sdf.ctypes.data_as(C.c_void_p)))
    dims = tuple(int(v) * smooth + 1 for v in grid.N)
    fine = np.empty(dims[0] * dims[1] * dims[2], dtype=np.float32); c.check(c.lib.r2s_download_fine_sdf(c.h, fine.ctypes.data_as(C.c_void_p)))
    return sdf, fine.reshape(dims[::-1]), rep


@pytest.mark.parametrize("n", [64, 128])
def test_large_pipeline_properties(r2s, n):
    X, IEN, rho = simp_hex8(n)
    mesh = r2s.Mesh(X, IEN, rho)
    grid = r2s.Grid(X.min(0), X.max(0), 2 * n, 3)
    rn = r2s.DenseInNodes(mesh, rho)
    sdf, fine, rep = _run_pipeline(r2s, mesh, grid, rn)
    sdf2, fine2, rep2 = _run_pipeline(r2s, mesh, grid, rn)
    # determinism: two runs are bit-identical (no float atomics anywhere on the path)
    assert np.array_equal(sdf, sdf2) and np.array_equal(fine, fine2)
    assert rep.n_not_converged <= 1e-5 * rep.n_pairs
    # every element is a unit cube: points with a positive sign are exactly the points inside the mesh whose interpolated density >= 0.5
    far = np.abs(sdf) > 1e9
    assert (np.abs(sdf[~far]) <= np.sqrt(3) * (1 + 2 * 2.1 * grid.cell_size) + 1e-9).all()     # band: within the diagonal of an element grown by delta + 1 cell
    # idempotence of the artifact removal
    again = sdf.copy()
    assert r2s.remove_sdf_artifacts(again, grid, mesh=mesh) == 0 and np.array_equal(again, sdf)
    # volume matching: the fine field's volume is within a few percent of the target (the offset is matched on the coarse grid)
    target = mesh.V_frac * mesh.V_domain
    assert abs(rep.volume - target) / target < 0.05
    # the coarse samples of the fine grid agree with the :same evaluation
    _, same, _ = _run_pipeline(r2s, mesh, grid, rn, smooth=1)
    assert np.max(np.abs(fine[::2, ::2, ::2] - same)) <= 1e-5 * max(1.0, np.abs(same).max())
    # z-slab decomposition: distances/signs of a slab equal the same planes of the full run (multi-GPU sharding invariant)
    import ctypes as C
    nz = int(grid.N[2]) + 1
    k0, k1 = nz // 3, 2 * nz // 3
    c = mesh.ctx
    c.check(c.lib.r2s_set_slab(c.h, k0, k1))
    d_slab, _ = r2s.evalDistances(mesh, grid, None, rn, 0.5, want_xp=False)
    s_slab = r2s.Sign_Detection(mesh, grid, None, rn, 0.5)
    c.check(c.lib.r2s_set_slab(c.h, 0, nz))
    d_full, _ = r2s.evalDistances(mesh, grid, None, rn, 0.5, want_xp=False)
    s_full = r2s.Sign_Detection(mesh, grid, None, rn, 0.5)
    pl = int(grid.N[0] + 1) * int(grid.N[1] + 1)
    assert np.array_equal(d_slab[k0 * pl:k1 * pl], d_full[k0 * pl:k1 * pl])
    assert np.array_equal(s_slab[k0 * pl:k1 * pl], s_full[k0 * pl:k1 * pl])
    mesh.ctx.close()


def test_tet4_two_million_tets_public_api(r2s):
    """BASELINE configs[3]: synthetic TET4 SIMP field, 70^3 hex cells Schlaefli-split = 2 058 000 tets, explicit threshold (the reference's
    automatic threshold is HEX8-only), :automatic grid, through rho2sdf_tet4.  The oracle is too slow here: size-independent properties."""
    n = 70
    X, IEN, rn = schlafli_tet4(n, "simp")
    assert IEN.shape == (6 * n ** 3, 4)
    rho = rn[IEN - 1].mean(axis=1)
    out1 = r2s.rho2sdf_tet4("tet", X, IEN, rho, threshold_density=0.5, sdf_grid_setup="automatic", rbf_grid="fine", return_report=True)
    fine, fg, grid, sdf, rep = out1
    # grid step = median edge of the split (unit edges, face diagonals sqrt2, one body diagonal sqrt3 per tet path)
    assert abs(grid.cell_size - n / np.floor(n / np.median([1, 1, 1, np.sqrt(2), np.sqrt(2), np.sqrt(3)]))) < 1e-9
    assert fine.shape == tuple(int(v) * 2 + 1 for v in grid.N[::-1]) and fine.dtype == np.float32 and np.isfinite(fine).all()
    assert sdf.shape == (grid.ngp,) and np.isfinite(sdf).all() and rep["n_crossing"] > 0 and rep["cg_iters"] > 5
    inside = sdf > 0
    assert 0.05 < inside.mean() < 0.6                                   # the SIMP field fills a moderate fraction of the box
    band = np.abs(sdf) < 1e9
    assert np.abs(sdf[band]).max() <= np.sqrt(3) * (1 + 2 * 2.1 * grid.cell_size) + 1e-9
    # determinism through the public entry point
    fine2, _, _, sdf2, _ = r2s.rho2sdf_tet4("tet", X, IEN, rho, threshold_density=0.5, sdf_grid_setup="automatic", rbf_grid="fine", return_report=True)
    assert np.array_equal(sdf, sdf2) and np.array_equal(fine, fine2)


def _mixed_mesh(n=10):
    """Half axis-aligned boxes, half distorted hexes (interior nodes of the x > mid half jittered by +-0.12 h)."""
    X, IEN, rho = simp_hex8(n)
    X = X.copy()
    h = (X[:, 0].max() - X[:, 0].min()) / n
    rng = np.random.default_rng(7)
    lo, hi = X.min(0), X.max(0)
    inner = np.all((X > lo + 0.5 * h) & (X < hi - 0.5 * h), axis=1) & (X[:, 0] > 0.5 * (lo[0] + hi[0]) + 0.25 * h)
    X[inner] += rng.uniform(-0.12, 0.12, (int(inner.sum()), 3)) * h
    return X, IEN, rho


def test_mixed_box_and_distorted_hexes(r2s, monkeypatch):
    """A mesh holding both kinds of HEX8 elements -- axis-aligned boxes (pair-list path with lower-bound pruning) and distorted hexes
    (general trilinear chunk kernel): both run, each leaving the other kind alone; sending everything through the general kernel
    (R2S_PROJ_BOX=0, read when the context is created) gives the same field."""
    n = 10
    X, IEN, rho = _mixed_mesh(n)
    mesh = r2s.Mesh(X, IEN, rho)
    grid = r2s.Grid(X.min(0), X.max(0), 2 * n, 3)
    rn = r2s.DenseInNodes(mesh, rho)
    d, od = check_distances(r2s, mesh, X, IEN, grid, rn, 0.5, 1.1)
    assert mesh.ctx.report().n_pairs_pruned < mesh.ctx.report().n_pairs      # (on a mesh this small nearly every tile holds boundary faces: little to prune)
    mesh.ctx.close()
    monkeypatch.setenv("R2S_PROJ_BOX", "0")
    mesh0 = r2s.Mesh(X, IEN, rho)
    d0, _ = r2s.evalDistances(mesh0, grid, None, rn, 0.5, delta_factor=1.1, want_xp=False)
    assert mesh0.ctx.report().n_pairs_pruned == 0
    assert np.max(np.abs(d0 - od)) <= DIST_TOL * grid.cell_size and np.max(np.abs(d0 - d)) <= 1e-11 * grid.cell_size
    mesh0.ctx.close()


@pytest.mark.parametrize("case", ["simp16", "simp24_coarse_grid", "simp12_fine_grid", "mixed"])
def test_projection_pruning_is_exact(r2s, monkeypatch, case):
    """The pair-list path skips (element, point) pairs whose lower bound (distance to the tight box of the element's iso-patch) is not
    below the point's current minimum.  The result of evalDistances is a minimum over the pairs, so pruning must not change a single
    bit: R2S_PROJ_PRUNE=0 (every pair projected) against the default, on grids coarser and finer than the elements."""
    X, IEN, rho, nmax = {"simp16": simp_hex8(16) + (32,), "simp24_coarse_grid": simp_hex8(24) + (30,), "simp12_fine_grid": simp_hex8(12) + (60,),
                         "mixed": _mixed_mesh(10) + (20,)}[case]
    res = {}
    for knob in ("1", "0"):
        monkeypatch.setenv("R2S_PROJ_PRUNE", knob)
        mesh = r2s.Mesh(X, IEN, rho)
        grid = r2s.Grid(X.min(0), X.max(0), nmax, 3)
        rn = r2s.DenseInNodes(mesh, rho)
        res[knob] = [r2s.evalDistances(mesh, grid, None, rn, rt, delta_factor=df, want_xp=False)[0] for rt, df in ((0.5, 1.1), (0.3, 2.5))]
        rep = mesh.ctx.report()
        assert (rep.n_pairs_pruned > 0) == (knob == "1") and rep.n_pairs_pruned < rep.n_pairs
        mesh.ctx.close()
    for a, b in zip(res["1"], res["0"]):
        assert np.array_equal(a, b)
    od, _, _ = oracle.eval_distances(X, IEN, grid, rn, 0.3, 2.5, want_xp=False, nthreads=oracle.max_threads())
    assert np.max(np.abs(res["1"][1] - od)) <= DIST_TOL * grid.cell_size


def test_pipelined_host_buffer_calls(r2s):
    """r2s_pipeline_slab_begin / _wait: three consecutive calls on alternating buffer sets return what the synchronous call returns."""
    import ctypes as C
    n = 24
    X, IEN, rho = simp_hex8(n)
    mesh = r2s.Mesh(X, IEN, rho)
    grid = r2s.Grid(X.min(0), X.max(0), 2 * n, 3)
    rn = r2s.DenseInNodes(mesh, rho)
    sdf_ref, fine_ref, _ = _run_pipeline(r2s, mesh, grid, rn)
    c = mesh.ctx
    p = r2s.Params(); c.lib.r2s_default_params(C.byref(p))
    p.rho_t, p.smooth, p.rbf_interp, p.remove_artifacts = 0.5, 2, 1, 1
    p.target_volume, p.final_volume = mesh.V_frac * mesh.V_domain, 1
    bufs = [(np.full(sdf_ref.size, np.nan), np.full(fine_ref.size, np.nan, dtype=np.float32)) for _ in range(2)]
    rn2 = np.ascontiguousarray(rn)
    tickets = []
    for k in range(3):
        rep = r2s.Report(); t = C.c_int(-1)
        c.check(c.lib.r2s_pipeline_slab_begin(c.h, C.byref(p), rn2.ctypes.data_as(C.c_void_p), bufs[k % 2][0].ctypes.data_as(C.c_void_p),
                                              bufs[k % 2][1].ctypes.data_as(C.c_void_p), C.byref(rep), C.byref(t)))
        if tickets:
            kk, tt = tickets.pop()
            c.check(c.lib.r2s_pipeline_slab_wait(c.h, tt))
            assert np.array_equal(bufs[kk % 2][0], sdf_ref.ravel()) and np.array_equal(bufs[kk % 2][1], fine_ref.ravel())
            bufs[kk % 2][0][:] = np.nan; bufs[kk % 2][1][:] = np.nan
        tickets.append((k, t.value))
    kk, tt = tickets.pop()
    c.check(c.lib.r2s_pipeline_slab_wait(c.h, tt))
    assert np.array_equal(bufs[kk % 2][0], sdf_ref.ravel()) and np.array_equal(bufs[kk % 2][1], fine_ref.ravel())
    mesh.ctx.close()


def test_simp_hex8_64_pipeline_vs_oracle(r2s):
    """The 64^3 replica of BASELINE configs[4] through ONE device-resident pipeline call against the CPU oracle's pipeline on the same
    inputs (bench.py repeats this on the 96^3 replica and prints it as `parity`)."""
    n = 64
    X, IEN, rho = simp_hex8(n)
    mesh = r2s.Mesh(X, IEN, rho)
    grid = r2s.Grid(X.min(0), X.max(0), 2 * n, 3)
    rn = r2s.DenseInNodes(mesh, rho)
    assert mesh.is_lattice
    sdf, fine, rep = _run_pipeline(r2s, mesh, grid, rn)
    nt = oracle.max_threads()
    assert np.array_equal(rn, oracle.nodal_densities(X, IEN, rho))
    od, _, _ = oracle.eval_distances(X, IEN, grid, rn, 0.5, 1.1, nthreads=nt, want_xp=False)
    osg = oracle.sign_detection(X, IEN, grid, rn, 0.5, nthreads=nt)
    osdf, onf = oracle.remove_artifacts(od * osg, grid)
    assert np.array_equal(np.abs(sdf) > 1e9, np.abs(osdf) > 1e9) and np.array_equal(np.signbit(sdf), np.signbit(osdf)) and rep.n_flipped == onf
    assert np.max(np.abs(sdf - osdf)) <= DIST_TOL * grid.cell_size
    ofine, oinfo = oracle.rbf_smoothing(osdf, grid, True, 2, mesh.V_domain * mesh.V_frac, mode=0, nthreads=nt)
    assert rep.cg_iters == oinfo["cg_iters"] and abs(rep.th - oinfo["th"]) <= RBF_TOL * grid.cell_size
    assert np.max(np.abs(fine - ofine)) <= RBF_TOL * grid.cell_size
    mesh.ctx.close()


def test_sign_lattice_fast_path(r2s, monkeypatch):
    """Sign_Detection_HEX8 on tensor-product lattice meshes: the list-free kernel (cells around a point from per-axis tables) against
    the general kernel (R2S_SIGN_LATTICE=0: sorted candidate lists, density-class shortcut) and the oracle -- bit-identical signs on the
    plain cube, on a graded lattice with holes and shuffled numbering, and on sphere.mat; unstructured meshes never take it."""
    from fixtures import graded_lattice_hex8
    cases = [simp_hex8(16) + (32, True), graded_lattice_hex8(12) + (30, True), load_mesh("sphere") + (24, True), _mixed_mesh(10) + (20, False),
             load_mesh("chapadlo") + (40, False)]
    for X, IEN, rho, nmax, lattice in cases:
        res = {}
        for knob in ("1", "0"):
            monkeypatch.setenv("R2S_SIGN_LATTICE", knob)
            mesh = r2s.Mesh(X, IEN, rho)                     # knobs are read when the context is created
            assert mesh.is_lattice == lattice
            grid = r2s.Grid(*r2s.getMesh_AABB(X), nmax, 3)
            rn = r2s.DenseInNodes(mesh, rho)
            res[knob] = [r2s.Sign_Detection(mesh, grid, None, rn, rt) for rt in (0.5, 0.3)]
            if knob == "1":      # a z-slab of the lattice path equals the same planes of the full run
                nz, pl = int(grid.N[2]) + 1, int(grid.N[0] + 1) * int(grid.N[1] + 1)
                mesh.ctx.check(mesh.ctx.lib.r2s_set_slab(mesh.ctx.h, nz // 3, 2 * nz // 3))
                s_slab = r2s.Sign_Detection(mesh, grid, None, rn, 0.5)
                assert np.array_equal(s_slab[nz // 3 * pl:2 * nz // 3 * pl], res[knob][0][nz // 3 * pl:2 * nz // 3 * pl])
            mesh.ctx.close()
        monkeypatch.delenv("R2S_SIGN_LATTICE")
        for q, rt in enumerate((0.5, 0.3)):
            assert np.array_equal(res["1"][q], res["0"][q])
            if X.shape[0] < 10000:
                assert np.array_equal(res["1"][q], oracle.sign_detection(X, IEN, grid, rn, rt))
            assert (res["1"][q] > 0).any() and (res["1"][q] < 0).any()


def test_threshold_search_cache_is_exact(r2s, monkeypatch):
    """LS_Threshold keeps, per active cut cell, the cell's last quadrature and a margin within which no Gauss value can change sign; the
    volume is an exact integer sum, so the search must take bit-identical decisions with the cache (default) and without (R2S_VOL_CACHE=0).
    R2S_DEBUG_SYNC=1 (a synchronisation after every launch, for fault localisation) must not change anything either."""
    X, IEN, rho = simp_hex8(24)
    res = {}
    for name, env in (("cache", {}), ("nocache", {"R2S_VOL_CACHE": "0"}), ("debug", {"R2S_DEBUG_SYNC": "1"})):
        for k, v in env.items():
            monkeypatch.setenv(k, v)
        mesh = r2s.Mesh(X, IEN, rho)
        grid = r2s.Grid(X.min(0), X.max(0), 48, 3)
        rn = r2s.DenseInNodes(mesh, rho)
        res[name] = _run_pipeline(r2s, mesh, grid, rn)
        mesh.ctx.close()
        for k in env:
            monkeypatch.delenv(k)
    for name in ("nocache", "debug"):
        assert res[name][2].th == res["cache"][2].th and res[name][2].volume == res["cache"][2].volume and res[name][2].bisections == res["cache"][2].bisections
        assert np.array_equal(res[name][0], res["cache"][0]) and np.array_equal(res[name][1], res["cache"][1])
    # a 400^3-cell field on which every cell is cut and the fixed-point sum exceeds 2^64 (tests/test_volume_exact.py), approximation mode
    from test_volume_exact import rbf_on_grid, wrap_field
    f, n = wrap_field(400), 400
    big = {}
    for name, env in (("cache", {}), ("nocache", {"R2S_VOL_CACHE": "0"})):
        for k, v in env.items():
            monkeypatch.setenv(k, v)
        ctx = r2s.Context()
        fine, th, vol, rep, _ = rbf_on_grid(r2s, ctx, f, [n, n, n], 1.0, 1, False, 0.5 * n ** 3)
        big[name] = (fine, th, vol, rep.bisections)
        ctx.close()
        for k in env:
            monkeypatch.delenv(k)
    assert big["nocache"][1:] == big["cache"][1:] and np.array_equal(big["nocache"][0], big["cache"][0])
