"""GPU tests of the per-element volume fractions of the continuous smoothed SDF (r2s_element_volume_fractions, csrc/r2s_elemfrac.cu): the
fractions and element volumes equal the host replay (tests/host/elemfrac_host.cpp) on the downloaded weights bit for bit, on HEX8 pipelines
(sphere, SIMP, cantilever, the general hexes of chapadlo) and a TET4 one, at three quadrature orders and two isos; elements are skipped; the
volumes add up to the mesh volume; the solid volume against the fine grid's; several slabs; residency; errors."""
import ctypes as C

import numpy as np
import pytest

import elemfrac_ref as ef
from fixtures import load_mesh, schlafli_tet4
from test_isosurface import _device_lists
from test_sample_sdf import _host_field, _run_pipeline

pytestmark = pytest.mark.gpu
CASES = ["sphere", "sphere_same", "simp24", "cantilever", "chapadlo", "schlafli_tet4"]


def _pipeline(r2s, case):
    """(mesh, grid, smooth, fine) after the stage functions of rho2sdf() on one device"""
    if case not in ("chapadlo", "schlafli_tet4"):
        return _run_pipeline(r2s, case)
    if case == "chapadlo":
        X, IEN, rho = load_mesh("chapadlo")
        opts = r2s.Rho2sdfOptions(sdf_grid_setup="automatic", rbf_grid="fine")
    else:
        X, IEN, rn = schlafli_tet4(8, "radial")
        rho = rn[IEN - 1].mean(axis=1)
        opts = r2s.Rho2sdfOptions(threshold_density=0.5, sdf_grid_setup="automatic", rbf_grid="fine", element_type=r2s.TET4)
    mesh = r2s.Mesh(X, IEN, rho, element_type=opts.element_type)
    grid = r2s.noninteractive_sdf_grid_setup(mesh)
    rn = r2s.DenseInNodes(mesh, rho)
    rho_t = opts.threshold_density if opts.threshold_density is not None else r2s.find_threshold_for_volume(mesh, rn)
    d, _ = r2s.evalDistances(mesh, grid, None, rn, rho_t, want_xp=False)
    sdf = d * r2s.Sign_Detection(mesh, grid, None, rn, rho_t)
    r2s.remove_sdf_artifacts(sdf, grid, 0.0, opts.artifact_min_component_ratio, mesh=mesh)
    fine, _ = r2s.RBFs_smoothing(mesh, sdf, grid, opts.rbf_interp, 2, case)
    return mesh, grid, 2, fine


@pytest.mark.parametrize("case", CASES)
def test_equals_host_replay(r2s, case):
    mesh, grid, smooth, fine = _pipeline(r2s, case)
    F = _host_field(r2s, mesh, grid)
    IEN0 = mesh.IEN - 1
    rng = np.random.default_rng(1)
    for q in (1, 3, 15):
        # q = 15: a random third of the elements (at most 3000) is replayed, to keep the host side short
        sub = np.arange(mesh.nel) if q < 15 else np.sort(rng.choice(mesh.nel, min(mesh.nel, max(mesh.nel // 3, 1), 3000), replace=False))
        for iso in (0.0, 0.17 * grid.cell_size):
            iso = np.float32(iso)
            frac, vol, nev = r2s.element_volume_fractions(mesh, iso, q, return_volumes=True, stats=True)
            hf, hv, cls = ef.replay(F, mesh.X, IEN0[sub], q, iso)
            partial = int(((frac > 0) & (frac < 1)).sum())
            print("%s q=%d iso=%g: nel=%d, sampled %d (%.1f %%), host skips %d of the replayed, %d partial, solid %.6g of %.6g" %
                  (case, q, iso, mesh.nel, nev, 100.0 * nev / mesh.nel, int((cls != 0).sum()), partial, float((frac * vol).sum()), float(vol.sum())))
            assert np.array_equal(frac[sub], hf) and np.array_equal(vol[sub], hv), (q, iso)
            assert 0 < nev <= mesh.nel and (partial > 0 or q == 1)      # one point per element: every fraction is 0 or 1
            assert (frac[sub][cls == 1] == 1.0).all() and (frac[sub][cls == 2] == 0.0).all()
            assert np.array_equal(r2s.element_volume_fractions(mesh, iso, q), frac)
            if case.startswith("sphere"):
                assert nev < mesh.nel
        if q == 3 and mesh.nen == 8:      # the element volumes of calculate_mesh_volume's quadrature add up to its V_domain
            assert abs(vol.sum() - mesh.V_domain) <= 1e-12 * mesh.V_domain, (vol.sum(), mesh.V_domain)
        if mesh.nen == 4 and q > 1:       # the Duffy factor: each V_e is the tet's volume |det J| / 6 (one point is not exact for it)
            P = mesh.X[IEN0]
            v6 = np.abs(np.linalg.det(np.stack([P[:, 0] - P[:, 3], P[:, 1] - P[:, 3], P[:, 2] - P[:, 3]], 2))) / 6
            assert np.allclose(vol, v6, rtol=1e-13, atol=0)
    mesh.close()


def test_solid_volume_against_fine_grid(r2s):
    """On the sphere (:fine) the solid volume sum S_e of the continuous field against the fine grid's calculate_volume_from_sdf (the report's
    `volume`), and the convergence of the quadrature: the error at q = 20 against q = 32 is below the error at q = 5"""
    mesh, grid, smooth, fine = _pipeline(r2s, "sphere")
    vfine = float(r2s.calculate_volume_from_sdf(fine, r2s.FineGrid(grid, smooth)))
    S = {}
    for q in (5, 15, 20, 32):
        frac, vol = r2s.element_volume_fractions(mesh, 0.0, q, return_volumes=True)
        S[q] = float((frac * vol).sum())
    print("sphere: solid volume S(q) %s, fine grid %.8g, V_frac V_domain %.8g; |S(15) - fine| / fine = %.3g" %
          ({q: "%.10g" % v for q, v in S.items()}, vfine, mesh.V_frac * mesh.V_domain, abs(S[15] - vfine) / vfine))
    assert abs(S[20] - S[32]) < abs(S[5] - S[32])
    # the fine grid integrates the trilinear interpolant of the field sampled at cell / 2, the fractions the field itself, and only inside
    # the mesh: the two differ by the interpolation error of the surface position, O((cell / 2)^2 curvature) per unit area.  Measured on
    # this sphere (about 3 coarse cells across the solid, so the curvature term is large): 0.76 %; 1 % is the bound
    assert abs(S[15] - vfine) <= 0.01 * vfine
    mesh.close()


@pytest.mark.parametrize("case", ["sphere", "simp24"])
def test_multi_slabs(r2s, case):
    """2 and 3 slabs on one device: bit for bit the host replay on the multi handle's weights (and so any split of the elements)"""
    for devs in _device_lists():
        mesh, grid, _, _ = _run_pipeline(r2s, case, devices=devs)
        F = _host_field(r2s, mesh, grid)
        for q, iso in ((3, 0.0), (5, 0.17 * grid.cell_size)):
            iso = np.float32(iso)
            frac, vol, nev = r2s.element_volume_fractions(mesh, iso, q, return_volumes=True, stats=True)
            hf, hv, cls = ef.replay(F, mesh.X, mesh.IEN - 1, q, iso)
            print("%s %s q=%d: sampled %d of %d, host skips %d" % (case, devs, q, nev, mesh.nel, int((cls != 0).sum())))
            assert np.array_equal(frac, hf) and np.array_equal(vol, hv), devs
            assert 0 < nev <= mesh.nel
        mesh.close()


def test_residency(r2s, tmp_path):
    """the weights, th, sdf_dists, fine_sdf and a surface are as they were before the call"""
    mesh, grid, smooth, fine = _pipeline(r2s, "sphere_same")
    w0, th0 = r2s.rbf_weights(mesh)
    V0, T0 = r2s.isosurface(mesh)
    p0 = r2s.read_vti(r2s.export_device_result_to_vti(mesh, str(tmp_path / "d0"), fine=False))[4]
    r2s.element_volume_fractions(mesh, 0.0, 15)
    w1, th1 = r2s.rbf_weights(mesh)
    assert np.array_equal(w0, w1) and th0 == th1
    V1, T1 = np.empty_like(V0), np.empty_like(T0)
    mesh.ctx.check(mesh.ctx.lib.r2s_download_isosurface(mesh.ctx.h, V1.ctypes.data_as(C.c_void_p), T1.ctypes.data_as(C.c_void_p)))
    assert np.array_equal(V0, V1) and np.array_equal(T0, T1)
    assert np.array_equal(r2s.read_vti(r2s.export_device_result_to_vti(mesh, str(tmp_path / "f"), fine=True))[4], fine)
    assert np.array_equal(r2s.read_vti(r2s.export_device_result_to_vti(mesh, str(tmp_path / "d1"), fine=False))[4], p0)
    mesh.close()


def test_errors(r2s):
    X, IEN, rho = load_mesh("sphere")
    mesh = r2s.Mesh(X, IEN, rho)
    with pytest.raises(r2s.R2SError, match="r2s_set_grid|no smoothed field"):
        r2s.element_volume_fractions(mesh)
    mesh.close()
    c = r2s.Context()
    with pytest.raises(r2s.R2SError, match="r2s_set_mesh"):
        c.check(c.lib.r2s_element_volume_fractions(c.h, 0.0, 3, np.zeros(4).ctypes.data_as(C.c_void_p), None, None))
    c.close()
    mesh, grid, smooth, fine = _pipeline(r2s, "sphere_same")
    for q in (0, 33, -1):
        with pytest.raises(r2s.R2SError, match="quad_order must be in 1..32"):
            r2s.element_volume_fractions(mesh, 0.0, q)
    with pytest.raises(r2s.R2SError, match="iso must be finite"):
        r2s.element_volume_fractions(mesh, float("nan"))
    with pytest.raises(r2s.R2SError, match="iso must be finite"):
        r2s.element_volume_fractions(mesh, float("inf"))
    mc = mesh.ctx
    with pytest.raises(r2s.R2SError, match="fractions is required"):
        mc.check(mc.lib.r2s_element_volume_fractions(mc.h, 0.0, 3, None, None, None))
    assert r2s.element_volume_fractions(mesh, 0.0, 3).shape == (mesh.nel,)      # NULL volumes and n_evaluated are accepted
    mesh.close()
    mesh2, _, _, _ = _run_pipeline(r2s, "simp24_approx", devices=[0, 0])
    s1 = mesh2.multi.slab(1)
    with pytest.raises(r2s.R2SError, match="use r2s_multi_element_volume_fractions"):
        s1.check(s1.lib.r2s_element_volume_fractions(s1.h, 0.0, 3, np.zeros(mesh2.nel).ctypes.data_as(C.c_void_p), None, None))
    mesh2.close()
