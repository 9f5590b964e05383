"""GPU tests of evalDistances / Sign_Detection at arbitrary points (r2s_eval_distances_points, r2s_sign_detection_points; rule in
include/r2s.h): the grid's points passed as an array reproduce the grid path, edge-case point sets match the oracle's points functions,
the results are a function of the point alone, and a points call leaves the pipeline's resident results untouched."""
import ctypes as C

import numpy as np
import pytest

import oracle
import points_oracle
from points_cases import GRID_CASES, case, edge_points, grid_points

pytestmark = pytest.mark.gpu


def _mesh(r2s, X, IEN, rn, grid, is_tet):
    rho = rn[IEN - 1].mean(axis=1)
    mesh = r2s.Mesh(X, IEN, rho, element_type=r2s.TET4 if is_tet else r2s.HEX8)
    g = r2s.Grid(X.min(0), X.max(0), grid.nmax, 3)
    assert np.array_equal(g.AABB_min, grid.AABB_min) and np.array_equal(g.N, grid.N) and g.cell_size == grid.cell_size
    return mesh, g


def _grid_vs_points(r2s, mesh, g, rn, params):
    P = r2s.generateGridPoints(g)
    h = g.cell_size
    for rt, df in params:
        d, xp = r2s.evalDistances(mesh, g, None, rn, rt, delta_factor=df)
        pd, pxp = r2s.evalDistances(mesh, g, P, rn, rt, delta_factor=df)
        far = d > 1e9
        assert np.array_equal(pd > 1e9, far) and np.array_equal(pd[far], d[far])
        # the per-pair solvers are the grid path's xp kernels' arithmetic in another kernel; FMA contraction may differ in the last bit
        assert np.max(np.abs(pd - d)) <= 1e-11 * h
        assert np.max(np.abs(np.linalg.norm(P[~far] - pxp[~far], axis=1) - pd[~far]), initial=0.0) <= 1e-9 * h
        s = r2s.Sign_Detection(mesh, g, None, rn, rt)
        assert np.array_equal(r2s.Sign_Detection(mesh, g, P, rn, rt), s)
    return int(np.sum(pd == d)), pd.size


@pytest.mark.parametrize("name", GRID_CASES)
def test_grid_points_as_an_array_reproduce_the_grid_path(r2s, name):
    X, IEN, rn, grid, params, is_tet = case(name)
    mesh, g = _mesh(r2s, X, IEN, rn, grid, is_tet)
    eq, n = _grid_vs_points(r2s, mesh, g, rn, params)
    print("%s: %d of %d distances bit-equal to the grid path" % (name, eq, n))
    mesh.close()


def test_lattice_signs_with_the_general_grid_kernel(r2s, monkeypatch):
    """R2S_SIGN_LATTICE=0: the grid path takes the sorted-list sign kernel; the points path gives the same bits."""
    monkeypatch.setenv("R2S_SIGN_LATTICE", "0")
    X, IEN, rn, grid, params, is_tet = case("graded_lattice_hex8")
    mesh, g = _mesh(r2s, X, IEN, rn, grid, is_tet)
    P = r2s.generateGridPoints(g)
    for rt, _ in params:
        assert np.array_equal(r2s.Sign_Detection(mesh, g, P, rn, rt), r2s.Sign_Detection(mesh, g, None, rn, rt))
    mesh.close()


@pytest.mark.parametrize("name", ["simp", "graded_lattice_hex8", "chapadlo", "schlafli_tet4", "sphere5"])
def test_edge_case_points_against_the_oracle(r2s, name):
    X, IEN, rn, grid, params, is_tet = case(name)
    mesh, g = _mesh(r2s, X, IEN, rn, grid, is_tet)
    for rt, df in params:
        P = edge_points(X, IEN, grid, rn, rt)
        d, xp = r2s.evalDistances(mesh, g, P, rn, rt, delta_factor=df)
        od, oxp, _ = points_oracle.eval_distances_points(X, IEN, grid, rn, rt, P, df)
        far = od > 1e9
        assert np.array_equal(d > 1e9, far) and np.array_equal(d[far], od[far]) and not xp[far].any()
        assert np.max(np.abs(d - od)) <= 1e-9 * g.cell_size
        s = r2s.Sign_Detection(mesh, g, P, rn, rt)
        os_ = points_oracle.sign_detection_points(X, IEN, grid, rn, rt, P)
        assert np.array_equal(s, os_), "signs differ at %d points" % int((s != os_).sum())
        assert (~far).sum() > 100 and (s > 0).sum() > 10
    mesh.close()


def test_consistency_xp_prune_order_and_slab(r2s, monkeypatch):
    X, IEN, rn, grid, params, _ = case("simp")
    rt, df = params[0]
    mesh, g = _mesh(r2s, X, IEN, rn, grid, False)
    rng = np.random.default_rng(11)
    n = (1 << 22) + 3
    base = edge_points(X, IEN, grid, rn, rt)
    P = np.concatenate([base, rng.uniform(g.AABB_min - g.cell_size, g.AABB_max + g.cell_size, size=(n - base.shape[0], 3))])
    d, xp = r2s.evalDistances(mesh, g, P, rn, rt, delta_factor=df)
    rep = mesh.ctx.report()
    assert rep.n_pairs > 0 and rep.n_pairs_pruned > 0
    d0, _ = r2s.evalDistances(mesh, g, P, rn, rt, delta_factor=df, want_xp=False)
    assert np.array_equal(d0, d)
    s = r2s.Sign_Detection(mesh, g, P, rn, rt)
    for seed in (1, 2):
        perm = np.random.default_rng(seed).permutation(n)
        dp, xpp = r2s.evalDistances(mesh, g, P[perm], rn, rt, delta_factor=df)
        assert np.array_equal(dp, d[perm]) and np.array_equal(xpp, xp[perm])
        assert np.array_equal(r2s.Sign_Detection(mesh, g, P[perm], rn, rt), s[perm])
    Q = P[: 1 << 16]
    c = mesh.ctx
    nz = int(g.N[2]) + 1
    c.check(c.lib.r2s_set_slab(c.h, nz // 3, 2 * nz // 3))
    ds, xps = r2s.evalDistances(mesh, g, Q, rn, rt, delta_factor=df)
    assert np.array_equal(ds, d[: 1 << 16]) and np.array_equal(xps, xp[: 1 << 16])
    assert np.array_equal(r2s.Sign_Detection(mesh, g, Q, rn, rt), s[: 1 << 16])
    mesh.close()
    monkeypatch.setenv("R2S_PROJ_PRUNE", "0")
    mesh0, g0 = _mesh(r2s, X, IEN, rn, grid, False)
    dn, xpn = r2s.evalDistances(mesh0, g0, Q, rn, rt, delta_factor=df)
    assert mesh0.ctx.report().n_pairs_pruned == 0
    assert np.array_equal(dn, d[: 1 << 16]) and np.array_equal(xpn, xp[: 1 << 16])
    mesh0.close()


def test_points_calls_leave_resident_results_untouched(r2s):
    X, IEN, rn, grid, params, _ = case("simp")
    rt = params[0][0]
    mesh, g = _mesh(r2s, X, IEN, rn, grid, False)
    mesh._use_grid(g)
    c = mesh.ctx
    p = r2s.Params(); c.lib.r2s_default_params(C.byref(p))
    p.rho_t, p.smooth, p.rbf_interp, p.remove_artifacts = rt, 2, 1, 1
    p.target_volume, p.final_volume = mesh.V_frac * mesh.V_domain, 1
    fd = [int(v) * 2 + 1 for v in g.N]
    probe = edge_points(X, IEN, grid, rn, rt, n=300)

    def state():
        sdf = np.empty(g.ngp); c.check(c.lib.r2s_download_sdf(c.h, sdf.ctypes.data_as(C.c_void_p)))
        fine = np.empty(fd[0] * fd[1] * fd[2], dtype=np.float32); c.check(c.lib.r2s_download_fine_sdf(c.h, fine.ctypes.data_as(C.c_void_p)))
        V, T = r2s.isosurface(mesh, 0.0)
        w, th = r2s.rbf_weights(mesh)
        return [sdf, fine, r2s.sample_sdf(mesh, probe), V, T, w, np.array([th])]

    def pipeline():
        rep = r2s.Report()
        c.check(c.lib.r2s_upload_nodal_densities(c.h, rn.ctypes.data_as(C.c_void_p)))
        c.check(c.lib.r2s_pipeline_resident(c.h, C.byref(p), C.byref(rep)))
        return state()

    before = pipeline()
    other = np.clip(rn[::-1].copy(), 0.0, 1.0)      # a different density field
    P = r2s.generateGridPoints(g)[::7]
    r2s.evalDistances(mesh, g, P, other, rt)
    r2s.Sign_Detection(mesh, g, P, other, rt)
    after = state()
    for a, b in zip(before, after):
        assert np.array_equal(a, b)
    c.check(c.lib.r2s_pipeline_resident(c.h, C.byref(p), C.byref(r2s.Report())))      # resident rho_n is still the uploaded one
    for a, b in zip(before, state()):
        assert np.array_equal(a, b)
    mesh.close()


def test_invalid_inputs_are_rejected(r2s):
    X, IEN, rn, grid, params, _ = case("sphere")
    mesh, g = _mesh(r2s, X, IEN, rn, grid, False)
    rt = params[0][0]
    for bad in (np.nan, np.inf, -np.inf):
        P = np.zeros((5, 3)); P[3, 1] = bad
        with pytest.raises(r2s.R2SError):
            r2s.evalDistances(mesh, g, P, rn, rt)
        with pytest.raises(r2s.R2SError):
            r2s.Sign_Detection(mesh, g, P, rn, rt)
    c = mesh.ctx
    out = np.empty(4)
    with pytest.raises(r2s.R2SError):
        c.check(c.lib.r2s_eval_distances_points(c.h, rn.ctypes.data_as(C.c_void_p), rt, 1.1, None, 4, out.ctypes.data_as(C.c_void_p), None))
    with pytest.raises(r2s.R2SError):
        c.check(c.lib.r2s_sign_detection_points(c.h, rn.ctypes.data_as(C.c_void_p), rt, None, 4, out.ctypes.data_as(C.c_void_p)))
    mesh.close()
    bare = r2s.Context(0)
    P = np.zeros((2, 3))
    with pytest.raises(r2s.R2SError):      # no mesh, no grid
        bare.check(bare.lib.r2s_eval_distances_points(bare.h, rn.ctypes.data_as(C.c_void_p), rt, 1.1, P.ctypes.data_as(C.c_void_p), 2, out.ctypes.data_as(C.c_void_p), None))
    with pytest.raises(r2s.R2SError):
        bare.check(bare.lib.r2s_sign_detection_points(bare.h, rn.ctypes.data_as(C.c_void_p), rt, P.ctypes.data_as(C.c_void_p), 2, out.ctypes.data_as(C.c_void_p)))
    m2 = r2s.Mesh(X, IEN, rn[IEN - 1].mean(axis=1))      # mesh, no grid
    with pytest.raises(r2s.R2SError):
        m2.ctx.check(m2.ctx.lib.r2s_eval_distances_points(m2.ctx.h, rn.ctypes.data_as(C.c_void_p), rt, 1.1, P.ctypes.data_as(C.c_void_p), 2, out.ctypes.data_as(C.c_void_p), None))
    m2.close()
    bare.close()
