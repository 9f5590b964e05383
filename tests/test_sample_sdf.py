"""GPU tests of the sampler of the continuous smoothed SDF (csrc/r2s_sample.cu): bit equality with the host build (tests/host/sample_host.cpp)
given the weights the device holds, lattice against points, lattice against the resident fine_sdf, order and chunk independence, gradient
direction, several slabs, errors."""
import ctypes as C

import numpy as np
import pytest

import sample_ref as ref
from test_isosurface import _device_lists, _pipeline_case
from test_sample_host import _points
from test_volume_exact import CUTS, fine_eval_input, rbf_on_grid

pytestmark = pytest.mark.gpu
U = 2.0 ** -24


def _run_pipeline(r2s, case, devices=None):
    X, IEN, rho, opts = _pipeline_case(r2s, case)
    smooth = 2 if opts.rbf_grid == "fine" else 1
    mesh = r2s.Mesh(X, IEN, rho, element_type=opts.element_type, devices=devices)
    grid = r2s.noninteractive_sdf_grid_setup(mesh) if opts.sdf_grid_setup == "automatic" else r2s.Grid(X.min(0), X.max(0), int(np.floor(np.max(X.max(0) - X.min(0)) / opts.grid_step)), 3)
    rn = r2s.DenseInNodes(mesh, rho)
    rho_t = opts.threshold_density if opts.threshold_density is not None else r2s.find_threshold_for_volume(mesh, rn)
    if devices is None:
        d, _ = r2s.evalDistances(mesh, grid, None, rn, rho_t, want_xp=False)
        s = r2s.Sign_Detection(mesh, grid, None, rn, rho_t)
        sdf = d * s
        if opts.remove_artifacts:
            r2s.remove_sdf_artifacts(sdf, grid, 0.0, opts.artifact_min_component_ratio, mesh=mesh)
        fine, fg = r2s.RBFs_smoothing(mesh, sdf, grid, opts.rbf_interp, smooth, case)
    else:
        mesh._use_grid(grid)
        m = mesh.multi
        p = r2s.Params(); m.lib.r2s_default_params(C.byref(p))
        p.rho_t, p.smooth, p.rbf_interp, p.remove_artifacts, p.artifact_min_ratio = rho_t, smooth, int(opts.rbf_interp), int(opts.remove_artifacts), opts.artifact_min_component_ratio
        p.target_volume, p.final_volume = mesh.V_frac * mesh.V_domain, 0
        fine = np.empty(int(np.prod([int(v) * smooth + 1 for v in grid.N])), np.float32); sdf = np.empty(grid.ngp); rep = r2s.Report()
        m.check(m.lib.r2s_multi_pipeline(m.h, C.byref(p), rn.ctypes.data_as(C.c_void_p), sdf.ctypes.data_as(C.c_void_p), fine.ctypes.data_as(C.c_void_p), C.byref(rep)))
        fine = fine.reshape([int(v) * smooth + 1 for v in grid.N][::-1])
    return mesh, grid, smooth, fine


def _host_field(r2s, mesh, grid):
    w, th = r2s.rbf_weights(mesh)
    return ref.Field(w, grid.AABB_min, grid.AABB_max, grid.cell_size, 1e-3, th)


def _check_points(r2s, mesh, F, P):
    v, g = r2s.sample_sdf(mesh, P, gradient=True)
    hv, hg = F.host(P, gradient=True)
    assert np.array_equal(v, hv) and np.array_equal(g, hg)
    assert np.array_equal(r2s.sample_sdf(mesh, P), v)
    return v, g


def _lattice_points(o, h, shape):
    o32, h32 = np.float32(o), np.float32(h)
    ax = [(o32[d] + np.arange(shape[d], dtype=np.float32) * h32[d]).astype(np.float32) for d in range(3)]
    kk, jj, ii = np.meshgrid(np.arange(shape[2]), np.arange(shape[1]), np.arange(shape[0]), indexing="ij")
    return np.stack([ax[0][ii.ravel()], ax[1][jj.ravel()], ax[2][kk.ravel()]], 1).astype(np.float64)


@pytest.mark.parametrize("case", ["sphere", "cantilever", "simp24", "sphere_same"])
def test_pipeline_field_equals_host_build(r2s, case):
    mesh, grid, smooth, fine = _run_pipeline(r2s, case)
    F = _host_field(r2s, mesh, grid)
    rng = np.random.default_rng(3)
    P = _points(F, rng, n_random=20000)
    v, g = _check_points(r2s, mesh, F, P)
    # lattice == points at the documented lattice formula; an arbitrary lattice off the grid, crossing the border
    o, h, shape = grid.AABB_min - 1.3 * grid.cell_size, np.array([0.31, 0.29, 0.43]) * grid.cell_size, (37, 41, 29)
    lat = r2s.sample_sdf_lattice(mesh, o, h, shape)
    assert np.array_equal(lat.ravel(), F.host(_lattice_points(o, h, shape)))
    # lattice at origin AABB_min, spacing cell / smooth against the resident fine_sdf, at sampled fine points: the two definitions differ
    # by the round-off of each (sampler: (n + K) 2^-24 (A + |th|), k_fine_eval: (n + 2) 2^-24 (A + |th|)) and by sum |w| |phi - exp(-m)|,
    # phi from the Float32 offsets, m the ideal squared offset of k_fine_eval's table
    lat = r2s.sample_sdf_lattice(mesh, grid.AABB_min, [grid.cell_size / smooth] * 3, fine.shape[::-1])
    assert lat.shape == fine.shape
    idx = rng.integers(0, np.array(fine.shape), (300, 3))
    kap = float(F.kappa)
    for k, j, i in idx:
        p32 = (np.float32(grid.AABB_min) + np.float32([i, j, k]) * np.float32(grid.cell_size / smooth)).astype(np.float32)
        taps = F.taps(p32.astype(np.float64))
        A, D = 0.0, 0.0
        for ci, cj, ck, e in taps:
            e64 = e.astype(np.float64)
            m = (ci - i / smooth) ** 2 + (cj - j / smooth) ** 2 + (ck - k / smooth) ** 2
            wv = abs(float(F.w[ck, cj, ci]))
            A += wv * np.exp(-m); D += wv * abs(np.exp(-kap * float(e64 @ e64)) - np.exp(-m))
        bound = 2 * (len(taps) + ref.K_ROUNDOFF) * U * (1.01 * A + abs(float(F.th))) + D
        assert abs(float(lat[k, j, i]) - float(fine[k, j, i])) <= bound, (k, j, i, lat[k, j, i], fine[k, j, i], bound)
    if case == "sphere":
        # gradient direction: at the surface's vertices the gradient points into the solid, against the outward facet normals
        V, T = r2s.isosurface(mesh)
        vv, gv = r2s.sample_sdf(mesh, V.astype(np.float64), gradient=True)
        nrm = np.cross(V[T[:, 1]] - V[T[:, 0]], V[T[:, 2]] - V[T[:, 0]]).astype(np.float64)
        gt = gv[T].astype(np.float64).mean(1)
        frac = float(np.mean((gt * nrm).sum(1) < 0))
        print("sphere: %d triangles, gradient against the outward normal at %.4f of them" % (len(T), frac))
        assert frac >= 0.99
    mesh.close()


@pytest.mark.parametrize("cut", CUTS)
@pytest.mark.parametrize("interp", [False, True])
def test_smoothing_field_equals_host_build(r2s, cut, interp):
    """r2s_rbf_smoothing at the three cut-offs on grids that are no multiple of any tile, both modes"""
    ctx = r2s.Context()
    N = (33, 7, 17)
    rng = np.random.default_rng(int(cut * 1e6) + interp)
    sdf = fine_eval_input(tuple(v + 1 for v in N), rng)
    fine, tho, vol, rep, grid = rbf_on_grid(r2s, ctx, sdf, N, 0.7, 2, interp, 0.3 * np.prod(N) * 0.343, rbf_cut=cut)
    w = np.empty((N[2] + 1, N[1] + 1, N[0] + 1), np.float32); th = C.c_float()
    ctx.check(ctx.lib.r2s_download_rbf_weights(ctx.h, w.ctypes.data_as(C.c_void_p), C.byref(th)))
    assert th.value == np.float32(tho)
    F = ref.Field(w, grid.AABB_min, grid.AABB_max, 0.7, cut, th.value)
    P = _points(F, rng, n_random=5000)
    n = len(P)
    v = np.empty(n, np.float32); g = np.empty((n, 3), np.float32)
    p = np.ascontiguousarray(P)
    ctx.check(ctx.lib.r2s_sample_sdf(ctx.h, p.ctypes.data_as(C.c_void_p), n, v.ctypes.data_as(C.c_void_p), g.ctypes.data_as(C.c_void_p)))
    hv, hg = F.host(P, gradient=True)
    assert np.array_equal(v, hv) and np.array_equal(g, hg)
    if not interp:      # approximation mode: the weights are the processed Float32 SDF
        s = sdf.astype(np.float32); fin = np.abs(s) < 1e9
        assert np.array_equal(w, np.where(fin, s, np.sign(s) * np.abs(s[fin]).max()).astype(np.float32))
    ctx.close()


def test_order_and_chunk_independence(r2s):
    mesh, grid, smooth, fine = _run_pipeline(r2s, "sphere_same")
    F = _host_field(r2s, mesh, grid)
    rng = np.random.default_rng(11)
    n = (1 << 24) + 3
    P = rng.uniform(grid.AABB_min - 2 * grid.cell_size, grid.AABB_max + 2 * grid.cell_size, (n, 3))
    v, g = r2s.sample_sdf(mesh, P, gradient=True)
    perm = rng.permutation(n)
    vp, gp = r2s.sample_sdf(mesh, P[perm], gradient=True)
    assert np.array_equal(vp, v[perm]) and np.array_equal(gp, g[perm])
    for a, b in [(0, 5), (5, (1 << 22) + 7), ((1 << 22) + 7, n)]:
        vs, gs = r2s.sample_sdf(mesh, P[a:b], gradient=True)
        assert np.array_equal(vs, v[a:b]) and np.array_equal(gs, g[a:b])
    sel = rng.integers(0, n, 20000)
    hv, hg = F.host(P[sel], gradient=True)
    assert np.array_equal(v[sel], hv) and np.array_equal(g[sel], hg)
    e = r2s.sample_sdf(mesh, np.zeros((0, 3)))
    assert e.shape == (0,)
    mesh.close()


@pytest.mark.parametrize("case", ["simp24_approx", "simp24"])
def test_multi_slabs(r2s, case):
    mesh1, grid, smooth, fine1 = _run_pipeline(r2s, case)
    rng = np.random.default_rng(5)
    F1 = _host_field(r2s, mesh1, grid)
    P0 = _points(F1, rng, n_random=20000)
    o, h, shape = grid.AABB_min - 0.7 * grid.cell_size, [grid.cell_size / 3] * 3, (50, 47, int(grid.N[2]) * 3 + 6)
    v1, g1 = r2s.sample_sdf(mesh1, P0, gradient=True)
    lat1 = r2s.sample_sdf_lattice(mesh1, o, h, shape)
    for devs in _device_lists():
        mesh, _, _, fine = _run_pipeline(r2s, case, devices=devs)
        cuts = mesh.multi.slab_planes()
        # points on and next to every slab cut (the floor plane decides the slab)
        zc = []
        for k in cuts[1:-1]:
            z = F1.C[2][k]
            zc += [z, np.nextafter(z, np.float32(-np.inf)), np.nextafter(z, np.float32(np.inf)), z - 0.5 * grid.cell_size, z + 0.5 * grid.cell_size]
        Pc = np.stack([rng.uniform(grid.AABB_min[0], grid.AABB_max[0], len(zc)), rng.uniform(grid.AABB_min[1], grid.AABB_max[1], len(zc)), np.array(zc, np.float64)], 1)
        P = np.concatenate([P0, Pc])
        F = _host_field(r2s, mesh, grid)
        v, g = _check_points(r2s, mesh, F, P)
        lat = r2s.sample_sdf_lattice(mesh, o, h, shape)
        assert np.array_equal(lat.ravel(), F.host(_lattice_points(o, h, shape)))
        if case.endswith("approx"):      # no CG: the weights are the same on every layout, so are the results
            assert np.array_equal(F.w, F1.w) and F.th == F1.th
            assert np.array_equal(v[:len(P0)], v1) and np.array_equal(g[:len(P0)], g1) and np.array_equal(lat, lat1)
        mesh.close()
    mesh1.close()


def test_errors(r2s):
    c = r2s.Context()
    v = np.empty(4, np.float32); P = np.zeros((4, 3))
    with pytest.raises(r2s.R2SError, match="r2s_set_grid|no smoothed field"):
        c.check(c.lib.r2s_sample_sdf(c.h, P.ctypes.data_as(C.c_void_p), 4, v.ctypes.data_as(C.c_void_p), None))
    N = (9, 8, 7)
    sdf = fine_eval_input(tuple(n + 1 for n in N), np.random.default_rng(1))
    with pytest.raises(r2s.R2SError, match="no smoothed field"):
        amin = np.zeros(3); amax = np.array(N, np.float64); Nn = np.array(N, np.int64)
        c.check(c.lib.r2s_set_grid(c.h, amin.ctypes.data_as(C.c_void_p), amax.ctypes.data_as(C.c_void_p), Nn.ctypes.data_as(C.c_void_p), 1.0))
        c.check(c.lib.r2s_sample_sdf(c.h, P.ctypes.data_as(C.c_void_p), 4, v.ctypes.data_as(C.c_void_p), None))
    rbf_on_grid(r2s, c, sdf, N, 1.0, 1, False, 100.0)
    c.check(c.lib.r2s_sample_sdf(c.h, P.ctypes.data_as(C.c_void_p), 4, v.ctypes.data_as(C.c_void_p), None))
    for bad in (np.nan, np.inf, -np.inf):
        Q = P.copy(); Q[2, 1] = bad
        with pytest.raises(r2s.R2SError, match="NaN or infinite"):
            c.check(c.lib.r2s_sample_sdf(c.h, Q.ctypes.data_as(C.c_void_p), 4, v.ctypes.data_as(C.c_void_p), None))
    with pytest.raises(r2s.R2SError, match="required"):
        c.check(c.lib.r2s_sample_sdf(c.h, None, 4, v.ctypes.data_as(C.c_void_p), None))
    with pytest.raises(r2s.R2SError, match="required"):
        c.check(c.lib.r2s_sample_sdf(c.h, P.ctypes.data_as(C.c_void_p), 4, None, None))
    c.check(c.lib.r2s_sample_sdf(c.h, None, 0, None, None))
    o = np.zeros(3); h = np.ones(3); out = np.empty(8, np.float32)
    for dims in ([0, 2, 2], [2, -1, 2], [2, 2, 0]):
        d = np.array(dims, np.int64)
        with pytest.raises(r2s.R2SError, match="dims must be >= 1"):
            c.check(c.lib.r2s_sample_sdf_lattice(c.h, o.ctypes.data_as(C.c_void_p), h.ctypes.data_as(C.c_void_p), d.ctypes.data_as(C.c_void_p), out.ctypes.data_as(C.c_void_p)))
    d = np.array([2, 2, 2], np.int64); hn = np.array([1.0, np.nan, 1.0])
    with pytest.raises(r2s.R2SError, match="NaN or infinite"):
        c.check(c.lib.r2s_sample_sdf_lattice(c.h, o.ctypes.data_as(C.c_void_p), hn.ctypes.data_as(C.c_void_p), d.ctypes.data_as(C.c_void_p), out.ctypes.data_as(C.c_void_p)))
    amin = np.zeros(3); amax = np.array(N, np.float64); Nn = np.array(N, np.int64)
    c.check(c.lib.r2s_set_grid(c.h, amin.ctypes.data_as(C.c_void_p), amax.ctypes.data_as(C.c_void_p), Nn.ctypes.data_as(C.c_void_p), 1.0))
    with pytest.raises(r2s.R2SError, match="no smoothed field"):      # a new grid drops the field
        c.check(c.lib.r2s_sample_sdf(c.h, P.ctypes.data_as(C.c_void_p), 4, v.ctypes.data_as(C.c_void_p), None))
    with pytest.raises(r2s.R2SError, match="no smoothed field"):
        c.check(c.lib.r2s_download_rbf_weights(c.h, None, C.byref(C.c_float())))
    c.close()
