"""GPU tests of the zero surface of the continuous field on a lattice (r2s_isosurface_lattice, csrc/r2s_surf.cu + r2s_snap.cuh): triangles
equal to marching cubes on the sampled lattice field, vertices equal to the host replay of the search (tests/host/snap_host.cpp), vertices on
the zero set within the Float32 evaluation bound, chunk-size independence, several slabs, mesh properties, residency and errors."""
import ctypes as C
import os

import numpy as np
import pytest

import isosurface_ref as mref
import sample_ref
import snap_ref as ref
from test_isosurface import _device_lists
from test_sample_sdf import _host_field, _run_pipeline

pytestmark = pytest.mark.gpu
U = 2.0 ** -24


def _lattices(grid, smooth):
    """(name, origin, spacing, shape, isotropic): the fine lattice, a 2x refinement of it, an anisotropic one, one cutting the mesh box"""
    amin, amax, c = np.asarray(grid.AABB_min), np.asarray(grid.AABB_max), grid.cell_size
    N = np.array([int(v) for v in grid.N])
    out = [("fine", amin, [c / smooth] * 3, tuple(int(v) for v in N * smooth + 1), True),
           ("refine2", amin, [c / (2 * smooth)] * 3, tuple(int(v) for v in N * 2 * smooth + 1), True)]
    h = np.array([0.37, 0.29, 0.45]) * c
    o = amin - 0.6 * c
    out.append(("aniso", o, h, tuple(int(v) for v in np.ceil((amax + 0.6 * c - o) / h)), False))
    o = amin + 0.3 * (amax - amin)
    out.append(("cut", o, [c / 3] * 3, tuple(int(v) for v in np.ceil(0.55 * (amax - amin) / (c / 3))), True))
    return out


def _composition(r2s, mesh, o, h, shape, iso, ctx):
    lat = r2s.sample_sdf_lattice(mesh, o, h, shape)
    V, T = r2s.isosurface_from_sdf(lat, o, h, iso, ctx=ctx)
    return lat, V, T


def _zero_set_stats(F, V, Vlin, edges, tr, ev, iso, sel, h):
    """|f64 - iso| at snapped vertices against B = 2.2 eps + 0.55 |df/dx_d| ulp(x), eps = (n + K) 2^-24 (sum |w phi| + |th|) the sampler's
    round-off bound at the vertex (sample_ref.K_ROUNDOFF).  The vertex x is the end of an adjacent-float bracket (lo, hi) whose Float32
    values straddle iso with the smaller residual: |f32(x) - iso| <= |f32(lo) - f32(hi)| / 2 <= (eps(lo) + eps(hi) + |f64(lo) - f64(hi)|) / 2,
    and |f64 - f32| <= eps at x itself.  Skipped (and counted): searches stopped by the cap, and brackets whose ends have different tap
    sets (a tap crossing the cut radius between two adjacent floats makes f jump by w exp(-kappa t2))."""
    worst, skipped, lin = 0.0, 0, []
    for q in sel:
        ax = int(edges[q, 3])
        lo, hi = tr[q, 0], tr[q, 1]
        p = V[q].astype(np.float64)
        pl, ph = p.copy(), p.copy(); pl[ax] = lo; ph[ax] = hi
        vl = F.float64(Vlin[q].astype(np.float64))
        lin.append(abs(vl[0] - float(iso)) / h)
        if ev[q] >= ref.max_evals() or len(F.taps(pl)) != len(F.taps(ph)):
            skipped += 1
            continue
        val, grad, A, n = F.float64(p)
        eps = (n + sample_ref.K_ROUNDOFF) * U * (1.01 * A + abs(float(F.th)))
        ulp = float(np.spacing(np.abs(np.float32(p[ax]))))
        B = 2.2 * eps + 0.55 * abs(grad[ax]) * ulp
        r = abs(val - float(iso))
        assert r <= B, (q, V[q], r, B, eps, grad)
        worst = max(worst, r / B)
    return worst, skipped, np.array(lin)


@pytest.mark.parametrize("case", ["sphere", "sphere_same", "simp24", "cantilever"])
def test_lattice_surface(r2s, case, tmp_path):
    mesh, grid, smooth, fine = _run_pipeline(r2s, case)
    F = _host_field(r2s, mesh, grid)
    w0, th0 = r2s.rbf_weights(mesh)
    ctx = r2s.Context()
    rng = np.random.default_rng(len(case))
    for name, o, h, shape, iso_tropic in _lattices(grid, smooth):
        for iso in ([0.0, 0.17 * grid.cell_size] if name == "fine" else [0.0]):
            iso = np.float32(iso)
            V, T = r2s.isosurface_lattice(mesh, o, h, shape, iso)
            lat, Vlin, Tlin = _composition(r2s, mesh, o, h, shape, iso, ctx)
            # 1. triangles and vertex count of marching cubes on the sampled lattice field
            assert len(T) > 50 and np.array_equal(T, Tlin) and len(V) == len(Vlin), (name, len(V), len(Vlin))
            # 2. vertices: the host replay of the search on the downloaded weights
            E = ref.crossing_edges(lat, iso)
            Vh, tr, ev = ref.lattice_vertices(F, o, h, E, iso)
            assert np.array_equal(V, Vh), name
            # 3. on the zero set, within the Float32 evaluation bound
            sel = rng.choice(len(V), min(len(V), 100), replace=False)
            hmin = float(np.min(h))
            worst, skipped, lin = _zero_set_stats(F, V, Vlin, E, tr, ev, iso, sel, hmin)
            print("%s %s iso=%g: nv=%d nt=%d, evaluations mean %.2f max %d capped %d; snapped |f-iso| <= %.3f of the bound (%d skipped); "
                  "linear vertices |f-iso|/h median %.2e max %.2e" % (case, name, iso, len(V), len(T), ev.mean(), ev.max(), int((ev >= ref.max_evals()).sum()),
                                                                     worst, skipped, np.median(lin), lin.max()))
            # 6. mesh properties
            bad = mref.unpaired_edges(T)
            assert mref.on_boundary_face(V, T, bad, np.float32(o), np.float32(h), lat.shape).all() if len(bad) else True
            border_negative = all((b < iso).all() for b in (lat[0], lat[-1], lat[:, 0], lat[:, -1], lat[:, :, 0], lat[:, :, -1]))
            if iso_tropic and border_negative:
                assert len(bad) == 0
                # both approximate the volume of {f >= iso} at second order in the lattice step (divergence volume of the snapped surface,
                # the detailed quadrature of the same lattice field): a few per mille for these parts, 5 % leaves room for thin members
                vol = mref.divergence_volume(V, T)
                qv = r2s.calculate_volume_from_sdf(lat, float(h[0]), float(iso), ctx=ctx)
                qv = qv[0] if isinstance(qv, tuple) else qv
                print("%s %s: divergence volume %.6g, quadrature volume %.6g" % (case, name, vol, qv))
                assert abs(vol - qv) <= 0.05 * abs(qv), (vol, qv)
    # export round trip through the lattice path
    o, h, shape = _lattices(grid, smooth)[1][1:4]
    V, T = r2s.isosurface_lattice(mesh, o, h, shape)
    r2s.export_isosurface(mesh, str(tmp_path / "s.ply"), lattice=(o, h, shape))
    r2s.export_isosurface(mesh, str(tmp_path / "s.stl"), lattice=(o, h, shape))
    V2, T2 = r2s.read_ply(str(tmp_path / "s.ply"))
    assert np.array_equal(V2, V) and np.array_equal(T2, T)
    _, P = r2s.read_stl(str(tmp_path / "s.stl"))
    assert np.array_equal(P, V[T])
    # 7. residency: the weights, th and fine_sdf are as the pipeline left them
    w1, th1 = r2s.rbf_weights(mesh)
    assert np.array_equal(w0, w1) and th0 == th1
    p = r2s.export_device_result_to_vti(mesh, str(tmp_path / "fine"), "distance", fine=True)
    assert np.array_equal(r2s.read_vti(p)[4], fine)
    ctx.close()
    mesh.close()


def test_chunk_independence(r2s):
    """R2S_SURF_PLANES=3 against the default chunking (two chunks of the 1 GiB budget on this lattice): the same mesh bit for bit"""
    mesh, grid, smooth, fine = _run_pipeline(r2s, "sphere_same")
    amin, amax = np.asarray(grid.AABB_min), np.asarray(grid.AABB_max)
    shape = (700, 700, 600)
    o, h = amin, (amax - amin) / (np.array(shape) - 1)
    assert (1 << 28) // (shape[0] * shape[1]) - 2 < shape[2]      # the default chunk holds fewer planes than the lattice
    V, T = r2s.isosurface_lattice(mesh, o, h, shape)
    w, th = r2s.rbf_weights(mesh)
    os.environ["R2S_SURF_PLANES"] = "3"      # read by r2s_create: the next mesh's context
    try:
        mesh3, _, _, _ = _run_pipeline(r2s, "sphere_same")
    finally:
        os.environ.pop("R2S_SURF_PLANES", None)
    w3, th3 = r2s.rbf_weights(mesh3)
    assert np.array_equal(w, w3) and th == th3
    V3, T3 = r2s.isosurface_lattice(mesh3, o, h, shape)
    print("chunk independence: nv=%d nt=%d" % (len(V), len(T)))
    assert len(T) > 10 ** 5 and np.array_equal(V, V3) and np.array_equal(T, T3)
    # a small lattice through many 3-plane chunks against the host replay
    o2, h2, s2 = amin, [grid.cell_size / 2] * 3, tuple(int(v) * 2 + 1 for v in grid.N)
    V3, T3 = r2s.isosurface_lattice(mesh3, o2, h2, s2)
    V1, T1 = r2s.isosurface_lattice(mesh, o2, h2, s2)
    assert np.array_equal(V1, V3) and np.array_equal(T1, T3)
    mesh3.close()
    mesh.close()


@pytest.mark.parametrize("case", ["simp24_approx", "simp24"])
def test_multi_slabs(r2s, case, tmp_path):
    mesh1, grid, smooth, fine1 = _run_pipeline(r2s, case)
    c = grid.cell_size
    lats = [(grid.AABB_min, [c / 2] * 3, tuple(int(v) * 2 + 1 for v in grid.N)),
            (np.asarray(grid.AABB_min) - 0.7 * c, [c / 3, c / 3, 0.45 * c], (50, 47, int(int(grid.N[2]) / 0.45) + 4))]
    ref1 = [r2s.isosurface_lattice(mesh1, o, h, s) for o, h, s in lats]
    ctx = r2s.Context()
    for devs in _device_lists():
        mesh, _, _, _ = _run_pipeline(r2s, case, devices=devs)
        F = _host_field(r2s, mesh, grid)
        for (o, h, s), (V1, T1) in zip(lats, ref1):
            V, T = r2s.isosurface_lattice(mesh, o, h, s)
            lat, _, Tl = _composition(r2s, mesh, o, h, s, 0.0, ctx)
            Vh, _, _ = ref.lattice_vertices(F, o, h, ref.crossing_edges(lat, 0.0), 0.0)
            assert np.array_equal(T, Tl) and np.array_equal(V, Vh), devs      # each layout's mesh is the host replay of its own weights
            if case.endswith("approx"):      # no CG: the weights are the same on every layout, so is the mesh
                assert np.array_equal(V, V1) and np.array_equal(T, T1), devs
        o, h, s = lats[0]
        r2s.export_isosurface(mesh, str(tmp_path / "m.ply"), lattice=(o, h, s))
        V2, T2 = r2s.read_ply(str(tmp_path / "m.ply"))
        assert np.array_equal(V2, r2s.isosurface_lattice(mesh, o, h, s)[0]) and len(T2) > 0
        mesh.close()
    ctx.close()
    mesh1.close()


def test_errors(r2s):
    c = r2s.Context()
    o = np.zeros(3); h = np.ones(3); d = np.array([4, 4, 4], np.int64)
    nv, nt = C.c_int64(), C.c_int64()

    def call(ctx, o, h, d, iso=0.0):
        ctx.check(ctx.lib.r2s_isosurface_lattice(ctx.h, _p(o), _p(h), _p(d), iso, C.byref(nv), C.byref(nt)))

    def _p(a):
        return np.ascontiguousarray(a).ctypes.data_as(C.c_void_p)
    with pytest.raises(r2s.R2SError, match="r2s_set_grid|no smoothed field"):
        call(c, o, h, d)
    c.close()
    mesh, grid, smooth, fine = _run_pipeline(r2s, "sphere_same")
    mc = mesh.ctx
    w0, th0 = r2s.rbf_weights(mesh)
    r2s.isosurface(mesh)
    for bad_o, bad_h in ((np.array([0.0, np.nan, 0.0]), h), (o, np.array([1.0, 1.0, np.inf])), (o, np.array([1.0, 1e38, 1.0]))):
        with pytest.raises(r2s.R2SError, match="NaN or infinite"):
            call(mc, bad_o, bad_h, np.array([4, 10, 4], np.int64))
    with pytest.raises(r2s.R2SError, match="no surface"):      # a failed extraction leaves no mesh behind
        mc.check(mc.lib.r2s_download_isosurface(mc.h, None, None))
    for dims in ([1, 4, 4], [4, 4, 1]):
        with pytest.raises(r2s.R2SError, match="at least 2 points"):
            call(mc, o, h, np.array(dims, np.int64))
    with pytest.raises(r2s.R2SError, match="2\\^31 or more cells"):
        call(mc, o, h, np.array([2049, 2049, 2049], np.int64))
    with pytest.raises(r2s.R2SError, match="iso must be finite"):
        call(mc, o, h, d, float("nan"))
    w1, th1 = r2s.rbf_weights(mesh)
    assert np.array_equal(w0, w1) and th0 == th1
    mesh.close()
    mesh2, _, _, _ = _run_pipeline(r2s, "simp24_approx", devices=[0, 0])
    with pytest.raises(r2s.R2SError, match="use r2s_multi_isosurface_lattice"):
        call(mesh2.multi.slab(1), grid.AABB_min, h, d)
    mesh2.close()
