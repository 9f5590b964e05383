"""GPU tests of the band extraction of the continuous field's zero surface (r2s_isosurface_band, csrc/r2s_band.cuh + r2s_surf.cu): the mesh
equals r2s_isosurface_lattice's bit for bit on every lattice that call accepts (V and T, single context, chunked, several slabs), blocks are
skipped, a lattice past 2^31 cells is extracted and checked on a window against marching cubes and the host replay of the search, STL / PLY
round trips, residency and the errors."""
import ctypes as C
import os

import numpy as np
import pytest

import isosurface_ref as mref
import snap_ref as ref
from test_isosurface import _device_lists
from test_isosurface_lattice import _lattices
from test_sample_sdf import _host_field, _run_pipeline

pytestmark = pytest.mark.gpu


@pytest.mark.parametrize("case", ["sphere", "sphere_same", "simp24", "cantilever"])
def test_band_equals_lattice(r2s, case, tmp_path):
    mesh, grid, smooth, fine = _run_pipeline(r2s, case)
    w0, th0 = r2s.rbf_weights(mesh)
    for name, o, h, shape, _ in _lattices(grid, smooth):
        for iso in (0.0, 0.17 * grid.cell_size):
            iso = np.float32(iso)
            V, T = r2s.isosurface_lattice(mesh, o, h, shape, iso)
            Vb, Tb, ns = r2s.isosurface_band(mesh, o, h, shape, iso, stats=True)
            npts = int(np.prod(shape))
            print("%s %s iso=%g: nv=%d nt=%d, sampled %d of %d points (%.1f %%)" % (case, name, iso, len(V), len(T), ns, npts, 100.0 * ns / npts))
            assert len(T) > 50 and np.array_equal(Vb, V) and np.array_equal(Tb, T), (name, iso, len(V), len(Vb))
            assert 0 < ns <= npts
    # export round trips through the band path
    o, h, shape = _lattices(grid, smooth)[1][1:4]
    V, T = r2s.isosurface_band(mesh, o, h, shape)
    r2s.export_isosurface(mesh, str(tmp_path / "s.ply"), band=(o, h, shape))
    r2s.export_isosurface(mesh, str(tmp_path / "s.stl"), band=(o, h, shape))
    V2, T2 = r2s.read_ply(str(tmp_path / "s.ply"))
    assert np.array_equal(V2, V) and np.array_equal(T2, T)
    _, P = r2s.read_stl(str(tmp_path / "s.stl"))
    assert np.array_equal(P, V[T])
    # residency: the weights, th and fine_sdf are as the pipeline left them
    w1, th1 = r2s.rbf_weights(mesh)
    assert np.array_equal(w0, w1) and th0 == th1
    p = r2s.export_device_result_to_vti(mesh, str(tmp_path / "fine"), "distance", fine=True)
    assert np.array_equal(r2s.read_vti(p)[4], fine)
    mesh.close()


def test_chunk_independence(r2s):
    """R2S_SURF_PLANES=3 against the default chunking: the same mesh bit for bit, equal to the dense call's"""
    mesh, grid, smooth, fine = _run_pipeline(r2s, "sphere_same")
    amin, amax = np.asarray(grid.AABB_min), np.asarray(grid.AABB_max)
    shape = (700, 700, 600)
    o, h = amin, (amax - amin) / (np.array(shape) - 1)
    V, T, ns = r2s.isosurface_band(mesh, o, h, shape, stats=True)
    assert ns < int(np.prod(shape))      # skipping happens
    os.environ["R2S_SURF_PLANES"] = "3"      # read by r2s_create: the next mesh's context
    try:
        mesh3, _, _, _ = _run_pipeline(r2s, "sphere_same")
    finally:
        os.environ.pop("R2S_SURF_PLANES", None)
    assert np.array_equal(r2s.rbf_weights(mesh)[0], r2s.rbf_weights(mesh3)[0])
    V3, T3 = r2s.isosurface_band(mesh3, o, h, shape)
    Vd, Td = r2s.isosurface_lattice(mesh3, o, h, shape)
    assert len(T) > 10 ** 5 and np.array_equal(V, V3) and np.array_equal(T, T3) and np.array_equal(V, Vd) and np.array_equal(T, Td)
    mesh3.close()
    mesh.close()


@pytest.mark.parametrize("case", ["simp24_approx", "simp24"])
def test_multi_slabs(r2s, case, tmp_path):
    _, grid, _, _ = _run_pipeline(r2s, case)
    c = grid.cell_size
    lats = [(grid.AABB_min, [c / 2] * 3, tuple(int(v) * 2 + 1 for v in grid.N)),
            (np.asarray(grid.AABB_min) - 0.7 * c, [c / 3, c / 3, 0.45 * c], (50, 47, int(int(grid.N[2]) / 0.45) + 4))]
    for devs in _device_lists():
        mesh, _, _, _ = _run_pipeline(r2s, case, devices=devs)
        for o, h, s in lats:
            V, T = r2s.isosurface_lattice(mesh, o, h, s)
            Vb, Tb, ns = r2s.isosurface_band(mesh, o, h, s, stats=True)
            assert len(T) > 0 and np.array_equal(Vb, V) and np.array_equal(Tb, T), devs
            assert 0 < ns <= int(np.prod(s))
        o, h, s = lats[0]
        Vl, Tl = r2s.isosurface_lattice(mesh, o, h, s)
        r2s.export_isosurface(mesh, str(tmp_path / "m.ply"), band=(o, h, s))
        V2, T2 = r2s.read_ply(str(tmp_path / "m.ply"))
        assert np.array_equal(V2, Vl) and np.array_equal(T2, Tl)
        mesh.close()


def _lattice_points(o, h, ranges):
    """the Float32 lattice coordinates float(o) + float(i) * float(h) of the index ranges (x, y, z), as float64 points, x fastest"""
    o32, h32 = np.float32(o), np.float32(h)
    ax = [(o32[d] + np.arange(*ranges[d]).astype(np.float32) * h32[d]).astype(np.float32) for d in range(3)]
    z, y, x = np.meshgrid(ax[2], ax[1], ax[0], indexing="ij")
    return np.stack([x.ravel(), y.ravel(), z.ravel()], 1).astype(np.float64)


def test_past_2_31_cells(r2s):
    """sphere_same on a 1301^3 lattice (2.2e9 cells, which r2s_isosurface_lattice rejects): the band call succeeds, the mesh is closed,
    and on a window of planes its triangles equal marching cubes on the window's values (from sample_sdf at the lattice's Float32
    coordinates, bit for bit the lattice values) up to the id offset, and 1000 of its vertices equal the host replay of the search"""
    mesh, grid, smooth, fine = _run_pipeline(r2s, "sphere_same")
    n = 1301
    amin, amax = np.asarray(grid.AABB_min), np.asarray(grid.AABB_max)
    o, h, shape = amin, (amax - amin) / (n - 1), (n, n, n)
    assert (n - 1) ** 3 >= 1 << 31
    with pytest.raises(r2s.R2SError, match="2\\^31 or more cells"):
        r2s.isosurface_lattice(mesh, o, h, shape)
    V, T, ns = r2s.isosurface_band(mesh, o, h, shape, stats=True)
    print("1301^3: nv=%d nt=%d sampled %d of %d points (%.2f %%)" % (len(V), len(T), ns, n ** 3, 100.0 * ns / n ** 3))
    assert len(T) > 10 ** 6 and ns < n ** 3
    # closed: the border of the lattice is below iso
    border = np.concatenate([_lattice_points(o, h, [(0, n), (0, n), (k, k + 1)]) for k in (0, n - 1)] +
                            [_lattice_points(o, h, [(0, n), (j, j + 1), (0, n)]) for j in (0, n - 1)] +
                            [_lattice_points(o, h, [(i, i + 1), (0, n), (0, n)]) for i in (0, n - 1)])
    bad = mref.unpaired_edges(T)
    if len(bad):
        assert mref.on_boundary_face(V, T, bad, np.float32(o), np.float32(h), shape).all()
    if (r2s.sample_sdf(mesh, border) < 0).all():
        assert len(bad) == 0
    # a window of planes [k0, k1) through the middle of the sphere
    k0, k1 = n // 2 - 4, n // 2 + 4
    win = r2s.sample_sdf(mesh, _lattice_points(o, h, [(0, n), (0, n), (k0, k1)])).reshape(k1 - k0, n, n)
    o_w = np.array(o, np.float64); o_w[2] = float(np.float32(np.float32(o[2]) + np.float32(k0) * np.float32(h[2])))
    Vw, Tw = r2s.isosurface_from_sdf(win, o_w, h, 0.0)
    # the window's triangles of cell planes [k0, k1 - 3) are its first ones (cells in linear order); they reference vertices of planes
    # up to k1 - 2, all numbered in the window as in the whole lattice.  The band mesh's triangles of cell planes < k0: the band mesh of
    # the lattice's first k0 + 1 planes (same origin and spacing, so the same coordinates)
    _, Tp = r2s.isosurface_from_sdf(win[:-2], o_w, h, 0.0)
    _, Tb0 = r2s.isosurface_band(mesh, o, h, (n, n, k0 + 1))
    m = len(Tp)
    assert m > 1000
    band = T[len(Tb0):len(Tb0) + m].astype(np.int64)
    off = band - Tw[:m].astype(np.int64)
    assert (off == off[0, 0]).all(), "triangles differ from marching cubes on the window"
    # vertices: the host replay of the search on the window's crossing edges
    F = _host_field(r2s, mesh, grid)
    E = ref.crossing_edges(win, np.float32(0.0))
    used = np.unique(Tw[:m])
    pick = np.random.default_rng(0).choice(used, 1000, replace=False)
    Ew = E[pick].copy()
    Ew[:, 2] += k0
    Vh, _, _ = ref.lattice_vertices(F, o, h, Ew, np.float32(0.0))
    assert np.array_equal(V[pick + off[0, 0]], Vh)
    mesh.close()


def test_errors(r2s):
    c = r2s.Context()
    o = np.zeros(3); h = np.ones(3); d = np.array([4, 4, 4], np.int64)
    nv, nt, ns = C.c_int64(), C.c_int64(), C.c_int64()

    def _p(a):
        return np.ascontiguousarray(a).ctypes.data_as(C.c_void_p)

    def call(ctx, o, h, d, iso=0.0):
        ctx.check(ctx.lib.r2s_isosurface_band(ctx.h, _p(o), _p(h), _p(d), iso, C.byref(nv), C.byref(nt), C.byref(ns)))
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
    with pytest.raises(r2s.R2SError, match="dims must be < 2\\^31"):
        call(mc, o, h, np.array([4, 1 << 31, 4], np.int64))
    with pytest.raises(r2s.R2SError, match="iso must be finite"):
        call(mc, o, h, d, float("nan"))
    w1, th1 = r2s.rbf_weights(mesh)
    assert np.array_equal(w0, w1) and th0 == th1
    mesh.close()
    mesh2, _, _, _ = _run_pipeline(r2s, "simp24_approx", devices=[0, 0])
    with pytest.raises(r2s.R2SError, match="use r2s_multi_isosurface_band"):
        call(mesh2.multi.slab(1), grid.AABB_min, h, d)
    mesh2.close()
