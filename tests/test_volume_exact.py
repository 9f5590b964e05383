"""The volume stages on the GPU against the exact host reference (tests/volume_ref.py), bit for bit.

calculate_volume_from_sdf, the final fine-grid volume of the pipeline and the LS_Threshold search add up per-cell Float32 quadratures as
fixed-point integers, so their doubles are reproducible exactly on the host: any dropped, doubled or wrongly classified cell -- at a tile
seam, a slab boundary, a cut-list regrow, or a wrap of the integer sum -- changes the result.  The fine evaluation of the approximation
mode is compared with a float64 evaluation of the same taps under a rigorous Float32 round-off bound."""
import ctypes as C

import numpy as np
import pytest

import oracle
import volume_ref
from fixtures import simp_hex8

pytestmark = pytest.mark.gpu

ISOS = (0.0, 0.25, -1e-3)


def tool_volume(ctx, f, edge, iso=0.0, order=9):
    """r2s_volume_from_sdf's double (the Python wrapper rounds it to float32)."""
    a = np.ascontiguousarray(f, np.float32)
    nz, ny, nx = a.shape
    v = C.c_double()
    ctx.check(ctx.lib.r2s_volume_from_sdf(ctx.h, a.ctypes.data_as(C.c_void_p), nx, ny, nz, float(np.float32(edge)), float(np.float32(iso)), order, C.byref(v)))
    return v.value


def tool_fields(shape, rng):
    """shape = (nx, ny, nz); fields indexed [k, j, i]"""
    nx, ny, nz = shape
    k, j, i = np.meshgrid(np.arange(nz), np.arange(ny), np.arange(nx), indexing="ij")
    c = [(n - 1) / 2 for n in (nz, ny, nx)]
    r = np.sqrt((k - c[0]) ** 2 + (j - c[1]) ** 2 + (i - c[2]) ** 2)
    sz = (nz, ny, nx)
    yield "sphere", 0.35 * max(shape) - r
    yield "gyroid", np.sin(0.7 * i) * np.cos(0.6 * j) + np.sin(0.6 * j) * np.cos(0.5 * k) + np.sin(0.5 * k) * np.cos(0.7 * i)
    yield "noise", rng.uniform(-1, 1, sz)
    yield "quantised", rng.choice(np.array([-1.0, -0.25, -1e-3, 0.0, 0.25, 1.0], np.float32), sz)      # many corners exactly at an iso
    yield "signed_zeros", rng.choice(np.array([0.0, -0.0, 0.0, -0.0, -1e-3, 0.25, -1.0], np.float32), sz)
    yield "magnitudes", rng.choice([-1.0, 1.0], sz) * 10.0 ** rng.uniform(-30, 30, sz)
    yield "all_full", np.full(sz, 2.0)
    yield "all_empty", np.full(sz, -2.0)
    yield "checkerboard", np.where((i + j + k) % 2 == 0, 1.0, -1.0)      # every cell cut


# 2-point axes, partial 4-row y-tiles, x-tile seams at cell 63 / 126, 32-plane z-tiles with a remainder
@pytest.mark.parametrize("shape", [(2, 2, 2), (3, 130, 2), (66, 5, 34), (64, 65, 33), (129, 7, 65), (200, 3, 97)])
def test_volume_tool_is_bit_exact(r2s, shape):
    ctx = r2s.Context()
    rng = np.random.default_rng(sum(shape))
    edge = np.float32(0.37)
    for name, f in tool_fields(shape, rng):
        f = f.astype(np.float32)
        for iso in ISOS:
            ref = volume_ref.reference(f, edge, iso)[2]
            got = tool_volume(ctx, f, edge, iso)
            assert got == ref, "%s iso=%g: %r != %r" % (name, iso, got, ref)
    ctx.close()


def test_volume_tool_regrows_the_cut_list(r2s):
    """A fresh context starts with a 1024-entry cut list; more cut cells than that take the grow-and-repeat path."""
    rng = np.random.default_rng(2)
    shape = (40, 41, 39)
    for name, f in tool_fields(shape, rng):
        if name not in ("checkerboard", "noise", "gyroid"):
            continue
        f = f.astype(np.float32)
        for iso in ISOS:
            ctx = r2s.Context()
            c = [f[a:f.shape[0] - 1 + a, b:f.shape[1] - 1 + b, d:f.shape[2] - 1 + d] for a in (0, 1) for b in (0, 1) for d in (0, 1)]
            ncut = int(((np.min(c, axis=0) < np.float32(iso)) & ~(np.max(c, axis=0) < np.float32(iso))).sum())
            assert ncut > 4 * 1024, (name, iso, ncut)
            ref = volume_ref.reference(f, 0.5, iso)[2]
            assert tool_volume(ctx, f, 0.5, iso) == ref, (name, iso)
            ctx.close()


def alternating_tile():
    return np.array([1.0, -1.0], np.float32).reshape(1, 1, 2)


def test_volume_tool_sum_does_not_wrap(r2s):
    """401^3 points alternating along x: all 6.4e7 cells are cut, each with part ~ 4.66, so the fixed-point sum is ~2.2 * 2^64 (a single
    64-bit word wrapped twice here).  Order 9 against the exact class sum; order 20 (k_vol_cut_n) to 1e-6 against the oracle's value of
    each class's single cell times its count."""
    tile, shape, edge = alternating_tile(), (401, 401, 401), np.float32(0.25)
    f = volume_ref.periodic_field(tile, shape)
    nfull, S, ref = volume_ref.periodic_reference(tile, shape, edge)
    assert nfull == 0 and S > 2 ** 65
    ctx = r2s.Context()
    assert tool_volume(ctx, f, edge) == ref
    ref20 = sum(cnt * oracle.volume_from_sdf(cell, edge, order=20) for cnt, cell in volume_ref.periodic_classes(tile, shape))
    got20 = tool_volume(ctx, f, edge, order=20)
    assert abs(got20 - ref20) <= 1e-6 * ref20
    ctx.close()


# ---- the pipeline's final volume -------------------------------------------------------------------------------------------------------
def run_resident(r2s, mesh, grid, rn, smooth, interp):
    mesh._use_grid(grid)
    c = mesh.ctx
    p = r2s.Params(); c.lib.r2s_default_params(C.byref(p))
    p.rho_t, p.smooth, p.rbf_interp, p.target_volume, p.final_volume = 0.5, smooth, int(interp), mesh.V_frac * mesh.V_domain, 1
    c.check(c.lib.r2s_upload_nodal_densities(c.h, rn.ctypes.data_as(C.c_void_p)))
    rep = r2s.Report()
    c.check(c.lib.r2s_pipeline_resident(c.h, C.byref(p), C.byref(rep)))
    dims = tuple(int(v) * smooth + 1 for v in grid.N)
    fine = np.empty(dims[::-1], dtype=np.float32)
    c.check(c.lib.r2s_download_fine_sdf(c.h, fine.ctypes.data_as(C.c_void_p)))
    return fine, rep


@pytest.mark.parametrize("case", ["simp24", "simp64", "mixed"])
def test_pipeline_final_volume_is_exact(r2s, case):
    """rep.volume = float32 of the reference's volume of the returned field, for both smoothing grids and both RBF modes."""
    if case == "mixed":
        from test_gpu_parity import _mixed_mesh
        X, IEN, rho = _mixed_mesh(10)
        nmax = 20
    else:
        n = int(case[4:])
        X, IEN, rho = simp_hex8(n)
        nmax = 2 * n
    mesh = r2s.Mesh(X, IEN, rho)
    grid = r2s.Grid(X.min(0), X.max(0), nmax, 3)
    rn = r2s.DenseInNodes(mesh, rho)
    for smooth in (1, 2):
        for interp in (True, False):
            fine, rep = run_resident(r2s, mesh, grid, rn, smooth, interp)
            ref = volume_ref.reference(fine, volume_ref.fine_edge(grid, smooth))[2]
            assert rep.volume == np.float32(ref), (smooth, interp, rep.volume, ref)
    mesh.close()


# ---- LS_Threshold at a size where a single-word sum wraps ------------------------------------------------------------------------------
def wrap_field(n=400):
    """(n+1)^3 coarse points: +-1 alternating along x plus a small ramp in y and z with incommensurate slopes, so that every cell is cut
    for every threshold the search tries and the volume changes in steps of about one cell."""
    ax = np.arange(n + 1, dtype=np.float64)
    k, j, i = ax[:, None, None], ax[None, :, None], ax[None, None, :]
    return np.where(i % 2 == 0, 1.0, -1.0) + 0.1 * ((j / n - 0.5) + np.sqrt(2.0) * (k / n - 0.5)) / (1 + np.sqrt(2.0))


def rbf_on_grid(r2s, ctx, sdf, N, cell, smooth, interp, target, rbf_cut=1e-3):
    N = np.ascontiguousarray(N, np.int64)
    amin = np.zeros(3); amax = N * cell
    ctx.check(ctx.lib.r2s_set_grid(ctx.h, amin.ctypes.data_as(C.c_void_p), amax.ctypes.data_as(C.c_void_p), N.ctypes.data_as(C.c_void_p), float(cell)))
    d = np.ascontiguousarray(sdf, np.float64)
    dims = tuple(int(v) * smooth + 1 for v in N)
    fine = np.empty(dims[::-1], np.float32)
    th, vol = C.c_float(), C.c_float()
    ctx.check(ctx.lib.r2s_rbf_smoothing(ctx.h, d.ctypes.data_as(C.c_void_p), int(interp), int(smooth), float(rbf_cut), float(target),
                                        fine.ctypes.data_as(C.c_void_p), C.byref(th), C.byref(vol)))
    grid = type("G", (), {"N": N, "AABB_min": amin, "AABB_max": amax})
    return fine, th.value, vol.value, ctx.report(), grid


def test_threshold_search_at_wrap_size(r2s):
    """Approximation mode on :same over a 400^3-cell field whose cut cells add up to ~2^65 in fixed point: the search must hit half the
    box and report the exact volume of the field it returns (a wrapped sum steers the bisection to a wrong threshold and then confirms it)."""
    n, cell = 400, 1.0
    target = 0.5 * (n * cell) ** 3
    ctx = r2s.Context()
    fine, th, vol, rep, grid = rbf_on_grid(r2s, ctx, wrap_field(n), [n, n, n], cell, 1, False, target)
    nfull, S, ref = volume_ref.reference(fine, volume_ref.fine_edge(grid, 1))
    assert S > 2 ** 64
    assert vol == np.float32(ref)
    assert abs(vol - target) <= 1e-5 * target
    ctx.close()


# ---- fine evaluation against float64 ---------------------------------------------------------------------------------------------------
def taps(smooth, rbf_cut, cell=1.0):
    """Per phase (px, py, pz): the library's tap rule (float)(sqrt(m) * cell) <= (float)sqrt(-log(cut) * cell^2) over offsets -4..4."""
    maxd = np.float32(np.sqrt(-np.log(rbf_cut) * cell * cell))
    out = {}
    for pz in range(smooth):
        for py in range(smooth):
            for px in range(smooth):
                t = []
                for dk in range(-4, 5):
                    for dj in range(-4, 5):
                        for di in range(-4, 5):
                            m = (di - px / smooth) ** 2 + (dj - py / smooth) ** 2 + (dk - pz / smooth) ** 2
                            if np.float32(np.sqrt(m) * cell) <= maxd:
                                t.append((di, dj, dk, np.exp(-m)))
                out[(px, py, pz)] = t
    return out


def eval_f64(s, smooth, tp, probe=None):
    """Sum over the taps of exp(-m) s_t in float64 (zero outside the grid) and the sum of |exp(-m) s_t|, per fine point; with `probe`,
    for every tap of every phase: does some point see that tap's term above probe(point)?"""
    nz, ny, nx = s.shape
    P = 4
    sp = np.zeros((nz + 2 * P, ny + 2 * P, nx + 2 * P)); sp[P:-P, P:-P, P:-P] = s
    fz, fy, fx = ((n - 1) * smooth + 1 for n in (nz, ny, nx))
    E, A, NT = np.zeros((fz, fy, fx)), np.zeros((fz, fy, fx)), np.zeros((fz, fy, fx))
    seen = []
    for (px, py, pz), t in tp.items():
        cz, cy, cx = len(range(pz, fz, smooth)), len(range(py, fy, smooth)), len(range(px, fx, smooth))
        e, a = np.zeros((cz, cy, cx)), np.zeros((cz, cy, cx))
        for di, dj, dk, w in t:
            v = sp[P + dk:P + dk + cz, P + dj:P + dj + cy, P + di:P + di + cx]
            e += w * v; a += np.abs(w * v)
            if probe is not None:
                seen.append(bool((np.abs(w * v) > probe[pz::smooth, py::smooth, px::smooth]).any()))
        E[pz::smooth, py::smooth, px::smooth] = e; A[pz::smooth, py::smooth, px::smooth] = a; NT[pz::smooth, py::smooth, px::smooth] = len(t)
    if probe is not None:
        return seen
    return E, A, NT


def fine_eval_input(shape, rng):
    """A sparse signed field (15 % of the points nonzero, |v| in [0.25, 1]) with a few far values (+-1e10, replaced by the largest finite
    |v| before the evaluation).  Sparse, so that at many points a single tap carries most of the sum: every tap is then observable above
    the round-off bound (a dense field hides the smallest taps of the widest cut-off under the bound)."""
    nx, ny, nz = shape
    sz = (nz, ny, nx)
    s = np.where(rng.random(sz) < 0.15, rng.choice([-1.0, 1.0], sz) * rng.uniform(0.25, 1.0, sz), 0.0)
    far = rng.random(sz) < 0.01
    s[far] = rng.choice([-1e10, 1e10], int(far.sum()))
    return s


CUTS = (1e-3, float(np.exp(-6.1)), float(np.exp(-7.9)))


def test_fine_eval_cut_offs_differ():
    sets = [{(di, dj, dk, p) for p, t in taps(2, cut).items() for di, dj, dk, _ in t} for cut in CUTS]
    assert sets[1] < sets[0] < sets[2]


@pytest.mark.parametrize("N", [(5, 3, 2), (31, 4, 9), (32, 5, 8), (33, 7, 17), (40, 40, 70)])
def test_fine_eval_matches_float64(r2s, N):
    """Approximation mode: the weights are float32(sdf) with far values replaced, so the returned field is sum_t exp(-m) s_t + tho up to
    Float32 round-off, |err| <= (n_taps + 2) 2^-24 (sum |phi_t s_t| + |tho|) -- a bound that a single dropped or extra tap exceeds (the
    test checks that), at grid sizes that are no multiple of the kernels' tiles (32 x 4 x 4 and 32 x 4 x 8 outputs per block)."""
    rng = np.random.default_rng(N[0] * 100 + N[2])
    shape = tuple(v + 1 for v in N)
    sdf = fine_eval_input(shape, rng)
    s = sdf.astype(np.float32)
    finite = np.abs(s) < 1e9
    s = np.where(finite, s, np.sign(s) * np.abs(s[finite]).max()).astype(np.float32).astype(np.float64)
    ctx = r2s.Context()
    for smooth in (1, 2):
        for cut in CUTS:
            tp = taps(smooth, cut)
            E, A, NT = eval_f64(s, smooth, tp)
            fine, tho, vol, rep, grid = rbf_on_grid(r2s, ctx, sdf, N, 1.0, smooth, False, 0.3 * np.prod(N), rbf_cut=cut)
            bound = (NT + 2) * 2.0 ** -24 * (A + abs(tho))
            err = np.abs(fine.astype(np.float64) - (E + tho))
            assert (err <= bound).all(), (smooth, cut, float((err / bound).max()))
            # sensitivity: every tap of every phase (the smallest, e^-7.75 for the widest cut-off, included) contributes more than 20 times
            # the bound at some point, so dropping or adding any one tap fails the comparison above
            if min(N) >= 4:      # (on smaller grids some taps always fall outside)
                assert all(eval_f64(s, smooth, tp, probe=20 * bound)), (smooth, cut)
            wmin = min(w for t in tp.values() for _, _, _, w in t)
            near = np.abs(E + tho) < 0.5
            assert 20 * np.median(bound[near]) <= wmin * np.median(np.abs(s[s != 0])), (smooth, cut)
    ctx.close()
