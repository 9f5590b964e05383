"""The interpolation-mode solve of RBFs_smoothing (the CG of r2s_dev_rbf) and the coarse LSF against a float64 replay (tests/cg_ref.py),
point by point, at shapes that hit every edge of the stencil kernel's launch, on one context and on z-slabs.

Per case:
  1. the CG iteration count equals cg64's, unless cg64's residual at the iteration where the two could part lies within 1 % of the
     tolerance (then +-1, printed);
  2. max|w_gpu - cg64(s, iters=k_gpu)| <= tau max|cg64|, tau = 8 times the drift of a Float32 model of the same loop (cg_ref.tau; the
     host tests show that every kernel defect they model exceeds 10 tau);
  3. the true residual |s - K w_gpu| is below 1.05 sqrt(eps(Float32)) |s|: no convergence flag raised early;
  4. the coarse LSF and the threshold search: with L = K w in float64 and the rigorous Float32 bound delta of cg_ref.lsf_bounds, the
     quadrature volumes (tests/volume_ref.py) of the fields L - delta and L + delta, rounded outward to Float32, at the GPU's threshold
     bracket the target whenever the search stopped on its 1e-4 criterion.  The volume is monotone in the field values (rounding is
     monotone, the interpolation weights are nonnegative), so a kernel LSF within delta of L has a volume between the two."""
import ctypes as C
import time

import numpy as np
import pytest

import cg_ref as ref
import volume_ref
from fixtures import block_geometry
from test_volume_exact import rbf_on_grid

pytestmark = pytest.mark.gpu


def check_solve(label, s, k_gpu, w):
    """Assertions 1-3 for the weights w (float32 [k, j, i]) a GPU solve returned after k_gpu iterations on the processed field s."""
    x64, k64, hist = ref.cg64(s)
    tol = ref.CG_RELTOL * hist[0]
    if k_gpu != k64:
        near = hist[min(k_gpu, k64)] / tol
        print("%s: iterations %d, cg64 %d; cg64 residual at iteration %d = %.4f tol" % (label, k_gpu, k64, min(k_gpu, k64), near))
        assert abs(k_gpu - k64) <= 1 and abs(near - 1) <= 0.01, (label, k_gpu, k64, near)
    t, xk = ref.tau(s, k_gpu, x64 if k_gpu == k64 else None)
    err = float(np.abs(w.astype(np.float64) - xk).max() / np.abs(xk).max())
    sd = s.astype(np.float64)
    res = float(np.linalg.norm(sd - ref.K64(w)) / (ref.CG_RELTOL * np.linalg.norm(sd)))
    print("%s: iterations %d (cg64 %d)  weight error %.3g tau (tau %.2e)  true residual %.4f tol" % (label, k_gpu, k64, err / t, t, res))
    assert err <= t, (label, err, t)
    assert res <= 1.05, (label, res)
    return k64


def check_lsf(label, w, shape, th_gpu, target, rep):
    """Assertion 4 for weights w (the GPU's, or s in approximation mode) and the GPU's returned offset th_gpu (= -threshold).
    When the search stopped on eps (bisections < 40), |fl32(V_gpu(th)) - target| <= 1e-4 at its threshold th.  After 40 bisections the
    bracket [lo, hi] with fl32(V_gpu(lo)) > target >= fl32(V_gpu(hi)) has shrunk to at most g = 2^-39 (max - min of the LSF) around th
    (or to adjacent floats), so the same bracket is asserted at th - g for V+ and at th + g for V-."""
    nx = shape[0]
    L, delta = ref.lsf_bounds(w)
    lo32, hi32 = ref.round_down32(L - delta), ref.round_up32(L + delta)
    edge = ref.coarse_edge(0.0, float(nx - 1), nx)
    th = np.float32(-th_gpu)
    if rep.bisections < 40:
        t_lo = t_hi = th
    else:
        g = (float(hi32.max()) - float(lo32.min())) * 2.0 ** -39
        t_lo = np.nextafter(ref.round_down32(float(th) - g), np.float32(-np.inf))
        t_hi = np.nextafter(ref.round_up32(float(th) + g), np.float32(np.inf))
    vlo = volume_ref.reference(lo32, edge, 0.0, float(t_hi))[2]
    vhi = volume_ref.reference(hi32, edge, 0.0, float(t_lo))[2]
    print("%s: bisections %d  V- %.5f  target %.5f  V+ %.5f  (width %.2e of the target)" % (label, rep.bisections, vlo, target, vhi, (vhi - vlo) / target))
    assert vhi - vlo <= 0.02 * target, (label, vlo, vhi)      # the bracket says something: a thin band of cells around the level set
    assert float(np.float32(vlo)) - 1e-4 <= target <= float(np.float32(vhi)) + 1e-4, (label, vlo, target, vhi)


def zero_level_volume(s, shape):
    """The target of a case: the volume of {s >= 0} of the processed SDF, so that the threshold lies where the LSF has a slope."""
    return volume_ref.reference(s, ref.coarse_edge(0.0, float(shape[0] - 1), shape[0]))[2]


def single(r2s, ctx, shape, kind):
    sdf = ref.make_field(kind, shape)
    s = ref.process(sdf)
    N = [n - 1 for n in shape]
    target = zero_level_volume(s, shape)
    assert 0 < target < np.prod(N)
    for interp in (True, False):
        label = "%s %s %s" % ("x".join(map(str, shape)), kind, "interp" if interp else "approx")
        fine, th, vol, rep, grid = rbf_on_grid(r2s, ctx, sdf, N, 1.0, 1, interp, target)
        w = np.empty(s.shape, np.float32); thw = C.c_float()
        ctx.check(ctx.lib.r2s_download_rbf_weights(ctx.h, w.ctypes.data_as(C.c_void_p), C.byref(thw)))
        assert thw.value == np.float32(th)
        if interp:
            check_solve(label, s, rep.cg_iters, w)
        else:
            assert rep.cg_iters == 0 and np.array_equal(w, s)
        check_lsf(label, w, shape, th, target, rep)


@pytest.fixture(scope="module")
def ctx(r2s):
    c = r2s.Context()
    yield c
    c.close()


@pytest.mark.parametrize("shape", ref.SHAPES, ids=lambda s: "x".join(map(str, s)))
def test_cg_and_lsf_match_float64(r2s, ctx, shape):
    t0 = time.time()
    for kind in ref.FIELDS:
        single(r2s, ctx, shape, kind)
    print("%s: %.1f s" % (shape, time.time() - t0))


def test_cg_at_more_ctas_than_reduction_slots(r2s, ctx):
    """1.53 M points: 512 stencil CTAs (and 1184 update CTAs), more than the 256 strided slots cta_sum_last adds up."""
    nx, ny, nz = ref.LARGE
    assert -(-(nx + 2) // 32) * -(-ny // 16) > 256
    t0 = time.time()
    for kind in ref.fields_of(ref.LARGE):
        single(r2s, ctx, ref.LARGE, kind)
    print("%s: %.1f s" % (ref.LARGE, time.time() - t0))


# ---- z-slabs ------------------------------------------------------------------------------------------------------------------------------
# (points per axis, slab count, the cuts r2s_multi makes on its first call: even, at least 3 planes per slab)
SLAB_CASES = [
    ((33, 17, 12), 4, [0, 3, 6, 9, 12]),        # 3-plane slabs: a slab's CG halo (2 planes; 3 up for the weights) spans all of the adjacent slab
    ((31, 16, 130), 2, [0, 65, 130]),           # the cut lies on the 65-plane z-chunk boundary of the one-context launch
    ((63, 15, 9), 3, [0, 3, 6, 9]),
]


def slab_grid(shape, X):
    """A grid with `shape` points around the mesh X: the cell is the smallest that leaves a 10 % margin on every axis."""
    N = np.array([n - 1 for n in shape], np.int64)
    lo, hi = X.min(0), X.max(0)
    cell = float(np.max(1.2 * (hi - lo) / N))
    amin = (lo + hi) / 2 - N * cell / 2
    return type("SlabGrid", (), {"AABB_min": amin, "AABB_max": amin + N * cell, "N": N, "cell_size": cell, "ngp": int(np.prod(N + 1))})


def run_slabs(r2s, shape, devs, cuts_expected):
    X, IEN, rho = block_geometry([4, 4, 40] if shape[2] > 64 else [4, 4, 4])
    mesh = r2s.Mesh(X, IEN, rho, devices=devs)
    try:
        grid = slab_grid(shape, X)
        mesh._use_grid(grid)
        m = mesh.multi
        assert m.slab_planes() == cuts_expected
        rn = r2s.DenseInNodes(mesh, rho)
        p = r2s.Params(); m.lib.r2s_default_params(C.byref(p))
        p.rho_t, p.smooth, p.rbf_interp, p.remove_artifacts, p.final_volume = 0.5, 1, 1, 0, 0
        p.target_volume = 0.3 * float(np.prod(grid.N)) * grid.cell_size ** 3
        sdf = np.empty(grid.ngp); fine = np.empty(grid.ngp, np.float32); rep = r2s.Report()
        m.check(m.lib.r2s_multi_pipeline(m.h, C.byref(p), rn.ctypes.data_as(C.c_void_p), sdf.ctypes.data_as(C.c_void_p), fine.ctypes.data_as(C.c_void_p), C.byref(rep)))
        assert m.slab_planes() == cuts_expected      # the re-cut by measured cost applies from the next call on
        w, th = r2s.rbf_weights(mesh)
        s = ref.process(sdf.reshape(w.shape))
        assert (np.abs(sdf) > 1e9).any() and (np.abs(sdf) < 1e9).any()      # band and far values
        check_solve("%s on devices %s" % ("x".join(map(str, shape)), devs), s, rep.cg_iters, w)
    finally:
        mesh.close()


@pytest.mark.parametrize("case", SLAB_CASES, ids=lambda c: "%dslabs_%s" % (c[1], "x".join(map(str, c[0]))))
def test_cg_on_slabs_of_one_gpu(r2s, case):
    shape, n, cuts = case
    run_slabs(r2s, shape, [0] * n, cuts)


@pytest.mark.parametrize("case", SLAB_CASES, ids=lambda c: "%dslabs_%s" % (c[1], "x".join(map(str, c[0]))))
def test_cg_on_slabs_of_distinct_gpus(r2s, case):
    """The fused halo stores of the stencil kernel (peer memory between distinct GPUs, DESIGN.md section 6)."""
    import torch
    shape, n, cuts = case
    if torch.cuda.device_count() < n:
        pytest.skip("%d slabs on distinct GPUs need %d devices, %d visible" % (n, n, torch.cuda.device_count()))
    run_slabs(r2s, shape, list(range(n)), cuts)
