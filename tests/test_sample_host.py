"""CPU tests of the sampler of the continuous smoothed SDF (rho2sdf.jl_b200/csrc/r2s_sample.cuh, host build tests/host/sample_host.cpp):
the Float32 exponential, the squared cut radius, the 124-neighbour bound that makes "all points within maxd" the reference's set, and
the evaluator against float64 evaluations of the same definition and against a KD-tree restatement of rbf_interpolation_kdtree."""
import math

import numpy as np
import pytest

import sample_ref as ref
from test_volume_exact import CUTS, fine_eval_input

U = 2.0 ** -24


def test_exp_f32_error_bound_over_every_argument():
    """every float in [-16, 0] (the kernel uses [-8, 0]): |exp_f32(x) - exp(x)| <= 1.5 2^-24 exp(x), the bound r2s_sample.cuh states"""
    m, worst = ref.exp_scan(-16.0, 0.0)
    print("exp_f32: max relative error %.3f 2^-24 at x = %.9g" % (m / U, worst))
    assert m <= 1.5 * U
    assert ref.exp_f32(np.array([0.0, -0.0, -87.0, -1e30, -np.inf], np.float32)).tolist() == [1.0, 1.0, 0.0, 0.0, 0.0]


@pytest.mark.parametrize("cut", CUTS)
@pytest.mark.parametrize("cell", [1.0, 0.1, 0.37, 2.5e-3, 17.0])
def test_t2_is_the_largest_square_below_maxd(cut, cell):
    md = ref.maxd(cut, cell)
    t2 = ref.t2(md)
    assert md == np.float32(math.sqrt(-math.log(cut) * cell * cell))
    assert np.sqrt(t2) <= md < np.sqrt(np.nextafter(t2, np.float32(np.inf)))      # numpy's float32 sqrt is correctly rounded


def test_no_ball_of_the_cut_radius_holds_more_than_124_grid_points():
    """The reference sums the 124 nearest coarse points within maxd; the sampler sums all points within maxd.  The sets are equal if no
    ball of radius maxd holds more than 124 lattice points.  Covering argument in cell units: every centre x in the unit cell lies within
    delta sqrt(3) / 2 of a sample s of the delta-grid of cell centres, so a ball B(x, r) lies inside B(s, r + delta sqrt(3) / 2).  r is
    sqrt(ln(1/cut)) (1 + eps) for the widest supported cut, ln(1/cut) -> 8, with eps = 1e-3 covering the Float32 rounding of maxd and of
    the coordinate tables; counting is exact in float64 far from the squared-radius boundary (a margin of 1e-9 is added)."""
    delta = 1.0 / 40
    r = math.sqrt(8.0) * (1 + 1e-3) + delta * math.sqrt(3) / 2
    s = (np.arange(40) + 0.5) * delta
    sz, sy, sx = np.meshgrid(s, s, s, indexing="ij")
    S = np.stack([sx.ravel(), sy.ravel(), sz.ravel()], 1)
    o = np.arange(-3, 5)
    oz, oy, ox = np.meshgrid(o, o, o, indexing="ij")
    L = np.stack([ox.ravel(), oy.ravel(), oz.ravel()], 1).astype(np.float64)
    cnt = np.zeros(len(S), np.int64)
    for q in range(0, len(S), 4000):
        d2 = ((S[q:q + 4000, None, :] - L[None, :, :]) ** 2).sum(-1)
        cnt[q:q + 4000] = (d2 <= r * r + 1e-9).sum(1)
    print("largest count within r = %.4f cells: %d" % (r, cnt.max()))
    assert cnt.max() <= 124


def _field(shape, cut, seed, cell=1.0, amin=(0.0, 0.0, 0.0), th=0.3):
    rng = np.random.default_rng(seed)
    nz, ny, nx = shape
    w = fine_eval_input((nx, ny, nz), rng)
    w = np.where(np.abs(w) < 1e9, w, 0.5 * np.sign(w)).astype(np.float32)
    amin = np.asarray(amin, np.float64)
    amax = amin + cell * np.array([nx - 1, ny - 1, nz - 1], np.float64)
    return ref.Field(w, amin, amax, cell, cut, th)


def _points(F, rng, n_random=150):
    """random points, coarse lattice points, fine (:fine) lattice points, points within 3 cells of and beyond the border, far points"""
    lo, hi, c = F.amin, F.amax, F.cell
    pts = [rng.uniform(lo, hi, (n_random, 3))]
    idx = rng.integers(0, F.n, (40, 3))
    pts.append(np.stack([F.C[d][idx[:, d]] for d in range(3)], 1).astype(np.float64))
    pts.append(lo + 0.5 * c * rng.integers(0, 2 * (F.n - 1) + 1, (40, 3)))
    side = rng.integers(0, 2, (60, 3))
    pts.append(np.where(side, hi + rng.uniform(-3 * c, 3 * c, (60, 3)), lo + rng.uniform(-3 * c, 3 * c, (60, 3))))
    pts.append(np.array([[lo[0] - 4 * c, lo[1], lo[2]], [hi[0], hi[1] + 3.5 * c, hi[2]], lo - 1e6 * c, hi + 1e30]))
    return np.concatenate(pts)


@pytest.mark.parametrize("cut", CUTS)
@pytest.mark.parametrize("case", [((9, 7, 11), 1.0, (0, 0, 0)), ((6, 13, 8), 0.37, (-2.0, 5.0, 0.25)), ((5, 5, 5), 2.5e-3, (10.0, -3.0, 1.0))])
def test_host_evaluator_matches_float64(cut, case):
    """value and gradient against the same definition in float64 (same Float32 tap set and offsets e, exact arithmetic after):
    |value - v64| <= (n_taps + K) 2^-24 (sum |w phi| + |th|), K = sample_ref.K_ROUNDOFF derived there from the operation sequence.  The
    weights are sparse, so that dropping the smallest tap or adding the nearest excluded point breaks the bound at most points."""
    shape, cell, amin = case
    F = _field(shape, cut, seed=len(CUTS) * shape[0] + shape[2], cell=cell, amin=amin)
    rng = np.random.default_rng(shape[1])
    P = _points(F, rng)
    val, grad = F.host(P, gradient=True)
    assert np.array_equal(F.host(P), val)
    drop = add = total = 0
    for t, p in enumerate(P):
        v64, g64, A, nt = F.float64(p)
        bound = (nt + ref.K_ROUNDOFF) * U * (A + abs(float(F.th)))
        assert abs(float(val[t]) - v64) <= bound, (t, p, float(val[t]), v64, bound)
        # gradient: each term 2 kappa w phi e carries phi's error, e exact, two more roundings (w phi, the fma) and the final scaling
        assert np.all(np.abs(grad[t].astype(np.float64) - g64) <= (nt + ref.K_ROUNDOFF + 2) * U * 2 * float(F.kappa) * A * 3 * F.cell + 1e-30), (t, grad[t], g64)
        if nt == 0:
            assert val[t] == F.th and not grad[t].any()      # far away: exactly th
            continue
        total += 1
        d = F.float64(p, "drop")
        if d is not None and abs(d[0] - v64) > bound:
            drop += 1
        a = F.float64(p, "add")
        if a is not None and abs(a[0] - v64) > bound:
            add += 1
    print("cut %.4g: %d points with taps; one tap dropped breaks the bound at %d, one added at %d" % (cut, total, drop, add))
    assert drop >= 0.9 * total and add >= 0.9 * total


@pytest.mark.parametrize("cut", CUTS)
def test_host_evaluator_matches_kdtree_restatement(cut):
    """rbf_interpolation_kdtree restated with a 124-nearest-neighbour KD-tree query: the same set (the covering test above), so only the
    summation order and the kernel's Float32 round-off differ: within 1e-4 of the field's scale, the smoothing tolerance of
    tests/test_oracle_golden.py"""
    F = _field((12, 10, 14), cut, seed=5, cell=0.5, amin=(1.0, -1.0, 0.0))
    rng = np.random.default_rng(9)
    P = _points(F, rng, n_random=600)
    got = F.host(P)
    want = F.knn124(P)
    scale = float(np.abs(want).max())
    assert np.abs(got.astype(np.float64) - want).max() <= 1e-4 * scale
