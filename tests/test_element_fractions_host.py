"""CPU tests of the per-element volume fractions of r2s_element_volume_fractions (rho2sdf.jl_b200/csrc/r2s_elemfrac.cuh), built for the
host (tests/host/elemfrac_host.cpp): the rule against a plain numpy restatement on fuzzed general hexes and tets, the TET4 volume, the
split of the block classifier into a box form and its lattice wrapper, the element box against every Gauss point, and the soundness of
the skipping on the float64 CG weights of a sphere replica."""
import numpy as np
import pytest

import cg_ref
import elemfrac_ref as ef
import sample_ref

CUT = 1e-3
U = 2.0 ** -24


def _rotation(rng):
    q, r = np.linalg.qr(rng.normal(size=(3, 3)))
    return q * np.sign(np.diag(r))


def fuzz_mesh(rng, nen, m, center, size, thin=False):
    """m unconnected elements (nodes not shared): perturbed, rotated, scaled unit cubes (HEX8) or tets (TET4) around `center`, some of them
    nearly flat when `thin`.  Returns X (m nen, 3), IEN (m, nen) 0-based."""
    cube = np.array([[0, 0, 0], [1, 0, 0], [1, 1, 0], [0, 1, 0], [0, 0, 1], [1, 0, 1], [1, 1, 1], [0, 1, 1]], np.float64)
    tet = np.array([[1, 0, 0], [0, 1, 0], [0, 0, 1], [0, 0, 0]], np.float64)
    X = []
    for e in range(m):
        P = (cube if nen == 8 else tet) + rng.uniform(-0.2, 0.2, (nen, 3))
        if thin and e % 3 == 0:
            P[:, 2] *= 1e-2
        P = (P - 0.5) @ _rotation(rng).T * (size * rng.uniform(0.3, 1.0)) + center + rng.uniform(-1, 1, 3) * size
        X.append(P)
    return np.concatenate(X), np.arange(m * nen, dtype=np.int64).reshape(m, nen)


def mixed_field(rng, shape, cell, amin):
    w = rng.uniform(-1.0, 1.0, size=shape[::-1]).astype(np.float32)
    amin = np.asarray(amin, np.float64)
    return sample_ref.Field(w, amin, amin + cell * (np.array(shape) - 1), cell, CUT, np.float32(0.05))


@pytest.mark.parametrize("nen", [8, 4])
@pytest.mark.parametrize("origin", [0.0, 1000.0])
def test_numpy_restatement(nen, origin):
    """Gauss points and weights of the host rule against numpy (points to 1e-13 of the element size, V_e to 1e-13 relative), and the
    fractions against numpy's Heaviside of the float64 field at float(x), wherever no Gauss value lies within the sampler's Float32 bound
    of iso"""
    rng = np.random.default_rng(11 + nen + int(origin))
    cell = 0.37
    F = mixed_field(rng, (18, 18, 18), cell, (origin, origin - 0.3, origin + 0.6))
    center = F.amin + 9 * cell
    X, IEN = fuzz_mesh(rng, nen, 24, center, 2.5 * cell, thin=True)
    compared = 0
    for q in (2, 3):
        for iso in (0.0, 0.3):
            frac, vol, _ = ef.replay(F, X, IEN, q, np.float32(iso))
            for e in range(len(IEN)):
                x, W, ok = ef.points(X, IEN, e, q)
                xn, Wn = ef.numpy_points(X[IEN[e]], q)
                assert ok.all()
                assert np.abs(x - xn).max() <= 1e-13 * (np.abs(X[IEN[e]]).max() + 1.0)
                assert abs(vol[e] - Wn.sum()) <= 1e-13 * Wn.sum() and vol[e] == ef.replay(F, X, IEN[e:e + 1], q, iso)[1][0]
                f64 = [F.float64(p) for p in xn.astype(np.float32).astype(np.float64)]
                near = any(abs(v - float(np.float32(iso))) <= (n + sample_ref.K_ROUNDOFF) * U * (A + abs(float(F.th))) for v, _, A, n in f64)
                if near:
                    continue
                inside = np.array([v >= float(np.float32(iso)) for v, _, _, _ in f64])
                fn = (Wn * inside).sum() / Wn.sum()
                assert abs(frac[e] - fn) <= 1e-13, (e, q, iso, frac[e], fn)
                compared += 1
                assert 0.0 <= frac[e] <= 1.0
    partial = frac[(frac > 0) & (frac < 1)]
    print("nen=%d origin=%g: %d element fractions compared, %d partial at the last rule" % (nen, origin, compared, len(partial)))
    assert compared >= 60 and len(partial) > 0


@pytest.mark.parametrize("q", range(2, 9))
def test_tet4_volume(q):
    """sum W = |det J| / 6 (the Duffy factor (1 - xi)(1 - xi - eta) / 8), not the 3/4 of it that the reference's (1 - xi)^2 factor gives"""
    rng = np.random.default_rng(q)
    X, IEN = fuzz_mesh(rng, 4, 20, np.array([1000.0, -3.0, 50.0]), 1.7, thin=True)
    for e in range(len(IEN)):
        _, W, ok = ef.points(X, IEN, e, q)
        P = X[IEN[e]]
        v = abs(np.linalg.det(np.stack([P[0] - P[3], P[1] - P[3], P[2] - P[3]], 1))) / 6
        assert ok.all() and abs(W.sum() - v) <= 1e-13 * v, (q, e, W.sum(), v)


def test_classifier_split():
    """the lattice form of the block classifier equals its box form on the Float32 box of the lattice indices, bit for bit, on fuzzed
    lattices (same-signed weights, so that every answer occurs)"""
    rng = np.random.default_rng(5)
    seen = set()
    for trial in range(6):
        sign = 1 if trial % 2 else -1
        cell = [1.0, 0.37, 2.5][trial % 3]
        amin = np.array([0.0, 1000.0, -3.0])[[trial % 3, (trial + 1) % 3, (trial + 2) % 3]]
        w = (sign * rng.uniform(0.05, 1.0, size=(17, 18, 20))).astype(np.float32)
        F = sample_ref.Field(w, amin, amin + cell * (np.array([20, 18, 17]) - 1), cell, CUT, np.float32(-sign * 2.0))
        h = (cell * rng.uniform(0.05, 0.8, 3) * rng.choice([-1, 1], 3)).astype(np.float32)
        o = (F.amin + F.cell * 8.5).astype(np.float32)
        m = 400
        lo = rng.integers(-6, 6, (m, 3))
        hi = lo + rng.integers(0, 9, (m, 3))
        iso = (F.th + sign * rng.uniform(0, 4, m)).astype(np.float32)
        pa = (o + lo.astype(np.float32) * h).astype(np.float32)
        pb = (o + hi.astype(np.float32) * h).astype(np.float32)
        a, b = np.minimum(pa, pb), np.maximum(pa, pb)
        cl = ef.classify_lattice(F, o, h, lo, hi, iso)
        cb = ef.classify_box(F, a, b, iso)
        assert np.array_equal(cl, cb)
        seen |= set(cl.tolist())
    assert seen == {0, 1, 2}


def test_box_coverage():
    """every float(x) of every Gauss point lies in its element's box, on fuzzed general hexes and tets: rotated, nearly flat, near 1e3,
    straddling 0, tiny and large.  The analysis of r2s_elemfrac.cuh bounds the rounding of x far below a Float32 step wherever a Gauss point
    can come near the box's edge, so the fuzzing does not find a point outside the box without its margins either: that count is printed,
    and the margins are what the stated argument needs, not a fix for a case seen"""
    rng = np.random.default_rng(9)
    outside_bare = 0
    total = 0
    for nen in (8, 4):
        for center, size in ((np.zeros(3), 1.0), (np.full(3, 1000.0), 0.37), (np.array([1e-7, -1e-7, 0.0]), 1e-6), (np.array([0.0, 3e5, -2.0]), 50.0)):
            X, IEN = fuzz_mesh(rng, nen, 30, center, size, thin=True)
            a, b = ef.boxes(X, IEN)
            a0, b0 = ef.boxes(X, IEN, widen=False)
            for q in (1, 2, 5, 15, 32):
                for e in range(len(IEN)):
                    x, _, ok = ef.points(X, IEN, e, q)
                    p = x[ok].astype(np.float32)
                    assert (p >= a[e]).all() and (p <= b[e]).all(), (nen, center, q, e)
                    outside_bare += int(((p < a0[e]) | (p > b0[e])).sum())
                    total += len(p)
    print("box coverage: %d Gauss points, %d outside the box without its one-step widening" % (total, outside_bare))


def test_skip_soundness():
    """On the float64 CG weights of a sphere replica (tests/cg_ref.py) and a mesh of hexes two coarse cells wide (and the same cells split
    into tets), every element the classifier skips evaluates to exactly 1 or 0 in the replay, which evaluates every Gauss point, and a
    stated share is skipped"""
    shape = (40, 38, 36)
    s = cg_ref.process(cg_ref.make_field("smooth", shape)).astype(np.float64)
    w, _, _ = cg_ref.cg64(s)
    F = sample_ref.Field(w.astype(np.float32), np.zeros(3), np.array(shape, np.float64) - 1, 1.0, CUT, np.float32(0.0))
    n = (np.array(shape) - 1) // 2
    g = [np.arange(n[d] + 1) * 2.0 + 0.013 * d for d in range(3)]
    z, y, x = np.meshgrid(g[2], g[1], g[0], indexing="ij")
    X = np.stack([x.ravel(), y.ravel(), z.ravel()], 1)
    k, j, i = np.meshgrid(np.arange(n[2]), np.arange(n[1]), np.arange(n[0]), indexing="ij")
    b = ((k * (n[1] + 1) + j) * (n[0] + 1) + i).ravel()
    sx, sy = 1, n[0] + 1
    sz = sy * (n[1] + 1)
    H = np.stack([b, b + sx, b + sx + sy, b + sy, b + sz, b + sx + sz, b + sx + sy + sz, b + sy + sz], 1).astype(np.int64)
    T = np.concatenate([H[:, list(t)] for t in ([0, 1, 2, 6], [0, 2, 3, 6], [0, 4, 5, 6])])
    for IEN in (H, T):
        for q, iso in ((3, 0.0), (5, 0.17)):
            frac, vol, cls = ef.replay(F, X, IEN, q, np.float32(iso))
            assert (frac[cls == 1] == 1.0).all() and (frac[cls == 2] == 0.0).all()
            assert (vol > 0).all()
            share = float((cls != 0).mean())
            print("sphere replica, %s, q=%d iso=%g: %d elements, %.1f %% skipped (%d inside, %d outside), %d partial" %
                  ("HEX8" if IEN.shape[1] == 8 else "TET4", q, iso, len(cls), 100 * share, (cls == 1).sum(), (cls == 2).sum(),
                   ((frac > 0) & (frac < 1)).sum()))
            assert share >= 0.5 and (cls == 2).any() and ((frac > 0) & (frac < 1)).any()
            assert (cls == 1).any() or iso > 0      # above th = 0 only the lower bound of the sum can prove a box inside
