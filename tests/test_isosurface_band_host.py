"""CPU tests of the block classifier of r2s_isosurface_band (rho2sdf.jl_b200/csrc/r2s_band.cuh), built for the host with the host sampler
(tests/host/band_host.cpp): every block declared one-sided has every lattice point, evaluated bit for bit by the host sampler, on that
side -- at the exact boundary of the lower-bound branch, across the cut radius, at spacings from 1e-3 to 2 cells and origins near 1e3.
The same classifier without its rounding terms is caught by those cases, and on the float64 CG weights of a sphere replica (tests/cg_ref.py)
at a cell / 4 lattice most blocks are skipped."""
import ctypes as C
import os
import subprocess

import numpy as np
import pytest

import cg_ref
import sample_ref

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
CUT = 1e-3
_LIB = None


def lib():
    global _LIB
    if _LIB is None:
        src = os.path.join(HERE, "host", "band_host.cpp")
        so = os.path.join(HERE, "host", "libband_host.so")
        deps = [src] + [os.path.join(ROOT, "rho2sdf.jl_b200", "csrc", f) for f in ("r2s_sample.cuh", "r2s_band.cuh")]
        if not os.path.exists(so) or os.path.getmtime(so) < max(os.path.getmtime(d) for d in deps):
            subprocess.check_call(["g++", "-O2", "-std=c++17", "-ffp-contract=off", "-fopenmp", "-fPIC", "-shared", src, "-o", so])
        L = C.CDLL(so)
        fp = np.ctypeslib.ndpointer(np.float32, flags="C")
        dp = np.ctypeslib.ndpointer(np.float64, flags="C")
        ip = np.ctypeslib.ndpointer(np.int32, flags="C")
        lp = np.ctypeslib.ndpointer(np.int64, flags="C")
        L.band_host_block.restype = C.c_int
        L.band_host_classify.argtypes = [fp, ip, dp, dp, C.c_double, C.c_double, C.c_float, fp, fp, lp, C.c_long, fp, C.c_int, C.c_int, ip, lp, fp, fp]
        _LIB = L
    return _LIB


def classify(F, o, h, boxes, iso, exact=True, check=False):
    """(cls, wrong, vmin, vmax) per box of the lattice o + float(i) h (boxes: (m, 6) lo, hi) on the Field F, iso per box or one value"""
    boxes = np.ascontiguousarray(boxes, np.int64).reshape(-1, 6)
    m = len(boxes)
    iso = np.ascontiguousarray(np.broadcast_to(np.asarray(iso, np.float32), (m,)))
    cls = np.zeros(m, np.int32); wrong = np.zeros(m, np.int64); vmin = np.zeros(m, np.float32); vmax = np.zeros(m, np.float32)
    lib().band_host_classify(F.w, F.n, F.amin, F.amax, F.cell, F.cut, float(F.th), np.asarray(o, np.float32), np.asarray(h, np.float32), boxes, m, iso,
                             int(exact), int(check), cls, wrong, vmin, vmax)
    return cls, wrong, vmin, vmax


def key(x):
    u = np.asarray(x, np.float32).view(np.uint32).astype(np.int64)
    return np.where(u & 0x80000000, 0xffffffff - u, u | 0x80000000)


def unkey(k):
    k = np.asarray(k, np.int64)
    u = np.where(k & 0x80000000, k & 0x7fffffff, 0xffffffff - k).astype(np.uint32)
    return u.view(np.float32)


def boundary_iso(F, o, h, boxes, side, exact):
    """per box, the iso at the edge of the classifier's answer `side`: the largest iso declared inside (side 1) or the smallest declared
    outside (side 2), by bisection over the Float32 order; NaN where no iso in the searched range gets that answer"""
    m = len(boxes)
    th = np.float32(F.th)
    if side == 1:      # th >= iso: inside whenever the weights allow it; a large iso: never
        good, bad = np.full(m, key(th)), np.full(m, key(th + np.float32(1e6)))
    else:
        good, bad = np.full(m, key(np.nextafter(th, np.float32(np.inf)))), np.full(m, key(th - np.float32(1e6)))
    ok = classify(F, o, h, boxes, unkey(good), exact)[0] == side
    for _ in range(34):
        mid = np.where(good < bad, good + (bad - good) // 2, bad + (good - bad) // 2)
        c = classify(F, o, h, boxes, unkey(mid), exact)[0] == side
        good, bad = np.where(c, mid, good), np.where(c, bad, mid)
    return np.where(ok, unkey(good), np.nan)


def field(rng, shape, cell, amin, sign, lo=0.05, hi=1.0):
    w = (sign * rng.uniform(lo, hi, size=shape[::-1])).astype(np.float32)
    amin = np.asarray(amin, np.float64)
    return sample_ref.Field(w, amin, amin + cell * (np.array(shape) - 1), cell, CUT, np.float32(-sign * 3.0 * rng.uniform(0.5, 1.5)))


def boxes_in(rng, F, o, h, m, ext):
    """m boxes of extent ext (points - 1 per axis) at random lattice positions whose points stay inside the grid's interior"""
    a, b = F.amin + 2.5 * F.cell, F.amax - 2.5 * F.cell - ext * np.abs(h)
    i0 = np.ceil((a - o) / h)
    i1 = np.floor((b - o) / h)
    lo = np.stack([rng.integers(int(i0[d]), int(i1[d]) + 1, size=m) for d in range(3)], axis=1)
    return np.concatenate([lo, lo + np.asarray(ext, np.int64)], axis=1)


CASES = [  # (cell, grid origin, lattice spacing in cells, box extents)
    (1.0, (0.0, 0.0, 0.0), 0.25, [(0, 0, 0), (1, 1, 1), (8, 8, 8), (0, 3, 0)]),
    (0.37, (1000.0, 999.3, 1000.6), 1e-3, [(0, 0, 0), (2, 1, 1), (8, 8, 8)]),
    (1.0, (997.0, 1001.5, 1000.0), 2.0, [(0, 0, 0), (1, 1, 1), (3, 3, 3)]),
    (2.5, (-3.0, 1003.0, 0.5), 0.7, [(0, 0, 0), (8, 8, 8), (1, 0, 4)]),
]


@pytest.mark.parametrize("case", range(len(CASES)))
@pytest.mark.parametrize("sign", [1, -1])
def test_lower_bound_boundary(case, sign):
    """Same-signed weights and th on the other side of iso: the lower-bound branch decides.  At the boundary iso of every box (and a few
    ulps inside it) every lattice point is on the declared side; the variant without rounding terms puts points on the wrong side."""
    cell, amin, hc, exts = CASES[case]
    rng = np.random.default_rng(100 * case + (sign > 0))
    F = field(rng, (20, 18, 17), cell, amin, sign)
    side = 1 if sign > 0 else 2
    caught = 0
    for ext in exts:
        h = np.float32(hc * cell) * np.array([1.0, 0.93, 1.07], np.float32)
        o = (F.amin + rng.uniform(0, 1, 3) * cell).astype(np.float32)
        boxes = boxes_in(rng, F, o.astype(np.float64), h.astype(np.float64), 60, ext)
        for exact in (True, False):
            iso = boundary_iso(F, o, h, boxes, side, exact)
            sel = ~np.isnan(iso)
            assert sel.sum() >= 30 if exact else True, (ext, sel.sum())
            for step in ((0, -1, -2) if side == 1 else (0, 1, 2)):      # the boundary and iso moved towards the decided side
                isos = unkey(key(iso[sel]) + step)
                cls, wrong, vmin, vmax = classify(F, o, h, boxes[sel], isos, exact)
                assert (cls == side).all()
                if exact:
                    assert wrong.sum() == 0, (ext, step, np.flatnonzero(wrong))
                else:
                    caught += int(wrong.sum())
            if exact:      # one ulp past the boundary the block is sampled
                isos = unkey(key(iso[sel]) + (1 if side == 1 else -1))
                assert (classify(F, o, h, boxes[sel], isos, exact)[0] == 0).all()
                # the bound is tight where the box is a point: the decided iso is within 2^-13 of the sum |f - th| at the point
                _, _, vmin, vmax = classify(F, o, h, boxes[sel], iso[sel], exact, check=True)
                if ext == (0, 0, 0):
                    gap = np.abs(vmin.astype(np.float64) - iso[sel]) / np.abs(vmin.astype(np.float64) - float(F.th))
                    assert np.median(gap) < 2.0 ** -13, np.median(gap)
    assert caught > 0, "the classifier without rounding terms was not caught"


def _straddling_point(rng, F):
    """a point p and a coarse point c whose Float32 d2 (the sampler's) is <= t2 while the exact distance is beyond the cut radius"""
    c = np.array([F.n[d] // 2 for d in range(3)])
    C_ = np.array([F.C[d][c[d]] for d in range(3)], np.float32)
    t2 = np.float32(F.t2)
    for _ in range(20000):
        u = rng.normal(size=3); u /= np.linalg.norm(u)
        r = float(F.maxd) * (1.0 + rng.integers(-6, 7) * 2.0 ** -23)
        p = (C_.astype(np.float64) + r * u).astype(np.float32)
        e = (C_ - p).astype(np.float32)
        ee = (e * e).astype(np.float32)
        d2 = np.float32(np.float32(ee[0] + ee[1]) + ee[2])
        ex = np.sum((C_.astype(np.float64) - p.astype(np.float64)) ** 2)
        if d2 <= t2 and ex > float(t2) and len(F.taps(p)) > 0 and any(t[:3] == tuple(c) for t in F.taps(p)):
            return p, c
    raise AssertionError("no straddling point found")


@pytest.mark.parametrize("amin", [(0.0, 0.0, 0.0), (1000.0, 1000.0, 1000.0)])
def test_cut_radius(amin):
    """A tap the sampler includes although its exact distance is beyond the cut radius, with a large weight of the other sign: the
    classifier keeps it in the reach set and samples the block; without the margin it declares the block inside, and a point is not."""
    rng = np.random.default_rng(7)
    F = field(rng, (12, 12, 12), 1.0, amin, 1, lo=0.0, hi=1e-3)
    F.th = np.float32(0.0)
    p, c = _straddling_point(rng, F)
    F.w[c[2], c[1], c[0]] = -1000.0
    assert F.host(p[None].astype(np.float64))[0] < 0.0
    for h in (1e-3, 0.25):
        boxes = np.array([[0, 0, 0, 0, 0, 0], [0, 0, 0, 1, 1, 1]], np.int64)
        for exact in (True, False):
            cls, wrong, _, _ = classify(F, p, np.full(3, h, np.float32), boxes, 0.0, exact)
            if exact:
                assert (cls == 0).all()
            else:
                assert cls[0] == 1 and wrong[0] == 1


def test_nan_and_huge_weights_are_sampled():
    rng = np.random.default_rng(3)
    F = field(rng, (12, 12, 12), 1.0, (0, 0, 0), 1)
    o = (F.amin + 5.3).astype(np.float32)
    h = np.full(3, 0.2, np.float32)
    box = np.array([[0, 0, 0, 4, 4, 4]], np.int64)
    assert classify(F, o, h, box, F.th - 1)[0][0] == 1
    for bad in (np.nan, np.inf, 2.0 ** 101):
        w = F.w.copy()
        F.w[6, 6, 6] = bad
        assert classify(F, o, h, box, F.th - 1)[0][0] == 0, bad
        F.w = w


def test_sphere_replica_skips():
    """The float64 CG weights of the cg_ref sphere replica at a cell / 4 lattice: a stated share of the blocks is skipped, and every
    lattice point of a sample of the skipped blocks is on its block's side."""
    shape = (64, 60, 56)
    s = cg_ref.process(cg_ref.make_field("smooth", shape)).astype(np.float64)
    w, _, _ = cg_ref.cg64(s)
    F = sample_ref.Field(w[..., :].astype(np.float32), np.zeros(3), np.array(shape, np.float64) - 1, 1.0, CUT, np.float32(0.0))
    B = lib().band_host_block()
    dims = (np.array(shape) - 1) * 4 + 1
    nb = (dims - 2) // B + 1
    g = np.stack(np.meshgrid(np.arange(nb[2]), np.arange(nb[1]), np.arange(nb[0]), indexing="ij"), -1).reshape(-1, 3)[:, ::-1]
    lo = g * B
    boxes = np.concatenate([lo, np.minimum(lo + B, dims - 1)], axis=1)
    o, h = np.zeros(3, np.float32), np.full(3, 0.25, np.float32)
    cls, _, _, _ = classify(F, o, h, boxes, 0.0)
    share = float((cls != 0).mean())
    print("sphere replica, cell / 4 lattice %s: %d blocks, %.1f %% skipped (%d inside, %d outside)" % (tuple(dims), len(cls), 100 * share,
                                                                                                      (cls == 1).sum(), (cls == 2).sum()))
    assert share >= 0.6 and (cls == 1).any() and (cls == 2).any()
    rng = np.random.default_rng(0)
    pick = rng.choice(np.flatnonzero(cls != 0), 300, replace=False)
    c2, wrong, _, _ = classify(F, o, h, boxes[pick], 0.0, check=True)
    assert (c2 == cls[pick]).all() and wrong.sum() == 0
