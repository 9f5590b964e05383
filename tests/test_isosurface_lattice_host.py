"""CPU tests of the vertex search of r2s_isosurface_lattice (rho2sdf.jl_b200/csrc/r2s_snap.cuh, host build tests/host/snap_host.cpp): the
host build against a plain-Python restatement of the rule, and the properties include/r2s.h states -- the vertex lies on its edge, it is
an end of the final bracket, the bracket's ends straddle iso under the inside rule and are adjacent floats unless the evaluation cap
stopped the search, ties and exact-iso ends -- on constructed edges (monotone, non-monotone, noisy) and on lattice edges of random fields."""
import numpy as np
import pytest

import sample_ref
import snap_ref as ref
from test_sample_host import _field

f32 = np.float32


def _check(f, xa, xb, va, vb, iso, out):
    x, (lo, hi, flo, fhi), ev = out
    iso = f32(iso)
    assert min(xa, xb) <= x <= max(xa, xb)
    assert x == lo or x == hi
    # the invariant: s(lo) = s(a), s(hi) = s(b), with the bracket values f at the bracket ends (the lattice values at the start)
    assert (flo >= iso) == (va >= iso) and (fhi >= iso) == (vb >= iso)
    assert flo == (va if lo == xa else f(lo)) and fhi == (vb if hi == xb else f(hi))
    if ev < ref.max_evals():
        assert ref.adjacent(lo, hi)
    pick_hi = abs(float(fhi) - float(iso)) < abs(float(flo) - float(iso))
    assert x == (hi if pick_hi else lo)
    return ev


def _edges(rng, n):
    """random constructed edges: (Poly, xa, xb, iso) with the ends on different sides of iso"""
    out = []
    while len(out) < n:
        kind = rng.integers(0, 4)
        x0 = f32(rng.uniform(-50, 50))
        h = f32(10.0 ** rng.uniform(-6, 1)) * (1 if rng.random() < 0.85 else -1)      # a few edges run downwards
        xa, xb = x0, f32(x0 + h)
        r = f32(rng.uniform(min(xa, xb), max(xa, xb)))
        if kind == 0:      # linear, root r
            c = [-float(r) * 2.0, 2.0, 0.0, 0.0]; amp = 0.0
        elif kind == 1:    # cubic with a root in the edge (monotone or not across it)
            s = rng.uniform(-3, 3) / float(abs(h)) ** 2
            c = [-float(r) + s * float(r) ** 3, 1.0, -3 * s * float(r), s]; amp = 0.0
        elif kind == 2:    # steep linear plus hash noise: s(x) non-monotone near the root
            c = [-float(r), 1.0, 0.0, 0.0]; amp = float(abs(h)) * 10.0 ** rng.uniform(-9, -2)
        else:              # flat noise around iso: s(x) is random along the whole edge
            c = [0.0, 0.0, 0.0, 0.0]; amp = 1.0
        p = ref.Poly(c, amp)
        iso = f32(rng.choice([0.0, 1e-7, -0.25]) if kind != 3 else 0.0)
        if (p(xa) >= iso) != (p(xb) >= iso):
            out.append((p, xa, xb, iso))
    return out


def test_host_build_equals_python_restatement():
    rng = np.random.default_rng(1)
    caps = evs = 0
    edges = _edges(rng, 600)
    for p, xa, xb, iso in edges:
        va, vb = p(xa), p(xb)
        got = p.search(xa, xb, iso)
        want = ref.python_search(p, xa, xb, va, vb, iso, cap=ref.max_evals())
        assert got[0] == want[0] and got[1] == want[1] and got[2] == want[2], (p.c, p.amp, xa, xb, iso, got, want)
        ev = _check(p, xa, xb, va, vb, iso, got)
        caps += ev >= ref.max_evals(); evs += ev
    print("constructed edges: %d, mean evaluations %.2f, stopped by the cap: %d" % (len(edges), evs / len(edges), caps))


def test_monotone_edges_converge_to_adjacent_floats_at_the_root():
    """a linear function with a float root r inside the edge: the bracket closes on r; the vertex is r or its neighbour, whichever is nearer"""
    rng = np.random.default_rng(2)
    for _ in range(300):
        xa = f32(rng.uniform(-10, 10)); xb = f32(xa + f32(10.0 ** rng.uniform(-5, 0)))
        r = f32(rng.uniform(xa, xb))
        if not xa < r < xb:
            continue
        p = ref.Poly([-float(r), 1.0, 0.0, 0.0])
        x, (lo, hi, flo, fhi), ev = p.search(xa, xb, 0.0)
        assert ev < ref.max_evals() and ref.adjacent(lo, hi)
        assert hi == r and x == r and fhi == 0.0      # f(r) = 0 >= iso: r is the inside end (b's side), at zero residual


def test_ties_and_exact_iso_ends():
    # adjacent ends: no evaluation; equal residuals go to lo, a smaller one at b to hi
    xa = f32(1.0); xb = np.nextafter(xa, f32(2))
    p = ref.Poly([0.0, 0.0, 0.0, 0.0])
    assert p.search(xa, xb, 0.0, va=0.5, vb=-0.5) == (xa, (xa, xb, f32(0.5), f32(-0.5)), 0)
    assert p.search(xa, xb, 0.0, va=0.5, vb=-0.25)[0] == xb
    assert p.search(xb, xa, 0.0, va=-0.5, vb=0.5)[0] == xb      # a downward edge: lo is its first end
    assert p.search(xa, xa, 0.0, va=0.5, vb=-0.5)[0] == xa      # a zero-length edge (spacing below the coordinate's resolution)
    # f(x_a) == iso: a is inside and at zero residual; every interior point is outside, so the bracket closes on a and the vertex is a
    p = ref.Poly([1.0, -1.0, 0.0, 0.0])
    x, (lo, hi, flo, fhi), ev = p.search(1.0, 1.5, 0.0)
    assert x == f32(1.0) and lo == f32(1.0) and hi == np.nextafter(f32(1.0), f32(2)) and flo == 0.0
    # f(x_b) == iso and x_a outside: b is the inside end at zero residual
    p = ref.Poly([-1.5, 1.0, 0.0, 0.0])
    x, (lo, hi, flo, fhi), ev = p.search(1.0, 1.5, 0.0)
    assert x == f32(1.5) and hi == f32(1.5) and fhi == 0.0 and ref.adjacent(lo, hi)
    # iso = -0.0 against +-0 values: the inside rule is value >= iso, so -0.0 and +0.0 are both inside
    p = ref.Poly([1.0, -1.0, 0.0, 0.0])      # 1 - x: inside for x <= 1
    x, (lo, hi, flo, fhi), ev = p.search(0.5, 2.0, -0.0)
    assert x == f32(1.0) and ref.adjacent(lo, hi)


def test_non_monotone_edges_keep_the_bracket():
    """noise of every amplitude: the vertex is still an end of a straddling bracket, adjacent unless capped; the cap is reported"""
    rng = np.random.default_rng(3)
    caps = 0
    for amp in (1e-7, 1e-4, 1e-2, 1.0):
        for _ in range(100):
            xa = f32(rng.uniform(-1, 1)); xb = f32(xa + f32(rng.uniform(1e-3, 1)))
            p = ref.Poly([-float(xa + xb) / 2, 1.0, 0.0, 0.0], amp)
            va, vb = p(xa), p(xb)
            if (va >= 0) == (vb >= 0):
                continue
            out = p.search(xa, xb, 0.0)
            assert out == ref.python_search(p, xa, xb, va, vb, 0.0)
            caps += _check(p, xa, xb, va, vb, 0.0, out) >= ref.max_evals()
    print("noisy edges stopped by the cap: %d" % caps)


def _sphere_field(shape, cut, seed, cell=0.5):
    """approximation-mode-like weights: a sphere's signed distance on the coarse points, with noise"""
    rng = np.random.default_rng(seed)
    nz, ny, nx = shape
    z, y, x = np.meshgrid(np.arange(nz), np.arange(ny), np.arange(nx), indexing="ij")
    c = (np.array([nx, ny, nz]) - 1) / 2.0
    d = 0.35 * min(shape) - np.sqrt((x - c[0]) ** 2 + (y - c[1]) ** 2 + (z - c[2]) ** 2)
    w = (cell * d + 0.2 * cell * rng.standard_normal(d.shape)).astype(np.float32)
    amin = np.array([0.25, -1.0, 3.0])
    return sample_ref.Field(w, amin, amin + cell * (np.array([nx, ny, nz]) - 1), cell, cut, 0.0)


def _lattice_points(o, h, shape):
    o32, h32 = np.float32(o), np.float32(h)
    ax = [(o32[d] + np.arange(shape[d], dtype=np.float32) * h32[d]).astype(np.float32) for d in range(3)]
    kk, jj, ii = np.meshgrid(np.arange(shape[2]), np.arange(shape[1]), np.arange(shape[0]), indexing="ij")
    return np.stack([ax[0][ii.ravel()], ax[1][jj.ravel()], ax[2][kk.ravel()]], 1).astype(np.float64)


@pytest.mark.parametrize("kind", ["sphere", "random"])
@pytest.mark.parametrize("cut", [1e-3, 1e-2])
def test_lattice_edges_of_random_fields(kind, cut):
    """every crossing edge of a lattice over the field: vertex on the edge, an end of a straddling bracket whose values are the sampler's
    values at its ends, adjacent floats unless capped; 40 edges also against the Python restatement with the host sampler as f"""
    F = _sphere_field((12, 11, 13), cut, seed=4) if kind == "sphere" else _field((9, 8, 10), cut, seed=5, cell=0.7, amin=(-1.0, 2.0, 0.5))
    iso = f32(0.0) if kind == "sphere" else f32(0.3)
    o = F.amin - 0.8 * F.cell
    h = np.array([0.23, 0.31, 0.27]) * F.cell
    shape = tuple(int(v) for v in np.ceil((F.amax - o + 0.8 * F.cell) / h))
    val = F.host(_lattice_points(o, h, shape)).reshape(shape[::-1])
    E = ref.crossing_edges(val, iso)
    V, tr, ev = ref.lattice_vertices(F, o, h, E, iso)
    assert len(E) > 200
    o32, h32 = np.float32(o), np.float32(h)
    P = (o32[None, :] + E[:, :3].astype(np.float32) * h32[None, :]).astype(np.float32)
    ax = E[:, 3]
    rows = np.arange(len(E))
    xa = P[rows, ax]
    xb = (o32[ax] + (E[rows, ax] + 1).astype(np.float32) * h32[ax]).astype(np.float32)
    # off-axis coordinates are the lattice's; the axis coordinate is in [x_a, x_b] and is lo or hi
    Vo = V.copy(); Vo[rows, ax] = P[rows, ax]
    assert np.array_equal(Vo, P)
    x = V[rows, ax]
    assert ((x >= np.minimum(xa, xb)) & (x <= np.maximum(xa, xb))).all()
    assert ((x == tr[:, 0]) | (x == tr[:, 1])).all()
    # the bracket values are the sampler's at the bracket ends, and they straddle iso as the lattice ends do
    va = val.ravel()[(E[:, 2] * shape[1] + E[:, 1]) * shape[0] + E[:, 0]]
    for end, col in ((0, 2), (1, 3)):
        Q = P.astype(np.float64).copy(); Q[rows, ax] = tr[:, end]
        assert np.array_equal(F.host(Q), tr[:, col])
    assert np.array_equal(tr[:, 2] >= iso, va >= iso) and np.array_equal(tr[:, 3] >= iso, ~(va >= iso))
    capped = ev >= ref.max_evals()
    adj = np.array([ref.adjacent(a, b) for a, b in tr[:, :2]])
    assert (adj | capped).all()
    print("%s cut=%g: %d edges, evaluations mean %.2f max %d, stopped by the cap: %d" % (kind, cut, len(E), ev.mean(), ev.max(), capped.sum()))
    for q in np.random.default_rng(6).choice(len(E), 40, replace=False):
        def f(v, q=q):
            p = P[q].astype(np.float64).copy(); p[ax[q]] = v
            return F.host(p[None, :])[0]
        vb = F.host(np.where(np.arange(3) == ax[q], xb[q], P[q]).astype(np.float64)[None, :])[0]
        xq, brq, eq = ref.python_search(f, xa[q], xb[q], va[q], vb, iso)
        assert xq == x[q] and brq == tuple(tr[q]) and eq == ev[q]
