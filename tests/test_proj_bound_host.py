"""CPU tests of the lower bound the box projection prunes with (rho2sdf.jl_b200/csrc/r2s_bound.cuh, host build tests/host/bound_host.cpp):
the distance from a grid point to (tight box of the iso-patch) /\\ (slab that holds the patch) must never exceed the distance the solver
reports, must equal the exact distance to box /\\ slab up to its rounding margin, and, used with a per-point seed on a replica of the
bench workload, must prune only pairs that cannot change a point's minimum."""
import numpy as np
import pytest

import bound_ref as ref
import oracle
from fixtures import Grid, simp_hex8

SG = np.array([[-1, -1, -1], [1, -1, -1], [1, 1, -1], [-1, 1, -1], [-1, -1, 1], [1, -1, 1], [1, 1, 1], [-1, 1, 1]], float)
EDGES = [(0, 1), (1, 2), (2, 3), (3, 0), (4, 5), (5, 6), (6, 7), (7, 4), (0, 4), (1, 5), (2, 6), (3, 7)]


def _densities(rng, kind, rho_t):
    if kind == "random":
        return rng.uniform(0, 1, 8)
    if kind == "saddle":      # rho_t + a * xi0 xi1 xi2 (+ a little noise): the gradient vanishes at the centre
        return rho_t + rng.uniform(0.05, 0.5) * SG.prod(1) + rng.uniform(-1, 1, 8) * rng.choice([0.0, 1e-3, 0.05])
    if kind == "saddle2":     # rho_t + a * xi0 xi1: a saddle line through the element
        return rho_t + rng.uniform(0.05, 0.5) * SG[:, 0] * SG[:, 1] + rng.uniform(-1, 1, 8) * 1e-4
    if kind == "corners":     # iso through nodes
        re = rng.uniform(0, 1, 8); re[rng.choice(8, rng.integers(1, 4), replace=False)] = rho_t
        return re
    if kind == "edge":        # iso along an edge
        re = rng.uniform(0, 1, 8); a, b = EDGES[rng.integers(12)]; re[a] = re[b] = rho_t
        return re
    if kind == "flat":        # nearly no gradient
        return rho_t + rng.uniform(-1, 1, 8) * rng.choice([1e-6, 1e-9, 1e-12])
    raise ValueError(kind)


def _points(rng, c, h, m):
    """points inside, on the faces / edges / nodes of, and outside the element c + h [-1, 1]^3"""
    P = [c + rng.uniform(-1, 1, (m, 3)) * h, c + rng.uniform(-3, 3, (m, 3)) * h, c + SG * h, c + rng.integers(-3, 4, (m, 3)) * h / 2]
    Q = c + rng.uniform(-1, 1, (m, 3)) * h
    ax = rng.integers(0, 3, m); Q[np.arange(m), ax] = c[ax] + rng.choice([-1.0, 1.0], m) * h[ax]
    return np.concatenate(P + [Q])


@pytest.mark.parametrize("kind", ["random", "saddle", "saddle2", "corners", "edge", "flat"])
@pytest.mark.parametrize("far", [False, True])
def test_bound_never_exceeds_the_solver_distance(kind, far):
    rng = np.random.default_rng(1000 + 7 * ["random", "saddle", "saddle2", "corners", "edge", "flat"].index(kind) + int(far))
    n_el = n_pts = n_slab = n_bad = 0; worst = 0.0
    while n_el < 150:
        rho_t = float(rng.choice([0.3, 0.5]))
        h = rng.uniform(0.05, 2.0, 3) if rng.random() < 0.5 else np.full(3, rng.uniform(0.05, 2.0))
        c = rng.uniform(-1e3, 1e3, 3) if far else rng.uniform(-3, 3, 3)
        re = _densities(rng, kind, rho_t)
        if not (re.min() < rho_t < re.max()):      # crossing elements only (k_classify)
            continue
        Xe = c + SG * h
        rec = ref.element(Xe, re, rho_t)
        assert rec is not None
        P = _points(rng, c, h, 40)
        d, ok, _ = ref.project(Xe, re, rho_t, P)
        lb = ref.lb(P, rec)
        lb2g = ref.lb2_gap(P, rec)
        assert np.all(lb2g[ok] <= d[ok] ** 2)      # the cheap test before lb_box_slab is sound as well
        n_el += 1; n_pts += int(ok.sum()); n_slab += int(np.isfinite(rec[9])); n_bad += int((~ok).sum())
        assert np.all(lb >= 0.0)
        worst = max(worst, float(np.max(np.where(ok, lb - d, -np.inf))))
        assert np.all(lb[ok] <= d[ok]), (kind, far, Xe[0], re.tolist(), rho_t, float(np.max(lb[ok] - d[ok])))
    print("%s far=%s: %d elements (%d with a bounded slab), %d converged pairs, %d not converged, max(lb - d) = %.3g" % (kind, far, n_el, n_slab, n_pts, n_bad, worst))
    assert n_pts > (0.5 if kind == "flat" else 0.9) * 150 * 168      # the solver gives up on a part of the nearly flat elements
    if kind in ("random", "corners", "edge"):
        assert n_slab >= 10      # the slab is exercised, not only the tight box


def _random_box_slab(rng, far):
    o = rng.uniform(-1e3, 1e3, 3) if far else rng.uniform(-2, 2, 3)
    lo = o + rng.uniform(-1, 0, 3); hi = lo + rng.uniform(0.01, 2, 3)
    if rng.random() < 0.2:
        k = rng.integers(3); hi[k] = lo[k] + rng.uniform(1e-9, 1e-6)           # nearly flat box
    n = rng.normal(size=3)
    if rng.random() < 0.3:
        n[rng.integers(3)] = 0.0
    if rng.random() < 0.1:
        n[:2] *= 1e-7                                                            # nearly along an axis
    n /= np.linalg.norm(n)
    cs = SG * (hi - lo) / 2 + (hi + lo) / 2
    proj = cs @ n
    a, b = np.sort(rng.uniform(proj.min(), proj.max(), 2))
    if rng.random() < 0.2:
        b = a + rng.uniform(0, 1e-9)                                             # a thin slab
    P = np.concatenate([(hi + lo) / 2 + rng.uniform(-3, 3, (20, 3)) * (hi - lo), rng.uniform(-3, 3, (5, 3)) + lo])
    return lo, hi, n, float(a), float(b), P


@pytest.mark.parametrize("far", [False, True])
def test_bound_is_the_distance_to_box_and_slab(far):
    """lb_box_slab against the exact distance (active-set enumeration): never above it, and never below the distance to the box and the
    slab widened by the bound's rounding margin 1e-14 (|P|_1 + |tlo|_1 + |thi|_1) -- where the slab is nearly parallel to a face the
    point is clamped to, the root is ill-conditioned and only that weaker statement holds"""
    rng = np.random.default_rng(77 + int(far))
    worst = 0.0
    for _ in range(400):
        lo, hi, n, a, b, P = _random_box_slab(rng, far)
        rec = np.concatenate([lo, hi, n, [a, b]])
        got = ref.lb(P, rec)
        for q in range(len(P)):
            ex = ref.box_slab_distance(P[q], lo, hi, n, a, b)
            scale = np.abs(P[q]).sum() + np.abs(lo).sum() + np.abs(hi).sum()
            dl = 1e-14 * scale
            ex_w = ref.box_slab_distance(P[q], lo, hi, n, a - 2 * dl, b + 2 * dl)
            assert np.isfinite(ex)
            assert got[q] <= ex * (1 + 1e-15) + 1e-15 * scale, (P[q].tolist(), rec.tolist(), got[q], ex)
            assert got[q] >= ex_w * (1 - 2e-14) - 2 * dl, (P[q].tolist(), rec.tolist(), got[q], ex_w)
            worst = max(worst, (ex - got[q]) / (1e-14 * (ex + scale)))
    print("far=%s: largest shortfall against the exact distance %.3g x (1e-14 (d + scale))" % (far, worst))


def test_bound_against_a_scipy_qp():
    """the same distance from scipy's SLSQP on a sample (its own tolerance: 1e-7 relative)"""
    from scipy.optimize import minimize
    rng = np.random.default_rng(5)
    for _ in range(60):
        lo, hi, n, a, b, P = _random_box_slab(rng, False)
        if (hi - lo).min() < 1e-3 or b - a < 1e-6:
            continue
        got = ref.lb(P[:5], np.concatenate([lo, hi, n, [a, b]]))
        for q in range(5):
            y0 = np.clip(P[q], lo, hi)
            res = minimize(lambda y: float(((y - P[q]) ** 2).sum()), y0, jac=lambda y: 2 * (y - P[q]), method="SLSQP", bounds=list(zip(lo, hi)),
                           constraints=[{"type": "ineq", "fun": lambda y: float(n @ y - a), "jac": lambda y: n},
                                        {"type": "ineq", "fun": lambda y: float(b - n @ y), "jac": lambda y: -n}], options={"ftol": 1e-15, "maxiter": 500})
            ex = float(np.sqrt(res.fun))
            assert abs(got[q] - ex) <= 1e-6 * (1 + ex), (got[q], ex)


def _replica(n, period):
    X, IEN, rho = simp_hex8(n, period_frac=period / n)
    g = Grid(X.min(0), X.max(0), 2 * n, 3)
    rn = oracle.nodal_densities(X, IEN, rho)
    return X, IEN, g, rn


def test_seeded_pruning_on_the_replica():
    """Pass A solves, per grid point, the pair with the nearest tight box (Float32 distance rounded down, ties to the smaller element);
    pass B prunes a pair iff its tight-box bound, its box + slab-gap bound or its box /\\ slab bound is above the point's minimum after
    pass A (relative margin 1e-10, as the scans).  Every pruned pair must be at least the point's final minimum."""
    X, IEN, g, rn = _replica(24, 64.0)
    rho_t, delta = 0.5, 1.1 * g.cell_size
    re_all = rn[IEN - 1]
    crossing = np.nonzero((re_all.min(1) < rho_t) & (re_all.max(1) > rho_t))[0]
    npx = g.N + 1
    pc = [g.AABB_min[d] + g.cell_size * np.arange(npx[d]) for d in range(3)]
    vox, dist, lbs, lbb, lbg, eid = [], [], [], [], [], []
    for a, e in enumerate(crossing):
        Xe = X[IEN[e] - 1]; re = re_all[e]
        lo, hi = Xe.min(0), Xe.max(0)
        rng_ = [np.arange(max(int(np.floor(g.N[d] * ((lo[d] - delta) - g.AABB_min[d]) / (g.AABB_max[d] - g.AABB_min[d]))), 0),
                          min(int(np.floor(g.N[d] * ((hi[d] + delta) - g.AABB_min[d]) / (g.AABB_max[d] - g.AABB_min[d]))), g.N[d]) + 1) for d in range(3)]
        K, J, I = np.meshgrid(rng_[2], rng_[1], rng_[0], indexing="ij")
        P = np.stack([pc[0][I.ravel()], pc[1][J.ravel()], pc[2][K.ravel()]], 1)
        rec = ref.element(Xe, re, rho_t)
        d, ok, _ = ref.project(Xe, re, rho_t, P)
        assert ok.all()
        vox.append(((K * npx[1] + J) * npx[0] + I).ravel()); dist.append(d); lbs.append(ref.lb(P, rec)); lbg.append(ref.lb2_gap(P, rec))
        lbb.append(np.linalg.norm(np.maximum(np.maximum(rec[0:3] - P, P - rec[3:6]), 0), axis=1)); eid.append(np.full(len(P), a))
    vox, dist, lbs, lbb, lbg, eid = map(np.concatenate, (vox, dist, lbs, lbb, lbg, eid))
    assert np.all(lbs <= dist) and np.all(lbb <= lbs + 1e-10)
    # seed: smallest (float32 of the tight-box bound rounded down, element)
    f = lbb.astype(np.float32)
    f = np.where(f.astype(np.float64) > lbb, np.nextafter(f, np.float32(-np.inf)), f)
    order = np.lexsort((eid, f, vox))
    first = np.r_[True, vox[order][1:] != vox[order][:-1]]
    seed = np.zeros(len(vox), bool); seed[order[first]] = True
    cur = np.full(int(g.ngp), np.inf); np.minimum.at(cur, vox[seed], dist[seed])
    c2 = cur[vox] ** 2 * (1 + 1e-10)
    pruned = ~seed & ((lbb ** 2 > c2) | (lbg > c2) | (lbs ** 2 > c2))
    final = np.full(int(g.ngp), np.inf); np.minimum.at(final, vox, dist)
    assert np.all(dist[pruned] >= final[vox[pruned]])
    solved = 1 - pruned.mean()
    print("replica n=24: %d crossing elements, %d pairs, %.1f%% solved (seeds %.1f%%)" % (len(crossing), len(vox), 100 * solved, 100 * seed.mean()))
    assert solved < 0.35
