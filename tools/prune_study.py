#!/usr/bin/env python
"""Offline study (CPU only) of how many (element, grid point) projections the distance field really needs.

The reference projects every grid point of an element's (AABB +- delta) range onto the element's iso-patch and keeps the
minimum per grid point (evalDistances).  A pair whose lower bound -- the distance from the point to a box that contains the
element's iso-patch -- is not below the point's final minimum cannot change the result.  This script counts, on a replica of
the bench workload, how many pairs survive (a) best-first pruning per grid point with the element AABB as the box, (b) the
same with the tight box of the iso-patch (sub-boxes of the element whose 8 corner densities straddle rho_t: a trilinear
field takes its extrema over a box at the corners, so the other sub-boxes hold no iso-surface), and the iteration statistics
a warp of 32 lanes sees.  Uses the host build of the projection solver (tests/host/libiso_host.so).

The last block counts the schemes of the device's pair scans with the device's own rules (host build of rho2sdf.jl_b200/csrc/r2s_bound.cuh,
tests/host/bound_host.cpp): the tight box of k_box_records, the slab that holds the iso-patch, the distance to box /\ slab, and how pass A
is chosen (pairs inside the element's box, or one pair per point with the smallest bound).  Solver iterations are those of the kernel's
path (element phase 1, FAST restoration)."""
import argparse, ctypes as C, os, subprocess, sys
import numpy as np
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT); sys.path.insert(0, os.path.join(ROOT, "tests"))
from fixtures import Grid, simp_hex8
import bound_ref
import oracle


def host_lib():
    d = os.path.join(ROOT, "tests", "host")
    so = os.path.join(d, "libiso_host.so")
    src = os.path.join(d, "iso_host.cpp")
    hdr = os.path.join(ROOT, "rho2sdf.jl_b200", "csrc", "r2s_iso.cuh")
    if not os.path.exists(so) or os.path.getmtime(so) < max(os.path.getmtime(src), os.path.getmtime(hdr)):
        subprocess.check_call(["g++", "-O2", "-std=c++17", "-ffp-contract=off", "-fPIC", "-shared", "-I/usr/local/cuda/include", src, "-o", so])
    L = C.CDLL(so)
    dp = np.ctypeslib.ndpointer(np.float64, flags="C"); ip = np.ctypeslib.ndpointer(np.int32, flags="C")
    L.iso_host_project_many.argtypes = [dp, dp, C.c_long, dp, C.c_double, C.c_int, dp, ip]
    L.iso_host_counts.argtypes = [np.ctypeslib.ndpointer(np.int64, flags="C"), C.c_int]
    return L


def tight_box(Xe, re, rho_t, m):
    """AABB (in x) of the sub-boxes (m per axis) of a box element that can hold iso-surface."""
    lo, hi = Xe.min(0), Xe.max(0)
    t = np.linspace(-1, 1, m + 1)
    SG = np.array([[-1, -1, -1], [1, -1, -1], [1, 1, -1], [-1, 1, -1], [-1, -1, 1], [1, -1, 1], [1, 1, 1], [-1, 1, 1]], float)
    Z, E, Xi = np.meshgrid(t, t, t, indexing="ij")
    N = np.stack([(1 + SG[a, 0] * Xi) * (1 + SG[a, 1] * E) * (1 + SG[a, 2] * Z) / 8 for a in range(8)], axis=-1)
    v = N @ re - rho_t                                    # [z][e][x] lattice values
    c = np.stack([v[k:k + m, j:j + m, i:i + m] for k in (0, 1) for j in (0, 1) for i in (0, 1)], axis=-1)
    has = (c.min(-1) <= 0) & (c.max(-1) >= 0)
    kz, ky, kx = np.nonzero(has)
    if kx.size == 0:
        return lo, hi
    f = lambda a, b, d: (lo[d] + (hi[d] - lo[d]) * a.min() / m, lo[d] + (hi[d] - lo[d]) * (b.max() + 1) / m)
    bx, by, bz = f(kx, kx, 0), f(ky, ky, 1), f(kz, kz, 2)
    return np.array([bx[0], by[0], bz[0]]), np.array([bx[1], by[1], bz[1]])


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--n", type=int, default=40)
    ap.add_argument("--period", type=float, default=64.0, help="period of the SIMP pattern in elements (64 in the bench workload)")
    ap.add_argument("--sub", type=int, default=4, help="sub-boxes per axis for the tight box")
    args = ap.parse_args()
    L = host_lib()
    n = args.n
    X, IEN, rho = simp_hex8(n, period_frac=args.period / n)
    g = Grid(X.min(0), X.max(0), 2 * n, 3)
    rn = oracle.nodal_densities(X, IEN, rho)
    rho_t, delta = 0.5, 1.1 * g.cell_size
    re_all = rn[IEN - 1]
    crossing = np.nonzero((re_all.min(1) < rho_t) & (re_all.max(1) > rho_t))[0]
    np_ax = g.N + 1
    pc = [g.AABB_min[d] + g.cell_size * np.arange(np_ax[d]) for d in range(3)]
    best = np.full(int(g.ngp), np.inf)
    recs = []           # (voxel ids, dist, lb_aabb, lb_tight, its)
    dev = []            # device rules: (voxel ids, dist, its, lb tight box, lb slab only, lb box /\ slab, element index)
    for e in crossing:
        Xe = X[IEN[e] - 1]; re = re_all[e]
        lo, hi = Xe.min(0), Xe.max(0)
        rng = []
        for d in range(3):
            I0 = int(np.floor(g.N[d] * ((lo[d] - delta) - g.AABB_min[d]) / (g.AABB_max[d] - g.AABB_min[d])))
            I1 = int(np.floor(g.N[d] * ((hi[d] + delta) - g.AABB_min[d]) / (g.AABB_max[d] - g.AABB_min[d])))
            rng.append(np.arange(max(I0, 0), min(I1, g.N[d]) + 1))
        K, J, I = np.meshgrid(rng[2], rng[1], rng[0], indexing="ij")
        vox = ((K * np_ax[1] + J) * np_ax[0] + I).ravel()
        P = np.stack([pc[0][I.ravel()], pc[1][J.ravel()], pc[2][K.ravel()]], axis=1)
        dist = np.zeros(len(vox)); its = np.zeros(len(vox), dtype=np.int32)
        L.iso_host_project_many(np.ascontiguousarray(Xe), np.ascontiguousarray(re), len(vox), np.ascontiguousarray(P), rho_t, 1, dist, its)
        lb = np.linalg.norm(np.maximum(np.maximum(lo - P, P - hi), 0), axis=1)
        tlo, thi = tight_box(Xe, re, rho_t, args.sub)
        lbt = np.linalg.norm(np.maximum(np.maximum(tlo - P, P - thi), 0), axis=1)
        assert np.all(lbt <= dist * (1 + 1e-9) + 1e-12), (e, float((lbt - dist).max()))
        np.minimum.at(best, vox, dist)
        recs.append((vox, dist, lb, lbt, its))
        rec = bound_ref.element(Xe, re, rho_t)
        dd, _, itd = bound_ref.project(Xe, re, rho_t, P)
        lbx = np.linalg.norm(np.maximum(np.maximum(rec[0:3] - P, P - rec[3:6]), 0), axis=1)
        t = P @ rec[6:9]
        lbsl = np.maximum(np.maximum(rec[9] - t, t - rec[10]), 0) if np.isfinite(rec[9]) else np.zeros(len(P))
        lbs = bound_ref.lb(P, rec)
        assert np.all(lbs <= dd), e
        dev.append((vox, dd, itd, lbx, lbsl, lbs, np.full(len(P), len(dev))))
    vox = np.concatenate([r[0] for r in recs]); dist = np.concatenate([r[1] for r in recs]); lb = np.concatenate([r[2] for r in recs])
    lbt = np.concatenate([r[3] for r in recs]); its = np.concatenate([r[4] for r in recs])
    npairs = len(vox); band = int(np.isfinite(best).sum())
    print("n=%d period=%g: %d crossing elements of %d (%.1f%%), %d pairs (%.1f per element), %d band grid points (%.1f candidates each)" % (
        n, args.period, len(crossing), len(rho), 100 * len(crossing) / len(rho), npairs, npairs / len(crossing), band, npairs / band))
    cnt = np.zeros(8, dtype=np.int64); L.iso_host_counts(cnt, 1)
    print("per pair: eval_full %.2f  eval_g %.2f  eval_f %.2f  tangent steps %.2f  line-search trials %.2f  active-set passes %.2f" % tuple(cnt[:6] / npairs))
    print("iterations per pair: mean %.2f  p50 %d  p90 %d  p99 %d  max %d" % (its.mean(), *np.percentile(its, [50, 90, 99]).astype(int), its.max()))
    # warp view of the chunk kernel: 32 consecutive pairs of one element wait for their slowest lane
    tot_w = 0; tot_l = 0
    for r in recs:
        it = r[4]
        for c0 in range(0, len(it), 32):
            ch = it[c0:c0 + 32]; tot_w += int(ch.max()) * 32; tot_l += int(ch.sum())
    print("chunk kernel: lane utilisation at iteration granularity %.1f%% (sum of iterations / 32 x slowest lane)" % (100 * tot_l / tot_w))
    # lane-refill kernels at iteration granularity: a lane that finishes takes the next point.  (b) one warp per element, drained at
    # the element's end (k_project_hex8_min); (c) persistent warp that moves on to its next element without draining.
    def simulate(seqs):
        """seqs: list of per-warp work lists (iterations per pair, in order).  Returns (useful lane-iterations, issued warp-iterations x 32)."""
        useful = issued = 0
        for w in seqs:
            lanes = np.zeros(32, dtype=np.int64); q = 0; nw = len(w)
            while True:
                for l in np.nonzero(lanes == 0)[0]:
                    if q < nw:
                        lanes[l] = max(int(w[q]), 1); q += 1
                busy = lanes > 0
                if not busy.any():
                    break
                step = int(lanes[busy].min())            # advance until the next lane finishes
                useful += step * int(busy.sum()); issued += step * 32
                lanes[busy] -= step
        return useful, issued
    u_b, i_b = simulate([r[4] for r in recs])
    nwarps = 64
    per_warp = [np.concatenate([recs[e][4] for e in range(w, len(recs), nwarps)]) for w in range(nwarps)]
    u_c, i_c = simulate(per_warp)
    print("lane-refill, one warp per element (drained per element): lane utilisation %.1f%%;  persistent warps across elements: %.1f%%" % (100 * u_b / i_b, 100 * u_c / i_c))
    need_a = lb < best[vox]; need_t = lbt < best[vox]
    # best-first per grid point: sorted by bound, stop when bound >= running minimum
    order = np.lexsort((lbt, vox)); vs, ds, ls, its_s = vox[order], dist[order], lbt[order], its[order]
    starts = np.r_[0, np.nonzero(np.diff(vs))[0] + 1, len(vs)]
    done = 0; iters_bf = 0; per_vox = []
    for a, b in zip(starts[:-1], starts[1:]):
        cur = np.inf; k = 0
        for q in range(a, b):
            if ls[q] >= cur: break
            cur = min(cur, ds[q]); k += 1; iters_bf += int(its_s[q])
        done += k; per_vox.append(k)
    per_vox = np.array(per_vox)
    # two global passes: A = every pair whose point lies inside the element's AABB (bound 0, never skippable); B = the others, skipped when
    # their bound is not below the minimum pass A left for the point (points no pass-A pair reached keep +inf: nothing skipped for them)
    bestA = np.full(int(g.ngp), np.inf)
    inA = lb == 0.0
    np.minimum.at(bestA, vox[inA], dist[inA])
    for name, bound in (("element AABB", lb), ("tight box", lbt)):
        keepB = (~inA) & (bound < bestA[vox])
        kept = inA.sum() + keepB.sum()
        print("two global passes with the %s: pass A %d pairs, pass B keeps %d of %d -> %.1f%% of all pairs, %.1f%% of the iterations" % (
            name, inA.sum(), keepB.sum(), (~inA).sum(), 100 * kept / npairs, 100 * (its[inA].sum() + its[keepB].sum()) / its.sum()))
    print("pairs that can matter (bound < final minimum): element AABB %d (%.1f%%), tight box %d (%.1f%%)" % (
        need_a.sum(), 100 * need_a.mean(), need_t.sum(), 100 * need_t.mean()))
    print("best-first per grid point with the tight box: %d projections (%.1f%% of the pairs, %.2f per band point; p50 %d p90 %d max %d), %.1f%% of the iterations" % (
        done, 100 * done / npairs, done / band, *np.percentile(per_vox, [50, 90]).astype(int), per_vox.max(), 100 * iters_bf / its.sum()))
    device_schemes(dev, inA, int(g.ngp))


def device_schemes(dev, inner, ngp):
    """inner: the point lies in the element's box (today's pass A)"""
    vox, dist, its, lbx, lbsl, lbs, eid = (np.concatenate([r[k] for r in dev]) for k in range(7))
    final = np.full(ngp, np.inf); np.minimum.at(final, vox, dist)
    npairs, itall = len(vox), its.sum()

    def two_pass(seedA, bound):
        cur = np.full(ngp, np.inf); np.minimum.at(cur, vox[seedA], dist[seedA])
        keepB = ~seedA & ~(bound ** 2 > cur[vox] ** 2 * (1 + 1e-10))
        assert np.all(dist[~(seedA | keepB)] >= final[vox[~(seedA | keepB)]])
        solved = seedA | keepB
        return 100 * solved.mean(), 100 * its[solved].sum() / itall

    f = lbs.astype(np.float32)
    f = np.where(f.astype(np.float64) > lbs, np.nextafter(f, np.float32(-np.inf)), f)
    order = np.lexsort((eid, f, vox)); first = np.r_[True, vox[order][1:] != vox[order][:-1]]
    seed = np.zeros(npairs, bool); seed[order[first]] = True
    print("device rules (pairs solved, solver iterations; boundary-face tiles not modelled):")
    for name, A, b in (("pass A = pairs inside the element box, pass B by the tight box", inner, lbx),
                       ("pass A = inner, bound = max(tight box, slab)", inner, np.maximum(lbx, lbsl)),
                       ("pass A = inner, bound = distance to box /\\ slab", inner, lbs),
                       ("pass A = inner + per-point seed, bound = box /\\ slab", inner | seed, lbs),
                       ("pass A = per-point seed (smallest bound), bound = box /\\ slab  [the kernels]", seed, lbs)):
        print("  %-80s %5.1f%% %5.1f%%" % ((name,) + two_pass(A, b)))
    order = np.lexsort((lbs, vox)); vs, ds, ls, it_s = vox[order], dist[order], lbs[order], its[order]
    starts = np.r_[0, np.nonzero(np.diff(vs))[0] + 1, len(vs)]
    done = iters = 0
    for a, b in zip(starts[:-1], starts[1:]):
        cur = np.inf
        for q in range(a, b):
            if ls[q] ** 2 > cur ** 2 * (1 + 1e-10):
                break
            cur = min(cur, ds[q]); done += 1; iters += int(it_s[q])
    print("  %-80s %5.1f%% %5.1f%%" % ("floor: best-first per point with box /\\ slab", 100 * done / npairs, 100 * iters / itall))


if __name__ == "__main__":
    main()
