"""Time evalDistances / Sign_Detection at arbitrary points (r2s_eval_distances_points / r2s_sign_detection_points) on the bench workload:
bench.workload(n) (default 256: 256^3 SIMP), grid Grid(AABB, 2n, 3) (519^3 points for n = 256), rho_t = 0.5, delta = 1.1, after one
resident pipeline (:fine smoothing, interpolation, artifact removal), then:

  (a) 10^7 uniform random points in the AABB, and 10^7 points within one cell of the surface (coarse grid points with |sdf| < h, moved by
      a uniform offset in [-h/2, h/2]^3): ns per point (host clock around the call), pairs solved per point and the pruned share (report);
  (b) all coarse grid points through the points path against r2s_eval_distances / r2s_sign_detection (the price of generality), and
      whether the results agree (distances within 1e-11 h, signs equal);
  (c) the vertices of the :fine zero surface (r2s_isosurface at 0): the raw signed distance dist * sign there, max / median / p99 of
      |.| / h and the count outside the delta band -- how far smoothing and volume matching moved the boundary.

Kernel time: torch.profiler (CUDA activities) in a run of its own.  Call time: a host clock around whole calls (they end in a
synchronise) after a warm-up call.  GPU name and power limit are read in the same run.

    python tools/points_bench.py [--n 256] [--points 10000000] [--out profiles/r6a_points_n256.json]
"""
import argparse
import ctypes as C
import json
import os
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
sys.path.insert(0, os.path.join(ROOT, "tools"))

from sample_bench import gpu_info, kernel_ms      # noqa: E402


def main():
    ap = argparse.ArgumentParser(description=__doc__.split("\n")[0])
    ap.add_argument("--n", type=int, default=256)
    ap.add_argument("--points", type=int, default=10 ** 7)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r6a_points_n256.json"))
    args = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("points_bench.py: no CUDA device (the measurement has no CPU fallback)")
    import bench
    import rho2sdf_b200 as r2s
    info = gpu_info()
    X, IEN, rho = bench.workload(args.n)
    grid = r2s.Grid(X.min(0), X.max(0), 2 * args.n, 3)
    mesh = r2s.Mesh(X, IEN, rho, element_type=r2s.HEX8)
    rn = r2s.DenseInNodes(mesh, rho)
    mesh._use_grid(grid)
    c = mesh.ctx
    rt, delta, h = 0.5, 1.1, grid.cell_size
    c.check(c.lib.r2s_upload_nodal_densities(c.h, rn.ctypes.data_as(C.c_void_p)))
    p = r2s.Params(); c.lib.r2s_default_params(C.byref(p))
    p.rho_t, p.smooth, p.rbf_interp, p.remove_artifacts = rt, 2, 1, 1
    p.target_volume, p.final_volume = mesh.V_frac * mesh.V_domain, 1
    c.check(c.lib.r2s_pipeline_resident(c.h, C.byref(p), C.byref(r2s.Report())))
    sdf = np.empty(grid.ngp); c.check(c.lib.r2s_download_sdf(c.h, sdf.ctypes.data_as(C.c_void_p)))
    res = {"gpu": info, "n": args.n, "grid_N": [int(v) for v in grid.N], "ngp": grid.ngp, "cell": h, "rho_t": rt, "delta_factor": delta, "cases": {}}

    def timed(call):
        call()      # warm-up
        t0 = time.perf_counter(); call(); return time.perf_counter() - t0

    def points_case(name, P):
        n = P.shape[0]
        out = {"points": n}
        d = np.empty(n)
        t = timed(lambda: r2s.evalDistances(mesh, grid, P, rn, rt, delta_factor=delta, want_xp=False))
        rep = c.report()
        out.update(dist_s=t, dist_ns_per_point=t / n * 1e9, pairs_per_point=(rep.n_pairs - rep.n_pairs_pruned) / n, pairs_in_range_per_point=rep.n_pairs / n,
                   pruned_share=rep.n_pairs_pruned / max(rep.n_pairs, 1), not_converged=rep.n_not_converged)
        out["dist_kernel_ms"] = kernel_ms(lambda: r2s.evalDistances(mesh, grid, P, rn, rt, delta_factor=delta, want_xp=False), ["k_pt_dist", "k_pt_hex", "k_pt_keys"])
        t = timed(lambda: r2s.Sign_Detection(mesh, grid, P, rn, rt))
        out.update(sign_s=t, sign_ns_per_point=t / n * 1e9)
        out["sign_kernel_ms"] = kernel_ms(lambda: r2s.Sign_Detection(mesh, grid, P, rn, rt), ["k_pt_sign", "k_pt_keys"])
        res["cases"][name] = out
        print(name, json.dumps(out), flush=True)

    rng = np.random.default_rng(0)
    points_case("uniform_aabb", rng.uniform(grid.AABB_min, grid.AABB_max, (args.points, 3)))
    G = r2s.generateGridPoints(grid)
    band = np.nonzero(np.abs(sdf) < h)[0]
    near = G[rng.choice(band, size=args.points)] + rng.uniform(-0.5 * h, 0.5 * h, (args.points, 3))
    points_case("near_surface", near)
    del near

    # (b) the grid's own points through both entry points
    dg = np.empty(grid.ngp)
    tg = timed(lambda: c.check(c.lib.r2s_eval_distances(c.h, rn.ctypes.data_as(C.c_void_p), rt, delta, dg.ctypes.data_as(C.c_void_p), None)))
    sg = r2s.Sign_Detection(mesh, grid, None, rn, rt)
    tsg = timed(lambda: r2s.Sign_Detection(mesh, grid, None, rn, rt))
    dp = [None]
    tp = timed(lambda: dp.__setitem__(0, r2s.evalDistances(mesh, grid, G, rn, rt, delta_factor=delta, want_xp=False)[0]))
    sp = [None]
    tsp = timed(lambda: sp.__setitem__(0, r2s.Sign_Detection(mesh, grid, G, rn, rt)))
    far = dg > 1e9
    gridcase = {"points": grid.ngp, "grid_dist_s": tg, "points_dist_s": tp, "grid_sign_s": tsg, "points_sign_s": tsp,
                "dist_far_identical": bool(np.array_equal(dp[0] > 1e9, far) and np.array_equal(dp[0][far], dg[far])),
                "dist_max_abs_over_h": float(np.max(np.abs(dp[0] - dg)) / h), "dist_bit_equal_share": float(np.mean(dp[0] == dg)),
                "signs_equal": bool(np.array_equal(sp[0], sg))}
    res["cases"]["grid_points"] = gridcase
    print("grid_points", json.dumps(gridcase), flush=True)
    del G, dg, dp, sp, sg

    # (c) raw signed distance at the vertices of the :fine zero surface
    V, T = r2s.isosurface(mesh, 0.0)
    Vd = np.ascontiguousarray(V, dtype=np.float64)
    dv, _ = r2s.evalDistances(mesh, grid, Vd, rn, rt, delta_factor=delta, want_xp=False)
    sv = r2s.Sign_Detection(mesh, grid, Vd, rn, rt)
    a = np.abs(dv * sv) / h
    surf = {"vertices": int(Vd.shape[0]), "triangles": int(T.shape[0]), "max_over_h": float(a.max()), "median_over_h": float(np.median(a)),
            "p99_over_h": float(np.percentile(a, 99)), "outside_delta_band": int(np.sum(dv > delta * h)), "far_1e10": int(np.sum(dv > 1e9)),
            "inside_share": float(np.mean(sv > 0))}
    res["cases"]["fine_surface_vertices"] = surf
    print("fine_surface_vertices", json.dumps(surf), flush=True)
    os.makedirs(os.path.dirname(args.out), exist_ok=True)
    json.dump(res, open(args.out, "w"), indent=1)
    print("wrote", args.out)


if __name__ == "__main__":
    main()
