"""Time the sampler of the continuous smoothed SDF (r2s_sample_sdf / r2s_sample_sdf_lattice) on the bench workload: bench.workload(n)
(default 256), grid step 0.5, :fine smoothing with interpolation and artifact removal, then:

  * 10^8 uniformly random points in the AABB, in input order and sorted by coarse cell (gather locality), with and without gradients;
  * the lattice at the :fine spacing (origin AABB_min, spacing cell / 2: the points of fine_sdf), next to k_fine_eval2 of the same call;
  * the lattice at cell / 3 over a central sub-box.

Kernel time: torch.profiler (CUDA activities) in a run of its own, summed over the sampler's launches of one call.  Host-to-host call
time: a host clock around whole calls (they end in a synchronise), repeated --reps times for the spread.  HBM floor: the bytes the
kernels must move at 7.7 TB/s.  Issue estimate: the static SASS instruction count of the kernel (cuobjdump of libr2s.so) issued once
per point, 148 SMs x 4 warp instructions per clock at the SM clock nvidia-smi reports.  It is not a lower bound: the unrolled body
branches over coarse rows outside the cut radius, so a point issues fewer instructions than the static count.  GPU name and power
limit are read in the same run.

    python tools/sample_bench.py [--n 256] [--points 100000000] [--reps 3] [--out profiles/r5a_sample_n256.json]
"""
import argparse
import ctypes as C
import json
import os
import re
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))


def gpu_info():
    out = subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True, text=True)
    parts = [p.strip() for p in out.stdout.strip().split(",")] if out.returncode == 0 else []
    return {"name": parts[0] if parts else None, "power_limit": parts[1] if len(parts) > 1 else None, "sm_max_clock": parts[2] if len(parts) > 2 else None}


def sass_count(lib, kernel):
    """static SASS instruction count of one kernel in libr2s.so (None if cuobjdump is missing)"""
    try:
        out = subprocess.run(["cuobjdump", "-sass", lib], capture_output=True, text=True).stdout
    except OSError:
        return None
    cnt, on = 0, False
    for line in out.splitlines():
        if "Function :" in line:
            on = kernel in line
            continue
        if on and re.match(r"\s+/\*[0-9a-f]{4}\*/", line):
            cnt += 1
    return cnt or None


def kernel_ms(fn, names):
    import torch
    from torch.profiler import ProfilerActivity, profile
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        fn()
        torch.cuda.synchronize()
    tot = {}
    for e in prof.events():
        if e.device_type.name == "CUDA":
            for n in names:
                if n in e.name:
                    tot[n] = tot.get(n, 0.0) + e.device_time_total / 1000.0
    return tot


def main():
    ap = argparse.ArgumentParser(description=__doc__.split("\n")[0])
    ap.add_argument("--n", type=int, default=256)
    ap.add_argument("--points", type=int, default=10 ** 8)
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r5a_sample_n256.json"))
    args = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("sample_bench.py: no CUDA device (the measurement has no CPU fallback)")
    import bench
    import rho2sdf_b200 as r2s
    info = gpu_info()
    X, IEN, rho = bench.workload(args.n)
    grid = r2s.Grid(X.min(0), X.max(0), 2 * args.n, 3)
    mesh = r2s.Mesh(X, IEN, rho, element_type=r2s.HEX8)
    rho_n = r2s.DenseInNodes(mesh, rho)
    mesh._use_grid(grid)
    c = mesh.ctx
    c.check(c.lib.r2s_upload_nodal_densities(c.h, rho_n.ctypes.data_as(C.c_void_p)))
    p = r2s.Params(); c.lib.r2s_default_params(C.byref(p))
    p.rho_t, p.smooth, p.rbf_interp, p.remove_artifacts = 0.5, 2, 1, 1
    p.target_volume, p.final_volume = mesh.V_frac * mesh.V_domain, 1
    rep = r2s.Report()
    c.check(c.lib.r2s_pipeline_resident(c.h, C.byref(p), C.byref(rep)))
    fine_ms = kernel_ms(lambda: c.check(c.lib.r2s_pipeline_resident(c.h, C.byref(p), C.byref(rep))), ["k_fine_eval2"]).get("k_fine_eval2")
    lib = r2s.library_path()
    sass = {"points": sass_count(lib, "k_sample_pointsILb0"), "points_grad": sass_count(lib, "k_sample_pointsILb1"), "lattice": sass_count(lib, "k_sample_lattice")}
    clock = None
    try:
        clock = float(info["sm_max_clock"].split()[0]) * 1e6
    except Exception:
        pass
    res = {"gpu": info, "n": args.n, "grid_N": [int(v) for v in grid.N], "cell": grid.cell_size, "k_fine_eval2_ms": fine_ms, "sass_instructions": sass, "cases": {}}

    def run(name, call, npts, kname, hbm_bytes, sass_key):
        call()      # warm-up (and staging buffers)
        ts = []
        for _ in range(args.reps):
            t0 = time.perf_counter(); call(); ts.append(time.perf_counter() - t0)
        km = kernel_ms(call, [kname]).get(kname)
        r = {"points": npts, "host_s": ts, "host_points_per_s": npts / min(ts), "kernel_ms": km,
             "kernel_points_per_s": npts / (km / 1e3) if km else None, "hbm_floor_ms": hbm_bytes / 7.7e12 * 1e3}
        si = sass.get(sass_key)
        if si and clock:
            r["issue_estimate_ms"] = npts / 32 * si / (148 * 4 * clock) * 1e3
        res["cases"][name] = r
        print(name, json.dumps(r), flush=True)

    rng = np.random.default_rng(0)
    n = args.points
    P = rng.uniform(grid.AABB_min, grid.AABB_max, (n, 3))
    val = np.empty(n, np.float32); g = np.empty((n, 3), np.float32)
    f = lambda Q, G: c.check(c.lib.r2s_sample_sdf(c.h, Q.ctypes.data_as(C.c_void_p), n, val.ctypes.data_as(C.c_void_p), G.ctypes.data_as(C.c_void_p) if G is not None else None))
    run("points_random", lambda: f(P, None), n, "k_sample_points", n * 28, "points")
    run("points_random_grad", lambda: f(P, g), n, "k_sample_points", n * 40, "points_grad")
    cell = np.floor((P - grid.AABB_min) / grid.cell_size).astype(np.int64)
    key = (cell[:, 2] * (grid.N[1] + 1) + cell[:, 1]) * (grid.N[0] + 1) + cell[:, 0]
    P = np.ascontiguousarray(P[np.argsort(key, kind="stable")])
    run("points_sorted", lambda: f(P, None), n, "k_sample_points", n * 28, "points")
    run("points_sorted_grad", lambda: f(P, g), n, "k_sample_points", n * 40, "points_grad")
    del P, val, g
    dims = np.array([int(v) * 2 + 1 for v in grid.N], np.int64)
    out = np.empty(int(np.prod(dims)), np.float32)
    o = np.ascontiguousarray(grid.AABB_min, np.float64); h = np.full(3, grid.cell_size / 2)
    lat = lambda o_, h_, d_, out_: c.check(c.lib.r2s_sample_sdf_lattice(c.h, o_.ctypes.data_as(C.c_void_p), h_.ctypes.data_as(C.c_void_p), d_.ctypes.data_as(C.c_void_p), out_.ctypes.data_as(C.c_void_p)))
    run("lattice_fine", lambda: lat(o, h, dims, out), int(np.prod(dims)), "k_sample_lattice", int(np.prod(dims)) * 4, "lattice")
    fine = np.empty_like(out)
    c.check(c.lib.r2s_download_fine_sdf(c.h, fine.ctypes.data_as(C.c_void_p)))
    res["lattice_fine_vs_fine_sdf_max_abs"] = float(np.abs(out - fine).max())
    del out, fine
    d3 = np.array([800, 800, 800], np.int64)
    o3 = np.ascontiguousarray(grid.AABB_min + 0.5 * (grid.AABB_max - grid.AABB_min) - 400 * grid.cell_size / 3)
    h3 = np.full(3, grid.cell_size / 3)
    out3 = np.empty(int(np.prod(d3)), np.float32)
    run("lattice_cell3_800cube", lambda: lat(o3, h3, d3, out3), int(np.prod(d3)), "k_sample_lattice", int(np.prod(d3)) * 4, "lattice")
    os.makedirs(os.path.dirname(args.out), exist_ok=True)
    json.dump(res, open(args.out, "w"), indent=1)
    print("wrote", args.out)


if __name__ == "__main__":
    main()
