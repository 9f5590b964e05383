"""Time r2s_isosurface on the bench workload: bench.workload(n) (default 256), grid step 0.5, :fine smoothing with interpolation and
artifact removal, then the zero surface of the resident fine_sdf.

Reports nv / nt, the time per call (CUDA events on the context's stream around whole calls, after warm-up; the calls include their two
small host read-backs), the bytes the algorithm must move (fine_sdf read once per pass, the mesh written once) and the time those take at
the HBM rate measured in the same run (a device-to-device copy of a buffer the size of fine_sdf), the download of the mesh against the
download of fine_sdf (both into pageable host arrays), and the GPU name and power limit (nvidia-smi query).

    python tools/isosurface_bench.py [--n 256] [--calls 20] [--out profiles/r4a_isosurface_n256.json]
"""
import argparse
import ctypes as C
import json
import os
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


def main():
    ap = argparse.ArgumentParser(description=__doc__.split("\n")[0])
    ap.add_argument("--n", type=int, default=256)
    ap.add_argument("--calls", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r4a_isosurface_n256.json"))
    args = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("isosurface_bench.py: no CUDA device (the measurement has no CPU fallback)")
    import bench
    import rho2sdf_b200 as r2s
    stream = torch.cuda.Stream()
    X, IEN, rho = bench.workload(args.n)
    grid = r2s.Grid(X.min(0), X.max(0), 2 * args.n, 3)
    mesh = r2s.Mesh(X, IEN, rho, element_type=r2s.HEX8, stream=stream.cuda_stream)
    rho_n = r2s.DenseInNodes(mesh, rho)
    mesh._use_grid(grid)
    c = mesh.ctx
    c.check(c.lib.r2s_upload_nodal_densities(c.h, rho_n.ctypes.data_as(C.c_void_p)))
    p = r2s.Params(); c.lib.r2s_default_params(C.byref(p))
    p.rho_t, p.smooth, p.rbf_interp, p.remove_artifacts = 0.5, 2, 1, 1
    p.target_volume, p.final_volume = mesh.V_frac * mesh.V_domain, 1
    rep = r2s.Report()
    c.check(c.lib.r2s_pipeline_resident(c.h, C.byref(p), C.byref(rep)))
    dims = [int(v) * 2 + 1 for v in grid.N]
    npts = int(np.prod(dims))

    nv, nt = C.c_int64(), C.c_int64()
    for _ in range(args.warmup):
        c.check(c.lib.r2s_isosurface(c.h, 0.0, C.byref(nv), C.byref(nt)))
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    times = []
    for _ in range(args.calls):
        e0.record(stream)
        c.check(c.lib.r2s_isosurface(c.h, 0.0, C.byref(nv), C.byref(nt)))
        e1.record(stream)
        e1.synchronize()
        times.append(e0.elapsed_time(e1))
    nv, nt = nv.value, nt.value
    # per-kernel device times, in a pass of their own (torch.profiler, CUDA activities)
    from torch.profiler import profile, ProfilerActivity
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for _ in range(3):
            c.check(c.lib.r2s_isosurface(c.h, 0.0, C.byref(C.c_int64()), C.byref(C.c_int64())))
        torch.cuda.synchronize()
    kern = {}
    for ev in prof.key_averages():
        t = getattr(ev, "device_time_total", 0) or getattr(ev, "cuda_time_total", 0)
        if t > 0 and ev.count > 0:
            kern[ev.key[:80]] = {"calls": ev.count, "ms_per_call": t / ev.count / 1e3}

    # HBM rate of this card, measured here: device-to-device copy of a fine_sdf-sized buffer (read + write)
    with torch.cuda.stream(stream):
        a = torch.empty(npts, dtype=torch.float32, device="cuda").uniform_()
        b = torch.empty_like(a)
        for _ in range(3):
            b.copy_(a)
        cp = []
        for _ in range(10):
            e0.record(stream); b.copy_(a); e1.record(stream); e1.synchronize(); cp.append(e0.elapsed_time(e1))
        del a, b
    hbm_gbs = 2 * 4 * npts / (float(np.median(cp)) * 1e-3) / 1e9
    bytes_moved = 2 * 4 * npts + 12 * nv + 12 * nt      # two reads of fine_sdf, vertices and triangles written once

    V = np.empty((nv, 3), np.float32); T = np.empty((nt, 3), np.int32); F = np.empty(npts, np.float32)
    dl_mesh, dl_fine = [], []
    for _ in range(3):
        t0 = time.perf_counter(); c.check(c.lib.r2s_download_isosurface(c.h, V.ctypes.data_as(C.c_void_p), T.ctypes.data_as(C.c_void_p))); dl_mesh.append(time.perf_counter() - t0)
        t0 = time.perf_counter(); c.check(c.lib.r2s_download_fine_sdf(c.h, F.ctypes.data_as(C.c_void_p))); dl_fine.append(time.perf_counter() - t0)

    ms = float(np.median(times))
    res = {
        "workload": "bench.workload(%d): synthetic SIMP HEX8, grid step 0.5, :fine, interpolation, artifact removal; fine grid %s = %d points" % (args.n, "x".join(map(str, dims)), npts),
        "gpu": gpu_info(),
        "n_vertices": nv, "n_triangles": nt,
        "ms_isosurface_median": ms, "ms_isosurface_min": float(np.min(times)), "ms_isosurface_max": float(np.max(times)), "calls": args.calls,
        "bytes_moved": bytes_moved, "hbm_gbs_measured": hbm_gbs, "ms_at_measured_hbm": bytes_moved / (hbm_gbs * 1e9) * 1e3,
        "share_of_hbm_floor": bytes_moved / (hbm_gbs * 1e9) * 1e3 / ms,
        "ms_download_isosurface": 1e3 * float(np.median(dl_mesh)), "ms_download_fine_sdf": 1e3 * float(np.median(dl_fine)),
        "mesh_bytes": 12 * nv + 12 * nt, "fine_sdf_bytes": 4 * npts,
        "kernels_per_call": {k: dict(v, calls=v["calls"] / 3) for k, v in kern.items()},
        "pipeline_ms_total": rep.ms_total, "pipeline_volume": rep.volume,
        "note": "times are CUDA events around whole r2s_isosurface calls on the context's stream (two passes, two scans, two small read-backs); "
                "downloads are host wall-clock into pageable arrays",
    }
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(res, f, indent=1)
    print(json.dumps(res))
    mesh.close()


if __name__ == "__main__":
    main()
