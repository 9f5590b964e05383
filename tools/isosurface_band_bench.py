"""Time r2s_isosurface_band against r2s_isosurface_lattice on the bench workload: bench.workload(n) (default 256), grid step 0.5, :fine
smoothing with interpolation and artifact removal, then the zero surface of the continuous field on lattices origin AABB_min, spacing cell / r.

  cell / 2 (the :fine lattice): dense and band calls alternate (--calls each, after one warm-up of each); the two meshes are asserted equal.
  cell / 4 and cell / 8 (whole lattices, past 2^31 cells: the band path only): --calls band calls after a warm-up; a lattice whose mesh
    reaches 2^31 vertices is reported with the error.

Per lattice: points, nv / nt, wall time per call (host clock around whole calls, which end in a device synchronise), the share of lattice
points sampled (n_sampled / points: the points one of the two sweeps evaluates), the device memory a call takes at its peak (cudaMemGetInfo
polled from a host thread, against the free memory before it), and, with --profile, kernel time per pass in one profiled call of its own
(torch.profiler, CUDA activities).  GPU name and power limit from nvidia-smi, in the same run.

    python tools/isosurface_band_bench.py [--n 256] [--calls 3] [--refine 2,4,8] [--profile] [--out profiles/r8a_isosurface_band_n256.json]
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

PASSES = {"classify": "k_band_classify", "fill": "k_band_fill", "sampling_band": "k_band_sample", "sampling_dense": "k_sample_lattice",
          "count": "k_surf_count", "emit": "k_surf_emit", "snap": "k_surf_snap"}


def kernel_ms(call):
    import torch
    from torch.profiler import profile, ProfilerActivity
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        call()
        torch.cuda.synchronize()
    kern, other = {}, 0.0
    for ev in prof.key_averages():
        t = (getattr(ev, "device_time_total", 0) or getattr(ev, "cuda_time_total", 0)) / 1e3
        if t <= 0:
            continue
        name = next((k for k, s in PASSES.items() if s in ev.key), None)
        if name:
            kern[name] = kern.get(name, 0.0) + t
        else:
            other += t
    kern["other_ms"] = other
    return kern


def main():
    ap = argparse.ArgumentParser(description=__doc__.split("\n")[0])
    ap.add_argument("--n", type=int, default=256)
    ap.add_argument("--calls", type=int, default=3)
    ap.add_argument("--refine", default="2,4,8", help="lattice spacings cell / r for each r")
    ap.add_argument("--profile", action="store_true", help="kernel times from one profiled call per lattice (run separately from the timing)")
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r8a_isosurface_band_n256.json"))
    args = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("isosurface_band_bench.py: no CUDA device (the measurement has no CPU fallback)")
    import bench
    import rho2sdf_b200 as r2s
    from isosurface_bench import gpu_info
    from isosurface_lattice_bench import peak_during
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
    res = {"workload": "bench.workload(%d): synthetic SIMP HEX8, grid step 0.5, :fine, interpolation, artifact removal; coarse grid %s" %
                       (args.n, "x".join(str(int(v) + 1) for v in grid.N)),
           "gpu": info, "lattices": {}}
    for r in [int(v) for v in args.refine.split(",")]:
        o = np.asarray(grid.AABB_min, np.float64); h = np.array([grid.cell_size / r] * 3)
        dims = np.array([int(v) * r + 1 for v in grid.N], np.int64)
        npts = int(np.prod(dims))
        nv, nt, ns = C.c_int64(), C.c_int64(), C.c_int64()
        ptr = lambda a: a.ctypes.data_as(C.c_void_p)
        band = lambda: c.check(c.lib.r2s_isosurface_band(c.h, ptr(o), ptr(h), ptr(dims), 0.0, C.byref(nv), C.byref(nt), C.byref(ns)))
        dense = lambda: c.check(c.lib.r2s_isosurface_lattice(c.h, ptr(o), ptr(h), ptr(dims), 0.0, C.byref(nv), C.byref(nt)))
        ent = {"spacing": "cell / %d" % r, "dims": [int(v) for v in dims], "points": npts, "cells": int(np.prod(dims - 1))}
        try:
            _, peak = peak_during(band)
        except r2s.R2SError as e:
            ent["error"] = str(e)
            res["lattices"]["h/%d" % r] = ent
            print(json.dumps(ent), flush=True)
            continue
        ent.update({"n_vertices": nv.value, "n_triangles": nt.value, "n_sampled": ns.value, "sampled_share": ns.value / npts,
                    "peak_device_bytes_observed_band": int(peak)})
        with_dense = ent["cells"] < (1 << 31)
        if with_dense:
            def dl():
                V = np.empty((nv.value, 3), np.float32); T = np.empty((nt.value, 3), np.int32)
                c.check(c.lib.r2s_download_isosurface(c.h, ptr(V), ptr(T)))
                return V, T
            Vb, Tb = dl()
            _, peak_d = peak_during(dense)
            Vd, Td = dl()
            assert np.array_equal(Vb, Vd) and np.array_equal(Tb, Td), "band and dense meshes differ"
            ent["meshes_equal"] = True
            ent["peak_device_bytes_observed_dense"] = int(peak_d)
            del Vb, Tb, Vd, Td
        wb, wd = [], []
        for _ in range(args.calls):
            if with_dense:
                t0 = time.perf_counter(); dense(); wd.append(time.perf_counter() - t0)
            t0 = time.perf_counter(); band(); wb.append(time.perf_counter() - t0)
        ent["wall_s_band"] = wb; ent["wall_s_band_median"] = float(np.median(wb))
        if with_dense:
            ent["wall_s_dense"] = wd; ent["wall_s_dense_median"] = float(np.median(wd))
        if args.profile:
            ent["kernel_ms_band"] = kernel_ms(band)
            if with_dense:
                ent["kernel_ms_dense"] = kernel_ms(dense)
        res["lattices"]["h/%d" % r] = ent
        print(json.dumps(ent), flush=True)
    res["note"] = ("wall times: host clock around whole calls (they end in a device synchronise), dense and band alternating where both run; "
                   "sampled_share: lattice points evaluated by one sweep over the lattice's points; peak_device_bytes_observed: largest drop "
                   "of cudaMemGetInfo's free memory polled every 0.5 ms during the first call (includes the mesh buffers); kernel_ms: one "
                   "profiled call, summed per pass")
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(res, f, indent=1)
    print(json.dumps({"gpu": info, "out": args.out}))
    mesh.close()


if __name__ == "__main__":
    main()
