"""Time r2s_isosurface_lattice on the bench workload: bench.workload(n) (default 256), grid step 0.5, :fine smoothing with interpolation and
artifact removal, then the zero surface of the continuous field on the lattices origin AABB_min, spacing cell / 2 (the :fine lattice)
and cell / 4 (one refinement beyond it).

Per lattice: points, nv / nt, wall time per call (host clock around whole calls, which end in a device synchronise; after one warm-up call),
lattice points per second (every point is sampled twice: a count sweep and an emit sweep), kernel time per pass in a profiled call of its
own (torch.profiler, CUDA activities: sampling k_sample_lattice, count k_surf_count, emit k_surf_emit<true>, snap k_surf_snap, the rest),
the device memory the call takes at its peak (cudaMemGetInfo polled from a host thread during the call, against the free memory before it)
next to the bound the header states ((chunk planes + 2) plane buffers + row scratch + mesh), and the residuals |f - iso| in float64 (the
host definition of tests/sample_ref.py on the downloaded weights) at a sample of snapped vertices and at the linearly interpolated vertices
of the same edges, in units of the lattice step.  GPU name and power limit from nvidia-smi, in the same run.

    python tools/isosurface_lattice_bench.py [--n 256] [--calls 2] [--sample 400] [--out profiles/r7a_isosurface_lattice_n256.json]
"""
import argparse
import ctypes as C
import json
import os
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
sys.path.insert(0, os.path.join(ROOT, "tools"))

PASSES = {"sampling": "k_sample_lattice", "count": "k_surf_count", "emit": "k_surf_emit", "snap": "k_surf_snap"}


def peak_during(fn):
    """(result of fn(), largest drop of free device memory seen while fn ran, in bytes)"""
    import torch
    free0 = torch.cuda.mem_get_info()[0]
    low = [free0]
    stop = threading.Event()

    def poll():
        while not stop.is_set():
            low[0] = min(low[0], torch.cuda.mem_get_info()[0])
            time.sleep(0.0005)
    th = threading.Thread(target=poll)
    th.start()
    try:
        out = fn()
    finally:
        stop.set(); th.join()
    return out, free0 - low[0]


def residuals(r2s, mesh, F, V, o, h, iso, sample, rng):
    """|f64 - iso| / min(h) at `sample` snapped vertices and at the linear vertices of the same edges (t = (iso - va) / (vb - va) in double)"""
    o32, h32 = np.float32(o), np.float32(h)
    snap, lin, skipped = [], [], 0
    for q in rng.choice(len(V), min(sample, len(V)), replace=False):
        v = V[q]
        idx = np.round((v.astype(np.float64) - o32) / h32).astype(np.int64)
        on = (o32 + idx.astype(np.float32) * h32).astype(np.float32) == v
        if on.all():      # left at a lattice point: its edge is not recoverable from the coordinates alone
            skipped += 1
            continue
        d = int(np.nonzero(~on)[0][0])
        i0 = idx.copy(); i0[d] = int(np.floor((float(v[d]) - float(o32[d])) / float(h32[d])))
        pa = (o32 + i0.astype(np.float32) * h32).astype(np.float32)
        pb = pa.copy(); pb[d] = np.float32(o32[d] + np.float32(i0[d] + 1) * h32[d])
        va, vb = r2s.sample_sdf(mesh, np.stack([pa, pb]).astype(np.float64))
        t = (float(iso) - float(va)) / (float(vb) - float(va))
        pl = pa.astype(np.float64); pl[d] = float(pa[d]) + t * (float(pb[d]) - float(pa[d]))
        snap.append(abs(F.float64(v.astype(np.float64))[0] - float(iso)))
        lin.append(abs(F.float64(np.float32(pl).astype(np.float64))[0] - float(iso)))
    hm = float(np.min(h))
    st = lambda a: {"median_over_h": float(np.median(a)) / hm, "p99_over_h": float(np.percentile(a, 99)) / hm, "max_over_h": float(np.max(a)) / hm,
                    "median_abs": float(np.median(a))} if len(a) else {}
    return {"vertices": len(snap), "skipped_at_lattice_points": skipped, "snapped": st(np.array(snap)), "linear": st(np.array(lin))}


def main():
    ap = argparse.ArgumentParser(description=__doc__.split("\n")[0])
    ap.add_argument("--n", type=int, default=256)
    ap.add_argument("--calls", type=int, default=2)
    ap.add_argument("--sample", type=int, default=400)
    ap.add_argument("--refine", default="2,4", help="lattice spacings cell / r for each r")
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r7a_isosurface_lattice_n256.json"))
    args = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("isosurface_lattice_bench.py: no CUDA device (the measurement has no CPU fallback)")
    import bench
    import rho2sdf_b200 as r2s
    import sample_ref
    from isosurface_bench import gpu_info
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
    w, th = r2s.rbf_weights(mesh)
    F = sample_ref.Field(w, grid.AABB_min, grid.AABB_max, grid.cell_size, 1e-3, th)
    rng = np.random.default_rng(0)
    res = {"workload": "bench.workload(%d): synthetic SIMP HEX8, grid step 0.5, :fine, interpolation, artifact removal; coarse grid %s" %
                       (args.n, "x".join(str(int(v) + 1) for v in grid.N)),
           "gpu": info, "pipeline_ms_total": rep.ms_total, "lattices": {}}
    from torch.profiler import profile, ProfilerActivity
    for r in [int(v) for v in args.refine.split(",")]:
        o = np.asarray(grid.AABB_min, np.float64); h = np.array([grid.cell_size / r] * 3)
        dims = np.array([int(v) * r + 1 for v in grid.N], np.int64)
        full = [int(v) for v in dims]
        # the call accepts fewer than 2^31 cells: a lattice beyond that is measured on its slab of planes 0 .. k that stays below
        dims[2] = min(dims[2], ((1 << 31) - 1) // int((dims[0] - 1) * (dims[1] - 1)))
        npts = int(np.prod(dims))
        nv, nt = C.c_int64(), C.c_int64()
        call = lambda: c.check(c.lib.r2s_isosurface_lattice(c.h, o.ctypes.data_as(C.c_void_p), h.ctypes.data_as(C.c_void_p), dims.ctypes.data_as(C.c_void_p), 0.0,
                                                            C.byref(nv), C.byref(nt)))
        _, peak = peak_during(call)      # warm-up, and the memory peak of a call
        wall = []
        for _ in range(args.calls):
            t0 = time.perf_counter(); call(); wall.append(time.perf_counter() - t0)
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
            kern.setdefault("launches", {})[ev.key[:60]] = {"calls": ev.count, "ms": t}
        kern["other_ms"] = other
        pl = int(dims[0] * dims[1])
        planes = max(1, (1 << 30) // 4 // pl - 2)
        bound = 4 * (planes + 2) * pl + 8 * 4 * (planes + 1) * int(dims[1]) + 12 * nv.value + 12 * nt.value
        V = np.empty((nv.value, 3), np.float32)
        c.check(c.lib.r2s_download_isosurface(c.h, V.ctypes.data_as(C.c_void_p), None))
        ent = {"spacing": "cell / %d" % r, "dims": [int(v) for v in dims], "dims_whole_lattice": full, "points": npts, "n_vertices": nv.value, "n_triangles": nt.value,
               "wall_s": wall, "wall_s_median": float(np.median(wall)), "points_per_s": npts / float(np.median(wall)),
               "kernel_ms": kern, "chunk_planes_default": planes, "chunks": int(-(-int(dims[2]) // planes)),
               "peak_device_bytes_observed": int(peak), "device_bytes_bound": int(bound),
               "residuals": residuals(r2s, mesh, F, V, o, h, 0.0, args.sample, rng)}
        res["lattices"]["h/%d" % r] = ent
        print(json.dumps({k: v for k, v in ent.items() if k != "kernel_ms"}), flush=True)
        del V
    res["note"] = ("wall times: host clock around whole r2s_isosurface_lattice calls (they end in a device synchronise); kernel_ms: one profiled "
                   "call, summed per pass; peak_device_bytes_observed: largest drop of cudaMemGetInfo's free memory polled every 0.5 ms during "
                   "the first call (includes the mesh buffers, which stay allocated); residuals in float64 on the downloaded weights")
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(res, f, indent=1)
    print(json.dumps({"gpu": info, "out": args.out}))
    mesh.close()


if __name__ == "__main__":
    main()
