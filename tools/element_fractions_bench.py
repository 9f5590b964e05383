"""Time r2s_element_volume_fractions on the bench workload: bench.workload(n) (default 256: 1.68e7 HEX8 elements), grid step 0.5, :fine
smoothing with interpolation and artifact removal (one resident pipeline), then the solid volume fraction of every element at quadrature
orders 15 and 5.

Per order: wall time per call (host clock around whole calls, which end in a device synchronise; --calls calls after one warm-up, the
orders alternating), the elements sampled and the skipped share, the solid volume sum S_e against V_frac V_domain (the volume the
threshold search matched) and against the fine-grid volume of the pipeline's report, and, with --profile, the kernel time of the two passes
in one profiled call of its own (torch.profiler, CUDA activities).  GPU name and power limit from nvidia-smi, in the same run.

    python tools/element_fractions_bench.py [--n 256] [--calls 3] [--orders 15,5] [--profile] [--out profiles/r9a_element_fractions_n256.json]
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

PASSES = {"classify": "k_ef_classify", "evaluate": "k_ef_eval"}


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
    ap.add_argument("--orders", default="15,5")
    ap.add_argument("--profile", action="store_true", help="kernel times from one profiled call per order (run separately from the timing)")
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r9a_element_fractions_n256.json"))
    args = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("element_fractions_bench.py: no CUDA device (the measurement has no CPU fallback)")
    import bench
    import rho2sdf_b200 as r2s
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
    target = mesh.V_frac * mesh.V_domain
    res = {"workload": "bench.workload(%d): synthetic SIMP HEX8, %d elements, grid step 0.5, :fine, interpolation, artifact removal; coarse grid %s" %
                       (args.n, mesh.nel, "x".join(str(int(v) + 1) for v in grid.N)),
           "gpu": info, "V_domain": mesh.V_domain, "V_frac_V_domain": target, "fine_grid_volume": float(rep.volume), "th": float(rep.th), "orders": {}}
    orders = [int(v) for v in args.orders.split(",")]
    frac = np.empty(mesh.nel)
    vol = np.empty(mesh.nel)
    ne = C.c_int64()
    ptr = lambda a: a.ctypes.data_as(C.c_void_p)
    calls = {q: (lambda q=q: c.check(c.lib.r2s_element_volume_fractions(c.h, 0.0, q, ptr(frac), ptr(vol), C.byref(ne)))) for q in orders}
    for q in orders:
        calls[q]()
        S = float((frac * vol).sum())
        res["orders"][q] = {"n_evaluated": ne.value, "skipped_share": 1.0 - ne.value / mesh.nel, "gauss_points": mesh.nel * q ** 3,
                            "points_evaluated": ne.value * q ** 3, "solid_volume": S, "element_volume_sum": float(vol.sum()),
                            "solid_vs_V_frac_V_domain": S / target - 1.0, "solid_vs_fine_grid_volume": S / float(rep.volume) - 1.0,
                            "partial_elements": int(((frac > 0) & (frac < 1)).sum()), "wall_s": []}
        print(json.dumps({q: res["orders"][q]}), flush=True)
    for _ in range(args.calls):
        for q in orders:
            t0 = time.perf_counter(); calls[q](); res["orders"][q]["wall_s"].append(time.perf_counter() - t0)
    for q in orders:
        ent = res["orders"][q]
        ent["wall_s_median"] = float(np.median(ent["wall_s"]))
        ent["evaluated_points_per_s"] = ent["points_evaluated"] / ent["wall_s_median"]
        if args.profile:
            ent["kernel_ms"] = kernel_ms(calls[q])
        print(json.dumps({q: ent}), flush=True)
    res["note"] = ("wall_s: host clock around whole calls (they end in a device synchronise and the download of fractions and volumes), the "
                   "orders alternating after one warm-up call each; skipped_share: elements the band classifier proved one-sided, never sampled; "
                   "kernel_ms: one profiled call per order, summed per pass")
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(res, f, indent=1)
    print(json.dumps({"gpu": info, "out": args.out}))
    mesh.close()


if __name__ == "__main__":
    main()
