#!/usr/bin/env python
"""bench.py -- SDF voxels/s of the rho2sdf grid-sampling hot path on B200 (BASELINE.json metric).

    python bench.py --gpus N --steps K --warmup W            # this repo's CUDA path (libr2s.so through its C ABI)
    python bench.py --impl reference --gpus N --steps K ...   # the reference algorithm on the host cores (CPU oracle port)
    python bench.py --gpus 1 --steps K --dump-outputs DIR     # also write the results of the last timed step to DIR/*.npy

Workload (BASELINE.json configs[4], SURVEY.md 8d-5): synthetic n^3 HEX8 SIMP density field (n = 256), grid step h_e/2,
rho_t = 0.5, remove_artifacts, rbf_interp, rbf_grid = :fine  ->  (2(2n+6)+1)^3 = 1037^3 fine voxels.
A "step" is one pass of the region the reference itself times (src/RhoToSDF.jl:164-227): grid points -> distances -> signs ->
artifact removal -> RBF smoothing on the fine grid.  `value` = fine voxels / step time with the nodal densities resident
in HBM; `e2e` = the same through r2s_pipeline() with pinned HOST buffers (H2D of rho_n, D2H of sdf_dists and fine_sdf).
For N > 1 the coarse grid is cut into z-slabs, one rank (process) per GPU; scaling is strong (fixed problem).
"""
import argparse
import ctypes as C
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

import numpy as np  # noqa: E402

METRIC = "sdf_voxels_per_sec"
UNIT = "voxels/s"
# algorithmic work per unit (SURVEY.md 8d, restated in DESIGN.md "Rooflines")
FLOP_PER_PAIR_SURVEY = 2100.0   # SURVEY 8(d) estimate: FP64 flop per (element, grid point) projection (about 6 SQP evaluations of 350 flop)
B_PER_VOXEL_MATVEC = 16.0       # CG mat-vec: read r, u_old; write u_new, c (Float32)
B_PER_VOXEL_UPDATE = 24.0       # CG update: read x, u, r, c; write x, r
B_PER_VOXEL_CG_ITER = B_PER_VOXEL_MATVEC + B_PER_VOXEL_UPDATE
B_PER_FINE_VOXEL = 4.5          # fine evaluation: 4 B write + 1/8 * 4 B weight read
FMA_PER_FINE_VOXEL = 79.75      # mean of the 8 polyphase tap counts (81 + 3*70 + 3*80 + 88) / 8
B_PER_VOXEL_SIGN = 8.0
B_PER_VOXEL_CC = 4 * 9.0 + 16.0  # 4 label passes x 9 B + the final sdf read-modify-write
DUMP_BYTES = 48 << 20            # --dump-outputs: data bytes of all files together, well under 64 MB with the .npy headers
DUMP_SEED = 20240517


def dump_outputs(out_dir, arrays, budget=DUMP_BYTES):
    """Write each result array of the timed path's last step as out_dir/<name>.npy (its own dtype, float64 or float32).  The arrays
    share `budget` equally; an array larger than its share is written as the 1-D vector of its values at a fixed, seeded set of flat
    indices (sorted; the same for every run with the same arguments), so that the outputs of two builds compare element for element."""
    os.makedirs(out_dir, exist_ok=True)
    share = budget // len(arrays)
    for name, a in arrays.items():
        if a.nbytes > share:
            idx = np.unique(np.random.default_rng(DUMP_SEED).integers(0, a.size, share // a.itemsize))
            a = a.reshape(-1)[idx]
        np.save(os.path.join(out_dir, name + ".npy"), a)


def load_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return float(d["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
    return 6650.0, "fallback (B200_PROFILING.md)"


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled every 200 ms during the timed region (B200_PROFILING.md recipe)."""
    Q = "index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"

    def __init__(self, index):
        self.index, self.proc, self.lines = index, None, []

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + self.Q, "--format=csv,noheader,nounits", "-lms", "200"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except OSError:
            self.proc = None

    def _read(self):
        for ln in self.proc.stdout:
            self.lines.append(ln.strip())

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.25)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, mx, pw, reasons = [], [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for ln in self.lines:
            f = [x.strip() for x in ln.split(",")]
            if len(f) < 9:
                continue
            try:
                sm.append(float(f[1])); mx.append(float(f[2])); pw.append(float(f[3]))
            except ValueError:
                continue
            for nm, v in zip(names, f[5:9]):
                if v.lower().startswith("active"):
                    reasons.add(nm)
        # samples under load = the upper half of the power readings (the sampler also sees the idle gaps between steps)
        if sm:
            order = np.argsort(pw)
            load = [sm[i] for i in order[len(order) // 2:]]
            return {"sm_mhz": float(np.median(load)), "sm_max_mhz": float(max(mx)), "power_w_max": float(max(pw)), "samples": len(sm), "reasons": sorted(reasons)}
        return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["no samples"]}


def host_threads():
    try:
        return max(1, len(os.sched_getaffinity(0)))
    except AttributeError:
        return max(1, os.cpu_count() or 1)


def workload(n):
    from fixtures import simp_hex8
    return simp_hex8(n)


def base_config(n):
    """The workload both arms are quoted on (BASELINE configs[4]); grid dims follow Grid(): N = 2n + 6 cells per axis."""
    f = 4 * n + 13
    return {"workload": "synthetic %d^3 HEX8 SIMP density (seed 20240517) -> %dx%dx%d fine SDF grid (BASELINE configs[4])" % (n, f, f, f),
            "coarse_points": (2 * n + 7) ** 3, "fine_voxels": f ** 3, "rho_t": 0.5, "delta_factor": 1.1, "rbf_interp": True, "rbf_grid": "fine",
            "remove_artifacts": True, "smoothing_dtype": "f32 (as the reference)"}


def rep_box_elements(mesh):
    """Number of axis-aligned box elements of the mesh (they take the HexBox variant of the projection kernel)."""
    n = C.c_int64(0)
    mesh.ctx.check(mesh.ctx.lib.r2s_mesh_box_elements(mesh.ctx.h, C.byref(n)))
    return int(n.value)


def fine_voxels(grid, smooth):
    return int(np.prod([int(v) * smooth + 1 for v in grid.N]))


# ----------------------------------------------------------------------------------------------------------------------
# CPU oracle arm (also the cpu_baseline leg).  Julia is not installable in this image (no network, no toolchain), so the
# "reference" here is the C/OpenMP restatement in oracle/ -- kind = "port".
# ----------------------------------------------------------------------------------------------------------------------
def cpu_pipeline(n):
    import oracle
    from fixtures import Grid
    X, IEN, rho = workload(n)
    g = Grid(X.min(0), X.max(0), 2 * n, 3)
    vd, vf = oracle.mesh_volume(X, IEN, rho)
    rn = oracle.nodal_densities(X, IEN, rho)
    # all host cores this process may use; torchrun exports OMP_NUM_THREADS=1 for nproc > 1, which the oracle's explicit
    # num_threads(nt) clauses override
    nt = host_threads()

    def step(keep=None):
        t0 = time.perf_counter()
        d, _, _ = oracle.eval_distances(X, IEN, g, rn, 0.5, 1.1, nthreads=nt, want_xp=False)
        s = oracle.sign_detection(X, IEN, g, rn, 0.5, nthreads=nt)
        sdf, _ = oracle.remove_artifacts(d * s, g)
        fine, info = oracle.rbf_smoothing(sdf, g, True, 2, vd * vf, mode=0, nthreads=nt)
        t = time.perf_counter() - t0
        if keep is not None:      # the parity leg of the GPU arm compares these with the CUDA path on the same replica
            keep.update(X=X, IEN=IEN, rho=rho, grid=g, sdf=sdf, fine=fine, cg_iters=info["cg_iters"], th=info["th"], target=vd * vf)
        return t, fine.size
    return step, nt, g


def gpu_parity_on_replica(r2s, ref, device, stream):
    """The CUDA path on the replica the CPU oracle just ran (same inputs), compared field by field: the `parity` object of the bench line."""
    X, IEN, rho, g = ref["X"], ref["IEN"], ref["rho"], ref["grid"]
    mesh = r2s.Mesh(X, IEN, rho, element_type=r2s.HEX8, device=device, stream=stream)
    grid = r2s.Grid(X.min(0), X.max(0), int(g.N[0]) - 6, 3)
    assert list(grid.N) == list(g.N) and grid.cell_size == g.cell_size
    rho_n = r2s.DenseInNodes(mesh, rho)
    mesh._use_grid(grid)
    c = mesh.ctx
    p = r2s.Params(); c.lib.r2s_default_params(C.byref(p))
    p.rho_t, p.smooth, p.rbf_interp, p.remove_artifacts = 0.5, 2, 1, 1
    p.target_volume, p.final_volume = mesh.V_frac * mesh.V_domain, 1
    sdf = np.empty(grid.ngp); fine = np.empty(ref["fine"].size, dtype=np.float32); rep = r2s.Report()
    c.check(c.lib.r2s_pipeline(c.h, C.byref(p), rho_n.ctypes.data_as(C.c_void_p), sdf.ctypes.data_as(C.c_void_p), fine.ctypes.data_as(C.c_void_p), C.byref(rep)))
    c.close()
    h = grid.cell_size
    osdf, ofine = ref["sdf"], ref["fine"].ravel()
    far_g, far_o = np.abs(sdf) > 1e9, np.abs(osdf) > 1e9
    band = ~(far_g | far_o)
    return {"replica_n": int(round(len(rho) ** (1 / 3))), "coarse_points": int(grid.ngp), "fine_voxels": int(fine.size),
            "max_dist_err_over_h": float(np.max(np.abs(np.abs(sdf[band]) - np.abs(osdf[band]))) / h), "band_mismatches": int(np.count_nonzero(far_g != far_o)),
            "sign_mismatches": int(np.count_nonzero(np.signbit(sdf) != np.signbit(osdf))), "cg_iters": [int(rep.cg_iters), int(ref["cg_iters"])],
            "cg_iters_equal": bool(rep.cg_iters == ref["cg_iters"]), "th_err_over_h": float(abs(rep.th - ref["th"]) / h),
            "fine_err_over_h": float(np.max(np.abs(fine - ofine)) / h), "tolerances": {"dist": 1e-9, "sign": 0, "fine": 1e-3},
            "checker": "oracle/r2s_oracle.c (CPU restatement), same seeded inputs"}


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return 0
    n = args.cpu_n
    step, nt, g = cpu_pipeline(n)
    for _ in range(max(0, min(args.warmup, 1))):
        step()
    ts, last = [], {}
    for k in range(args.steps):
        t, nv = step(last if k == args.steps - 1 else None)
        ts.append(t)
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, {"sdf_dists": last["sdf"].reshape([int(v) + 1 for v in g.N[::-1]]), "fine_sdf": last["fine"]})
    t = float(np.mean(ts))
    sample = "n=%d^3 HEX8 SIMP replica of the workload (%d coarse points, %d fine voxels), full timed region" % (n, g.ngp, nv)
    line = {"impl": "reference", "metric": METRIC, "value": nv / t, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps, "warmup": min(args.warmup, 1),
            "ms_per_step": 1e3 * t, "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
            "config": dict(base_config(args.n), parallelism="host threads", sample="each step = the bounded %d^3 replica of the workload" % n),
            "cpu_baseline": {"value": nv / t, "unit": UNIT, "cores": nt, "kind": "port", "sample": sample},
            "e2e": {"value": nv / t, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}, "gpu_launches": 0}
    print(json.dumps(line), flush=True)
    return 0


# ----------------------------------------------------------------------------------------------------------------------
def run_gpu(args):
    import torch
    import torch.distributed as dist
    import rho2sdf_b200 as r2s

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if world != args.gpus:
        if world == 1 and args.gpus > 1:
            raise SystemExit("launch with: python -m torch.distributed.run --nnodes=1 --nproc-per-node %d --master-addr 127.0.0.1 bench.py --gpus %d ..." % (args.gpus, args.gpus))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device -- this framework has no CPU fallback (use --impl reference for the CPU arm)")
    torch.cuda.set_device(local)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    stream = torch.cuda.Stream(device=local)
    n = args.n
    with torch.cuda.stream(stream):
        X, IEN, rho = workload(n)
        grid = r2s.Grid(X.min(0), X.max(0), 2 * n, 3)
        nz = int(grid.N[2]) + 1

        def build():      # untimed: the reference builds Mesh before its timer
            mesh = r2s.Mesh(X, IEN, rho, element_type=r2s.HEX8, device=local, stream=stream.cuda_stream)
            rho_n = r2s.DenseInNodes(mesh, rho)
            mesh._use_grid(grid)
            c = mesh.ctx
            c.check(c.lib.r2s_upload_nodal_densities(c.h, rho_n.ctypes.data_as(C.c_void_p)))
            k0, k1 = 0, nz
            if world > 1:
                k0, k1 = r2s.slab_partition(nz, world)[rank]
                r2s.init_slab_comm(c, rank, world, k0, k1)
            return mesh, rho_n, c, k0, k1
        mesh, rho_n, c, k0, k1 = build()
        p = r2s.Params(); c.lib.r2s_default_params(C.byref(p))
        p.rho_t, p.smooth, p.rbf_interp, p.remove_artifacts = 0.5, 2, 1, 1
        p.target_volume, p.final_volume = mesh.V_frac * mesh.V_domain, 1
        n_balance = 0
        transport = None
        if world > 1:
            # One untimed call first.  If the peer-memory transport fails on this box (an error on any rank: time-out, diverging CG), every
            # rank abandons its context and continues on a fresh one with NCCL only (R2S_P2P=0); the line says which transport was measured.
            transport = "nccl" if os.environ.get("R2S_P2P", "1") == "0" else "peer-memory + nccl"
            ok, err = 1.0, ""
            try:
                rep = r2s.Report()
                c.check(c.lib.r2s_pipeline_resident(c.h, C.byref(p), C.byref(rep)))
            except r2s.R2SError as e:
                ok, err = 0.0, str(e)
            flag = torch.tensor([ok], dtype=torch.float64, device="cuda")
            dist.all_reduce(flag, op=dist.ReduceOp.MIN)
            if flag.item() < 0.5:
                if transport == "nccl":
                    raise SystemExit("bench.py: the multi-GPU pipeline failed on the NCCL transport: %s" % err)
                print("rank %d: peer-memory transport failed (%s); continuing with R2S_P2P=0" % (rank, err or "another rank failed"), file=sys.stderr, flush=True)
                os.environ["R2S_P2P"] = "0"
                failed = (mesh, c)      # kept alive on purpose: tearing a failed communicator down is not worth the risk inside a benchmark
                mesh, rho_n, c, k0, k1 = build()
                transport = "nccl (peer-memory transport failed: %s)" % (err or "on another rank")[:160]
            # load balancing during warm-up: the planes next to the mesh boundary carry the boundary-face work, so equal plane
            # counts are not equal work.  Measure the collective-free stages per rank, re-cut the slabs by cumulative cost.  The transport
            # check above is the first of these warm-up calls.
            n_balance = 0 if args.no_balance else min(2, max(0, args.warmup - 1))
            parts = r2s.slab_partition(nz, world)
            first = rep if flag.item() >= 0.5 else None
            for it in range(n_balance):
                if it > 0 or first is None:
                    rep = r2s.Report()
                    c.check(c.lib.r2s_pipeline_resident(c.h, C.byref(p), C.byref(rep)))
                free = rep.ms_bin + rep.ms_project + rep.ms_assemble + rep.ms_sign
                rbf = rep.ms_rbf_prep + rep.ms_cg + rep.ms_lsf + rep.ms_threshold + rep.ms_fine + rep.ms_volume
                mine = torch.tensor([free, rbf, float(k0), float(k1)], dtype=torch.float64, device="cuda")
                allr = [torch.zeros_like(mine) for _ in range(world)]
                dist.all_gather(allr, mine)
                rows = [a.tolist() for a in allr]
                cu = min(rw[1] / (rw[3] - rw[2]) for rw in rows)          # smoothing cost per plane (the rank that waited least)
                cost = np.zeros(nz)
                for rw in rows:
                    cost[int(rw[2]):int(rw[3])] = rw[0] / (rw[3] - rw[2]) + cu
                parts = r2s.slab_partition(nz, world, plane_cost=cost)
                k0, k1 = parts[rank]
                c.check(c.lib.r2s_set_slab(c.h, k0, k1))
            if n_balance == 0 and first is not None:
                n_balance = 1      # the check itself was a warm-up call
        nfine = fine_voxels(grid, 2)
        fdims = [int(v) * 2 + 1 for v in grid.N]
        # slab-local output sizes (planes this rank returns to the host in the e2e leg)
        kf0, kf1 = 2 * k0, (2 * k1 if k1 < nz else fdims[2])
        n_sdf_local = (k1 - k0) * int(grid.N[0] + 1) * int(grid.N[1] + 1)
        n_fine_local = (kf1 - kf0) * fdims[0] * fdims[1]
        # pinned host buffers for the e2e leg
        h_rho = torch.from_numpy(rho_n).pin_memory()
        h_sdf = torch.empty(n_sdf_local, dtype=torch.float64).pin_memory()
        h_fine = torch.empty(n_fine_local, dtype=torch.float32).pin_memory()

        def barrier():
            stream.synchronize()
            if world > 1:
                dist.barrier()
            torch.cuda.synchronize()

        def step_resident():
            rep = r2s.Report()
            c.check(c.lib.r2s_pipeline_resident(c.h, C.byref(p), C.byref(rep)))
            return rep

        def step_e2e():
            rep = r2s.Report()
            c.check(c.lib.r2s_pipeline_slab(c.h, C.byref(p), C.c_void_p(h_rho.data_ptr()), C.c_void_p(h_sdf.data_ptr()), C.c_void_p(h_fine.data_ptr()), C.byref(rep)))
            return rep

        for _ in range(args.warmup - n_balance):
            step_resident()
        # ---- timed region: exactly K steps, CUDA events on the launching stream, barrier + synchronize on both sides ----
        sampler = ClockSampler(local) if rank == 0 else None
        if sampler:
            sampler.start()
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(stream)
        reps = [step_resident() for _ in range(args.steps)]
        e1.record(stream)
        barrier()
        ms = e0.elapsed_time(e1)
        if args.dump_outputs:      # the device results of the last timed step, through the pinned buffers before the e2e leg reuses them
            c.check(c.lib.r2s_download_sdf(c.h, C.c_void_p(h_sdf.data_ptr())))
            c.check(c.lib.r2s_download_fine_sdf(c.h, C.c_void_p(h_fine.data_ptr())))
            dump_outputs(args.dump_outputs, {"sdf_dists": h_sdf.numpy().reshape([int(v) + 1 for v in grid.N[::-1]]), "fine_sdf": h_fine.numpy().reshape(fdims[::-1])})
        # ---- e2e: the same K steps through the host-buffer entry point ----
        step_e2e()
        barrier()
        f0, f1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        w0 = time.perf_counter()
        f0.record(stream)
        ereps = [step_e2e() for _ in range(args.steps)]
        f1.record(stream)
        barrier()
        wall_e2e = (time.perf_counter() - w0) * 1e3
        ms_e2e = max(f0.elapsed_time(f1), 0.0)
        # ---- extra: the same K steps through the pipelined host-buffer calls (two buffer sets; the downloads of step k drain
        # while step k+1 computes): the throughput of a batch of density fields.  Reported as "e2e_pipelined" beside the per-call "e2e".
        ms_pipe = None
        if args.pipelined_e2e and not args.no_pipelined_e2e and world == 1:      # (single GPU only: the multi-rank runs keep to the per-call API)
            try:
                h_sdf2 = torch.empty(n_sdf_local, dtype=torch.float64).pin_memory()
                h_fine2 = torch.empty(n_fine_local, dtype=torch.float32).pin_memory()
                bufs = [(h_sdf, h_fine), (h_sdf2, h_fine2)]

                def begin(k):
                    rep = r2s.Report(); t = C.c_int(-1)
                    c.check(c.lib.r2s_pipeline_slab_begin(c.h, C.byref(p), C.c_void_p(h_rho.data_ptr()), C.c_void_p(bufs[k % 2][0].data_ptr()), C.c_void_p(bufs[k % 2][1].data_ptr()),
                                                          C.byref(rep), C.byref(t)))
                    return t.value
                c.check(c.lib.r2s_pipeline_slab_wait(c.h, begin(0)))
                barrier()
                w1 = time.perf_counter()
                tk = begin(0)
                for k in range(1, args.steps):
                    tn = begin(k)
                    c.check(c.lib.r2s_pipeline_slab_wait(c.h, tk))
                    tk = tn
                c.check(c.lib.r2s_pipeline_slab_wait(c.h, tk))
                barrier()
                ms_pipe = (time.perf_counter() - w1) * 1e3
            except Exception as e:      # noqa: BLE001 -- an extra figure must not take the measured line down
                ms_pipe = None; print("pipelined leg failed: %r" % (e,), file=sys.stderr)
        clocks = sampler.stop() if sampler else None
        per_rank = None
        if world > 1:
            t = torch.tensor([ms, ms_e2e, wall_e2e, ms_pipe if ms_pipe is not None else 0.0], dtype=torch.float64, device="cuda")
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            ms, ms_e2e, wall_e2e, mp = (float(v) for v in t.tolist())
            ms_pipe = mp if ms_pipe is not None else None
            # per-rank stage times of the last timed step (load-balance evidence)
            keys = ("ms_bin", "ms_project", "ms_assemble", "ms_sign", "ms_cc", "ms_cg", "ms_threshold", "ms_total")
            mine = torch.tensor([getattr(reps[-1], k) for k in keys] + [float(k1 - k0)] + [float(v) for v in reps[-1].cg_probe], dtype=torch.float64, device="cuda")
            allr = [torch.zeros_like(mine) for _ in range(world)]
            dist.all_gather(allr, mine)
            per_rank = [dict(zip(keys + ("planes", "cg_matvec", "cg_xchg1", "cg_update", "cg_xchg2"), [round(float(v), 3) for v in a.tolist()])) for a in allr]
        # ---- roofline denominators measured on this device ----
        fp64, fp32 = C.c_double(), C.c_double()
        c.check(c.lib.r2s_measure_fma_peak(c.h, 1, C.byref(fp64)))
        c.check(c.lib.r2s_measure_fma_peak(c.h, 0, C.byref(fp32)))
    hbm, hbm_src = load_peaks()
    if rank == 0:
        K = args.steps
        step_ms = ms / K
        e2e_ms = max(ms_e2e, wall_e2e) / K       # host-blocking copies: the wall clock is the honest figure
        d = {k: float(np.mean([getattr(r, k) for r in reps])) for k in ("ms_bin", "ms_project", "ms_assemble", "ms_sign", "ms_cc", "ms_rbf_prep", "ms_cg", "ms_lsf",
                                                                         "ms_threshold", "ms_fine", "ms_volume", "ms_total")}
        rep = reps[-1]
        ngp_local = n_sdf_local
        # k_project_list: EXECUTED FP64 flop per solved pair, measured with ncu on this workload (tools/extract_counts.py -> profiles/project_list_counts.json;
        # thread-level dfma x 2 + dadd + dmul with the predicate on).  Pruned pairs are never projected, so they carry no work.
        counts = None
        cp = os.path.join(ROOT, "profiles", "project_list_counts.json")
        if os.path.exists(cp):
            try:
                counts = json.load(open(cp))
            except Exception:
                counts = None
        solved = int(rep.n_pairs - rep.n_pairs_pruned)
        ms_solve = float(np.mean([r.ms_solve for r in reps]))
        ms_scan = float(np.mean([r.ms_scan for r in reps]))
        box_variant = ms_solve > 0
        fpp = counts["fp64_flop_per_solved_pair"] if (counts and box_variant and "fp64_flop_per_solved_pair" in counts) else None
        ngp_pad = int((grid.N[0] + 1 + 3) // 4 * 4) * int(grid.N[1] + 1) * (k1 - k0)      # CG fields carry a row pitch that is a multiple of 4 floats
        mv_ms, up_ms = float(rep.cg_probe[0]), float(rep.cg_probe[2])
        stages = {
            "project_list": {"bound": "fp64", "ms": ms_solve, "achieved": (fpp * solved / (ms_solve * 1e-3) / 1e12) if (fpp and ms_solve > 0) else None, "peak": fp64.value, "unit": "TFLOP/s",
                             "pairs_solved": solved, "pairs_pruned": int(rep.n_pairs_pruned), "flop_per_solved_pair_measured": fpp,
                             "survey_estimate_tflops": FLOP_PER_PAIR_SURVEY * rep.n_pairs / (d["ms_project"] * 1e-3) / 1e12 if d["ms_project"] > 0 else None},
            "pair_scan": {"bound": "latency", "ms": ms_scan},
            "cg_matvec_tma": {"bound": "hbm", "ms": mv_ms, "achieved": B_PER_VOXEL_MATVEC * ngp_pad / (mv_ms * 1e-3) / 1e9 if mv_ms > 0 else None, "peak": hbm, "unit": "GB/s"},
            "cg_update": {"bound": "hbm", "ms": up_ms, "achieved": B_PER_VOXEL_UPDATE * ngp_pad / (up_ms * 1e-3) / 1e9 if up_ms > 0 else None, "peak": hbm, "unit": "GB/s"},
            "cg_total": {"bound": "hbm", "ms": d["ms_cg"], "achieved": B_PER_VOXEL_CG_ITER * ngp_pad * rep.cg_iters / (d["ms_cg"] * 1e-3) / 1e9 if d["ms_cg"] > 0 else None, "peak": hbm, "unit": "GB/s"},
            "fine_eval": {"bound": "fp32 issue", "ms": d["ms_fine"], "achieved": B_PER_FINE_VOXEL * n_fine_local / (d["ms_fine"] * 1e-3) / 1e9 if d["ms_fine"] > 0 else None,
                          "peak": hbm, "unit": "GB/s", "fp32_tflops": 2 * FMA_PER_FINE_VOXEL * n_fine_local / (d["ms_fine"] * 1e-3) / 1e12 if d["ms_fine"] > 0 else None,
                          "fp32_peak": fp32.value},
            "sign": {"bound": "hbm", "ms": d["ms_sign"], "achieved": 2 * B_PER_VOXEL_SIGN * ngp_local / (d["ms_sign"] * 1e-3) / 1e9 if d["ms_sign"] > 0 else None, "peak": hbm, "unit": "GB/s"},
            "cc": {"bound": "hbm", "ms": d["ms_cc"], "achieved": B_PER_VOXEL_CC * ngp_local / (d["ms_cc"] * 1e-3) / 1e9 if d["ms_cc"] > 0 else None, "peak": hbm, "unit": "GB/s"},
        }
        for s_ in stages.values():
            s_["frac"] = (s_["achieved"] / s_["peak"]) if s_.get("achieved") and s_.get("peak") else None
        dom = stages["project_list"]
        traffic = counts["dram_bytes_per_step"] if (counts and box_variant) else None
        traffic_note = ("measured DRAM bytes of the two k_project_list launches of one step (ncu --set full, %s); algorithmic: 8 B list entry + 16 B atomicMin per solved pair + 208 B record per "
                        "crossing element = %.2f GB" % (counts.get("source", "?"), (24.0 * solved + 208.0 * rep.n_crossing) / 1e9)) if traffic else "no ncu capture of the kernel that ran (profiles/project_list_counts.json missing)"
        line = {
            "metric": METRIC, "value": nfine / (step_ms * 1e-3), "unit": UNIT, "n_gpus": world, "steps": K, "warmup": args.warmup, "ms_per_step": step_ms,
            "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
            "config": dict(base_config(n), parallelism="zslab%d" % world, slab_planes=[int(b - a) for a, b in parts] if world > 1 else [nz], **({"transport": transport} if transport else {}), l2_policy="inputs larger than L2 (working set %.1f GB per step)" % ((rep.n_pairs * 8 + grid.ngp * 40 + nfine * 4) / 1e9)),
            "e2e": {"value": nfine / (e2e_ms * 1e-3), "unit": UNIT, "ms_per_step": e2e_ms, "h2d_bytes_per_step": int(rho_n.nbytes) * world,
                    "d2h_bytes_per_step": int(grid.ngp * 8 + nfine * 4), "api": "r2s_pipeline_slab (pinned host buffers)"},
            "gpu_launches": int(sum(r.launches for r in reps)),
            "roofline": {"kernel": "k_project_list (two launches per step: pairs inside the element box, then the pruned rest)", "bound": "fp64", "achieved": dom["achieved"], "peak": dom["peak"],
                         "unit": "TFLOP/s", "frac": dom["frac"], "traffic": traffic, "traffic_note": traffic_note,
                         "peak_source": "FP64 FMA chain micro-kernel measured in this run (r2s_measure_fma_peak; MEASURED_PEAKS.json has no FP64 figure); HBM peak %s" % hbm_src,
                         "algorithmic": "%s executed FP64 flop per solved pair (ncu: dfma x 2 + dadd + dmul, profiles/project_list_counts.json) x %d pairs solved of %d candidates (%d pruned by their lower bound) / %.2f ms of k_project_list (CUDA events around the two launches)"
                                        % ("%.0f" % fpp if fpp else "n/a", solved, rep.n_pairs, rep.n_pairs_pruned, ms_solve),
                         "ncu": {"lanes_per_warp_instruction": [round(l["lanes_per_warp_inst"], 2) for l in counts["launches"]], "fp64_pipe_pct": [round(l["fp64_pipe_pct"], 1) for l in counts["launches"]]} if counts else None},
            "stages_ms": d, "kernels": stages, "cg_iteration_ms": dict(zip(("matvec", "exchange1", "update", "exchange2"), [round(float(v), 4) for v in rep.cg_probe])),
            "report": {"pairs": int(rep.n_pairs), "pairs_pruned": int(rep.n_pairs_pruned), "ms_solve": ms_solve, "ms_scan": ms_scan, "newton_iters": int(rep.n_newton_iters), "not_converged": int(rep.n_not_converged), "cg_iters": int(rep.cg_iters),
                       "bisections": int(rep.bisections), "flipped": int(rep.n_flipped), "th": float(rep.th), "volume": float(rep.volume),
                       "target_volume": float(p.target_volume), "solid": int(rep.n_solid), "crossing": int(rep.n_crossing)},
            "clocks": clocks,
        }
        if ms_pipe is not None:
            line["e2e_pipelined"] = {"value": nfine / (ms_pipe / K * 1e-3), "unit": UNIT, "ms_per_step": ms_pipe / K, "api": "r2s_pipeline_slab_begin / _wait, two pinned buffer sets",
                                     "h2d_bytes_per_step": int(rho_n.nbytes) * world, "d2h_bytes_per_step": int(grid.ngp * 8 + nfine * 4)}
        if per_rank is not None:
            line["per_rank"] = per_rank
        if not args.no_cpu_baseline and world == 1:
            # the two checker legs never take the measured line down with them: a failure is reported in their own objects
            ref = {}
            try:
                step, nt, g = cpu_pipeline(args.cpu_n)
                t, nv = step(ref)
                line["cpu_baseline"] = {"value": nv / t, "unit": UNIT, "cores": nt, "kind": "port",
                                        "sample": "one pass of the timed region on the %d^3 replica of the workload (%d fine voxels) with the C/OpenMP oracle, %.1f s" % (args.cpu_n, nv, t)}
            except Exception as e:      # noqa: BLE001
                line["cpu_baseline"] = {"error": repr(e)[:300]}
            try:
                line["parity"] = gpu_parity_on_replica(r2s, ref, local, None) if ref else {"error": "no CPU reference"}
            except Exception as e:      # noqa: BLE001
                line["parity"] = {"error": repr(e)[:300]}
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()
    return 0


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--n", type=int, default=256, help="elements per axis of the synthetic HEX8 SIMP field")
    ap.add_argument("--cpu-n", type=int, default=96, help="replica size for the CPU oracle leg")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--pipelined-e2e", action="store_true", default=True, help="also time the pipelined host-buffer calls (r2s_pipeline_slab_begin/_wait) -> e2e_pipelined (default)")
    ap.add_argument("--no-pipelined-e2e", action="store_true", help="skip the pipelined host-buffer leg")
    ap.add_argument("--no-balance", action="store_true", help="keep equal plane counts per slab (no cost-based re-cut during warm-up)")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write sdf_dists.npy (float64) and fine_sdf.npy (float32) of the last timed step to DIR; "
                    "an output too large for %d MiB in all is written as a fixed, seeded sample of its values" % (DUMP_BYTES >> 20))
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.gpus != 1:
        ap.error("--dump-outputs needs --gpus 1")
    if args.impl == "reference":
        return run_reference(args)
    return run_gpu(args)


if __name__ == "__main__":
    sys.exit(main())
