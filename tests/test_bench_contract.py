"""bench.py output contract: the reference arm prints one JSON line with the keys its readers use (CPU); --dump-outputs writes the
results of the last timed step (the reference arm on CPU, the CUDA arm on a GPU)."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_reference_arm_json_line():
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "1", "--warmup", "0", "--cpu-n", "12"],
                         capture_output=True, text=True, timeout=600)
    assert out.returncode == 0, out.stderr[-2000:]
    lines = [ln for ln in out.stdout.splitlines() if ln.strip()]
    assert len(lines) == 1
    d = json.loads(lines[0])
    assert d["impl"] == "reference" and d["metric"] == "sdf_voxels_per_sec" and d["unit"] == "voxels/s" and d["higher_is_better"] is True
    assert d["value"] > 0 and d["steps"] == 1 and d["vs_baseline"] is None and d["data"] == "synthetic"
    assert d["cpu_baseline"]["kind"] == "port" and d["cpu_baseline"]["cores"] >= 1 and d["cpu_baseline"]["value"] == d["value"]
    assert d["e2e"] == {"value": d["value"], "unit": "voxels/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    assert "256^3" in d["config"]["workload"] and d["config"]["fine_voxels"] == 1037 ** 3


def test_reference_arm_other_ranks_exit_quietly():
    env = dict(os.environ, RANK="1", WORLD_SIZE="2", LOCAL_RANK="1")
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--gpus", "2", "--steps", "1", "--warmup", "0", "--cpu-n", "12"],
                         capture_output=True, text=True, timeout=120, env=env)
    assert out.returncode == 0 and out.stdout.strip() == ""


def test_reference_arm_uses_all_cores_under_torchrun_env():
    """torch.distributed.run exports OMP_NUM_THREADS=1 for nproc > 1; the CPU arm must still use every core of its affinity mask
    (round 1: the reference arm ran single-threaded under torchrun and hit the driver's time limit at N = 2, 4, 8)."""
    env = dict(os.environ, OMP_NUM_THREADS="1", RANK="0", WORLD_SIZE="2", LOCAL_RANK="0")
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--gpus", "2", "--steps", "1", "--warmup", "0", "--cpu-n", "12"],
                         capture_output=True, text=True, timeout=600, env=env)
    assert out.returncode == 0, out.stderr[-2000:]
    d = json.loads([ln for ln in out.stdout.splitlines() if ln.strip()][-1])
    assert d["cpu_baseline"]["cores"] == len(os.sched_getaffinity(0)) and d["n_gpus"] == 2


def _bench(*args, timeout=600):
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), *args], capture_output=True, text=True, timeout=timeout)
    assert out.returncode == 0, out.stderr[-3000:]
    return json.loads([ln for ln in out.stdout.splitlines() if ln.strip()][-1])


def _load_dump(d):
    assert sorted(os.listdir(d)) == ["fine_sdf.npy", "sdf_dists.npy"]
    assert sum(os.path.getsize(os.path.join(d, f)) for f in os.listdir(d)) <= 64 * 10 ** 6
    sdf, fine = np.load(os.path.join(d, "sdf_dists.npy")), np.load(os.path.join(d, "fine_sdf.npy"))
    assert sdf.dtype == np.float64 and fine.dtype == np.float32
    return sdf, fine


def test_reference_arm_dump_outputs(tmp_path):
    """--dump-outputs writes the results of the last timed step; with the same arguments two runs write the same arrays."""
    import oracle
    from fixtures import Grid, simp_hex8
    n = 12
    for run in ("a", "b"):
        d = _bench("--impl", "reference", "--steps", "2", "--warmup", "0", "--cpu-n", str(n), "--dump-outputs", str(tmp_path / run))
        assert d["steps"] == 2
    sdf, fine = _load_dump(tmp_path / "a")
    sdf_b, fine_b = _load_dump(tmp_path / "b")
    assert np.array_equal(sdf, sdf_b) and np.array_equal(fine, fine_b)
    X, IEN, rho = simp_hex8(n)
    g = Grid(X.min(0), X.max(0), 2 * n, 3)
    nt = len(os.sched_getaffinity(0))          # the reference arm's thread count (its distance buffers are per thread)
    rn = oracle.nodal_densities(X, IEN, rho)
    dist, _, _ = oracle.eval_distances(X, IEN, g, rn, 0.5, 1.1, nthreads=nt, want_xp=False)
    osdf, _ = oracle.remove_artifacts(dist * oracle.sign_detection(X, IEN, g, rn, 0.5, nthreads=nt), g)
    vd, vf = oracle.mesh_volume(X, IEN, rho)
    ofine, _ = oracle.rbf_smoothing(osdf, g, True, 2, vd * vf, mode=0, nthreads=nt)
    assert sdf.shape == tuple(int(v) + 1 for v in g.N[::-1]) and np.array_equal(sdf.ravel(), osdf)
    assert fine.shape == ofine.shape and np.array_equal(fine, ofine)


def test_dump_outputs_samples_what_exceeds_the_budget(tmp_path):
    import bench
    big = np.arange(10 ** 6, dtype=np.float32).reshape(100, 100, 100)
    small = np.linspace(-1.0, 1.0, 1000).reshape(10, 10, 10)
    for run in ("a", "b"):
        bench.dump_outputs(str(tmp_path / run), {"big": big, "small": small}, budget=1 << 20)
    a, b = np.load(tmp_path / "a" / "big.npy"), np.load(tmp_path / "b" / "big.npy")
    assert np.array_equal(a, b) and a.dtype == np.float32 and a.ndim == 1
    assert 0.9 * (1 << 17) < a.size <= 1 << 17 and np.all(np.diff(a) > 0)          # sorted distinct flat positions, values at those positions
    assert np.array_equal(np.load(tmp_path / "a" / "small.npy"), small)             # within its share: written whole, shape kept


def test_steps_must_be_positive():
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "0"], capture_output=True, text=True, timeout=120)
    assert out.returncode != 0 and "--steps" in out.stderr


@pytest.mark.gpu
def test_gpu_arm_dump_outputs_are_the_pipeline_results(r2s, tmp_path):
    """The CUDA arm times exactly --steps pipeline calls and --dump-outputs holds what the last of them computed: the same bits as a
    device-resident pipeline call on the same inputs in this process."""
    import ctypes as C
    from fixtures import simp_hex8
    n, steps = 12, 3
    d = _bench("--n", str(n), "--steps", str(steps), "--warmup", "1", "--no-cpu-baseline", "--dump-outputs", str(tmp_path / "out"))
    sdf, fine = _load_dump(tmp_path / "out")
    X, IEN, rho = simp_hex8(n)
    mesh = r2s.Mesh(X, IEN, rho)
    grid = r2s.Grid(X.min(0), X.max(0), 2 * n, 3)
    rn = r2s.DenseInNodes(mesh, rho)
    mesh._use_grid(grid)
    c = mesh.ctx
    c.check(c.lib.r2s_upload_nodal_densities(c.h, rn.ctypes.data_as(C.c_void_p)))
    p = r2s.Params(); c.lib.r2s_default_params(C.byref(p))
    p.rho_t, p.smooth, p.rbf_interp, p.remove_artifacts = 0.5, 2, 1, 1
    p.target_volume, p.final_volume = mesh.V_frac * mesh.V_domain, 1
    for _ in range(2):
        rep = r2s.Report()
        c.check(c.lib.r2s_pipeline_resident(c.h, C.byref(p), C.byref(rep)))
    osdf = np.empty(grid.ngp); c.check(c.lib.r2s_download_sdf(c.h, osdf.ctypes.data_as(C.c_void_p)))
    ofine = np.empty(int(np.prod(grid.N * 2 + 1)), dtype=np.float32); c.check(c.lib.r2s_download_fine_sdf(c.h, ofine.ctypes.data_as(C.c_void_p)))
    mesh.ctx.close()
    assert d["steps"] == steps and d["gpu_launches"] == steps * rep.launches
    assert sdf.shape == tuple(int(v) + 1 for v in grid.N[::-1]) and np.array_equal(sdf.ravel(), osdf)
    assert fine.shape == tuple(int(v) * 2 + 1 for v in grid.N[::-1]) and np.array_equal(fine.ravel(), ofine)
