"""z-slab decomposition: host-side logic on CPU (gloo, world_size 2) and the multi-GPU parity run (needs >= 2 GPUs)."""
import os
import subprocess
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_slab_partition_tiles_the_planes(r2s):
    for nz in (3, 7, 11, 67, 519):
        for world in (1, 2, 3, 4, 8):
            if nz < 3 * world:
                continue
            parts = r2s.slab_partition(nz, world)
            assert parts[0][0] == 0 and parts[-1][1] == nz and len(parts) == world
            assert all(a[1] == b[0] for a, b in zip(parts, parts[1:]))
            sizes = [b - a for a, b in parts]
            assert max(sizes) - min(sizes) <= 1 and min(sizes) >= 3
    with pytest.raises(r2s.R2SError):
        r2s.slab_partition(2, 4)


def test_weighted_slab_partition_equalises_cost(r2s):
    nz, world = 519, 8
    cost = np.ones(nz); cost[:12] = 3.0; cost[-12:] = 3.0          # expensive end planes (mesh boundary faces)
    parts = r2s.slab_partition(nz, world, plane_cost=cost)
    assert parts[0][0] == 0 and parts[-1][1] == nz and all(a[1] == b[0] for a, b in zip(parts, parts[1:]))
    loads = [cost[a:b].sum() for a, b in parts]
    assert max(loads) / (cost.sum() / world) < 1.03
    assert parts[0][1] - parts[0][0] < parts[3][1] - parts[3][0]  # the end slabs are thinner
    assert min(b - a for a, b in parts) >= 3
    uniform = r2s.slab_partition(nz, world, plane_cost=np.ones(nz))
    assert max(b - a for a, b in uniform) - min(b - a for a, b in uniform) <= 1


_GLOO_WORKER = r"""
import os, sys
sys.path.insert(0, %(root)r); sys.path.insert(0, os.path.join(%(root)r, "tests"))
import numpy as np, torch, torch.distributed as dist
import rho2sdf_b200 as r2s, oracle
from fixtures import simp_hex8, Grid
rank, world = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"])
dist.init_process_group("gloo")
# 1. the communicator id travels from rank 0 to every rank unchanged
made = []
uid = r2s.broadcast_unique_id(lambda: (made.append(1), bytes(range(128)))[1], rank, world)
assert uid == bytes(range(128)) and (len(made) == 1) == (rank == 0)
# 2. slabs computed independently (here with the CPU oracle standing in for the device) assemble into the single-rank result:
#    distances and signs need no exchange when every rank sees the whole mesh
n = 6
X, IEN, rho = simp_hex8(n)
g = Grid(X.min(0), X.max(0), 2 * n, 3)
rn = oracle.nodal_densities(X, IEN, rho)
d, _, _ = oracle.eval_distances(X, IEN, g, rn, 0.5, 1.1, want_xp=False)
s = oracle.sign_detection(X, IEN, g, rn, 0.5)
full = (d * s).reshape(int(g.N[2]) + 1, -1)
k0, k1 = r2s.slab_partition(full.shape[0], world)[rank]
mine = torch.from_numpy(full[k0:k1].copy())
sizes = [b - a for a, b in r2s.slab_partition(full.shape[0], world)]
parts = [torch.empty(sz, full.shape[1], dtype=torch.float64) for sz in sizes]
dist.all_gather(parts, mine) if len(set(sizes)) == 1 else [dist.broadcast(parts[r] if r != rank else mine, src=r) for r in range(world)]
parts[rank] = mine
assert np.array_equal(torch.cat(parts).numpy(), full)
# 3. a size-independent invariant of the interior mask: the all-gathered 1-bit mask has the same popcount as the full mask
cnt = torch.tensor([int((mine.numpy() >= 0).sum())]); dist.all_reduce(cnt)
assert int(cnt.item()) == int((full >= 0).sum())
dist.barrier(); dist.destroy_process_group()
print("GLOO OK", rank)
"""


def test_slab_host_logic_gloo_world2(tmp_path):
    script = tmp_path / "w.py"
    script.write_text(_GLOO_WORKER % {"root": ROOT})
    env = dict(os.environ, OMP_NUM_THREADS="2")
    out = subprocess.run([sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", "2", "--master-addr", "127.0.0.1", "--master-port", "29731", str(script)],
                         capture_output=True, text=True, timeout=600, env=env)
    assert out.returncode == 0, out.stdout[-2000:] + out.stderr[-4000:]
    assert out.stdout.count("GLOO OK") == 2


@pytest.mark.gpu
@pytest.mark.parametrize("p2p", ["1", "0"])
def test_slab_parity_multi_gpu(p2p):
    """p2p = 1: scalar all-reduces and CG halo planes over the peer-memory mailbox; R2S_P2P=0: everything through NCCL."""
    import torch
    ngpu = torch.cuda.device_count()
    if ngpu < 2:
        pytest.skip("needs at least 2 GPUs")
    world = 2 if ngpu < 4 else 4
    out = subprocess.run([sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", str(world), "--master-addr", "127.0.0.1", "--master-port", "29732",
                          os.path.join(ROOT, "tests", "slab_parity_ranks.py"), "48"], capture_output=True, text=True, timeout=900, env=dict(os.environ, R2S_P2P=p2p))
    assert out.returncode == 0 and "SLAB PARITY OK" in out.stdout, out.stdout[-3000:] + out.stderr[-3000:]
