#!/usr/bin/env python
"""Side-by-side timing of the A/B knobs on the bench workload (one process; a fresh context per variant, because r2s_create reads the
knobs once).

    python tools/ab_variants.py [--n 256] [--steps 2] [--variants "name:K=V,K=V;name2:..."]

For every variant: 1 warm-up + `steps` timed passes of r2s_pipeline_resident; prints the stage times, the iteration counters and
max |sdf - sdf(first variant)| / h.  One JSON line per variant on stdout."""
import argparse, ctypes as C, json, os, sys
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT); sys.path.insert(0, os.path.join(ROOT, "tests"))
import numpy as np

DEFAULT = "default:;no_prune:R2S_PROJ_PRUNE=0;general_proj:R2S_PROJ_BOX=0;sign_lists:R2S_SIGN_LATTICE=0"
KNOBS = ("R2S_PROJ_BOX", "R2S_PROJ_PRUNE", "R2S_SIGN_LATTICE", "R2S_P2P", "R2S_SURF_PLANES")      # cleared before every variant (R2S_SURF_PLANES: no effect on the pipeline)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--n", type=int, default=256)
    ap.add_argument("--steps", type=int, default=2)
    ap.add_argument("--variants", default=DEFAULT)
    args = ap.parse_args()
    import torch
    import rho2sdf_b200 as r2s
    from fixtures import simp_hex8
    n = args.n
    X, IEN, rho = simp_hex8(n)
    ref = None
    grid = r2s.Grid(X.min(0), X.max(0), 2 * n, 3)
    buf = torch.empty(int(grid.ngp), dtype=torch.float64).pin_memory()
    for spec in args.variants.split(";"):
        name, _, kv = spec.partition(":")
        for k in KNOBS:
            os.environ.pop(k, None)
        for item in filter(None, kv.split(",")):
            k, _, v = item.partition("=")
            os.environ[k] = v
        mesh = r2s.Mesh(X, IEN, rho, element_type=r2s.HEX8)
        rho_n = r2s.DenseInNodes(mesh, rho)
        mesh._use_grid(grid)
        c = mesh.ctx
        p = r2s.Params(); c.lib.r2s_default_params(C.byref(p))
        p.rho_t, p.smooth, p.rbf_interp, p.remove_artifacts = 0.5, 2, 1, 1
        p.target_volume, p.final_volume = mesh.V_frac * mesh.V_domain, 1
        c.check(c.lib.r2s_upload_nodal_densities(c.h, rho_n.ctypes.data_as(C.c_void_p)))
        reps = []
        for it in range(1 + args.steps):
            rep = r2s.Report()
            c.check(c.lib.r2s_pipeline_resident(c.h, C.byref(p), C.byref(rep)))
            if it:
                reps.append(rep)
        c.check(c.lib.r2s_download_sdf(c.h, C.c_void_p(buf.data_ptr())))
        sdf = buf.numpy()
        if ref is None:
            ref = sdf.copy(); diff = 0.0; sign_diff = 0
        else:
            diff = float(np.max(np.abs(sdf - ref))) / grid.cell_size; sign_diff = int(np.count_nonzero(np.signbit(sdf) != np.signbit(ref)))
        out = {"variant": name, "knobs": kv, "n": n}
        for k in ("ms_bin", "ms_project", "ms_assemble", "ms_sign", "ms_cc", "ms_cg", "ms_lsf", "ms_threshold", "ms_fine", "ms_volume", "ms_total"):
            out[k] = round(float(np.mean([getattr(r, k) for r in reps])), 3)
        out.update(pairs=int(reps[-1].n_pairs), pruned=int(reps[-1].n_pairs_pruned), newton_iters=int(reps[-1].n_newton_iters), not_converged=int(reps[-1].n_not_converged),
                   cg_iters=int(reps[-1].cg_iters), th=float(reps[-1].th), max_diff_over_h=diff, sign_diff=sign_diff)
        print(json.dumps(out), flush=True)
        c.close()


if __name__ == "__main__":
    main()
