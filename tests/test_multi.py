"""r2s_multi: the single-call multi-GPU entry (one process, one z-slab per entry of `devices`, in-process exchanges over peer memory).
Device ids may repeat, so the multi-slab code path -- slab binning, stitched artifact removal, CG halo exchange, all-reduces, re-cut by
measured cost, piece-wise VTI export -- is exercised on a one-GPU box as well; with >= 2 GPUs the same tests also run on distinct devices."""
import ctypes as C

import numpy as np
import pytest

import volume_ref
from fixtures import load_mesh, simp_hex8

pytestmark = pytest.mark.gpu


def _device_lists():
    import torch
    n = torch.cuda.device_count()
    lists = [[0, 0], [0, 0, 0]]
    if n >= 2:
        lists += [[0, 1], list(range(min(n, 4)))]
    return lists


@pytest.mark.parametrize("case", ["simp24", "chapadlo", "simp24_approx"])
def test_multi_pipeline_matches_single_device(r2s, case, tmp_path):
    if case.startswith("simp24"):
        X, IEN, rho = simp_hex8(24)
        opts = dict(threshold_density=0.5, sdf_grid_setup="manual", grid_step=0.5, rbf_interp=case == "simp24", rbf_grid="fine", remove_artifacts=True,
                    artifact_min_component_ratio=0.3)
    else:
        X, IEN, rho = load_mesh("chapadlo")
        opts = dict(sdf_grid_setup="automatic", rbf_interp=True, rbf_grid="fine", remove_artifacts=True)
    fine1, fg1, grid1, sdf1, rep1 = r2s.rho2sdf(case, X, IEN, rho, options=r2s.Rho2sdfOptions(**opts), return_report=True)
    scale = max(1.0, float(np.abs(fine1).max()))
    assert rep1["volume"] == np.float32(volume_ref.reference(fine1, volume_ref.fine_edge(grid1, 2))[2])
    for devs in _device_lists():
        base = str(tmp_path / ("out%d" % len(devs)))
        fine, fg, grid, sdf, rep = r2s.rho2sdf(case, X, IEN, rho, options=r2s.Rho2sdfOptions(**opts), return_report=True, devices=devs, export_vti=base)
        assert list(grid.N) == list(grid1.N) and rep["rho_t"] == rep1["rho_t"]
        assert np.array_equal(sdf, sdf1), "distances / signs / artifact removal must not depend on the slab count"
        assert rep["n_flipped"] == rep1["n_flipped"] and rep["cg_iters"] == rep1["cg_iters"] and rep["bisections"] == rep1["bisections"]
        # Float32 smoothing: the CG dot products are summed slab by slab, so the fields agree to round-off, not bit for bit
        assert np.max(np.abs(fine - fine1)) <= 1e-5 * scale and abs(rep["th"] - rep1["th"]) <= 1e-5 * scale
        assert abs(rep["volume"] - rep1["volume"]) <= 1e-5 * abs(rep1["volume"]) and rep["collectives"] > 0
        # the final volume is exact for the field each layout returns: the slabs' cell ranges (kf0 / kf1, the halo plane) add up to the grid
        assert rep["volume"] == np.float32(volume_ref.reference(fine, volume_ref.fine_edge(grid, 2))[2])
        if not opts["rbf_interp"]:      # no CG: the threshold search is an integer sum and the evaluation is per point, so nothing may differ
            assert np.array_equal(fine, fine1) and rep["th"] == rep1["th"] and rep["volume"] == rep1["volume"]
        # exportSdfToVTI of a result that lives on several slabs: pieces + index reassemble to the returned field
        dims, origin, spacing, label, arr = r2s.read_pvti(base + ".pvti")
        assert label == "distance" and arr.shape == fine.shape and np.array_equal(arr, fine)
        assert np.allclose(origin, grid.AABB_min) and np.allclose(spacing, [grid.cell_size / 2] * 3)


def test_multi_rebalance_and_repeat_calls(r2s):
    """Several pipeline calls on one handle: the slabs are re-cut by measured cost between calls, results stay identical; a new grid
    resets the partition; errors come back through r2s_multi_last_error."""
    X, IEN, rho = simp_hex8(32)
    mesh = r2s.Mesh(X, IEN, rho, devices=[0, 0, 0, 0])
    m = mesh.multi
    rn = r2s.DenseInNodes(mesh, rho)
    p = r2s.Params(); m.lib.r2s_default_params(C.byref(p))
    p.rho_t, p.smooth, p.rbf_interp, p.remove_artifacts = 0.5, 2, 1, 1
    p.target_volume, p.final_volume = mesh.V_frac * mesh.V_domain, 1
    outs = []
    for nmax in (64, 64, 64, 48):
        grid = r2s.Grid(X.min(0), X.max(0), nmax, 3)
        mesh._use_grid(grid)
        cuts0 = m.slab_planes()
        assert cuts0[0] == 0 and cuts0[-1] == int(grid.N[2]) + 1 and all(b - a >= 3 for a, b in zip(cuts0, cuts0[1:]))
        sdf = np.empty(grid.ngp); fine = np.empty(int(np.prod(grid.N * 2 + 1)), dtype=np.float32); rep = r2s.Report()
        m.check(m.lib.r2s_multi_pipeline(m.h, C.byref(p), rn.ctypes.data_as(C.c_void_p), sdf.ctypes.data_as(C.c_void_p), fine.ctypes.data_as(C.c_void_p), C.byref(rep)))
        outs.append((nmax, sdf, fine, rep.cg_iters, m.slab_planes()))
    assert np.array_equal(outs[0][1], outs[1][1]) and np.array_equal(outs[1][1], outs[2][1]) and outs[0][3] == outs[1][3] == outs[2][3]
    scale = max(1.0, float(np.abs(outs[0][2]).max()))
    assert np.max(np.abs(outs[0][2] - outs[1][2])) <= 1e-5 * scale and np.max(np.abs(outs[1][2] - outs[2][2])) <= 1e-5 * scale
    assert outs[3][1].size != outs[0][1].size and np.isfinite(outs[3][2]).all()
    bad = r2s.Params(); m.lib.r2s_default_params(C.byref(bad)); bad.smooth = 7
    with pytest.raises(r2s.R2SError, match="smooth"):
        m.check(m.lib.r2s_multi_pipeline(m.h, C.byref(bad), rn.ctypes.data_as(C.c_void_p), None, None, None))
    mesh.close()
