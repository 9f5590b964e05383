"""GPU tests of the seeded, slab-bounded pruning of the box projection (r2s_dist.cu: k_pair_scan<0/1/2>, r2s_bound.cuh): the distance
field must be bit-identical to projecting every (element, point) pair (R2S_PROJ_PRUNE=0) across SIMP sizes, grid ratios, thresholds and
candidate ranges, and on the workload's pattern most pairs must go unsolved."""
import numpy as np
import pytest

from fixtures import simp_hex8

pytestmark = pytest.mark.gpu

CASES = {      # (n elements per axis, SIMP period in elements, grid points along the longest axis, void border of 2 elements)
    "simp12_fine_grid": (12, 24.0, 60, False),
    "simp16": (16, 32.0, 32, False),
    "simp20_coarse_grid": (20, 16.0, 17, False),
    "simp24": (24, 64.0, 48, False),
    "simp32_p64": (32, 64.0, 64, False),
    "simp32_p64_void_border": (32, 64.0, 64, True),
}


def _fields(r2s, monkeypatch, case, knob):
    n, period, nmax, border = CASES[case]
    X, IEN, rho = simp_hex8(n, period_frac=period / n)
    if border:      # no active element on the mesh boundary: no tile holds boundary faces, so every pair can be pruned
        r = rho.reshape(n, n, n).copy()
        for ax in range(3):
            sl = [slice(None)] * 3
            sl[ax] = np.r_[0:2, n - 2:n]
            r[tuple(sl)] = 0.0
        rho = r.ravel()
    monkeypatch.setenv("R2S_PROJ_PRUNE", knob)
    mesh = r2s.Mesh(X, IEN, rho)
    grid = r2s.Grid(X.min(0), X.max(0), nmax, 3)
    rn = r2s.DenseInNodes(mesh, rho)
    out = []
    for rt in (0.3, 0.5):
        for df in (1.1, 2.5):
            d, _ = r2s.evalDistances(mesh, grid, None, rn, rt, delta_factor=df, want_xp=False)
            rep = mesh.ctx.report()
            out.append((rt, df, d, int(rep.n_pairs), int(rep.n_pairs_pruned)))
    mesh.ctx.close()
    return out


@pytest.mark.parametrize("case", sorted(CASES))
def test_seeded_pruning_is_exact(r2s, monkeypatch, case):
    on, off = _fields(r2s, monkeypatch, case, "1"), _fields(r2s, monkeypatch, case, "0")
    for (rt, df, d1, np1, pr1), (_, _, d0, np0, pr0) in zip(on, off):
        assert np1 == np0 > 0 and pr0 == 0 and pr1 < np1, (case, rt, df, np1, pr1)
        assert np.array_equal(d1, d0), (case, rt, df, float(np.max(np.abs(d1 - d0))))
        print("%s rho_t=%.1f delta=%.1f: %d pairs, %.1f%% solved" % (case, rt, df, np1, 100.0 * (np1 - pr1) / np1))


def test_solved_fraction_on_the_workload_pattern(r2s, monkeypatch):
    """simp32 with the bench workload's 64-element period, rho_t = 0.5, delta = 1.1, and a void border so that no pair goes to the pair
    buffer unpruned (tiles with boundary faces are solved in full; on a mesh this small they would hold most pairs): the seed and the
    bounds leave fewer than 35 % of the candidate pairs to the solver (23.0 % in the host replay of the same rules; the counts are
    deterministic)"""
    rt, df, _, npairs, pruned = _fields(r2s, monkeypatch, "simp32_p64_void_border", "1")[2]
    assert (rt, df) == (0.5, 1.1)
    print("simp32, period 64, void border: %d pairs, %d solved (%.1f%%)" % (npairs, npairs - pruned, 100.0 * (npairs - pruned) / npairs))
    assert npairs - pruned < 0.35 * npairs
