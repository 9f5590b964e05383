"""Meshes, grids and point sets of the evalDistances / Sign_Detection points tests (tests/test_points_*.py)."""
import numpy as np

import oracle
from fixtures import BLOCK_RHO_N, Grid, block_geometry, graded_lattice_hex8, load_mesh, schlafli_tet4, simp_hex8


def grid_points(grid):
    """generateGridPoints (Grid.jl:81-93): amin + cell * i per axis, x fastest -- the coordinates the grid entry points use."""
    ax = [grid.AABB_min[d] + grid.cell_size * np.arange(int(grid.N[d]) + 1, dtype=np.float64) for d in range(3)]
    k, j, i = np.meshgrid(np.arange(ax[2].size), np.arange(ax[1].size), np.arange(ax[0].size), indexing="ij")
    return np.stack([ax[0][i.ravel()], ax[1][j.ravel()], ax[2][k.ravel()]], axis=1)


def case(name):
    """(X, IEN, rho_n, grid, [(rho_t, delta_factor), ...], is_tet); grid.nmax = the N_max it was built with"""
    out = _case(name)
    out[3].nmax = {"block": 20, "sphere": 10, "sphere5": 5, "schlafli_tet4": 14, "graded_lattice_hex8": 24, "simp": 24}.get(name, 30)
    return out


def _case(name):
    if name == "block":
        X, IEN, _ = block_geometry([2, 1, 1])
        return X, IEN, BLOCK_RHO_N, Grid(X.min(0), X.max(0), 20, 3), [(0.5, 1.1), (0.5, 2.5)], False
    if name == "sphere":
        X, IEN, rho = load_mesh("sphere")
        return X, IEN, oracle.nodal_densities(X, IEN, rho), Grid(X.min(0), X.max(0), 10, 3), [(0.5, 1.1), (0.5, 2.5)], False
    if name == "sphere5":
        X, IEN, rho = load_mesh("sphere")
        return X, IEN, oracle.nodal_densities(X, IEN, rho), Grid(X.min(0), X.max(0), 5, 3), [(0.1, 1.1), (0.9, 1.1)], False
    if name in ("cantilever_beam_vfrac_03", "chapadlo"):
        X, IEN, rho = load_mesh(name)
        return X, IEN, oracle.nodal_densities(X, IEN, rho), Grid(X.min(0), X.max(0), 30, 3), [(0.5, 1.1)], False
    if name == "graded_lattice_hex8":
        X, IEN, rho = graded_lattice_hex8(10)
        return X, IEN, oracle.nodal_densities(X, IEN, rho), Grid(X.min(0), X.max(0), 24, 3), [(0.5, 1.1)], False
    if name == "simp":
        X, IEN, rho = simp_hex8(12)
        return X, IEN, oracle.nodal_densities(X, IEN, rho), Grid(X.min(0), X.max(0), 24, 3), [(0.5, 1.1)], False
    if name == "schlafli_tet4":
        X, IEN, rn = schlafli_tet4(6, "simp")
        return X, IEN, rn, Grid(X.min(0), X.max(0), 14, 3), [(0.5, 1.1)], True
    raise KeyError(name)


GRID_CASES = ["block", "sphere", "sphere5", "cantilever_beam_vfrac_03", "chapadlo", "graded_lattice_hex8", "schlafli_tet4"]


def edge_points(X, IEN, grid, rn, rho_t, seed=7, n=4000):
    """Point sets that hit the edge cases of the binning and of the per-pair rules: uniform in the grid box widened by two cells, clustered
    within 0.1 h of the iso surface (edge crossings of rho_t), exactly on cell boundaries amin + c (amax - amin) / N, on element nodes,
    edge midpoints and face centres, at the centres of lattice holes (elements' boxes that hold no element), and duplicates."""
    rng = np.random.default_rng(seed)
    h = grid.cell_size
    lo, hi = grid.AABB_min - 2 * h, grid.AABB_max + 2 * h
    sets = [rng.uniform(lo, hi, size=(n, 3))]
    E = X[IEN - 1]                                     # (nel, nen, 3)
    r = rn[IEN - 1]
    a, b = r[:, :-1], r[:, 1:]
    el, k = np.nonzero((a - rho_t) * (b - rho_t) < 0)
    if el.size:
        pick = rng.choice(el.size, size=min(n, el.size), replace=el.size < n)
        t = (rho_t - a[el[pick], k[pick]]) / (b[el[pick], k[pick]] - a[el[pick], k[pick]])
        P = E[el[pick], k[pick]] + t[:, None] * (E[el[pick], k[pick] + 1] - E[el[pick], k[pick]])
        sets.append(P + rng.uniform(-0.1 * h, 0.1 * h, size=P.shape))
    c = np.stack([rng.integers(0, int(grid.N[d]) + 1, size=n) for d in range(3)], axis=1)
    sets.append(grid.AABB_min + c * (grid.AABB_max - grid.AABB_min) / grid.N)
    nodes = X[rng.choice(X.shape[0], size=min(n, X.shape[0]), replace=False)]
    ie = rng.choice(IEN.shape[0], size=min(n, IEN.shape[0]), replace=False)
    sets += [nodes, 0.5 * (E[ie, 0] + E[ie, 1]), E[ie, :4].mean(axis=1), E[ie].mean(axis=1)]
    if IEN.shape[1] == 8:      # centres of lattice cells without an element (holes), from the node coordinate tables
        ax = [np.unique(X[:, d]) for d in range(3)]
        if max(a_.size for a_ in ax) < 64:
            cc = np.stack(np.meshgrid(*[0.5 * (a_[1:] + a_[:-1]) for a_ in ax], indexing="ij"), axis=-1).reshape(-1, 3)
            have = {tuple(np.round(v, 12)) for v in E.mean(axis=1)}
            holes = np.array([v for v in cc if tuple(np.round(v, 12)) not in have]).reshape(-1, 3)
            if holes.size:
                sets.append(holes)
    P = np.concatenate(sets, axis=0)
    return np.concatenate([P, P[rng.choice(P.shape[0], size=P.shape[0] // 10)]], axis=0)
