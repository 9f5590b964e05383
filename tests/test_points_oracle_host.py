"""CPU tests of the CPU reference of evalDistances / Sign_Detection at a list of points (tests/host/points_oracle.c, built on the oracle):
on the grid's own points they equal the grid functions bit for bit, their results are a function of the point alone, and points outside
the grid box get the far value."""
import numpy as np
import pytest

import oracle
import points_oracle
from points_cases import GRID_CASES, case, edge_points, grid_points


@pytest.mark.parametrize("name", GRID_CASES)
def test_grid_points_equal_grid_functions(name):
    X, IEN, rn, grid, params, _ = case(name)
    P = grid_points(grid)
    for rt, df in params:
        d, xp, st = oracle.eval_distances(X, IEN, grid, rn, rt, df)
        pd, pxp, pst = points_oracle.eval_distances_points(X, IEN, grid, rn, rt, P, df)
        assert np.array_equal(pd, d) and np.array_equal(pxp, xp) and pst == st
        s = oracle.sign_detection(X, IEN, grid, rn, rt)
        assert np.array_equal(points_oracle.sign_detection_points(X, IEN, grid, rn, rt, P), s)


@pytest.mark.parametrize("name", ["sphere", "graded_lattice_hex8", "schlafli_tet4"])
def test_permutation_and_duplication_invariance(name):
    X, IEN, rn, grid, params, _ = case(name)
    rt, df = params[0]
    P = edge_points(X, IEN, grid, rn, rt, n=600)
    d, xp, _ = points_oracle.eval_distances_points(X, IEN, grid, rn, rt, P, df)
    s = points_oracle.sign_detection_points(X, IEN, grid, rn, rt, P)
    rng = np.random.default_rng(1)
    idx = rng.integers(0, P.shape[0], size=2 * P.shape[0])      # a permutation with repeats
    d2, xp2, _ = points_oracle.eval_distances_points(X, IEN, grid, rn, rt, P[idx], df)
    assert np.array_equal(d2, d[idx]) and np.array_equal(xp2, xp[idx])
    assert np.array_equal(points_oracle.sign_detection_points(X, IEN, grid, rn, rt, P[idx]), s[idx])
    assert (d < 1e9).any() and (s > 0).any()


@pytest.mark.parametrize("name", ["sphere", "schlafli_tet4"])
def test_points_outside_the_grid_box(name):
    X, IEN, rn, grid, params, _ = case(name)
    rt, df = params[0]
    h = grid.cell_size
    c = 0.5 * (grid.AABB_min + grid.AABB_max)
    P = np.array([[grid.AABB_min[0] - 0.5 * h, c[1], c[2]], [c[0], grid.AABB_max[1] + 1.5 * h, c[2]], [c[0], c[1], grid.AABB_min[2] - 3 * h],
                  [1e30, -1e30, 1e30], [grid.AABB_max[0] + 1e3, c[1], c[2]]])
    d, xp, _ = points_oracle.eval_distances_points(X, IEN, grid, rn, rt, P, df)
    assert np.array_equal(d, np.full(len(P), 1e10)) and not xp.any()
    assert np.array_equal(points_oracle.sign_detection_points(X, IEN, grid, rn, rt, P), -np.ones(len(P)))
