"""The cut-cell quadrature of the volume kernels (rho2sdf.jl_b200/csrc/r2s_volq.cuh: packed f32x2 lerps, explicit fma) compiled for the
HOST and compared bit for bit with the loop it replaced, as nvcc had contracted it.  Threshold search and final volume are only exact
(integer sums of per-cell Float32 results) if every cell's sum is unchanged.

The whole-grid host reference built on it (tests/volume_ref.py) is checked here against the CPU oracle, analytic planar volumes and its
own periodic-class shortcut; tests/test_volume_exact.py compares the GPU with it bit for bit."""
import numpy as np
import pytest

import oracle
import volume_ref


@pytest.fixture(scope="module")
def host():
    return volume_ref.lib()


def gauss9():
    x, w = np.polynomial.legendre.leggauss(9)
    return np.ascontiguousarray(x, np.float32), np.ascontiguousarray(w, np.float32)


def run(host, cells, iso):
    cells = np.ascontiguousarray(cells, np.float32)
    n = cells.shape[0]
    gx, gw = gauss9()
    out = [np.empty(n, np.float32) for _ in range(4)]
    host.vol_host_quad9(cells, n, gx, gw, iso, *out)
    return out


def edge_cells(rng):
    cells = []
    for _ in range(2000):      # corners equal to the threshold (values are corner - th, so exactly 0), of either sign of zero
        c = rng.normal(size=8).astype(np.float32)
        k = rng.integers(1, 8)
        c[rng.choice(8, k, replace=False)] = rng.choice(np.array([0.0, -0.0], np.float32), k)
        cells.append(c)
    for _ in range(2000):      # all-zero and ±0 mixtures
        cells.append(rng.choice(np.array([0.0, -0.0], np.float32), 8))
    for _ in range(2000):      # planar cuts with Gauss values that are exactly 0: c = a (x - 1/2) with the midplane through Gauss points
        a = np.float32(rng.choice([1.0, 2.0, 0.5, 4.0]))
        s = np.array([-1, 1, -1, 1, -1, 1, -1, 1], np.float32) * a
        cells.append(s if rng.random() < 0.5 else np.roll(s.reshape(2, 2, 2), 1, axis=rng.integers(3)).ravel())
    for _ in range(4000):      # mixed magnitudes 1e-30 .. 1e30
        mag = 10.0 ** rng.uniform(-30, 30, 8)
        cells.append((rng.choice([-1.0, 1.0], 8) * mag).astype(np.float32))
    return np.array(cells, np.float32)


@pytest.mark.parametrize("iso", [0.0, 0.25, -1e-3])
def test_cut_cell_quadrature_is_bit_identical_to_the_old_loop(host, iso):
    rng = np.random.default_rng(7)
    rand = rng.normal(size=(100000, 8)).astype(np.float32) + rng.normal(size=(100000, 1)).astype(np.float32) * 0.5
    cells = np.concatenate([rand, edge_cells(rng)])
    part_new, m_new, part_old, m_old = run(host, cells, iso)
    assert np.array_equal(part_new.view(np.uint32), part_old.view(np.uint32))
    assert np.array_equal(m_new.view(np.uint32), m_old.view(np.uint32))
    assert 0.2 < np.mean((part_new > 0) & (part_new < 7.99)) < 1.0      # the fuzz does exercise cut cells


def test_library_gauss_table_is_numpys():
    x, w = np.empty(9, np.float32), np.empty(9, np.float32)
    volume_ref.lib().vol_host_gauss9(x, w)
    gx, gw = gauss9()
    assert np.array_equal(x, gx) and np.array_equal(w, gw)


def _fields(rng):
    n = (23, 17, 29)      # (nz, ny, nx)
    k, j, i = np.meshgrid(*[np.linspace(-1, 1, m) for m in n], indexing="ij")
    yield "noise", rng.uniform(-1, 1, n).astype(np.float32), 0.0
    yield "sphere", (0.7 - np.sqrt(i * i + j * j + k * k)).astype(np.float32), 0.0
    yield "gyroid", (np.sin(5 * i) * np.cos(4 * j) + np.sin(4 * j) * np.cos(5 * k) + np.sin(5 * k) * np.cos(4 * i)).astype(np.float32), 0.25
    yield "sphere_iso", (0.7 - np.sqrt(i * i + j * j + k * k)).astype(np.float32), -1e-3


@pytest.mark.parametrize("edge", [1.0, 0.0625, 0.37])
def test_reference_matches_oracle(edge):
    """The oracle (r2s_oracle.c) restates the reference's loop with its own arithmetic and sums cell by cell in double: agreement to
    Float32 round-off of the per-cell sums (the tolerance of test_volume_from_sdf_convergence)."""
    for name, f, iso in _fields(np.random.default_rng(3)):
        nfull, S, v = volume_ref.reference(f, edge, iso)
        ov = oracle.volume_from_sdf(f, np.float32(edge), iso=iso)
        assert abs(v - ov) <= 2e-6 * abs(ov), name      # the oracle scales every Gauss weight by jac in float: ~1e-6 at edges that are not powers of 2
        assert v == volume_ref.volume_of(nfull, S, edge)
        assert 0 < S and nfull > 0, name      # cut and full cells both occur


@pytest.mark.parametrize("axis", [0, 1, 2])
@pytest.mark.parametrize("t", [0.3, 0.55, 0.9])
def test_reference_planar_field(axis, t):
    """f = x_axis - c with the plane at a fraction t of cell m: every cut cell holds the Gauss points on the far side of the plane, so the
    volume is the full cells plus the cut slab times the 1-D Gauss sum of the step, and within half the largest weight of the analytic one."""
    shape, edge, m = [18, 13, 21], 0.5, 6
    c = (m + t) * edge
    ax = np.arange(shape[2 - axis], dtype=np.float64) * edge
    f = np.moveaxis(np.broadcast_to((ax - c)[:, None, None], (shape[2 - axis],) + tuple(s for d, s in enumerate(shape) if d != 2 - axis)), 0, 2 - axis)
    f = np.ascontiguousarray(f, np.float32)
    nfull, S, v = volume_ref.reference(f, edge)
    cells_across = int(np.prod([s - 1 for d, s in enumerate(shape) if d != 2 - axis]))
    gx, gw = np.polynomial.legendre.leggauss(9)
    step = gw[(gx + 1) / 2 >= t].sum() / 2
    ncells_full = (shape[2 - axis] - 2 - m) * cells_across
    assert nfull == ncells_full
    ev = edge ** 3
    assert abs(v - (ncells_full + cells_across * step) * ev) <= 1e-6 * v
    analytic = (shape[2 - axis] - 1 - m - t) * edge * cells_across * edge ** 2
    assert abs(v - analytic) <= 0.5 * gw.max() / 2 * cells_across * ev + 1e-9


def test_periodic_shortcut_matches_direct_reference():
    """The class shortcut (one single-cell reference per corner pattern, times its cell count) against the direct sum, with and without
    the per-thread memo, on small periodic grids whose sizes leave partial periods; includes a pattern with corners exactly at iso."""
    rng = np.random.default_rng(11)
    tiles = [np.array([1.0, -1.0], np.float32).reshape(1, 1, 2), rng.uniform(-1, 1, (3, 2, 5)).astype(np.float32),
             np.array([[[0.0, -0.0, 0.5]], [[-0.25, 0.0, 1.0]]], np.float32)]
    for tile in tiles:
        for shape in [(7, 6, 9), (4, 11, 16), (2, 2, 2)]:
            f = volume_ref.periodic_field(tile, shape)
            for iso in (0.0, 0.25):
                direct = volume_ref.reference(f, 0.5, iso, memo=False)
                assert volume_ref.reference(f, 0.5, iso, memo=True) == direct
                assert volume_ref.periodic_reference(tile, shape, 0.5, iso) == direct


def test_two_word_fixed_point_conversion_rounds_once():
    """vol_fixed_value (r2s_volq.cuh): the two accumulator words -> S / 2^37, against the compiler's 128-bit integer conversion; sums
    below 2^64 (where it must be the single-word value), just above, at the largest sum 2^31 cells can reach, and at rounding ties."""
    rng = np.random.default_rng(5)
    n = 200000
    s0 = rng.integers(0, 2 ** 63, n, dtype=np.uint64)
    s1 = rng.integers(0, 2 ** 39, n, dtype=np.uint64)
    s1[: n // 4] = rng.integers(0, 2 ** 20, n // 4, dtype=np.uint64)      # below 2^64
    ties = []
    for e in range(1, 9):      # S = 2^(64 + e - 1) + (2k + 1) * 2^(e + 10): exactly halfway between two doubles
        for k in (0, 1, 12345):
            S = (1 << (63 + e)) + (2 * k + 1) * (1 << (e + 10))
            ties += [S, S + 1, S - 1]
    tw = np.array([[S & 0xffffffff, S >> 32] for S in ties], dtype=np.uint64)
    s0 = np.concatenate([s0, tw[:, 0], np.array([2 ** 63 - 1], np.uint64)])
    s1 = np.concatenate([s1, tw[:, 1], np.array([2 ** 39 - 1], np.uint64)])
    got, ref = np.empty(s0.size), np.empty(s0.size)
    volume_ref.lib().vol_host_fixed_value(s0, s1, s0.size, got, ref)
    assert np.array_equal(got, ref)
    exact = [float(((int(b) << 32) + int(a))) / 2.0 ** 37 for a, b in zip(s0[-len(ties) - 1:], s1[-len(ties) - 1:])]
    assert np.array_equal(got[-len(ties) - 1:], np.array(exact))      # Python's int -> float is correctly rounded too
