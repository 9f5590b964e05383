"""The cut-cell quadrature of the volume kernels (rho2sdf.jl_b200/csrc/r2s_volq.cuh: packed f32x2 lerps, explicit fma) compiled for the
HOST and compared bit for bit with the loop it replaced, as nvcc had contracted it.  Threshold search and final volume are only exact
(integer sums of per-cell Float32 results) if every cell's sum is unchanged."""
import ctypes as C
import os
import subprocess

import numpy as np
import pytest

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)


@pytest.fixture(scope="module")
def host():
    src = os.path.join(HERE, "host", "vol_host.cpp")
    so = os.path.join(HERE, "host", "libvol_host.so")
    hdr = os.path.join(ROOT, "rho2sdf.jl_b200", "csrc", "r2s_volq.cuh")
    if not os.path.exists(so) or os.path.getmtime(so) < max(os.path.getmtime(src), os.path.getmtime(hdr)):
        subprocess.check_call(["g++", "-O2", "-std=c++17", "-ffp-contract=off", "-fPIC", "-shared", src, "-o", so])
    L = C.CDLL(so)
    fp = np.ctypeslib.ndpointer(np.float32, flags="C")
    L.vol_host_quad9.argtypes = [fp, C.c_long, fp, fp, C.c_float, fp, fp, fp, fp]
    return L


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
