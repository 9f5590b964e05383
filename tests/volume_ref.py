"""Exact host reference of the library's cut-cell volume (tests/host/vol_host.cpp, built on first use with OpenMP).

`reference` restates calculate_volume_from_sdf at quadrature order 9 as the library computes it: per cut cell the Float32 sum of
cut_cell_quad9 (the library's own header), as the integer llrint(part * 2^37), added without wrap-around into a Python int; the volume is
nfull * ev + (S / 2^37) * jac with S rounded to double once.  `periodic_reference` gets the same numbers for a field that repeats a small
tile, from one single-cell reference per corner pattern times the number of cells with that pattern."""
import ctypes as C
import os
import subprocess

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
_LIB = None


def lib():
    global _LIB
    if _LIB is None:
        src = os.path.join(HERE, "host", "vol_host.cpp")
        so = os.path.join(HERE, "host", "libvol_host.so")
        deps = [src] + [os.path.join(ROOT, "rho2sdf.jl_b200", "csrc", h) for h in ("r2s_volq.cuh", "r2s_tables.cuh")]
        if not os.path.exists(so) or os.path.getmtime(so) < max(os.path.getmtime(d) for d in deps):
            subprocess.check_call(["g++", "-O2", "-std=c++17", "-ffp-contract=off", "-fopenmp", "-fPIC", "-shared", src, "-o", so])
        L = C.CDLL(so)
        fp = np.ctypeslib.ndpointer(np.float32, flags="C")
        up = np.ctypeslib.ndpointer(np.uint64, flags="C")
        dp = np.ctypeslib.ndpointer(np.float64, flags="C")
        L.vol_host_quad9.argtypes = [fp, C.c_long, fp, fp, C.c_float, fp, fp, fp, fp]
        L.vol_host_gauss9.argtypes = [fp, fp]
        L.vol_host_grid.argtypes = [fp, C.c_long, C.c_long, C.c_long, C.c_long, C.c_float, C.c_float, C.c_float, C.c_int, C.POINTER(C.c_longlong),
                                    C.POINTER(C.c_ulonglong), C.POINTER(C.c_ulonglong), C.POINTER(C.c_double)]
        L.vol_host_fixed_value.argtypes = [up, up, C.c_long, dp, dp]
        _LIB = L
    return _LIB


def reference(sdf3, edge, iso=0.0, th=0.0, memo=True):
    """sdf3: float32 [k, j, i] (x fastest).  Returns (nfull, S, volume) with S the exact fixed-point sum (int)."""
    a = np.ascontiguousarray(sdf3, dtype=np.float32)
    nz, ny, nx = a.shape
    nf, lo, hi, v = C.c_longlong(), C.c_ulonglong(), C.c_ulonglong(), C.c_double()
    lib().vol_host_grid(a.ravel(), nx, ny, nz, nx, float(np.float32(iso)), float(np.float32(th)), float(np.float32(edge)), int(memo),
                        C.byref(nf), C.byref(lo), C.byref(hi), C.byref(v))
    return nf.value, (hi.value << 64) | lo.value, v.value


def volume_of(nfull, S, edge):
    """The library's conversion: float32 ev = edge^3, jac = ev / 8; nfull * ev + (S / 2^37) * jac in double, S rounded once."""
    e = np.float32(edge)
    ev = np.float32(np.float32(e * e) * e)
    jac = np.float32(ev / np.float32(8.0))
    return float(nfull) * float(ev) + (float(S) / 2.0 ** 37) * float(jac)


def fine_edge(grid, smooth):
    """The cell edge the pipeline's final volume uses: Float32 range of the x axis on the fine grid, norm of its first step."""
    fx = int(grid.N[0]) * smooth + 1
    a, b = np.float32(grid.AABB_min[0]), np.float32(grid.AABB_max[0])
    dxf = np.float32((b - a) / np.float32(fx - 1))
    d = np.float32(np.float32(a + np.float32(1.0) * dxf) - a)
    return np.float32(np.sqrt(np.float32(d * d)))


def _class_counts(n, p):
    """Number of cell origins i in [0, n - 1) with i % p == r, for r in range(p)."""
    return [len(range(r, n - 1, p)) for r in range(p)]


def periodic_classes(tile, shape):
    """Cells of the field f[k, j, i] = tile[k % pz, j % py, i % px] on `shape` = (nz, ny, nx) points, grouped by corner pattern:
    yields (count, 2x2x2 single-cell field)."""
    tile = np.asarray(tile, np.float32)
    pz, py, px = tile.shape
    cz, cy, cx = (_class_counts(n, p) for n, p in zip(shape, tile.shape))
    for rk in range(pz):
        for rj in range(py):
            for ri in range(px):
                cnt = cz[rk] * cy[rj] * cx[ri]
                if cnt:
                    idx = np.ix_([(rk + d) % pz for d in (0, 1)], [(rj + d) % py for d in (0, 1)], [(ri + d) % px for d in (0, 1)])
                    yield cnt, np.ascontiguousarray(tile[idx])


def periodic_reference(tile, shape, edge, iso=0.0):
    """(nfull, S, volume) of the periodic field, from the single-cell references of its corner patterns."""
    nfull, S = 0, 0
    for cnt, cell in periodic_classes(tile, shape):
        f, s, _ = reference(cell, edge, iso)
        nfull += cnt * f
        S += cnt * s
    return nfull, S, volume_of(nfull, S, edge)


def periodic_field(tile, shape):
    tile = np.asarray(tile, np.float32)
    nz, ny, nx = shape
    k, j, i = np.ogrid[:nz, :ny, :nx]
    return tile[k % tile.shape[0], j % tile.shape[1], i % tile.shape[2]]
