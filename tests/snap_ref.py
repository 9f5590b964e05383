"""Host build of the vertex search of r2s_isosurface_lattice (tests/host/snap_host.cpp on rho2sdf.jl_b200/csrc/r2s_snap.cuh and
r2s_sample.cuh, built on first use with OpenMP and -ffp-contract=off), a plain-Python restatement of the same rule (the header comment of
r2s_snap.cuh, step by step), and the lattice helpers the GPU tests share: the crossing edges of a lattice field in vertex order, and the
host replay of a whole lattice surface's vertices."""
import ctypes as C
import os
import struct
import subprocess

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
_LIB = None


def lib():
    global _LIB
    if _LIB is None:
        src = os.path.join(HERE, "host", "snap_host.cpp")
        so = os.path.join(HERE, "host", "libsnap_host.so")
        deps = [src] + [os.path.join(ROOT, "rho2sdf.jl_b200", "csrc", f) for f in ("r2s_sample.cuh", "r2s_snap.cuh")]
        if not os.path.exists(so) or os.path.getmtime(so) < max(os.path.getmtime(d) for d in deps):
            subprocess.check_call(["g++", "-O2", "-std=c++17", "-ffp-contract=off", "-fopenmp", "-fPIC", "-shared", src, "-o", so])
        L = C.CDLL(so)
        fp = np.ctypeslib.ndpointer(np.float32, flags="C")
        dp = np.ctypeslib.ndpointer(np.float64, flags="C")
        ip = np.ctypeslib.ndpointer(np.int32, flags="C")
        lp = np.ctypeslib.ndpointer(np.int64, flags="C")
        L.snap_host_max_evals.restype = C.c_int
        L.snap_host_poly_f.argtypes = [dp, C.c_double, C.c_float]
        L.snap_host_poly_f.restype = C.c_float
        L.snap_host_poly.argtypes = [dp, C.c_double, C.c_float, C.c_float, C.c_float, C.c_float, C.c_float, fp, C.POINTER(C.c_int)]
        L.snap_host_poly.restype = C.c_float
        L.snap_host_lattice.argtypes = [fp, ip, dp, dp, C.c_double, C.c_double, C.c_float, fp, fp, lp, C.c_long, C.c_float, fp, fp, ip]
        _LIB = L
    return _LIB


def max_evals():
    return int(lib().snap_host_max_evals())


# ---- constructed edges ------------------------------------------------------------------------------------------------------------------
class Poly:
    """f(x) = float(c0 + x (c1 + x (c2 + x c3)) + amp * noise(x)), noise a hash of the bits of x in [-1, 1] (snap_host.cpp)"""

    def __init__(self, c, amp=0.0):
        self.c = np.ascontiguousarray(c, np.float64)
        self.amp = float(amp)

    def __call__(self, x):
        return np.float32(lib().snap_host_poly_f(self.c, self.amp, float(np.float32(x))))

    def search(self, xa, xb, iso, va=None, vb=None):
        """the host build on the edge [xa, xb]: (x, (lo, hi, flo, fhi), evals); va / vb default to f at the ends"""
        xa, xb = np.float32(xa), np.float32(xb)
        va = self(xa) if va is None else np.float32(va)
        vb = self(xb) if vb is None else np.float32(vb)
        tr = np.zeros(4, np.float32)
        ev = C.c_int()
        x = lib().snap_host_poly(self.c, self.amp, float(xa), float(xb), float(va), float(vb), float(np.float32(iso)), tr, C.byref(ev))
        return np.float32(x), tuple(np.float32(v) for v in tr), ev.value


def key(x):
    u = struct.unpack("<I", struct.pack("<f", float(np.float32(x))))[0]
    return (~u & 0xffffffff) if u & 0x80000000 else (u | 0x80000000)


def unkey(k):
    u = (k & 0x7fffffff) if k & 0x80000000 else (~k & 0xffffffff)
    return np.float32(struct.unpack("<f", struct.pack("<I", u))[0])


def python_search(f, xa, xb, va, vb, iso, cap=48):
    """The rule of r2s_snap.cuh restated in Python (Python floats are IEEE doubles, np.float32 rounds once): (x, (lo, hi, flo, fhi), evals)"""
    iso = np.float32(iso)
    sa = bool(np.float32(va) >= iso)
    lo, hi, flo, fhi = np.float32(xa), np.float32(xb), np.float32(va), np.float32(vb)
    glo, ghi = float(flo) - float(iso), float(fhi) - float(iso)
    last, n = 0, 0
    while n < cap:
        klo, khi = key(lo), key(hi)
        kmin, kmax = min(klo, khi), max(klo, khi)
        if kmax - kmin <= 1:
            break
        t = glo / (glo - ghi)
        x = np.float32(float(lo) + (float(hi) - float(lo)) * t)
        kx = key(x)
        if not (kmin < kx < kmax):
            x = unkey(kmin + (kmax - kmin) // 2)
        fx = np.float32(f(x))
        r = float(fx) - float(iso)
        n += 1
        if bool(fx >= iso) == sa:
            lo, flo, glo = x, fx, r
            if last == 1:
                ghi *= 0.5
            last = 1
        else:
            hi, fhi, ghi = x, fx, r
            if last == 2:
                glo *= 0.5
            last = 2
    x = hi if abs(float(fhi) - float(iso)) < abs(float(flo) - float(iso)) else lo
    return x, (lo, hi, flo, fhi), n


# ---- lattice surfaces -------------------------------------------------------------------------------------------------------------------
def crossing_edges(field, iso):
    """(nv, 4) int64 rows (i, j, k, axis) of the lattice edges of field[k, j, i] whose ends lie on different sides of iso (inside iff
    value >= iso), in the library's vertex order: linear id of the lower point, then axis x < y < z"""
    f = np.asarray(field, np.float32)
    nz, ny, nx = f.shape
    ins = f >= np.float32(iso)
    rows = []
    for ax, (sl_a, sl_b) in enumerate([((slice(None), slice(None), slice(0, -1)), (slice(None), slice(None), slice(1, None))),
                                       ((slice(None), slice(0, -1), slice(None)), (slice(None), slice(1, None), slice(None))),
                                       ((slice(0, -1), slice(None), slice(None)), (slice(1, None), slice(None), slice(None)))]):
        k, j, i = np.nonzero(ins[sl_a] != ins[sl_b])
        rows.append(np.stack([i, j, k, np.full_like(i, ax)], 1).astype(np.int64))
    e = np.concatenate(rows)
    lin = (e[:, 2] * ny + e[:, 1]) * nx + e[:, 0]
    return np.ascontiguousarray(e[np.lexsort((e[:, 3], lin))])


def lattice_vertices(F, origin, spacing, edges, iso):
    """the host replay of the vertices of `edges` on the field F (sample_ref.Field): (V (n, 3) float32, brackets (n, 4) float32, evals (n,))"""
    e = np.ascontiguousarray(edges, np.int64)
    n = len(e)
    V = np.zeros((n, 3), np.float32)
    tr = np.zeros((n, 4), np.float32)
    ev = np.zeros(n, np.int32)
    o32 = np.ascontiguousarray(np.broadcast_to(np.asarray(origin, np.float64), (3,)).astype(np.float32))
    h32 = np.ascontiguousarray(np.broadcast_to(np.asarray(spacing, np.float64), (3,)).astype(np.float32))
    if n:
        lib().snap_host_lattice(F.w, F.n, F.amin, F.amax, F.cell, F.cut, float(F.th), o32, h32, e, n, float(np.float32(iso)), V.reshape(-1), tr.reshape(-1), ev)
    return V, tr, ev


def adjacent(a, b):
    return abs(key(a) - key(b)) <= 1
