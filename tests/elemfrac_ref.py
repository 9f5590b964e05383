"""Host build of the per-element volume fractions of r2s_element_volume_fractions (tests/host/elemfrac_host.cpp on
rho2sdf.jl_b200/csrc/r2s_elemfrac.cuh, built on first use with OpenMP and -ffp-contract=off), plus a plain numpy restatement of the
Gauss-point rule for the tests."""
import ctypes as C
import os
import subprocess

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
CSRC = os.path.join(ROOT, "rho2sdf.jl_b200", "csrc")
_LIB = None


def lib():
    global _LIB
    if _LIB is None:
        src = os.path.join(HERE, "host", "elemfrac_host.cpp")
        so = os.path.join(HERE, "host", "libelemfrac_host.so")
        deps = [src] + [os.path.join(CSRC, f) for f in ("r2s_elemfrac.cuh", "r2s_tables.cuh", "r2s_sample.cuh", "r2s_band.cuh")]
        if not os.path.exists(so) or os.path.getmtime(so) < max(os.path.getmtime(d) for d in deps):
            subprocess.check_call(["g++", "-O2", "-std=c++17", "-ffp-contract=off", "-fopenmp", "-fPIC", "-shared", src, "-o", so])
        L = C.CDLL(so)
        fp = np.ctypeslib.ndpointer(np.float32, flags="C")
        dp = np.ctypeslib.ndpointer(np.float64, flags="C")
        ip = np.ctypeslib.ndpointer(np.int32, flags="C")
        lp = np.ctypeslib.ndpointer(np.int64, flags="C")
        field = [fp, ip, dp, dp, C.c_double, C.c_double, C.c_float]
        L.ef_host_eval.argtypes = field + [C.c_int, dp, lp, C.c_long, C.c_int, C.c_float, dp, dp, ip]
        L.ef_host_points.argtypes = [C.c_int, dp, lp, C.c_long, C.c_int, dp, dp, ip]
        L.ef_host_box.argtypes = [C.c_int, dp, lp, C.c_long, C.c_int, fp, fp]
        L.ef_host_classify.argtypes = field + [C.c_int, fp, fp, fp, fp, lp, lp, C.c_long, fp, ip]
        _LIB = L
    return _LIB


def _mesh(X, IEN):
    """X (nnp, 3) float64 and IEN (nel, nen) 0-based int64, contiguous"""
    return np.ascontiguousarray(X, np.float64), np.ascontiguousarray(IEN, np.int64)


def _field(F):
    return (F.w, F.n, F.amin, F.amax, F.cell, F.cut, float(F.th))


def replay(F, X, IEN, q, iso):
    """(fractions, volumes, cls) of every element (IEN 0-based) on the sample_ref.Field F, every Gauss point evaluated"""
    X, IEN = _mesh(X, IEN)
    nel, nen = IEN.shape
    frac, vol, cls = np.empty(nel), np.empty(nel), np.empty(nel, np.int32)
    lib().ef_host_eval(*_field(F), nen, X, IEN, nel, int(q), float(iso), frac, vol, cls)
    return frac, vol, cls


def points(X, IEN, e, q):
    """(x (q^3, 3), W (q^3,), ok (q^3,) bool) of element e in the order t = (k q + j) q + i"""
    X, IEN = _mesh(X, IEN)
    n = q ** 3
    x, W, ok = np.empty((n, 3)), np.empty(n), np.empty(n, np.int32)
    lib().ef_host_points(IEN.shape[1], X, IEN, int(e), int(q), x, W, ok)
    return x, W, ok.astype(bool)


def boxes(X, IEN, widen=True):
    X, IEN = _mesh(X, IEN)
    nel, nen = IEN.shape
    a, b = np.empty((nel, 3), np.float32), np.empty((nel, 3), np.float32)
    lib().ef_host_box(nen, X, IEN, nel, int(widen), a, b)
    return a, b


def classify_box(F, a, b, iso):
    m = len(a)
    cls = np.empty(m, np.int32)
    iso = np.ascontiguousarray(np.broadcast_to(np.asarray(iso, np.float32), (m,)))
    z3, zi = np.zeros(3, np.float32), np.zeros((m, 3), np.int64)
    lib().ef_host_classify(*_field(F), 0, np.ascontiguousarray(a, np.float32), np.ascontiguousarray(b, np.float32), z3, z3, zi, zi, m, iso, cls)
    return cls


def classify_lattice(F, o, h, lo, hi, iso):
    m = len(lo)
    cls = np.empty(m, np.int32)
    iso = np.ascontiguousarray(np.broadcast_to(np.asarray(iso, np.float32), (m,)))
    z = np.zeros((m, 3), np.float32)
    lib().ef_host_classify(*_field(F), 1, z, z, np.asarray(o, np.float32), np.asarray(h, np.float32), np.ascontiguousarray(lo, np.int64),
                           np.ascontiguousarray(hi, np.int64), m, iso, cls)
    return cls


# ---- numpy restatement of the Gauss-point rule (written independently of the header's operation order) ----------------------------------
def gauss(q):
    g, w = np.polynomial.legendre.leggauss(q)
    return g, w


def numpy_points(Xe, q):
    """Gauss points (q^3, 3) and weights (q^3,) of one element with nodes Xe (nen, 3), order t = (k q + j) q + i"""
    g, w = gauss(q)
    k, j, i = np.meshgrid(np.arange(q), np.arange(q), np.arange(q), indexing="ij")
    i, j, k = i.ravel(), j.ravel(), k.ravel()
    Wq = w[i] * w[j] * w[k]
    if len(Xe) == 8:
        s = np.array([[-1, -1, -1], [1, -1, -1], [1, 1, -1], [-1, 1, -1], [-1, -1, 1], [1, -1, 1], [1, 1, 1], [-1, 1, 1]], np.float64)
        xi = np.stack([g[i], g[j], g[k]], 1)
        N = np.prod(1 + xi[:, None, :] * s[None], axis=2) / 8                                         # (n, 8)
        dN = np.empty((len(xi), 8, 3))
        for c in range(3):
            o = [d for d in range(3) if d != c]
            dN[:, :, c] = s[None, :, c] * np.prod(1 + xi[:, None, o] * s[None][:, :, o], axis=2) / 8
        J = np.einsum("ar,nac->nrc", Xe, dN)
        return N @ Xe, Wq * np.abs(np.linalg.det(J))
    u, v, z = (g[i] + 1) / 2, (g[j] + 1) / 2, (g[k] + 1) / 2
    xi = u
    eta = v * (1 - xi)
    zeta = z * (1 - xi - eta)
    N = np.stack([xi, eta, zeta, 1 - xi - eta - zeta], 1)
    J = np.stack([Xe[0] - Xe[3], Xe[1] - Xe[3], Xe[2] - Xe[3]], 1)
    return N @ Xe, Wq * abs(np.linalg.det(J)) * (1 - xi) * (1 - xi - eta) / 8
