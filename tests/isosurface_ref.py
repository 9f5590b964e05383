"""Host reference of the isosurface stage (tests/host/mc_host.cpp, built on first use with OpenMP and -ffp-contract=off), plus the mesh
checks the tests share: directed-edge pairing, Euler characteristic, connected components, divergence-theorem volume."""
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
        src = os.path.join(HERE, "host", "mc_host.cpp")
        so = os.path.join(HERE, "host", "libmc_host.so")
        deps = [src, os.path.join(ROOT, "rho2sdf.jl_b200", "csrc", "r2s_mc.cuh")]
        if not os.path.exists(so) or os.path.getmtime(so) < max(os.path.getmtime(d) for d in deps):
            subprocess.check_call(["g++", "-O2", "-std=c++17", "-ffp-contract=off", "-fopenmp", "-fPIC", "-shared", src, "-o", so])
        L = C.CDLL(so)
        fp = np.ctypeslib.ndpointer(np.float32, flags="C")
        dp = np.ctypeslib.ndpointer(np.float64, flags="C")
        ip = np.ctypeslib.ndpointer(np.int32, flags="C")
        L.mc_host_table.argtypes = [np.ctypeslib.ndpointer(np.uint8, flags="C")]
        L.mc_host_face_segments.argtypes = [C.c_int, C.c_int, ip]
        L.mc_host_face.argtypes = [C.c_int, ip]
        L.mc_host_edge.argtypes = [C.c_int, C.POINTER(C.c_int), C.POINTER(C.c_int)]
        L.mc_host_count.argtypes = [fp, C.c_longlong, C.c_longlong, C.c_longlong, C.c_float, C.POINTER(C.c_longlong), C.POINTER(C.c_longlong)]
        L.mc_host_extract.argtypes = [fp, C.c_longlong, C.c_longlong, C.c_longlong, dp, dp, C.c_float, fp, ip]
        _LIB = L
    return _LIB


def table():
    """[(tuple of triangles (e0, e1, e2))] for the 256 cases."""
    raw = np.zeros(256 * 16, dtype=np.uint8)
    lib().mc_host_table(raw)
    raw = raw.reshape(256, 16)
    return [tuple(tuple(int(v) for v in raw[c, 1 + 3 * t:4 + 3 * t]) for t in range(raw[c, 0])) for c in range(256)]


def edges():
    """cube edge e -> (start corner, axis)"""
    out = []
    for e in range(12):
        c, a = C.c_int(), C.c_int()
        lib().mc_host_edge(e, C.byref(c), C.byref(a))
        out.append((c.value, a.value))
    return out


def face(f):
    cyc = np.zeros(4, np.int32)
    lib().mc_host_face(f, cyc)
    return [int(v) for v in cyc]


def face_segments(case, f):
    seg = np.zeros(4, np.int32)
    n = lib().mc_host_face_segments(case, f, seg)
    return [(int(seg[2 * q]), int(seg[2 * q + 1])) for q in range(n)]


def reference(sdf3, origin=(0.0, 0.0, 0.0), spacing=(1.0, 1.0, 1.0), iso=0.0):
    """sdf3: float32 [k, j, i] (x fastest).  Returns (V (nv, 3) float32, T (nt, 3) int32) in the library's order."""
    a = np.ascontiguousarray(sdf3, dtype=np.float32)
    nz, ny, nx = a.shape
    nv, nt = C.c_longlong(), C.c_longlong()
    lib().mc_host_count(a.ravel(), nx, ny, nz, float(np.float32(iso)), C.byref(nv), C.byref(nt))
    V = np.zeros((nv.value, 3), np.float32)
    T = np.zeros((nt.value, 3), np.int32)
    lib().mc_host_extract(a.ravel(), nx, ny, nz, np.ascontiguousarray(origin, np.float64), np.ascontiguousarray(spacing, np.float64), float(np.float32(iso)),
                          V.reshape(-1), T.reshape(-1))
    return V, T


# ---- mesh checks ----------------------------------------------------------------------------------------------------------------------
def unpaired_edges(T):
    """Directed edges (a, b) whose reverse (b, a) is not used exactly once, or that are used more than once: [] for a closed, consistently
    oriented surface.  Returns the offending directed edges."""
    if len(T) == 0:
        return np.zeros((0, 2), np.int64)
    d = np.concatenate([T[:, [0, 1]], T[:, [1, 2]], T[:, [2, 0]]]).astype(np.int64)
    n = int(T.max()) + 1
    key = d[:, 0] * n + d[:, 1]
    uk, cnt = np.unique(key, return_counts=True)

    def count(k):
        idx = np.minimum(np.searchsorted(uk, k), len(uk) - 1)
        return np.where(uk[idx] == k, cnt[idx], 0)
    bad = (count(key) != 1) | (count(d[:, 1] * n + d[:, 0]) != 1)
    return d[bad]


def euler_characteristic(T):
    d = np.concatenate([T[:, [0, 1]], T[:, [1, 2]], T[:, [2, 0]]]).astype(np.int64)
    e = np.unique(np.sort(d, axis=1), axis=0)
    return len(np.unique(T)) - len(e) + len(T)


def components(T):
    """number of connected components of the triangles (sharing a vertex)"""
    import scipy.sparse as sp
    import scipy.sparse.csgraph as cg
    nv = int(T.max()) + 1
    r = np.concatenate([T[:, 0], T[:, 1]])
    c = np.concatenate([T[:, 1], T[:, 2]])
    g = sp.coo_matrix((np.ones(len(r)), (r, c)), shape=(nv, nv))
    n, lab = cg.connected_components(g, directed=False)
    return len(np.unique(lab[np.unique(T)]))


def divergence_volume(V, T):
    """sum v0 . (v1 x v2) / 6 in double: the enclosed volume of a closed surface oriented outwards"""
    v = V.astype(np.float64)
    a, b, c = v[T[:, 0]], v[T[:, 1]], v[T[:, 2]]
    return float(np.sum(np.einsum("ij,ij->i", a, np.cross(b, c))) / 6.0)


def on_boundary_face(V, T, edges_, origin, spacing, shape):
    """True for each directed edge whose two vertices lie in one and the same boundary face of the grid (shape = (nz, ny, nx) points)"""
    v = (V.astype(np.float64) - np.asarray(origin)) / np.asarray(spacing)
    hi = np.array([shape[2] - 1, shape[1] - 1, shape[0] - 1], np.float64)
    p, q = v[edges_[:, 0]], v[edges_[:, 1]]
    ok = np.zeros(len(edges_), bool)
    for d in range(3):
        for b in (0.0, hi[d]):
            ok |= (np.abs(p[:, d] - b) < 1e-4) & (np.abs(q[:, d] - b) < 1e-4)
    return ok


def stl_normals(V, T):
    """unit normals as the STL writer computes them: double cross product (v1 - v0) x (v2 - v0), 0 for a degenerate triangle"""
    v = V.astype(np.float64)
    n = np.cross(v[T[:, 1]] - v[T[:, 0]], v[T[:, 2]] - v[T[:, 0]])
    ln = np.linalg.norm(n, axis=1)
    out = np.zeros_like(n)
    nz = ln > 0
    out[nz] = n[nz] / ln[nz, None]
    return out.astype(np.float32)
