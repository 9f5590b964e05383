"""ctypes binding of tests/host/points_oracle.c: the CPU reference of evalDistances / Sign_Detection at a list of points (n, 3), built on
the CPU oracle.  TEST INFRASTRUCTURE ONLY.  The library is compiled once per process into a temporary directory (the tree may be
read-only), with the oracle's flags."""
import ctypes as C
import os
import subprocess
import tempfile

import numpy as np

import oracle

HERE = os.path.dirname(os.path.abspath(__file__))
_LIB = None
_dp = np.ctypeslib.ndpointer(dtype=np.float64, flags="C_CONTIGUOUS")
_ip = np.ctypeslib.ndpointer(dtype=np.int64, flags="C_CONTIGUOUS")


def lib():
    global _LIB
    if _LIB is None:
        cc = "/usr/bin/gcc" if os.path.exists("/usr/bin/gcc") else "gcc"
        so = os.path.join(tempfile.mkdtemp(prefix="r2s_points_oracle_"), "libpoints_oracle.so")
        src = os.path.join(HERE, "host", "points_oracle.c")
        flags = ["-O2", "-fPIC", "-std=c11", "-ffp-contract=off", "-fno-fast-math", "-fvisibility=hidden", "-w", "-shared"]
        try:
            subprocess.check_call([cc] + flags + ["-fopenmp", src, "-o", so, "-lm"])
        except subprocess.CalledProcessError:      # no libgomp: serial
            subprocess.check_call([cc] + flags + [src, "-o", so, "-lm"])
        L = C.CDLL(so)
        c_i64 = C.c_int64
        L.r2so_eval_distances_points.argtypes = [c_i64, _dp, c_i64, C.c_int, _ip, _dp, _dp, _ip, C.c_double, _dp, C.c_double, C.c_double,
                                                 _dp, c_i64, _dp, C.c_void_p, C.c_void_p]
        L.r2so_sign_detection_points.argtypes = [c_i64, _dp, c_i64, C.c_int, _ip, _dp, _dp, _ip, C.c_double, _dp, C.c_double, _dp, c_i64, C.c_int, _dp]
        _LIB = L
    return _LIB


def _points(points):
    P = np.ascontiguousarray(points, dtype=np.float64).reshape(-1, 3)
    return P, P.shape[0]


def eval_distances_points(X, IEN, grid, rho_n, rho_t, points, delta_factor=1.1, want_xp=True):
    """evalDistances at a list of points (n, 3): (dist (n,), xp (n, 3) or None, stats)."""
    X, IEN, nnp, nel, nen = oracle._mesh(X, IEN)
    amin, amax, N, cell = oracle._grid(grid)
    P, n = _points(points)
    dist = np.zeros(n)
    xp = np.zeros((n, 3)) if want_xp else None
    stats = np.zeros(3, dtype=np.int64)
    lib().r2so_eval_distances_points(nnp, X, nel, nen, IEN, amin, amax, N, cell, np.ascontiguousarray(rho_n, dtype=np.float64), float(rho_t),
                                     float(delta_factor), P, n, dist, xp.ctypes.data if want_xp else None, stats.ctypes.data)
    return dist, xp, {"pairs": int(stats[0]), "iters": int(stats[1]), "not_converged": int(stats[2])}


def sign_detection_points(X, IEN, grid, rho_n, rho_t, points, nthreads=None):
    """Sign_Detection at a list of points (n, 3) -> signs (n,)."""
    X, IEN, nnp, nel, nen = oracle._mesh(X, IEN)
    amin, amax, N, cell = oracle._grid(grid)
    P, n = _points(points)
    signs = np.zeros(n)
    lib().r2so_sign_detection_points(nnp, X, nel, nen, IEN, amin, amax, N, cell, np.ascontiguousarray(rho_n, dtype=np.float64), float(rho_t), P, n,
                                     int(nthreads or oracle.max_threads()), signs)
    return signs
