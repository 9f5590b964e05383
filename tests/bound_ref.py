"""Host build of the box projection's lower bounds (rho2sdf.jl_b200/csrc/r2s_bound.cuh, tests/host/bound_host.cpp) and an independent
restatement of the distance from a point to (box /\\ slab) by enumeration of the active sets of the quadratic program."""
import ctypes as C
import itertools
import os
import subprocess

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
_L = None


def lib():
    global _L
    if _L is None:
        d = os.path.join(HERE, "host")
        src, so = os.path.join(d, "bound_host.cpp"), os.path.join(d, "libbound_host.so")
        hdrs = [os.path.join(ROOT, "rho2sdf.jl_b200", "csrc", h) for h in ("r2s_iso.cuh", "r2s_bound.cuh")]
        if not os.path.exists(so) or os.path.getmtime(so) < max(os.path.getmtime(p) for p in [src] + hdrs):
            subprocess.check_call(["g++", "-O2", "-std=c++17", "-ffp-contract=off", "-fPIC", "-shared", "-I/usr/local/cuda/include", src, "-o", so])
        L = C.CDLL(so)
        dp = np.ctypeslib.ndpointer(np.float64, flags="C"); ip = np.ctypeslib.ndpointer(np.int32, flags="C")
        L.bnd_host_element.argtypes = [dp, dp, C.c_double, dp]
        L.bnd_host_lb.argtypes = [C.c_long, dp, dp, dp]
        L.bnd_host_lb2gap.argtypes = [C.c_long, dp, dp, dp]
        L.bnd_host_project.argtypes = [dp, dp, C.c_double, C.c_long, dp, dp, ip, ip]
        _L = L
    return _L


def element(Xe, re, rho_t):
    """tlo, thi, n, A, B of a box element as k_box_records stores them (None if the element is not an axis-aligned box)"""
    out = np.zeros(11)
    if not lib().bnd_host_element(np.ascontiguousarray(Xe, np.float64), np.ascontiguousarray(re, np.float64), rho_t, out):
        return None
    return out


def lb(P, rec):
    """lb_box_slab for the points P (n, 3) and an element record of element()"""
    P = np.ascontiguousarray(np.atleast_2d(P), np.float64)
    out = np.zeros(len(P))
    lib().bnd_host_lb(len(P), P, np.ascontiguousarray(rec), out)
    return out


def lb2_gap(P, rec):
    """lb2_box_gap (squared box distance + slab gap) for the points P (n, 3)"""
    P = np.ascontiguousarray(np.atleast_2d(P), np.float64)
    out = np.zeros(len(P))
    lib().bnd_host_lb2gap(len(P), P, np.ascontiguousarray(rec), out)
    return out


def project(Xe, re, rho_t, P):
    """distances k_project_list reports for the points P (n, 3) of one box element, converged flags, phase-2 iterations"""
    P = np.ascontiguousarray(np.atleast_2d(P), np.float64)
    d = np.zeros(len(P)); ok = np.zeros(len(P), np.int32); it = np.zeros(len(P), np.int32)
    rc = lib().bnd_host_project(np.ascontiguousarray(Xe, np.float64), np.ascontiguousarray(re, np.float64), rho_t, len(P), P, d, ok, it)
    assert rc == 0
    return d, ok.astype(bool), it


def box_slab_distance(P, tlo, thi, n, A, B):
    """min |y - P| over tlo <= y <= thi, A <= n.y <= B, by enumerating the active sets: every coordinate free, at its lower or at its
    upper face, the slab constraint inactive or at A or at B.  Each equality-constrained subproblem is solved in closed form (the free
    coordinates move along n); the answer is the smallest distance among the feasible candidates (the optimum is one of them)."""
    P = np.asarray(P, np.float64)
    best = np.inf
    tol = 1e-12 * (1 + np.abs(P).sum() + np.abs(tlo).sum() + np.abs(thi).sum())
    planes = [None] + [v for v in (A, B) if np.isfinite(v)]
    for fix in itertools.product((0, 1, 2), repeat=3):
        y0 = np.array([P[d] if fix[d] == 0 else (tlo[d] if fix[d] == 1 else thi[d]) for d in range(3)])
        free = np.array([f == 0 for f in fix])
        for c in planes:
            y = y0.copy()
            if c is not None:
                nf = np.where(free, n, 0.0)
                s = float(nf @ nf)
                if s == 0.0:
                    continue
                y = y0 + nf * (c - float(n @ y0)) / s
            if np.all(y >= tlo - tol) and np.all(y <= thi + tol) and (not np.isfinite(A) or n @ y >= A - tol) and (not np.isfinite(B) or n @ y <= B + tol):
                best = min(best, float(np.linalg.norm(y - P)))
    return best
