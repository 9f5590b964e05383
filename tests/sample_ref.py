"""Host build of the sampler of the continuous smoothed SDF (tests/host/sample_host.cpp on rho2sdf.jl_b200/csrc/r2s_sample.cuh, built on
first use with OpenMP and -ffp-contract=off), plus float64 restatements of the same definition and of the reference's
rbf_interpolation_kdtree (RBFs4Smoothing.jl:219-248) for the tests."""
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
        src = os.path.join(HERE, "host", "sample_host.cpp")
        so = os.path.join(HERE, "host", "libsample_host.so")
        deps = [src, os.path.join(ROOT, "rho2sdf.jl_b200", "csrc", "r2s_sample.cuh")]
        if not os.path.exists(so) or os.path.getmtime(so) < max(os.path.getmtime(d) for d in deps):
            subprocess.check_call(["g++", "-O2", "-std=c++17", "-ffp-contract=off", "-fopenmp", "-fPIC", "-shared", src, "-o", so])
        L = C.CDLL(so)
        fp = np.ctypeslib.ndpointer(np.float32, flags="C")
        dp = np.ctypeslib.ndpointer(np.float64, flags="C")
        ip = np.ctypeslib.ndpointer(np.int32, flags="C")
        L.smp_host_exp.argtypes = [fp, C.c_long, fp]
        L.smp_host_exp_scan.argtypes = [C.c_float, C.c_float, C.POINTER(C.c_double), C.POINTER(C.c_float)]
        L.smp_host_maxd.argtypes = [C.c_double, C.c_double]
        L.smp_host_maxd.restype = C.c_float
        L.smp_host_t2.argtypes = [C.c_float]
        L.smp_host_t2.restype = C.c_float
        L.smp_host_range.argtypes = [C.c_double, C.c_double, C.c_int, fp]
        L.smp_host_eval.argtypes = [fp, ip, dp, dp, C.c_double, C.c_double, C.c_float, dp, C.c_long, fp, C.c_void_p]
        _LIB = L
    return _LIB


def exp_f32(x):
    x = np.ascontiguousarray(x, np.float32)
    out = np.empty_like(x)
    lib().smp_host_exp(x, x.size, out)
    return out


def exp_scan(lo, hi):
    m, w = C.c_double(), C.c_float()
    lib().smp_host_exp_scan(lo, hi, C.byref(m), C.byref(w))
    return m.value, w.value


def maxd(cut, cell):
    return np.float32(lib().smp_host_maxd(cut, cell))


def t2(md):
    return np.float32(lib().smp_host_t2(md))


def table(amin, amax, n):
    out = np.empty(int(n), np.float32)
    lib().smp_host_range(float(amin), float(amax), int(n), out)
    return out


class Field:
    """A weight array w[k, j, i] on the grid (amin, amax, N), with cell size `cell`, cut-off `cut` and offset th."""

    def __init__(self, w, amin, amax, cell, cut, th):
        self.w = np.ascontiguousarray(w, np.float32)
        self.amin, self.amax = np.asarray(amin, np.float64), np.asarray(amax, np.float64)
        self.n = np.array(self.w.shape[::-1], np.int32)
        self.cell, self.cut, self.th = float(cell), float(cut), np.float32(th)
        self.C = [table(self.amin[d], self.amax[d], self.n[d]) for d in range(3)]
        self.kappa = np.float32(1.0 / (self.cell * self.cell))
        self.maxd = maxd(self.cut, self.cell)
        self.t2 = t2(self.maxd)

    def host(self, pts, gradient=False):
        """the host build: values (n,) float32 and, if asked, gradients (n, 3)"""
        p = np.ascontiguousarray(pts, np.float64).reshape(-1, 3)
        val = np.empty(len(p), np.float32)
        g = np.empty((len(p), 3), np.float32) if gradient else None
        lib().smp_host_eval(self.w, self.n, self.amin, self.amax, self.cell, self.cut, float(self.th), p, len(p), val,
                            g.ctypes.data_as(C.c_void_p) if gradient else None)
        return (val, g) if gradient else val

    def taps(self, p):
        """the definition's tap set at one point: [(i, j, k, e (3,) float32)] in ascending (k, j, i), decided in Float32 as the header does"""
        p = np.asarray(p, np.float64).astype(np.float32)
        out = []
        with np.errstate(over="ignore"):
            e = [self.C[d] - p[d] for d in range(3)]                                     # Float32
            ee = [(x * x).astype(np.float32) for x in e]
        # a window of 4 points around the floor plane per axis holds every point within maxd < 3 cells
        win = [range(max(0, int(np.searchsorted(self.C[d], p[d], side="right")) - 5), min(self.n[d], int(np.searchsorted(self.C[d], p[d], side="right")) + 5))
               for d in range(3)]
        xi = np.array(list(win[0]), np.int64)
        for k in win[2]:
            if ee[2][k] > self.t2:
                continue
            for j in win[1]:
                if ee[1][j] > self.t2:
                    continue
                d2 = ((ee[0][xi] + ee[1][j]).astype(np.float32) + ee[2][k]).astype(np.float32)
                for i in xi[d2 <= self.t2]:
                    out.append((int(i), j, k, np.array([e[0][i], e[1][j], e[2][k]], np.float32)))
        return out

    def float64(self, p, perturb=None):
        """value, gradient, sum |w phi|, tap count of the same definition in float64 (same Float32 tap set and e, exact arithmetic after)
        perturb: None, "drop" (leave out the smallest nonzero |w phi|) or "add" (add the nearest excluded coarse point)"""
        taps = self.taps(p)
        kap = float(self.kappa)
        val, grad, A = 0.0, np.zeros(3), 0.0
        terms = []
        for i, j, k, e in taps:
            e64 = e.astype(np.float64)
            phi = np.exp(-kap * float(e64 @ e64))
            t = float(self.w[k, j, i]) * phi
            terms.append(t)
            val += t; grad += 2 * kap * t * e64; A += abs(t)
        if perturb == "drop":
            nz = [abs(t) for t in terms if t != 0.0]
            if not nz:
                return None
            s = min(range(len(terms)), key=lambda q: abs(terms[q]) if terms[q] != 0.0 else np.inf)
            val -= terms[s]
        elif perturb == "add":
            pf = np.asarray(p, np.float64).astype(np.float32).astype(np.float64)
            inc = {(i, j, k) for i, j, k, _ in taps}
            best = None
            lo = [max(0, int(np.searchsorted(self.C[d], pf[d])) - 4) for d in range(3)]
            for k in range(lo[2], min(self.n[2], lo[2] + 9)):
                for j in range(lo[1], min(self.n[1], lo[1] + 9)):
                    for i in range(lo[0], min(self.n[0], lo[0] + 9)):
                        if (i, j, k) in inc or self.w[k, j, i] == 0:
                            continue
                        e = np.array([self.C[0][i], self.C[1][j], self.C[2][k]], np.float64) - pf
                        d2 = float(e @ e)
                        if best is None or d2 < best[0]:
                            best = (d2, float(self.w[k, j, i]))
            if best is None:
                return None
            val += best[1] * np.exp(-kap * best[0])
        return val + float(self.th), grad, A, len(taps)

    def knn124(self, Q):
        """rbf_interpolation_kdtree (RBFs4Smoothing.jl:219-248) restated as in tests/test_oracle_golden.py: the 124 nearest coarse points
        (scipy's cKDTree for NearestNeighbors.jl), kept if their Float32 distance is <= maxd, summed in ascending distance, plus th"""
        from scipy.spatial import cKDTree
        f32 = np.float32
        kk, jj, ii = np.meshgrid(np.arange(self.n[2]), np.arange(self.n[1]), np.arange(self.n[0]), indexing="ij")
        P = np.stack([self.C[0][ii.ravel()], self.C[1][jj.ravel()], self.C[2][kk.ravel()]], axis=1).astype(np.float64)
        wf = self.w.ravel()
        tree = cKDTree(P)
        Qf = np.asarray(Q, np.float64).astype(f32).astype(np.float64)
        dist, idx = tree.query(Qf, k=min(124, len(P)))
        sigma = self.cell
        out = np.zeros(len(Q), f32)
        for t in range(dist.shape[1]):
            dt = dist[:, t].astype(f32)
            term = wf[idx[:, t]].astype(np.float64) * np.exp(-(dt.astype(np.float64) / sigma) ** 2)
            out = np.where(dt <= self.maxd, (out.astype(np.float64) + term).astype(f32), out)
        return (out + self.th).astype(f32)


# the round-off constant K of the bound (n_taps + K) 2^-24 (sum |w phi| + |th|) on value - float64 value.  Per tap, phi carries
#   e^2 (1 rounding) and kappa e^2 (1) per axis: the argument of exp is off by up to 2 m_d 2^-24 relative, m_d = kappa e_d^2, i.e. the
#   factor a_d by 2 m_d 2^-24, and sum_d m_d = kappa |e|^2 <= kappa t2 <= ln(1/cut) < 8 for an included tap: 16;
#   exp_f32 on each axis: 3 * 1.5 (header bound); the two products (a_x a_y) a_z: 2;
# so |phi - exp(-kappa |e|^2)| <= 22.5 2^-24 phi.  The fma chain adds n_taps 2^-24 (sum |w phi|) (gamma_n, first order), the final + th one
# more rounding of |acc| + |th|.  K = 16 + 4.5 + 2 + 1 = 23.5, rounded up to 24.
K_ROUNDOFF = 24
