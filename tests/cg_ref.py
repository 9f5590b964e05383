"""Host reference of the interpolation-mode solve of RBFs_smoothing (RBFs4Smoothing.jl:199, r2s_dev_rbf in csrc/r2s_rbf.cu) and of the
coarse LSF, in numpy, for tests/test_cg_ref_host.py and tests/test_cg_float64.py.

* `process`: the input processing of k_to_f32 / k_replace_far (RBFs4Smoothing.jl:15-22).
* `K64`: the 81-point kernel matrix (weights exp(-m), m = |d|^2 <= 6, zero outside the grid) applied in float64 with shifted slices.
* `cg64`: IterativeSolvers' `cg` in float64 -- the solve the Float32 kernels approximate.
* `cg32`: the same loop in Float32 arithmetic with float64 dot products and the kernel's factorised weights.  It is a drift model, not an
  emulation: its distance from `cg64` calibrates the tolerance `tau` of the GPU comparison per case, and its `mutate` argument injects the
  defects a subtly wrong kernel would have, so the host tests can show that each one moves the result by far more than `tau`.
* `lsf_bounds`: the coarse LSF K w in float64 and a rigorous bound on the kernel's Float32 error per point.

Fields are indexed [k, j, i] (x fastest), like the library's arrays."""
import numpy as np

EPS32 = float(np.finfo(np.float32).eps)
U = 2.0 ** -24                                                    # unit round-off of Float32
CG_RELTOL = float(np.sqrt(np.float32(EPS32)))                    # IterativeSolvers' default reltol for Float32, sqrt(eps(Float32))

# the 81 offsets (dk, dj, di) with m = dk^2 + dj^2 + di^2 <= 6
OFFSETS = [(dk, dj, di) for dk in range(-2, 3) for dj in range(-2, 3) for di in range(-2, 3) if dk * dk + dj * dj + di * di <= 6]
# in-plane taps of the kernel's S9 (m2 <= 2) and S12 (m2 in {4, 5}) sums, in the kernel's loop order (dj outer, di inner)
_PLANE = [(dj, di, dj * dj + di * di) for dj in range(-2, 3) for di in range(-2, 3) if dj * dj + di * di <= 6]

# the kernel's weight table: W.w[m] = (float)exp(-(double)m) (r2s_dev_rbf)
W32 = np.array([np.float32(np.exp(-float(m))) for m in range(8)], np.float32)

MUTATIONS = ("seam_x", "row_y", "chunk_plane", "pad_column", "stale_u")


# ---- input processing -------------------------------------------------------------------------------------------------------------------
def process(sdf):
    """k_to_f32 + k_replace_far: round to Float32, then replace every value that is isapprox(|v|, 1f10) (default rtol sqrt(eps(Float32)),
    evaluated in Float32 as the kernel does) by sign(v) times the largest finite |v| (|v| < 1e9)."""
    s = np.asarray(sdf, np.float64).astype(np.float32)
    a = np.abs(s)
    fin = a < np.float32(1e9)
    if not fin.any():
        raise ValueError("the SDF holds no finite value")
    maxv = a[fin].max()
    big, rt = np.float32(1e10), np.float32(np.sqrt(np.float32(EPS32)))
    far = np.abs(a - big) <= rt * np.maximum(a, big)
    return np.where(far, np.sign(s) * maxv, s).astype(np.float32)


# ---- geometry of the kernel launch (r2s_dev_rbf) ------------------------------------------------------------------------------------------
def z_chunks(nz):
    """Even z-chunks of the mat-vec launch: nchunk = max(1, (nz + 32) / 64) chunks of zc = cdiv(nz, nchunk) planes.  Returns the chunk
    boundaries strictly inside the grid."""
    nchunk = max(1, (nz + 32) // 64)
    zc = -(-nz // nchunk)
    return list(range(zc, nz, zc))


def row_pitch(nx):
    return (nx + 3) & ~3


# ---- K in float64 -------------------------------------------------------------------------------------------------------------------------
def _padded(u, P=2, dtype=np.float64):
    nz, ny, nx = u.shape
    p = np.zeros((nz + 2 * P, ny + 2 * P, nx + 2 * P), dtype)
    p[P:P + nz, P:P + ny, P:P + nx] = u
    return p


def K64(u):
    """sum over the 81 offsets of exp(-m) u[. + d], zero outside the grid, in float64.  The taps of equal in-plane distance are added
    first and weighted once, then the planes are combined -- exactly K u in exact arithmetic, float64 round-off otherwise."""
    u = np.asarray(u, np.float64)
    nz, ny, nx = u.shape
    p = _padded(u)
    groups = {}
    for dj, di, m2 in _PLANE:
        sl = p[:, 2 + dj:2 + dj + ny, 2 + di:2 + di + nx]
        if m2 in groups:
            groups[m2] += sl
        else:
            groups[m2] = sl.copy()
    s9 = groups[0] + np.exp(-1.0) * groups[1] + np.exp(-2.0) * groups[2]
    s21 = s9 + np.exp(-4.0) * groups[4] + np.exp(-5.0) * groups[5]
    out = s21[2:2 + nz] + np.exp(-1.0) * (s21[1:1 + nz] + s21[3:3 + nz])
    out += np.exp(-4.0) * (s9[0:nz] + s9[4:4 + nz])
    return out


def K64_literal(u):
    """The same operator written tap by tap: sum over OFFSETS of exp(-m) u[. + d] (for the host test that pins K64)."""
    u = np.asarray(u, np.float64)
    nz, ny, nx = u.shape
    p = _padded(u)
    out = np.zeros_like(u)
    for dk, dj, di in OFFSETS:
        out += np.exp(-float(dk * dk + dj * dj + di * di)) * p[2 + dk:2 + dk + nz, 2 + dj:2 + dj + ny, 2 + di:2 + di + nx]
    return out


# ---- CG in float64 ------------------------------------------------------------------------------------------------------------------------
def cg64(s, iters=None, reltol=CG_RELTOL):
    """IterativeSolvers.cg(K, s) in float64: x0 = 0, u = r + beta u, c = K u, alpha = rho / (u . c), x += alpha u, r -= alpha c, stop when
    |r| <= reltol |r0| or after maxiter = n iterations.  With `iters`, exactly that many iterations are run instead (the stopping test is
    not applied).  Returns (x, k, hist): the iterate, the iteration count and the residual norms |r_0| .. |r_k|."""
    s = np.asarray(s, np.float64)
    x = np.zeros_like(s); r = s.copy(); u = np.zeros_like(s)
    res = float(np.sqrt(np.vdot(r, r))); prev = 1.0
    tol = reltol * res
    hist = [res]
    k, maxiter = 0, s.size
    while (k < iters) if iters is not None else (k < maxiter and res > tol):
        beta = res * res / (prev * prev)
        u *= beta; u += r
        c = K64(u)
        uc = float(np.vdot(u, c))
        if uc == 0.0:      # r = 0: x is the exact solution (only with `iters` beyond convergence on tiny grids)
            break
        alpha = res * res / uc
        x += alpha * u
        r -= alpha * c
        prev, res = res, float(np.sqrt(np.vdot(r, r)))
        hist.append(res)
        k += 1
    return x, k, np.array(hist)


# ---- CG in Float32 (drift model of the kernels) ---------------------------------------------------------------------------------------------
def _fma(a, b, c, fused):
    """a * b + c in Float32: rounded once (fused, as fmaf: the float64 product of two floats is exact, the float64 sum is rounded to Float32
    -- a double rounding, which differs from fmaf in rare ties only) or product and sum rounded separately (numpy's float32)."""
    if fused:
        return (np.float64(a) * np.asarray(b, np.float64) + np.asarray(c, np.float64)).astype(np.float32)
    return np.float32(a) * b + c


def matvec32(u, mutate=None, fused=False):
    """K u in Float32 as k_stencil81_tma forms it: per input plane the in-plane sums S9 (m2 <= 2) and S12 (m2 in {4, 5}), S21 = S9 + S12,
    and per output plane 0 + e^-4 S9[k-2] + e^-1 S21[k-1] + S21[k] + e^-1 S21[k+1] + e^-4 S9[k+2] in input-plane order, with the
    factorised weights w[m2] w[dz^2] (r2s_rbf.cu, plane marching).  `fused` selects one rounding per multiply-add (the kernel's fmaf) or
    two.  `mutate` injects one of the defects of MUTATIONS that live in the mat-vec (see cg32)."""
    u = np.asarray(u, np.float32)
    nz, ny, nx = u.shape
    p = _padded(u, dtype=np.float32)
    s9 = np.zeros((nz + 4, ny, nx), np.float32); s12 = np.zeros_like(s9)
    for dj, di, m2 in _PLANE:
        v = p[:, 2 + dj:2 + dj + ny, 2 + di:2 + di + nx]
        if m2 <= 2:
            s9 = _fma(W32[m2], v, s9, fused)
        else:
            s12 = _fma(W32[m2], v, s12, fused)
    s21 = s9 + s12
    e1, e4 = W32[1], W32[4]
    out = _fma(e4, s9[0:nz], np.zeros((nz, ny, nx), np.float32), fused)
    out = _fma(e1, s21[1:1 + nz], out, fused)
    out = out + s21[2:2 + nz]
    out = _fma(e1, s21[3:3 + nz], out, fused)
    out = _fma(e4, s9[4:4 + nz], out, fused)
    if mutate == "seam_x":           # (a) outputs in columns x = 29, 30 (mod 32), at the seam of the shifted CTA columns, lose the tap (0, 0, +1)
        x = np.arange(nx)
        sel = (x % 32 == 29) | (x % 32 == 30)
        out[:, :, sel] -= e1 * p[2:2 + nz, 2:2 + ny, 3:3 + nx][:, :, sel]
    elif mutate == "row_y":          # (b) outputs in rows y = 15 (mod 16), the last row of a CTA, lose the tap (0, +1, 0)
        y = np.arange(ny)
        sel = y % 16 == 15
        out[:, sel, :] -= e1 * p[2:2 + nz, 3:3 + ny, 2:2 + nx][:, sel, :]
    elif mutate == "chunk_plane":    # (c) the CTAs below a z-chunk boundary b see input plane b as zero
        for b in z_chunks(nz):
            out[b - 1] -= e1 * s21[2 + b]
            out[b - 2] -= e4 * s9[2 + b]
    return out


def mutation_site_exists(shape, mutate):
    """Does the defect change K on a grid of shape (nz, ny, nx)?  (a) needs an output column x = 29, 30 (mod 32) with x + 1 inside the grid,
    (b) a row y = 15 (mod 16) with y + 1 inside, (c) a z-chunk boundary, (d) pad columns (nx not a multiple of 4); (e) always exists."""
    nz, ny, nx = shape
    if mutate == "seam_x":
        return any(x % 32 in (29, 30) and x + 1 < nx for x in range(nx))
    if mutate == "row_y":
        return any(y % 16 == 15 and y + 1 < ny for y in range(ny))
    if mutate == "chunk_plane":
        return len(z_chunks(nz)) > 0
    if mutate == "pad_column":
        return row_pitch(nx) > nx
    return True


def cg32(s, iters=None, mutate=None, fused=False, maxiter=None):
    """The CG of r2s_dev_rbf in Float32: the vectors and the mat-vec (matvec32) in Float32, the dot products u.c and r.r summed in float64
    (the kernels convert each product to double), and the scalar steps as k_cg_init / k_cg_update / cg_close_iteration do them:
    res = float(sqrt(rr)), tol = sqrtf(eps) res0, alpha = res * res / float(uc), beta = res * res / (prev * prev), all in Float32; like
    the kernels, the run stops when the residual is not below 1e8 |r0| (divergence guard).  `iters` as in cg64; `maxiter` (default n) caps
    the run without `iters`; `fused` as in matvec32, for the mat-vec and the vector updates.  `mutate` injects one defect (MUTATIONS):
      seam_x, row_y, chunk_plane -- in the mat-vec (matvec32);
      pad_column -- the mat-vec also stores its outputs in the pad columns x = nx .. px - 1 of c (K u of the zero-extended u there), so
                    the element-wise update leaves -alpha c in r's pad and |r|^2 sums it;
      stale_u    -- the stencil input plane nz / 2 is u_old instead of u_new = r + beta u_old, and so is the u_new written back.
    Returns (x, k, hist) like cg64."""
    s = np.asarray(s, np.float32)
    nz, ny, nx = s.shape
    px = row_pitch(nx)
    x = np.zeros_like(s); r = s.copy(); u = np.zeros_like(s)
    rpad = np.zeros((nz, ny, px - nx), np.float32)
    dot = lambda a, b: float(np.vdot(a.astype(np.float64), b.astype(np.float64)))
    res = np.float32(np.sqrt(dot(r, r))); prev = np.float32(1.0)
    tol = np.float32(np.sqrt(np.float32(EPS32))) * res
    hist = [float(res)]
    k, beta = 0, np.float32(0.0)
    maxiter = s.size if maxiter is None else maxiter
    with np.errstate(over="ignore", invalid="ignore"):
        while (k < iters) if iters is not None else (k < maxiter and not res <= tol):
            unew = _fma(beta, u, r, fused)
            if mutate == "stale_u":
                unew[nz // 2] = u[nz // 2]
            u = unew
            c = matvec32(u, mutate, fused)
            alpha = np.float32(res * res) / np.float32(dot(u, c))
            x = _fma(alpha, u, x, fused)
            r = _fma(-alpha, c, r, fused)
            rr = dot(r, r)
            if mutate == "pad_column" and px > nx:
                up = np.zeros((nz, ny, px), np.float32); up[:, :, :nx] = u
                rpad = _fma(-alpha, matvec32(up, None, fused)[:, :, nx:], rpad, fused)
                rr += dot(rpad, rpad)
            prev, res = res, np.float32(np.sqrt(rr))
            beta = np.float32(res * res) / np.float32(prev * prev)
            hist.append(float(res))
            k += 1
            if iters is None and not res < np.float32(1e8) * np.float32(hist[0]):
                break
    return x, k, np.array(hist)


def drift(s, k, x64=None):
    """max|cg32 - cg64| / max|cg64| after k iterations, for both roundings of the multiply-adds (separate, fused): how far two Float32
    runs of the same loop land from the float64 iterate.  Returns ((drift_separate, drift_fused), x64)."""
    if x64 is None:
        x64 = cg64(s, iters=k)[0]
    m = float(np.abs(x64).max())
    return tuple(float(np.abs(cg32(s, iters=k, fused=f)[0] - x64).max()) / m for f in (False, True)), x64


def tau(s, k, x64=None):
    """Tolerance of a Float32 solve of K w = s after k iterations, relative to max|cg64(s, iters=k)|: 8 times the larger of the two drifts
    of the Float32 model (`drift`).  Returns (tau, x64)."""
    d, x64 = drift(s, k, x64)
    return 8.0 * max(d), x64


# ---- coarse LSF -----------------------------------------------------------------------------------------------------------------------
# Bound on |L_kernel - K w| per point, as a multiple of 2^-24 sum_t exp(-m_t) |w_t| (the 81 taps of the point).  In k_stencil81_tma a
# tap's term passes through at most
#   12 roundings in the in-plane fma chain (S12 has 12 taps, S9 9), 1 in S21 = S9 + S12, 5 in the output plane's chain over the five input
#   planes (the products w[dz^2] S inside fmaf are not rounded separately)                                                    -> 18,
# and its weight is w[m2] w[dz^2] with each factor (float)exp(-m) within 2^-24 relative of exp(-m): the factorised weight differs from
# exp(-m) by at most (1 + 2^-24)^2 - 1 < 2.0001 2^-24 relative (about 1.2e-7; r2s_rbf.cu quotes 4e-7 for the whole mat-vec)  -> 2.0001.
# So every term is within (1 + 2^-24)^20.0001 - 1 < 20.001 2^-24 of its exact value.  The constant used is the cruder (81 + 4) for the
# rounding of a sum of 81 terms with 4 more operations, plus 3 for the weights: 88, more than four times the derived 20.001.  A sum of
# terms each within gamma |t| is within gamma sum |t|: delta = 88 2^-24 sum |phi w|.  Values outside the grid are zero-filled by TMA and
# contribute exactly zero.
LSF_ROUNDOFF = 81 + 4 + 3


def lsf_bounds(w):
    """(L, delta): L = K w in float64 and delta = LSF_ROUNDOFF 2^-24 sum_t exp(-m_t) |w_t| per point, with |L_kernel - L| <= delta."""
    w = np.asarray(w, np.float64)
    return K64(w), LSF_ROUNDOFF * U * (1.0 + 1e-6) * K64(np.abs(w))


def round_down32(v):
    """Largest float32 <= v (elementwise)."""
    f = np.asarray(v, np.float64).astype(np.float32)
    return np.where(f.astype(np.float64) > v, np.nextafter(f, np.float32(-np.inf)), f).astype(np.float32)


def round_up32(v):
    """Smallest float32 >= v (elementwise)."""
    f = np.asarray(v, np.float64).astype(np.float32)
    return np.where(f.astype(np.float64) < v, np.nextafter(f, np.float32(np.inf)), f).astype(np.float32)


def coarse_edge(amin, amax, nx):
    """The coarse cell edge of the threshold search as r2s_dev_rbf measures it: norm(grid[2,1,1] - grid[1,1,1]) with Float32 range()
    coordinates (RBFs4Smoothing.jl:41-43)."""
    a, b = np.float32(amin), np.float32(amax)
    x1 = np.float32(float(a) + 1.0 * ((float(b) - float(a)) / float(nx - 1))) if nx > 1 else a
    if nx == 2:
        x1 = b
    ex = np.float32(x1 - a)
    return np.float32(np.sqrt(np.float32(ex * ex)))


# ---- the cases of the tests ----------------------------------------------------------------------------------------------------------------
# Points per axis (nx, ny, nz), chosen so that every edge of the mat-vec launch is hit at least once (r2s_dev_rbf, plane marching):
#   x: 2, 3, 5 (fewer columns than the 40-float TMA box), 30 (nx + 2 = 32: one CTA column), 31 (a second column with one output), 33, 62,
#      63, 94 -- and every x but 2 leaves pad columns (row pitch a multiple of 4);
#   y: 2, 15, 16, 17 (one row in a second CTA row), 33;
#   z: 2, 3, 4, 5 (fewer planes than the 4 TMA stages), 65 (one chunk), 96 and 97 (two chunks of 48 / 49), 160 (three chunks).
SHAPES = [(2, 2, 2), (2, 33, 97), (3, 16, 160), (5, 33, 65), (30, 17, 96), (31, 15, 65), (33, 2, 97), (62, 16, 5), (63, 33, 4),
          (94, 17, 3), (94, 15, 2)]
# 16 x 32 CTA columns x rows of one chunk: 512 partial sums, more than the 256 strided slots of cta_sum_last
LARGE = (510, 500, 6)
FIELDS = ("smooth", "sparse", "checker")


def fields_of(shape):
    """The fields run on a shape: all three, and the checkerboard alone (the most iterations) on the large case."""
    return ("checker",) if shape == LARGE else FIELDS


def make_field(kind, shape, seed=0):
    """The SDF handed to the smoothing, float64 [k, j, i] on `shape` = (nx, ny, nz) points:
      smooth  -- signed distance to a sphere (off centre, both signs on every grid) inside a band of 3.5 cells, +-1e10 outside (far values, as evalDistances leaves them);
      sparse  -- the field of test_volume_exact.fine_eval_input: 15 % of the points nonzero, 1 % far values;
      checker -- +-1 checkerboard with a small ramp: high frequencies are the smallest eigenvalues of K, so CG needs the most iterations."""
    nx, ny, nz = shape
    k, j, i = np.meshgrid(np.arange(nz), np.arange(ny), np.arange(nx), indexing="ij")
    if kind == "smooth":
        c = [0.25 * (n - 1) for n in (nz, ny, nx)]
        d = 0.35 * (max(shape) - 1) + 0.3 - np.sqrt((k - c[0]) ** 2 + (j - c[1]) ** 2 + (i - c[2]) ** 2)
        return np.where(np.abs(d) > 3.5, np.sign(d) * 1e10, d)
    if kind == "sparse":
        from test_volume_exact import fine_eval_input
        f = fine_eval_input(shape, np.random.default_rng(seed + nx * 10007 + ny * 101 + nz))
        f[0, 0, 0] = -0.75      # at least one finite nonzero value, and both signs, also on the smallest grids
        return f
    return np.where((i + j + k) % 2 == 0, 1.0, -1.0) + 0.05 * (i / nx + 2.0 * j / ny + 3.0 * k / nz)
