"""CPU tests of the host reference of the smoothing solve (tests/cg_ref.py) that tests/test_cg_float64.py compares the GPU with:
K64 is the reference's kernel matrix, cg64 solves it like an independent sparse solver, the Float32 drift model stays small at every case
of the GPU test (so its tolerance is not vacuous), and every defect the kernel could have moves the solution by far more than that
tolerance (so the GPU comparison would catch it)."""
import functools

import numpy as np
import pytest
import scipy.sparse
import scipy.sparse.linalg

import cg_ref as ref


def assembled_K(shape):
    """The reference's kernel matrix restated literally (RBFs4Smoothing.jl:142-176 with sigma = cell = 1 and cut 1e-3): entry
    exp(-|p_a - p_b|^2) for every pair of grid points with |p_a - p_b| <= sqrt(ln 1000), from all pairwise distances."""
    nz, ny, nx = shape
    k, j, i = np.meshgrid(np.arange(nz), np.arange(ny), np.arange(nx), indexing="ij")
    P = np.stack([i.ravel(), j.ravel(), k.ravel()], 1).astype(np.float64)
    d2 = ((P[:, None, :] - P[None, :, :]) ** 2).sum(-1)
    a, b = np.nonzero(np.sqrt(d2) <= np.sqrt(-np.log(1e-3)))
    return scipy.sparse.csr_matrix((np.exp(-d2[a, b]), (a, b)), shape=(len(P), len(P)))


@pytest.mark.parametrize("shape", [(2, 2, 2), (3, 5, 4), (9, 9, 9), (4, 9, 7)])
def test_K64_is_the_kernel_matrix(shape):
    A = assembled_K(shape)
    n = A.shape[0]
    assert (A != A.T).nnz == 0 and A.diagonal().min() == 1.0
    E = np.eye(n).reshape((n,) + shape)
    lit = np.stack([ref.K64_literal(e).ravel() for e in E], 1)
    assert np.array_equal(lit, A.toarray())      # tap by tap: the same entries, bit for bit
    assert len(ref.OFFSETS) == 81 and (A.getnnz(axis=1).max() == 81 if min(shape) >= 5 else True)
    u = np.random.default_rng(n).standard_normal(shape)
    assert np.abs(ref.K64(u).ravel() - A @ u.ravel()).max() <= 1e-14 * np.abs(A).sum(1).max() * np.abs(u).max()


@pytest.mark.parametrize("shape", [(2, 2, 2), (3, 5, 4), (9, 9, 9), (4, 9, 7)])
@pytest.mark.parametrize("kind", ref.FIELDS)
def test_cg64_matches_spsolve(shape, kind):
    A = assembled_K(shape)
    s = ref.process(ref.make_field(kind, shape[::-1])).astype(np.float64)
    x_direct = scipy.sparse.linalg.spsolve(A.tocsc(), s.ravel())
    x, k, hist = ref.cg64(s, reltol=1e-13)
    assert hist[-1] <= 1e-13 * hist[0] and k < s.size
    assert np.abs(x.ravel() - x_direct).max() <= 1e-10 * np.abs(x_direct).max()
    # with the library's tolerance: the iterate stops once, and running on with iters= reproduces the history
    x1, k1, h1 = ref.cg64(s)
    x2, k2, h2 = ref.cg64(s, iters=k1)
    assert k2 == k1 and np.array_equal(x1, x2) and np.array_equal(h1, h2)
    assert h1[-1] <= ref.CG_RELTOL * h1[0] < h1[-2]


def test_process_replaces_far_values():
    """The kernel's isapprox rule equals the simple one the sampler tests assert (|v| < 1e9 finite, the rest replaced) on their inputs."""
    for shape in [(5, 4, 3), (34, 8, 18)]:
        f = ref.make_field("sparse", shape)
        s = f.astype(np.float32)
        fin = np.abs(s) < 1e9
        assert np.array_equal(ref.process(f), np.where(fin, s, np.sign(s) * np.abs(s[fin]).max()).astype(np.float32))
    # isapprox(|v|, 1f10) with rtol sqrt(eps(Float32)) = 3.45e-4: 1e10 (1 + 1e-3) stays, 1e10 (1 + 3e-4) is replaced
    got = ref.process(np.array([1e10 * (1 + 1e-3), 1e10 * (1 + 3e-4), -1e10, 3.0, -0.5]))
    assert got.tolist() == [np.float32(1e10 * (1 + 1e-3)), 3.0, -3.0, 3.0, -0.5]


@functools.lru_cache(maxsize=None)
def solved(shape, kind):
    """(s, k64, hist64, x64 at k64, drifts) for one case of the GPU test"""
    s = ref.process(ref.make_field(kind, shape))
    x64, k64, hist = ref.cg64(s)
    d, _ = ref.drift(s, k64, x64)
    return s, k64, hist, x64, d


@pytest.mark.parametrize("shape", ref.SHAPES + [ref.LARGE], ids=lambda s: "x".join(map(str, s)))
def test_drift_model_is_small(shape):
    """cg32 (both roundings) stays within 1e-4 relative of cg64 at cg64's iteration count, and its converged solution has a true residual
    below 1.05 times the tolerance -- the bound test_cg_float64 holds the GPU to."""
    for kind in ref.fields_of(shape):
        s, k64, hist, x64, d = solved(shape, kind)
        print("%s %-7s k64 %3d  drift %.2e / %.2e  tau %.2e" % (shape, kind, k64, d[0], d[1], 8 * max(d)))
        assert max(d) <= 1e-4, (kind, d)
        assert 0 < k64 < s.size
        if shape != ref.LARGE:
            for fused in (False, True):
                x, k, h = ref.cg32(s, fused=fused)
                assert abs(k - k64) <= 1, (kind, fused, k, k64)
                r = np.linalg.norm(s.astype(np.float64) - ref.K64(x))
                assert r <= 1.05 * ref.CG_RELTOL * np.linalg.norm(s.astype(np.float64)), (kind, fused)


@pytest.mark.parametrize("shape", ref.SHAPES, ids=lambda s: "x".join(map(str, s)))
def test_every_mutation_is_caught(shape):
    """Each defect of cg32's `mutate` whose site exists on the grid fails the GPU comparison of test_cg_float64 (tau = 8 max drift):
    run to its own stopping point k' (capped at 4 k64 + 8 iterations), the mutated iterate is at least 10 tau away from cg64(s, iters=k')
    somewhere.  Two kinds of run pass this assertion, and the log tells them apart:
      * runs that stop within an iteration of cg64's count -- chunk_plane on every field, seam_x and row_y on the smooth field -- show
        weight sensitivity proper: their iterate is at least 3.5e4 tau from the float64 iterate at the same count;
      * the other runs (stale_u and pad_column everywhere, seam_x and row_y on the sparse and checkerboard fields) stop at the cap or far
        from cg64's count: the defect keeps CG from converging.  Their ratios of 1e6 to 1e14 tau measure that, not the weights; the
        iteration-count assertion of test_cg_float64 catches these defects on its own.  (A nonzero pad column of r inflates |r|^2, which
        also enters beta and so every later search direction.)"""
    nsites = 0
    for kind in ref.FIELDS:
        s, k64, hist, x64, d = solved(shape, kind)
        tau = 8 * max(d)
        for mut in ref.MUTATIONS:
            if not ref.mutation_site_exists(s.shape, mut):
                continue
            nsites += 1
            xm, km, _ = ref.cg32(s, mutate=mut, maxiter=4 * k64 + 8)
            xk = x64 if km == k64 else ref.cg64(s, iters=km)[0]
            with np.errstate(over="ignore", invalid="ignore"):
                err = np.abs(xm.astype(np.float64) - xk).max() / np.abs(xk).max()
            err = np.inf if not np.isfinite(err) else err
            kind_of_run = "same count" if abs(km - k64) <= 1 else ("capped" if km == 4 * k64 + 8 else "count differs")
            print("%s %-7s %-11s iterations %3d (cg64 %3d, %s)  %.3g tau" % (shape, kind, mut, km, k64, kind_of_run, err / tau))
            assert err >= 10 * tau, (kind, mut, err, tau, km, k64)
    assert nsites >= 2 * len(ref.FIELDS)
