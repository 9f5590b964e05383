"""CPU tests of the isosurface stage's case table (rho2sdf.jl_b200/csrc/r2s_mc.cuh, compiled for the host) and of the whole-grid host
reference the GPU tests compare against (tests/host/mc_host.cpp): the table is checked exhaustively over the 256 cases, the reference
on analytic fields (closedness, orientation, topology, volume convergence) and against a literal restatement of the output contract."""
import itertools
import math

import numpy as np
import pytest

import isosurface_ref as ref

CORNER = np.array([[c & 1, c >> 1 & 1, c >> 2 & 1] for c in range(8)], np.float64)


def edge_mid(e):
    c, a = ref.edges()[e]
    p = CORNER[c].copy()
    p[a] += 0.5
    return p


# ---- the table ------------------------------------------------------------------------------------------------------------------------
def test_table_sizes_and_edges():
    E = ref.edges()
    assert sorted((c, c | (1 << a)) for c, a in E) == [(a, b) for a in range(8) for b in range(a + 1, 8) if bin(a ^ b).count("1") == 1]
    tab = ref.table()
    assert max(len(t) for t in tab) == 5 and len(tab[0]) == 0 and len(tab[255]) == 0
    for case, tris in enumerate(tab):
        for t in tris:
            assert len(set(t)) == 3
            for e in t:      # every vertex of the case sits on an edge whose corners lie on different sides
                c, a = E[e]
                assert (case >> c & 1) != (case >> (c | 1 << a) & 1)


def test_table_is_closed_within_the_cube_and_matches_the_face_rule():
    E = ref.edges()
    faces = [ref.face(f) for f in range(6)]
    for case, tris in enumerate(ref.table()):
        directed = {}
        for t in tris:
            for q in range(3):
                d = (t[q], t[(q + 1) % 3])
                directed[d] = directed.get(d, 0) + 1
        assert all(v == 1 for v in directed.values()), case
        # an edge between two triangles is used once in each direction; what is left over is the loop boundary = the face segments
        boundary = {d for d in directed if (d[1], d[0]) not in directed}
        want = set()
        for f in range(6):
            segs = ref.face_segments(case, f)
            on_face = {e for e in range(12) if E[e][0] in faces[f] and (E[e][0] | 1 << E[e][1]) in faces[f]}
            for a, b in segs:
                assert a in on_face and b in on_face
            want |= set(segs)
        assert boundary == want, case


def test_no_triangle_edge_runs_inside_a_cube_face_unless_it_is_a_face_segment():
    """A chord between two edges of one face would lie in that face; if the neighbouring cell drew it too, four triangles would share
    the edge.  Every triangle edge of the table is either a face-rule segment or crosses the cube's interior."""
    E = ref.edges()
    faces = [ref.face(f) for f in range(6)]
    on = lambda e: {f for f in range(6) if E[e][0] in faces[f] and (E[e][0] | 1 << E[e][1]) in faces[f]}
    for case, tris in enumerate(ref.table()):
        segs = {s for f in range(6) for s in ref.face_segments(case, f)}
        for t in tris:
            for q in range(3):
                a, b = t[q], t[(q + 1) % 3]
                assert (a, b) in segs or (b, a) in segs or not (on(a) & on(b)), (case, t)


def test_face_rule_separates_diagonal_corners_and_depends_on_the_face_only():
    faces = [ref.face(f) for f in range(6)]
    for f in range(6):
        cyc = faces[f]
        for case in range(256):
            segs = ref.face_segments(case, f)
            ins = [case >> c & 1 for c in cyc]
            runs = sum(1 for q in range(4) if ins[q] and not ins[q - 1])
            assert len(segs) == runs
            if ins in ([1, 0, 1, 0], [0, 1, 0, 1]):
                assert len(segs) == 2      # ambiguous face: the two inside corners are separated
            # the same four corners with any other corners off the face give the same segments
            other = [c for c in range(8) if c not in cyc]
            for bits in itertools.product((0, 1), repeat=4):
                c2 = sum(ins[q] << cyc[q] for q in range(4)) + sum(b << c for b, c in zip(bits, other))
                assert ref.face_segments(c2, f) == segs


def test_single_and_three_corner_normals_point_away_from_the_inside_corners():
    for case, tris in enumerate(ref.table()):
        ins = [c for c in range(8) if case >> c & 1]
        if len(ins) not in (1, 3):
            continue
        for t in tris:
            p = [edge_mid(e) for e in t]
            n = np.cross(p[1] - p[0], p[2] - p[1])
            ctr = sum(p) / 3
            near = min(ins, key=lambda c: np.linalg.norm(CORNER[c] - ctr))
            assert n @ (ctr - CORNER[near]) > 0, (case, t)


# ---- the whole-grid reference -----------------------------------------------------------------------------------------------------------
def contract_restatement(f, origin, spacing, iso):
    """The output contract written out point by point (slow; small grids)."""
    nz, ny, nx = f.shape
    ins = f >= np.float32(iso)
    vid, V = {}, []
    for k in range(nz):
        for j in range(ny):
            for i in range(nx):
                for a, (di, dj, dk) in enumerate(((1, 0, 0), (0, 1, 0), (0, 0, 1))):
                    if i + di < nx and j + dj < ny and k + dk < nz and ins[k, j, i] != ins[k + dk, j + dj, i + di]:
                        va, vb = float(f[k, j, i]), float(f[k + dk, j + dj, i + di])
                        t = (float(np.float32(iso)) - va) / (vb - va)
                        p = [i, j, k]
                        V.append([np.float32(origin[d] + spacing[d] * (p[d] + t if d == a else p[d])) for d in range(3)])
                        vid[(i, j, k, a)] = len(V) - 1
    E, tab, T = ref.edges(), ref.table(), []
    for k in range(nz - 1):
        for j in range(ny - 1):
            for i in range(nx - 1):
                case = sum(int(ins[k + (c >> 2 & 1), j + (c >> 1 & 1), i + (c & 1)]) << c for c in range(8))
                for t in tab[case]:
                    T.append([vid[(i + (E[e][0] & 1), j + (E[e][0] >> 1 & 1), k + (E[e][0] >> 2 & 1), E[e][1])] for e in t])
    return np.array(V, np.float32).reshape(-1, 3), np.array(T, np.int32).reshape(-1, 3)


@pytest.mark.parametrize("shape,iso", [((2, 2, 2), 0.0), ((3, 5, 7), 0.37), ((6, 4, 9), -1.5), ((5, 7, 3), 0.0)])
def test_reference_equals_the_contract_restatement(shape, iso):
    rng = np.random.default_rng(sum(shape))
    f = rng.uniform(-3, 3, shape).astype(np.float32)
    f.ravel()[::7] = np.float32(iso)          # corners exactly on iso
    origin, spacing = (0.5, -1.25, 3.0), (0.1, 0.2, 0.3)
    V, T = ref.reference(f, origin, spacing, iso)
    V2, T2 = contract_restatement(f, origin, spacing, iso)
    assert np.array_equal(V, V2) and np.array_equal(T, T2)


def grid_field(n, fn, h=1.0):
    c = (n - 1) / 2.0
    z, y, x = np.meshgrid(*(np.arange(n) - c,) * 3, indexing="ij")
    return fn(x * h, y * h, z * h).astype(np.float32)


def sphere(R):
    return lambda x, y, z: R - np.sqrt(x * x + y * y + z * z)


def torus(R, r):
    return lambda x, y, z: r - np.sqrt((np.sqrt(x * x + y * y) - R) ** 2 + z * z)


def gyroid(x, y, z, w=0.45):
    return np.sin(w * x) * np.cos(w * y) + np.sin(w * y) * np.cos(w * z) + np.sin(w * z) * np.cos(w * x)


def closed(T):
    return len(ref.unpaired_edges(T)) == 0


def test_sphere_and_torus_are_closed_with_their_euler_characteristic():
    V, T = ref.reference(grid_field(33, sphere(11.3)))
    assert closed(T) and ref.euler_characteristic(T) == 2 and ref.components(T) == 1
    V, T = ref.reference(grid_field(41, torus(11.0, 4.2)))
    assert closed(T) and ref.euler_characteristic(T) == 0 and ref.components(T) == 1


def test_gyroid_and_noise_with_a_negative_border_are_closed():
    n = 40
    f = grid_field(n, lambda x, y, z: gyroid(x, y, z) - 0.2)
    f[[0, -1], :, :] = f[:, [0, -1], :] = f[:, :, [0, -1]] = -1
    V, T = ref.reference(f, iso=0.0)
    assert len(T) > 1000 and closed(T)
    rng = np.random.default_rng(1)
    f = rng.uniform(-1, 1, (23, 17, 29)).astype(np.float32)
    f[[0, -1], :, :] = f[:, [0, -1], :] = f[:, :, [0, -1]] = -1
    for iso in (0.0, 0.37, -0.5):
        V, T = ref.reference(f, iso=iso)
        assert len(T) > 1000 and closed(T)


@pytest.mark.parametrize("pts", [[(1, 1, 1), (2, 2, 1)], [(1, 1, 1), (2, 2, 2)]], ids=["face_diagonal", "body_diagonal"])
def test_diagonal_inside_points_give_two_components(pts):
    f = -np.ones((4, 4, 4), np.float32)
    for i, j, k in pts:
        f[k, j, i] = 1
    V, T = ref.reference(f)
    assert closed(T) and ref.components(T) == 2 and len(T) == 16


def test_field_touching_the_border_leaves_only_boundary_edges_unpaired():
    origin, spacing = (1.0, 2.0, 3.0), (0.5, 0.5, 0.5)
    f = grid_field(24, sphere(14.0))      # the ball is cut by all six faces of the grid
    V, T = ref.reference(f, origin, spacing)
    bad = ref.unpaired_edges(T)
    assert len(bad) > 0 and ref.on_boundary_face(V, T, bad, origin, spacing, f.shape).all()


def test_divergence_volume_converges_at_second_order():
    errs = []
    for R in (10, 20, 40):
        f = grid_field(2 * R + 7, sphere(R + 0.2))      # off the lattice, so no corner sits exactly on the sphere
        V, T = ref.reference(f)
        assert closed(T)
        exact = 4.0 / 3.0 * math.pi * (R + 0.2) ** 3
        errs.append(abs(ref.divergence_volume(V, T) - exact) / exact)
    assert errs[2] < 1e-3
    for a, b in zip(errs, errs[1:]):
        assert a / b > 3.0, errs      # second order: the error falls about fourfold per halving of h
