"""The numpy reference of the surface smoothing (scan3d_voxel_surface_smooth, scan3d_mesh_smooth_dev), restated from
the rules in include/scan3d.h: np.unique edges, np.add.at int64 sums.  The tests here check it against a plain
per-vertex Python loop and check the properties the rules promise: quantisation only below 2^(E - 17), held and
isolated vertices untouched, a flat grid stays flat, lambda|mu does not shrink a noisy sphere while mu = 0 does, and
degenerate and non-manifold faces follow the rules.  tests/test_gpu_smooth.py compares the GPU with smooth_ref."""
import math

import numpy as np
import pytest

F32, F64 = np.float32, np.float64
P = 40
Q_LIMIT = 1 << 42
DEGREE_LIMIT = 1 << 20
NQ = 2.0 ** 24                                           # the merge's fixed point of unit normals


class SmoothError(Exception):
    """code: "arg" (SCAN3D_ERR_ARG) or "config" (SCAN3D_ERR_CONFIG)"""

    def __init__(self, code):
        super().__init__(code)
        self.code = code


def exponent_ref(xyz):
    """E: 2^E is the smallest power of two above every |coordinate|"""
    field = (np.ascontiguousarray(xyz, F32).view(np.uint32) >> 23) & 0xff
    return int(field.max(initial=0)) - 126


def quantise_ref(x, E):
    return np.rint(np.asarray(x, F32).astype(F64) * math.ldexp(1.0, P - E)).astype(np.int64)


def dequantise_ref(q, E):
    return (np.asarray(q, np.int64).astype(F64) * math.ldexp(1.0, E - P)).astype(F32)


def update_ref(q, s, d, k):
    """one axis of one pass, elementwise: Q + rint(k ((double)S / d - (double)Q))"""
    m = np.asarray(s, np.int64).astype(F64) / np.asarray(d).astype(F64)
    return np.asarray(q, np.int64) + np.rint(F64(k) * (m - np.asarray(q, np.int64).astype(F64))).astype(np.int64)


def normal_fixed_ref(n):
    """the merge's fixed point of float normals [k][3]: clamp to [-1, 1], rint(v 2^24); a non-finite row gives 0"""
    n = np.asarray(n, F32)
    m = np.rint(np.clip(n, -1, 1).astype(F64) * NQ).astype(np.int64)
    m[~np.isfinite(n).all(1)] = 0
    return m


def face_normals_ref(p, tri):
    """(ok [f], fixed-point unit normals [f][3]) of faces tri over float positions p"""
    x = np.asarray(p, F32).astype(F64)
    a, b, c = x[tri[:, 0]], x[tri[:, 1]], x[tri[:, 2]]
    d1, d2 = b - a, c - a
    n = np.stack([d1[:, 1] * d2[:, 2] - d1[:, 2] * d2[:, 1], d1[:, 2] * d2[:, 0] - d1[:, 0] * d2[:, 2],
                  d1[:, 0] * d2[:, 1] - d1[:, 1] * d2[:, 0]], 1)
    l2 = (n[:, 0] * n[:, 0] + n[:, 1] * n[:, 1]) + n[:, 2] * n[:, 2]
    ok = (l2 > 0) & np.isfinite(l2)
    with np.errstate(invalid="ignore", divide="ignore"):
        u = (n / np.sqrt(l2)[:, None]).astype(F32)
    m = normal_fixed_ref(np.where(ok[:, None], u, 0))
    return ok, m


def normal_out_ref(s):
    """the merge's normalisation of int64 sums [k][3] (rows of zeros give zeros)"""
    X = np.asarray(s, np.int64).astype(F64)
    l2 = (X[:, 0] * X[:, 0] + X[:, 1] * X[:, 1]) + X[:, 2] * X[:, 2]
    with np.errstate(invalid="ignore", divide="ignore"):
        out = (X / np.sqrt(l2)[:, None]).astype(F32)
    out[l2 == 0] = 0
    return out


def displacement_ref(a, b):
    d = np.asarray(b, F32).astype(F64) - np.asarray(a, F32).astype(F64)
    return np.sqrt((d[:, 0] * d[:, 0] + d[:, 1] * d[:, 1]) + d[:, 2] * d[:, 2])


def edges_ref(faces, n):
    """(undirected edges [e][2] with min first, their side counts, degree [n], held [n])"""
    f = np.asarray(faces, np.int64).reshape(-1, 3)
    sides = np.concatenate([f[:, [0, 1]], f[:, [1, 2]], f[:, [2, 0]]])
    sides = sides[sides[:, 0] != sides[:, 1]]
    und, cnt = np.unique(np.sort(sides, 1), axis=0, return_counts=True)
    und = und.reshape(-1, 2)
    deg = np.bincount(und.ravel(), minlength=n).astype(np.int64)
    held = np.zeros(n, bool)
    held[und[cnt != 2].ravel()] = True
    return und, cnt, deg, held


def passes_of(iterations, mu):
    return iterations * (1 if F32(mu) == 0 else 2)


def smooth_ref(xyz, normals, faces, iterations=10, lam=0.5, mu=-0.53):
    """(xyz float32 [v][3], normals float32 [v][3] or None, result dict) after the call; raises SmoothError"""
    xyz = np.ascontiguousarray(xyz, F32).reshape(-1, 3)
    faces = np.ascontiguousarray(faces, np.int32).reshape(-1, 3)
    n = len(xyz)
    if not np.isfinite(xyz).all() or ((faces < 0) | (faces >= n)).any():
        raise SmoothError("arg")
    und, _, deg, held = edges_ref(faces, n)
    free = (deg > 0) & ~held
    if (deg[free] > DEGREE_LIMIT).any():
        raise SmoothError("config")
    E = exponent_ref(xyz)
    q = quantise_ref(xyz, E)
    k_lam, k_mu = F64(F32(lam)), F64(F32(mu))
    passes = passes_of(iterations, mu)
    for p in range(passes):
        k = k_lam if k_mu == 0 or p % 2 == 0 else k_mu
        s = np.zeros((n, 3), np.int64)
        np.add.at(s, und[:, 0], q[und[:, 1]])
        np.add.at(s, und[:, 1], q[und[:, 0]])
        q2 = q.copy()
        q2[free] = update_ref(q[free], s[free], deg[free, None], k)
        if (np.abs(q2[free]) > Q_LIMIT).any():
            raise SmoothError("config")
        q = q2
    out = xyz.copy()
    out[free] = dequantise_ref(q[free], E)
    if not np.isfinite(out).all():
        raise SmoothError("config")
    nrm = None
    if normals is not None:
        nrm = np.ascontiguousarray(normals, F32).reshape(-1, 3).copy()
        tri = faces[(faces[:, 0] != faces[:, 1]) & (faces[:, 1] != faces[:, 2]) & (faces[:, 0] != faces[:, 2])]
        ok, m = face_normals_ref(out, tri)
        sums = np.zeros((n, 3), np.int64)
        for c in range(3):
            np.add.at(sums, tri[ok, c], m[ok])
        has = (sums != 0).any(1)
        nrm[has] = normal_out_ref(sums[has])
    move = float(displacement_ref(xyz[free], out[free]).max(initial=0.0))
    return out, nrm, dict(vertices=n, faces=len(faces), held_vertices=int(held.sum()),
                          isolated_vertices=int((deg == 0).sum()), passes=passes, max_displacement=move)


# ---- a plain per-vertex restatement: Python ints and floats (IEEE doubles; round() ties to even) ----------------------
def smooth_loop(xyz, normals, faces, iterations, lam, mu):
    xyz = np.asarray(xyz, F32)
    n = len(xyz)
    nb = [set() for _ in range(n)]
    count = {}
    for f in np.asarray(faces).tolist():
        for a, b in ((f[0], f[1]), (f[1], f[2]), (f[2], f[0])):
            if a != b:
                nb[a].add(b)
                nb[b].add(a)
                e = (min(a, b), max(a, b))
                count[e] = count.get(e, 0) + 1
    held = [False] * n
    for (a, b), c in count.items():
        if c != 2:
            held[a] = held[b] = True
    free = [len(nb[v]) > 0 and not held[v] for v in range(n)]
    E = max([(int(x) >> 23) & 0xff for x in xyz.view(np.uint32).ravel()] + [0]) - 126
    q = [[round(float(x) * 2.0 ** (P - E)) for x in row] for row in xyz.tolist()]
    ks = [float(F32(lam)), float(F32(mu))]
    for p in range(passes_of(iterations, mu)):
        k = ks[0] if ks[1] == 0 or p % 2 == 0 else ks[1]
        q2 = [list(r) for r in q]
        for v in range(n):
            if free[v]:
                for a in range(3):
                    m = float(sum(q[w][a] for w in nb[v])) / float(len(nb[v]))
                    q2[v][a] = q[v][a] + round(k * (m - float(q[v][a])))
        q = q2
    out = xyz.copy()
    for v in range(n):
        if free[v]:
            out[v] = [F32(float(c) * 2.0 ** (E - P)) for c in q[v]]
    nrm = np.asarray(normals, F32).copy()
    sums = [[0, 0, 0] for _ in range(n)]
    for f in np.asarray(faces).tolist():
        if len(set(f)) < 3:
            continue
        a, b, c = (out[i].astype(F64).tolist() for i in f)
        d1 = [b[i] - a[i] for i in range(3)]
        d2 = [c[i] - a[i] for i in range(3)]
        nn = [d1[1] * d2[2] - d1[2] * d2[1], d1[2] * d2[0] - d1[0] * d2[2], d1[0] * d2[1] - d1[1] * d2[0]]
        l2 = (nn[0] * nn[0] + nn[1] * nn[1]) + nn[2] * nn[2]
        if not (l2 > 0 and math.isfinite(l2)):
            continue
        u = [float(F32(x / math.sqrt(l2))) for x in nn]
        m = [round(min(max(x, -1.0), 1.0) * NQ) for x in u]
        for i in f:
            for a_ in range(3):
                sums[i][a_] += m[a_]
    for v in range(n):
        if any(sums[v]):
            X = [float(x) for x in sums[v]]
            l = math.sqrt((X[0] * X[0] + X[1] * X[1]) + X[2] * X[2])
            nrm[v] = [F32(x / l) for x in X]
    return out, nrm


def _same(a, b):
    assert a.shape == b.shape and a.dtype == b.dtype
    assert np.array_equal(a.view(np.uint8), b.view(np.uint8))


# ---- meshes --------------------------------------------------------------------------------------------------------
def grid_mesh(nx, ny, h=1.0, z=None):
    """a flat nx x ny grid of two triangles per cell; z [ny][nx] heights or None"""
    y, x = np.mgrid[0:ny, 0:nx]
    zz = np.zeros((ny, nx)) if z is None else z
    xyz = np.stack([x * h, y * h, zz], -1).reshape(-1, 3).astype(F32)
    g = np.arange(nx * ny, dtype=np.int32).reshape(ny, nx)
    a, b, c, d = g[:-1, :-1].ravel(), g[:-1, 1:].ravel(), g[1:, :-1].ravel(), g[1:, 1:].ravel()
    faces = np.concatenate([np.stack([a, b, d], 1), np.stack([a, d, c], 1)]).astype(np.int32)
    return xyz, faces


def icosphere(level):
    """a closed unit icosphere (vertices, faces outward)"""
    t = (1 + 5 ** 0.5) / 2
    v = [[-1, t, 0], [1, t, 0], [-1, -t, 0], [1, -t, 0], [0, -1, t], [0, 1, t], [0, -1, -t], [0, 1, -t],
         [t, 0, -1], [t, 0, 1], [-t, 0, -1], [-t, 0, 1]]
    f = [[0, 11, 5], [0, 5, 1], [0, 1, 7], [0, 7, 10], [0, 10, 11], [1, 5, 9], [5, 11, 4], [11, 10, 2], [10, 7, 6],
         [7, 1, 8], [3, 9, 4], [3, 4, 2], [3, 2, 6], [3, 6, 8], [3, 8, 9], [4, 9, 5], [2, 4, 11], [6, 2, 10],
         [8, 6, 7], [9, 8, 1]]
    v = [np.array(p, F64) / np.linalg.norm(p) for p in v]
    for _ in range(level):
        mid = {}

        def m(a, b):
            key = (min(a, b), max(a, b))
            if key not in mid:
                p = v[a] + v[b]
                v.append(p / np.linalg.norm(p))
                mid[key] = len(v) - 1
            return mid[key]
        f = [g for a, b, c in f for g in ([a, m(a, b), m(c, a)], [b, m(b, c), m(a, b)], [c, m(c, a), m(b, c)],
                                          [m(a, b), m(b, c), m(c, a)])]
    return np.array(v), np.array(f, np.int32)


def noisy_sphere(level, r, centre, sigma, seed):
    u, faces = icosphere(level)
    rng = np.random.default_rng(seed)
    xyz = (np.asarray(centre) + u * (r + sigma * rng.normal(size=(len(u), 1)))).astype(F32)
    return xyz, u.astype(F32), faces


def odd_mesh(rng, n=60, f=150):
    """random faces with degenerate ones, repeated sides (non-manifold edges) and isolated vertices"""
    used = rng.permutation(n)[:n - 7]
    faces = rng.choice(used, (f, 3)).astype(np.int32)
    faces[::9, 1] = faces[::9, 0]                        # (a, a, b)
    faces[::13] = faces[::13, [0, 0, 0]]                 # (a, a, a)
    faces = np.concatenate([faces, faces[:10], faces[5:8, ::-1]])   # repeated sides: counts of 3 and 4
    xyz = rng.normal(size=(n, 3)).astype(F32)
    nrm = rng.normal(size=(n, 3)).astype(F32)
    return xyz, nrm, faces


# ---- the reference against the loop -------------------------------------------------------------------------------
@pytest.mark.parametrize("iterations,lam,mu", [(0, 0.5, -0.53), (1, 0.5, -0.53), (3, 0.5, -0.53), (4, 0.7, 0.0),
                                               (2, 1.0, -1.0)])
def test_reference_matches_the_loop(iterations, lam, mu):
    rng = np.random.default_rng(iterations)
    for xyz, nrm, faces in (odd_mesh(rng), noisy_sphere(1, 2.0, (0.3, -0.2, 0.1), 0.05, 3)):
        got_x, got_n, info = smooth_ref(xyz, nrm, faces, iterations, lam, mu)
        want_x, want_n = smooth_loop(xyz, nrm, faces, iterations, lam, mu)
        _same(got_x, want_x)
        _same(got_n, want_n)
        assert info["passes"] == passes_of(iterations, mu)


def test_zero_iterations_quantise_only_below_2_to_the_E_minus_17():
    rng = np.random.default_rng(4)
    xyz, faces = grid_mesh(30, 30)
    xyz[:, 2] = rng.normal(size=len(xyz)) * np.exp2(rng.integers(-30, 3, len(xyz)))
    xyz[::7, 2] = -0.0
    xyz[::11, 2] = np.float32(1e-42)                     # subnormal
    E = exponent_ref(xyz)
    out, _, info = smooth_ref(xyz, None, faces, 0)
    assert info["passes"] == 0 and info["max_displacement"] >= 0
    exact = (np.abs(xyz) >= 2.0 ** (E - 17)) | (xyz == 0)
    assert (~exact).any()
    assert np.array_equal(out[exact], xyz[exact])
    assert np.array_equal(out.view(np.uint32)[exact & (xyz != 0)], xyz.view(np.uint32)[exact & (xyz != 0)])
    # below that the error is at most half a step of 2^(E - 40)
    assert (np.abs(out.astype(F64) - xyz.astype(F64)) <= 2.0 ** (E - 41)).all()


def test_held_and_isolated_vertices_keep_their_bytes():
    rng = np.random.default_rng(5)
    xyz, nrm, faces = odd_mesh(rng, 200, 400)
    und, cnt, deg, held = edges_ref(faces, len(xyz))
    assert held.any() and (deg == 0).any() and (cnt >= 3).any()
    out, _, info = smooth_ref(xyz, nrm, faces, 10)
    fixed = held | (deg == 0)
    assert np.array_equal(out[fixed].view(np.uint32), xyz[fixed].view(np.uint32))
    assert info["held_vertices"] == held.sum() and info["isolated_vertices"] == (deg == 0).sum()
    # an open grid: the border is held, the inside moves
    gx, gf = grid_mesh(12, 9, z=rng.normal(size=(9, 12)))
    out, _, info = smooth_ref(gx, None, gf, 5)
    border = np.zeros((9, 12), bool)
    border[[0, -1], :] = border[:, [0, -1]] = True
    assert info["held_vertices"] == border.sum()
    assert np.array_equal(out[border.ravel()], gx[border.ravel()])
    assert not np.array_equal(out[~border.ravel()], gx[~border.ravel()])


def test_flat_grid_stays_flat():
    rng = np.random.default_rng(6)
    xyz, faces = grid_mesh(40, 30, h=0.25)
    xyz[:, :2] += (0.05 * rng.normal(size=(len(xyz), 2))).astype(F32)
    nrm = np.zeros_like(xyz)
    out, n2, info = smooth_ref(xyz, nrm, faces, 20)
    assert (out[:, 2] == 0).all() and info["max_displacement"] > 0
    assert np.array_equal(np.abs(n2), np.tile(np.array([0, 0, 1], F32), (len(xyz), 1)))


def _radii(xyz, centre):
    return np.linalg.norm(xyz.astype(F64) - centre, axis=1)


def test_taubin_does_not_shrink_a_noisy_sphere_but_laplacian_does():
    centre, r = np.array([10.0, -4.0, 2.5]), 2.0
    xyz, u, faces = noisy_sphere(4, r, centre, 0.02, 7)
    rms0 = float(np.sqrt(np.mean((_radii(xyz, centre) - r) ** 2)))
    out, nrm, info = smooth_ref(xyz, u, faces, 10)
    assert info["held_vertices"] == 0 and info["isolated_vertices"] == 0 and info["passes"] == 20
    rad = _radii(out, centre)
    rms = float(np.sqrt(np.mean((rad - rad.mean()) ** 2)))
    # Taubin's pass band (k_PB = 1 / lambda + 1 / mu = 0.11) keeps the low frequencies of white noise: 10 iterations
    # remove 2.6x of it here (3.7x at 50), while plain Laplacian smoothing at 20 passes loses 1.5 % of the radius
    assert rms < rms0 / 2.4
    assert abs(rad.mean() - r) < 0.01 * r
    lap, _, _ = smooth_ref(xyz, None, faces, 20, 0.5, 0.0)
    shrink_lap = r - _radii(lap, centre).mean()
    assert shrink_lap > 5 * abs(rad.mean() - r) and shrink_lap > 0.005 * r
    print(f"sphere r {r}, sigma 0.02, {len(xyz)} vertices: radial RMS {rms0:.4g} -> {rms:.4g}; mean radius "
          f"{rad.mean():.5f} (lambda|mu) vs {_radii(lap, centre).mean():.5f} (mu = 0, 20 passes)")
    # the recomputed normals are closer to radial than the noisy geometry's
    radial = (out.astype(F64) - centre) / rad[:, None]
    assert np.mean(np.sum(nrm * radial, 1)) > 0.999


def test_degenerate_and_non_manifold_faces():
    # a fan of three faces on the edge (0, 1) holds 0 and 1; (2, 2, 3) adds the edge {2, 3} with count 2 and no normal;
    # (4, 4, 4) adds nothing and leaves 4 isolated
    xyz = np.array([[0, 0, 0], [1, 0, 0], [0, 1, 0], [0, 0, 1], [5, 5, 5], [0.3, -1, 0.2]], F32)
    faces = np.array([[0, 1, 2], [1, 0, 3], [0, 1, 5], [2, 2, 3], [4, 4, 4]], np.int32)
    und, cnt, deg, held = edges_ref(faces, 6)
    counts = {tuple(e): c for e, c in zip(und.tolist(), cnt.tolist())}
    assert counts == {(0, 1): 3, (0, 2): 1, (1, 2): 1, (0, 3): 1, (1, 3): 1, (2, 3): 2, (0, 5): 1, (1, 5): 1}
    assert held.tolist() == [True, True, True, True, False, True]
    assert deg.tolist() == [4, 4, 3, 3, 0, 2]
    nrm = np.full((6, 3), 7, F32)
    out, n2, info = smooth_ref(xyz, nrm, faces, 3)
    assert np.array_equal(out, xyz) and info["held_vertices"] == 5 and info["isolated_vertices"] == 1
    assert np.array_equal(n2[4], nrm[4])                 # no face with three distinct vertices
    assert not np.array_equal(n2[0], nrm[0])
    # a closed tetrahedron with one extra degenerate face: (0, 0, 1) adds two sides on {0, 1}, which then has count 4
    tet = np.array([[1, 1, 1], [1, -1, -1], [-1, 1, -1], [-1, -1, 1]], F32)
    tf = np.array([[0, 1, 2], [0, 3, 1], [0, 2, 3], [1, 3, 2]], np.int32)
    out, _, info = smooth_ref(tet, None, tf, 1)
    assert info["held_vertices"] == 0 and not np.array_equal(out, tet)
    out, _, info = smooth_ref(tet, None, np.concatenate([tf, [[0, 0, 1]]]), 1)
    assert info["held_vertices"] == 2


def test_errors():
    xyz, faces = grid_mesh(5, 5)
    bad = xyz.copy()
    bad[3, 1] = np.nan
    for x, f in ((bad, faces), (xyz, np.concatenate([faces, [[0, 1, 25]]])), (xyz, np.concatenate([faces, [[-1, 1, 2]]]))):
        with pytest.raises(SmoothError) as e:
            smooth_ref(x, None, f, 1)
        assert e.value.code == "arg"
    # lambda = 1, mu = -1 multiplies the highest frequency of this mesh (eigenvalue 1.49 of the umbrella operator) by
    # |1 - 1.49^2| = 1.21 per iteration, until some |Q| passes 2^42
    xyz, _, faces = noisy_sphere(2, 1.9, (0, 0, 0), 0.4, 0)
    with pytest.raises(SmoothError) as e:
        smooth_ref(xyz, None, faces, 100, 1.0, -1.0)
    assert e.value.code == "config"
