"""The numpy reference of the hole filling (scan3d_voxel_surface_fill_holes, scan3d_mesh_fill_holes_dev), as
include/scan3d.h states it: hole edges, regular vertices, the holes with their smallest vertex first, and Liepa's
minimum-weight triangulation per hole, vectorised over each diagonal of the DP.  CPU checks: the reference against a
plain per-loop Python walk and DP on random meshes, and the properties the rules promise (closed results, the area of
a planar patch, holes that stay open and why, a second fill that adds nothing).  tests/test_fill_math_host.py compares
the shared header with the triangle terms and the per-hole DP below; tests/test_gpu_fill.py compares the GPU with
fill_ref."""
import math

import numpy as np
import pytest

from test_smooth_ref import grid_mesh, icosphere, odd_mesh

F32, F64 = np.float32, np.float64
NETS_MAX_EDGES, MAX_EDGES = 22, 1024


# ---- the rules, vectorised -----------------------------------------------------------------------------------------
def triangle_ref(a, b, c):
    """unit normals u [..., 3] (0 where undefined), has [...], area [...] of the float triangles (a, b, c)"""
    a, b, c = (np.asarray(x, F32).astype(F64) for x in (a, b, c))
    d1, d2 = b - a, c - a
    n = np.stack([d1[..., 1] * d2[..., 2] - d1[..., 2] * d2[..., 1],
                  d1[..., 2] * d2[..., 0] - d1[..., 0] * d2[..., 2],
                  d1[..., 0] * d2[..., 1] - d1[..., 1] * d2[..., 0]], -1)
    l2 = (n[..., 0] * n[..., 0] + n[..., 1] * n[..., 1]) + n[..., 2] * n[..., 2]
    ln = np.sqrt(l2)
    has = l2 > 0
    with np.errstate(invalid="ignore", divide="ignore"):
        u = np.where(has[..., None], n / ln[..., None], 0.0)
    return u, has, ln * 0.5


def cos_ref(u1, h1, u2, h2):
    c = (u1[..., 0] * u2[..., 0] + u1[..., 1] * u2[..., 1]) + u1[..., 2] * u2[..., 2]
    return np.where(h1 & h2, c, -1.0)


def polygon_ref(p, rim_u, rim_has, exists):
    """the DP of one hole: p [n][3] float32, rim normals [n][3] / [n], exists [n][n] bool.  Returns (faces [n - 2][3]
    of local ids in preorder or None when unfillable, cmin, area, k [n][n])."""
    n = len(p)
    cmin, area = np.zeros((n, n)), np.zeros((n, n))
    U, H, K = np.zeros((n, n, 3)), np.zeros((n, n), bool), np.full((n, n), -1, np.int64)
    t = np.arange(n - 1)
    cmin[t, t + 1], U[t, t + 1], H[t, t + 1], K[t, t + 1] = np.inf, rim_u[:-1], rim_has[:-1], 0
    for d in range(2, n):
        i = np.arange(n - d)
        j = i + d
        I, J = i[:, None], j[:, None]
        k = I + np.arange(1, d)[None, :]
        Ib, Jb = np.broadcast_to(I, k.shape), np.broadcast_to(J, k.shape)
        u, has, a = triangle_ref(p[Ib], p[k], p[Jb])
        c = np.minimum(cos_ref(u, has, U[Ib, k], H[Ib, k]), cos_ref(u, has, U[k, Jb], H[k, Jb]))
        closing = (i == 0) & (j == n - 1)
        c[closing] = np.minimum(c[closing], cos_ref(u[closing], has[closing], rim_u[n - 1], rim_has[n - 1]))
        cm = np.minimum(np.minimum(cmin[Ib, k], cmin[k, Jb]), c)
        ar = (area[Ib, k] + area[k, Jb]) + a
        feas = (K[Ib, k] >= 0) & (K[k, Jb] >= 0) & ~(exists[i, j] & ~closing)[:, None]
        best_c = np.where(feas, cm, -np.inf).max(1)
        t1 = feas & (cm == best_c[:, None])
        best_a = np.where(t1, ar, np.inf).min(1)
        t2 = t1 & (ar == best_a[:, None])
        ok = t2.any(1)
        col = np.argmax(t2, 1)
        r = np.arange(len(i))
        cmin[i, j] = np.where(ok, cm[r, col], 0.0)
        area[i, j] = np.where(ok, ar[r, col], 0.0)
        U[i, j] = np.where((ok & has[r, col])[:, None], u[r, col], 0.0)
        H[i, j] = ok & has[r, col]
        K[i, j] = np.where(ok, k[r, col], -1)
    if K[0, n - 1] < 0:
        return None, cmin, area, K
    faces, stack = [], [(0, n - 1)]
    while stack:
        i, j = stack.pop()
        if j - i < 2:
            continue
        k = K[i, j]
        faces.append((i, k, j))
        stack += [(k, j), (i, k)]
    return np.array(faces, np.int64), cmin, area, K


def hole_edges_ref(faces):
    """(tails, heads, rim faces) of the hole edges, in no particular order"""
    f = np.asarray(faces, np.int64).reshape(-1, 3)
    a, c = f.reshape(-1), f[:, [1, 2, 0]].reshape(-1)
    fid = np.repeat(np.arange(len(f)), 3)
    keep = a != c
    a, c, fid = a[keep], c[keep], fid[keep]
    key = np.minimum(a, c) << 32 | np.maximum(a, c)
    _, inv, cnt = np.unique(key, return_inverse=True, return_counts=True)
    b = cnt[inv.reshape(-1)] == 1
    return c[b], a[b], fid[b], np.unique(key)


def holes_ref(n, faces, max_edges):
    """(holes: list of vertex loops, v_0 the smallest, in ascending v_0; tails, heads, rims, edge keys)"""
    tails, heads, rims, keys = hole_edges_ref(faces)
    out_n, in_n = np.bincount(tails, minlength=n), np.bincount(heads, minlength=n)
    regular = (out_n == 1) & (in_n == 1)
    nxt = np.full(n, -1, np.int64)
    rim = np.full(n, -1, np.int64)
    nxt[tails], rim[tails] = heads, rims
    seen = np.zeros(n, bool)
    holes = []
    for v in np.flatnonzero(regular):
        if seen[v]:
            continue
        loop, u, ok = [v], nxt[v], True
        seen[v] = True
        while u != v:
            if not regular[u] or len(loop) == max_edges:
                ok = False
                break
            seen[u] = True
            loop.append(u)
            u = nxt[u]
        if ok:
            holes.append(np.array(loop, np.int64))
    return holes, rim, tails, keys


def polygon_faces_ref(p, rims, exists):
    """the faces of one hole (local ids) or None, by polygon_ref; rims [n][3][3] are the rim faces' corners"""
    ru, rh, _ = triangle_ref(rims[:, 0], rims[:, 1], rims[:, 2])
    return polygon_ref(p, ru, rh, exists)[0]


def fill_ref(xyz, faces, max_edges, polygon=polygon_faces_ref):
    """(added faces int32 [m][3], info dict with the fields of scan3d_fill_result); polygon(p, rims, exists) gives
    one hole's faces"""
    xyz = np.asarray(xyz, F32).reshape(-1, 3)
    f = np.asarray(faces, np.int64).reshape(-1, 3)
    holes, rim, tails, keys = holes_ref(len(xyz), f, max_edges)
    added, filled = [], 0
    for loop in holes:
        n = len(loop)
        rims = xyz[f[rim[loop]]]
        lo, hi = np.minimum.outer(loop, loop), np.maximum.outer(loop, loop)
        q = lo << 32 | hi
        exists = keys[np.minimum(np.searchsorted(keys, q), len(keys) - 1)] == q   # keys are sorted and unique
        tri = polygon(xyz[loop], rims, exists)
        if tri is not None:
            added.append(loop[tri])
            filled += 1
    add = np.concatenate(added).astype(np.int32) if added else np.zeros((0, 3), np.int32)
    # a filled hole of n edges adds n - 2 faces and closes its n hole edges
    info = dict(vertices=len(xyz), faces=len(f) + len(add), boundary_edges=len(tails), holes=len(holes),
                filled=filled, faces_added=len(add), open_edges=len(tails) - (len(add) + 2 * filled))
    return add, info


# ---- an independent plain-Python loop, for small meshes ------------------------------------------------------------
def _tri_loop(a, b, c):
    a, b, c = ([float(x) for x in q] for q in (a, b, c))
    d1 = [b[k] - a[k] for k in range(3)]
    d2 = [c[k] - a[k] for k in range(3)]
    n = [d1[1] * d2[2] - d1[2] * d2[1], d1[2] * d2[0] - d1[0] * d2[2], d1[0] * d2[1] - d1[1] * d2[0]]
    l2 = (n[0] * n[0] + n[1] * n[1]) + n[2] * n[2]
    ln = math.sqrt(l2)
    return ([x / ln for x in n] if l2 > 0 else None), ln * 0.5


def _cos_loop(u, w):
    if u is None or w is None:
        return -1.0
    return (u[0] * w[0] + u[1] * w[1]) + u[2] * w[2]


def fill_loop(xyz, faces, max_edges):
    faces = [tuple(int(v) for v in t) for t in np.asarray(faces).reshape(-1, 3)]
    count, side_face = {}, {}
    for fi, t in enumerate(faces):
        for a, c in ((t[0], t[1]), (t[1], t[2]), (t[2], t[0])):
            if a != c:
                e = (min(a, c), max(a, c))
                count[e] = count.get(e, 0) + 1
                side_face[e] = (a, c, fi)
    out_e, in_n = {}, {}
    for e, m in count.items():
        if m == 1:
            a, c, fi = side_face[e]
            out_e.setdefault(c, []).append((a, fi))
            in_n[a] = in_n.get(a, 0) + 1
    reg = {v for v in out_e if len(out_e[v]) == 1 and in_n.get(v, 0) == 1}
    added, holes, filled = [], 0, 0
    for v0 in sorted(reg):
        loop, u = [v0], out_e[v0][0][0]
        while u != v0 and u in reg and u > v0 and len(loop) < max_edges:
            loop.append(u)
            u = out_e[u][0][0]
        if u != v0:
            continue
        holes += 1
        n = len(loop)
        P = [xyz[v] for v in loop]
        cell = {}
        for t in range(n):
            r = faces[out_e[loop[t]][0][1]]
            cell[(t, t + 1)] = (math.inf, 0.0, _tri_loop(xyz[r[0]], xyz[r[1]], xyz[r[2]])[0], 0)
        close = cell.pop((n - 1, n))[2]
        for d in range(2, n):
            for i in range(n - d):
                j = i + d
                closing = (i, j) == (0, n - 1)
                best = None
                if closing or (min(loop[i], loop[j]), max(loop[i], loop[j])) not in count:
                    for k in range(i + 1, j):
                        L, R = cell[(i, k)], cell[(k, j)]
                        if L is None or R is None:
                            continue
                        u, a = _tri_loop(P[i], P[k], P[j])
                        c = min(_cos_loop(u, L[2]), _cos_loop(u, R[2]))
                        if closing:
                            c = min(c, _cos_loop(u, close))
                        w = (min(L[0], R[0], c), (L[1] + R[1]) + a)
                        if best is None or w[0] > best[0] or (w[0] == best[0] and w[1] < best[1]):
                            best = (w[0], w[1], u, k)
                cell[(i, j)] = best
        if cell[(0, n - 1)] is None:
            continue
        filled += 1
        stack = [(0, n - 1)]
        while stack:
            i, j = stack.pop()
            if j - i >= 2:
                k = cell[(i, j)][3]
                added.append((loop[i], loop[k], loop[j]))
                stack += [(k, j), (i, k)]
    return np.array(added, np.int32).reshape(-1, 3), holes, filled


# ---- meshes --------------------------------------------------------------------------------------------------------
def punched_sphere(level, holes, seed, r=2.0, sigma=0.0):
    """an icosphere with the faces around `holes` random vertices removed (their umbrella: a hole of their link)"""
    u, faces = icosphere(level)
    rng = np.random.default_rng(seed)
    xyz = (u * (r + sigma * rng.normal(size=(len(u), 1)))).astype(F32)
    centres = rng.choice(len(u), holes, replace=False)
    keep = ~np.isin(faces, centres).any(1)
    return xyz, faces[keep].astype(np.int32)


def cube_without_a_face():
    v = np.array([[x, y, z] for x in (0, 1) for y in (0, 1) for z in (0, 1)], F32)
    # outward quads (counter-clockwise seen from outside), the top (z = 1) left out
    quads = [(0, 1, 3, 2), (4, 6, 7, 5), (0, 4, 5, 1), (2, 3, 7, 6), (0, 2, 6, 4)]
    f = [t for a, b, c, d in quads for t in ((a, b, c), (a, c, d))]
    return v, np.array(f, np.int32)


def annulus(n_in, r_in=1.0, r_out=2.0):
    """a flat ring (normal +z) around a regular n_in-gon hole; its outer loop has 2 n_in edges"""
    th_in = 2 * np.pi * np.arange(n_in) / n_in
    th_out = 2 * np.pi * np.arange(2 * n_in) / (2 * n_in)
    xyz = np.concatenate([np.stack([r_in * np.cos(th_in), r_in * np.sin(th_in), 0 * th_in], 1),
                          np.stack([r_out * np.cos(th_out), r_out * np.sin(th_out), 0 * th_out], 1)]).astype(F32)
    f = []
    for i in range(n_in):
        a, a1 = i, (i + 1) % n_in
        o0, o1, o2 = n_in + 2 * i, n_in + 2 * i + 1, n_in + (2 * i + 2) % (2 * n_in)
        f += [(a, o0, o1), (a, o1, a1), (a1, o1, o2)]
    return xyz, np.array(f, np.int32)


def edge_counts(faces):
    f = np.asarray(faces, np.int64).reshape(-1, 3)
    a, c = f.reshape(-1), f[:, [1, 2, 0]].reshape(-1)
    k = a != c
    und = np.unique(np.minimum(a[k], c[k]) << 32 | np.maximum(a[k], c[k]), return_counts=True)[1]
    directed = np.unique(a[k] << 32 | c[k], return_counts=True)[1]
    return und, directed


def assert_closed(xyz, faces):
    und, directed = edge_counts(faces)
    assert (und == 2).all() and (directed == 1).all()
    used = len(np.unique(faces))
    assert used - len(und) + len(faces) == 2


def _check_against_loop(xyz, faces, max_edges):
    add, info = fill_ref(xyz, faces, max_edges)
    want, holes, filled = fill_loop(xyz, faces, max_edges)
    assert np.array_equal(add, want)
    assert info["holes"] == holes and info["filled"] == filled
    return add, info


# ---- tests ---------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("seed", range(4))
def test_reference_matches_the_loop_on_punched_spheres(seed):
    xyz, faces = punched_sphere(2, 6, seed, sigma=0.05 * seed)
    for m in (3, 6, 22):
        add, info = _check_against_loop(xyz, faces, m)
    assert info["filled"] >= 1


def test_reference_matches_the_loop_on_odd_and_random_meshes():
    rng = np.random.default_rng(11)
    for _ in range(3):
        xyz, _, faces = odd_mesh(rng, 40, 60)
        _check_against_loop(xyz, faces, 22)
    xyz, faces = grid_mesh(7, 5, 0.5, rng.normal(size=(5, 7)) * 0.1)
    add, info = _check_against_loop(xyz, faces, 24)          # the grid's rim: one loop of 20 edges
    assert info["holes"] == 1 and info["filled"] == 1 and len(add) == 18
    add, info = _check_against_loop(xyz, faces, 19)
    assert info["holes"] == 0 and info["open_edges"] == 20


def test_cube_and_punched_sphere_become_closed():
    xyz, faces = cube_without_a_face()
    add, info = _check_against_loop(xyz, faces, 4)
    assert info == dict(vertices=8, faces=12, boundary_edges=4, holes=1, filled=1, faces_added=2, open_edges=0)
    assert_closed(xyz, np.concatenate([faces, add]))
    # the new faces point up, out of the cube
    u = triangle_ref(xyz[add[:, 0]], xyz[add[:, 1]], xyz[add[:, 2]])[0]
    assert np.allclose(u, [0, 0, 1])
    xyz, faces = punched_sphere(3, 12, 5, sigma=0.02)
    add, info = fill_ref(xyz, faces, 22)
    assert info["holes"] == 12 and info["filled"] == 12 and info["open_edges"] == 0
    assert_closed(xyz, np.concatenate([faces, add]))


def test_planar_convex_patch_has_the_polygon_area():
    for n in (5, 12, 40):
        xyz, faces = annulus(n)
        add, info = fill_ref(xyz, faces, n)
        assert info["holes"] == 1 and info["filled"] == 1 and len(add) == n - 2
        assert info["open_edges"] == 2 * n                    # the outer loop is longer than max_edges
        u, has, a = triangle_ref(xyz[add[:, 0]], xyz[add[:, 1]], xyz[add[:, 2]])
        p = xyz[:n].astype(F64)
        shoelace = 0.5 * np.sum(p[:, 0] * np.roll(p[:, 1], -1) - np.roll(p[:, 0], -1) * p[:, 1])
        assert abs(a.sum() - shoelace) <= 1e-12 * shoelace * n
        assert has.all() and np.array_equal(u, np.tile([0.0, 0.0, 1.0], (n - 2, 1)))   # winding of the rim


def test_a_hole_whose_triangulations_all_need_an_existing_edge_stays_open():
    # two faces of a tetrahedron leave the loop 0 1 2 3, whose diagonal {0, 2} they hold; a closed tetrahedron on
    # (1, 3, 4, 5) holds the other diagonal
    xyz = np.array([[0, 0, 0], [1, 0, 0], [1, 1, 0.2], [0, 1, 0], [0.5, 0.5, 2], [0.5, -1, 1]], F32)
    faces = np.array([[0, 1, 2], [0, 2, 3], [1, 3, 4], [1, 4, 5], [1, 5, 3], [3, 5, 4]], np.int32)
    add, info = _check_against_loop(xyz, faces, 22)
    assert info == dict(vertices=6, faces=6, boundary_edges=4, holes=1, filled=0, faces_added=0, open_edges=4)
    # without the second diagonal the loop 0 3 2 1 closes the first tetrahedron
    add, info = _check_against_loop(xyz, faces[:2], 22)
    assert info["filled"] == 1 and sorted(map(tuple, add)) == [(0, 3, 1), (3, 2, 1)]


def test_shared_vertices_and_long_loops_stay_open_and_are_counted():
    # a bow tie: two triangles sharing vertex 0 (not regular); a lone triangle (its back face closes it); an annulus
    bow = np.array([[0, 1, 2], [0, 3, 4], [5, 6, 7]], np.int32)
    ring_xyz, ring = annulus(8)
    xyz = np.concatenate([np.random.default_rng(0).normal(size=(8, 3)).astype(F32), ring_xyz])
    faces = np.concatenate([bow, ring + 8])
    add, info = _check_against_loop(xyz, faces, 8)
    assert info == dict(vertices=32, faces=len(faces) + 1 + 6, boundary_edges=9 + 8 + 16, holes=2, filled=2,
                        faces_added=7, open_edges=6 + 16)
    assert [tuple(t) for t in add[:1]] == [(5, 7, 6)]


def test_second_fill_adds_nothing_and_empty_mesh():
    xyz, faces = punched_sphere(2, 5, 1)
    xyz2, faces2 = annulus(30)
    xyz = np.concatenate([xyz, xyz2])
    faces = np.concatenate([faces, faces2 + len(xyz) - len(xyz2)])
    add, info = fill_ref(xyz, faces, 22)
    assert info["filled"] >= 3 and info["open_edges"] >= 90
    again, info2 = fill_ref(xyz, np.concatenate([faces, add]), 22)
    assert len(again) == 0 and info2["boundary_edges"] == info2["open_edges"] == info["open_edges"]
    assert info2["holes"] == info["holes"] - info["filled"] and info2["filled"] == 0
    add, info = fill_ref(np.zeros((0, 3), F32), np.zeros((0, 3), np.int32), 22)
    assert len(add) == 0 and info == dict(vertices=0, faces=0, boundary_edges=0, holes=0, filled=0, faces_added=0,
                                          open_edges=0)
