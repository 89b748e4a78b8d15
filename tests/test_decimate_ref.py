"""CPU checks of the whole-surface simplification reference (scan3d_voxel_surface_decimate): decimate_ref below, a
vectorised numpy restatement of the rules in include/scan3d.h (np.unique on the cluster keys, first-index order), is
compared bit for bit with a plain per-face Python loop on small surface-nets meshes and small hand-made meshes.
tests/test_gpu_decimate.py holds the GPU to decimate_ref."""
import math

import numpy as np
import pytest

from test_surface_math_host import extract_ref, random_model, sphere_model

F32, F64 = np.float32, np.float64
Q = 2.0 ** 24
SCALE = 2.0 ** 40
DAMPING = 1e-3


def clusters_ref(xyz, H):
    """(cluster ordinal of each vertex, integer coordinates [c][3], position steps q [v][3], fractions f [v][3])"""
    t = np.asarray(xyz, F32).astype(F64) / H
    i = np.floor(t)
    f = t - i
    q = np.minimum(np.floor(f * Q), Q - 1).astype(np.uint64)
    if len(t) == 0:
        return np.zeros(0, np.int64), np.zeros((0, 3), np.int64), q, f
    uniq, first, inv = np.unique(i.astype(np.int64), axis=0, return_index=True, return_inverse=True)
    order = np.argsort(first)
    rank = np.empty_like(order)
    rank[order] = np.arange(order.size)
    return rank[inv.reshape(-1)], uniq[order], q, f


def face_planes_ref(xyz, faces, H):
    """(u [f][3], w [f], has a plane [f]) of each face"""
    p = np.asarray(xyz, F32).astype(F64)
    a, b, c = p[faces[:, 0]], p[faces[:, 1]], p[faces[:, 2]]
    d1, d2 = b - a, c - a
    n = np.stack([d1[:, 1] * d2[:, 2] - d1[:, 2] * d2[:, 1],
                  d1[:, 2] * d2[:, 0] - d1[:, 0] * d2[:, 2],
                  d1[:, 0] * d2[:, 1] - d1[:, 1] * d2[:, 0]], 1)
    l2 = (n[:, 0] * n[:, 0] + n[:, 1] * n[:, 1]) + n[:, 2] * n[:, 2]
    ok = l2 != 0
    with np.errstate(invalid="ignore", divide="ignore"):
        l = np.sqrt(l2)
        u = n / l[:, None]
        w = (l * 0.5) / (H * H)
    return u, w, ok


def corner_coeffs_ref(u, w, f):
    """int64 [n][10] of corners with unit normals u [n][3], weights w [n] and fractions f [n][3]"""
    e = (u[:, 0] * f[:, 0] + u[:, 1] * f[:, 1]) + u[:, 2] * f[:, 2]
    c = np.stack([u[:, 0] * u[:, 0], u[:, 0] * u[:, 1], u[:, 0] * u[:, 2], u[:, 1] * u[:, 1], u[:, 1] * u[:, 2],
                  u[:, 2] * u[:, 2], u[:, 0] * e, u[:, 1] * e, u[:, 2] * e, e * e], 1)
    return np.rint((w[:, None] * c) * SCALE).astype(np.int64)


def place_ref(qs, sq, n):
    """(y [c][3], status [c]: 0 solved, 1 trace 0, 2 fallback) from the quadric sums qs int64 [c][10], the position
    sums sq uint64 [c][3] and the counts n [c]"""
    a = qs[:, :9].astype(F64) * 2.0 ** -40
    ybar = sq.astype(F64) / (Q * n.astype(F64))[:, None]
    tr = (a[:, 0] + a[:, 3]) + a[:, 5]
    with np.errstate(all="ignore"):
        mu = DAMPING * (tr / 3.0)
        h = mu * 0.5
        D0 = a[:, 0] + mu
        L10, L20 = a[:, 1] / D0, a[:, 2] / D0
        D1 = (a[:, 3] + mu) - (L10 * L10) * D0
        L21 = (a[:, 4] - (L20 * L10) * D0) / D1
        D2 = ((a[:, 5] + mu) - (L20 * L20) * D0) - (L21 * L21) * D1
        z0 = a[:, 6] + mu * ybar[:, 0]
        z1 = (a[:, 7] + mu * ybar[:, 1]) - L10 * z0
        z2 = ((a[:, 8] + mu * ybar[:, 2]) - L20 * z0) - L21 * z1
        x2 = z2 / D2
        x1 = z1 / D1 - L21 * x2
        x0 = (z0 / D0 - L10 * x1) - L20 * x2
        x = np.stack([x0, x1, x2], 1)
        ok = (mu > 0) & np.isfinite(mu) & (D0 > h) & (D1 > h) & (D2 > h) & ((x >= 0) & (x <= 1)).all(1) & (tr != 0)
    y = np.where(ok[:, None], x, ybar)
    status = np.where(tr == 0, 1, np.where(ok, 0, 2))
    return y, status


def canonical_ref(t):
    """the cyclic rotation of each row of distinct ints t [f][3] that puts the smallest first"""
    k = np.argmin(t, axis=1)
    return t[np.arange(len(t))[:, None], (k[:, None] + np.arange(3)) % 3]


def decimate_ref(mesh, voxel_size, cell_size):
    """(xyz, normals, rgb, faces, collapsed, duplicates, fallbacks, extra) of the simplified mesh (xyz f32 [v][3],
    normals f32 [v][3], rgb u8 [v][3], faces int32 [f][3]); extra holds the clusters' means and integer coordinates"""
    xyz, nrm, rgb, faces = mesh
    H = F64(F32(cell_size))
    faces = np.asarray(faces, np.int64).reshape(-1, 3)
    cid, iv, q, f = clusters_ref(xyz, H)
    nc = len(iv)
    cnt = np.bincount(cid, minlength=nc).astype(np.uint64)
    sq, sm, sc = np.zeros((nc, 3), np.uint64), np.zeros((nc, 3), np.int64), np.zeros((nc, 3), np.uint64)
    np.add.at(sq, cid, q)
    m = np.rint(np.clip(np.asarray(nrm, F32), -1, 1).astype(F64) * Q).astype(np.int64)
    np.add.at(sm, cid, m)
    np.add.at(sc, cid, np.asarray(rgb, np.uint8).astype(np.uint64))
    u, w, ok = face_planes_ref(xyz, faces, H)
    qs = np.zeros((nc, 10), np.int64)
    for k in range(3):
        corner = faces[ok, k]
        np.add.at(qs, cid[corner], corner_coeffs_ref(u[ok], w[ok], f[corner]))
    y, status = place_ref(qs, sq, cnt)
    out_xyz = ((iv.astype(F64) + y) * H).astype(F32)
    mean = ((iv.astype(F64) + sq.astype(F64) / (Q * cnt.astype(F64))[:, None]) * H).astype(F32)
    X = sm.astype(F64)
    l2 = (X[:, 0] * X[:, 0] + X[:, 1] * X[:, 1]) + X[:, 2] * X[:, 2]
    with np.errstate(invalid="ignore", divide="ignore"):
        out_nrm = np.where((l2 != 0)[:, None], X / np.sqrt(l2)[:, None], 0.0).astype(F32)
    with np.errstate(divide="ignore"):
        out_rgb = ((sc + (cnt // np.uint64(2))[:, None]) // np.maximum(cnt, 1)[:, None]).astype(np.uint8)
    C = cid[faces] if len(faces) else np.zeros((0, 3), np.int64)
    col = (C[:, 0] == C[:, 1]) | (C[:, 1] == C[:, 2]) | (C[:, 0] == C[:, 2])
    keep = np.zeros(len(C), bool)
    live = np.flatnonzero(~col)
    if len(live):
        _, first = np.unique(canonical_ref(C[live]), axis=0, return_index=True)
        keep[live[first]] = True
    return (out_xyz, out_nrm, out_rgb, C[keep].astype(np.int32), int(col.sum()), int(len(live) - keep.sum()),
            int((status == 2).sum()), dict(mean=mean, ijk=iv, cluster=cid))


def decimate_loop(mesh, voxel_size, cell_size):
    """the same, one vertex, face and cluster at a time with Python floats (IEEE doubles, no FMA)"""
    xyz, nrm, rgb, faces = mesh
    H = float(F32(cell_size))
    key, cl, frac, qv = {}, [], [], []
    for p in xyz:
        t = [float(x) / H for x in p]
        i = tuple(math.floor(v) for v in t)
        fr = [v - math.floor(v) for v in t]
        frac.append(fr)
        qv.append([min(int(math.floor(v * Q)), int(Q) - 1) for v in fr])
        cl.append(key.setdefault(i, len(key)))
    nc = len(key)
    ijk = [None] * nc
    for i, c in key.items():
        ijk[c] = i
    n = [0] * nc
    sq, sm, sc = [[0] * 3 for _ in range(nc)], [[0] * 3 for _ in range(nc)], [[0] * 3 for _ in range(nc)]
    for v, c in enumerate(cl):
        n[c] += 1
        for a in range(3):
            sq[c][a] += qv[v][a]
            sm[c][a] += int(round(max(-1.0, min(1.0, float(nrm[v][a]))) * Q))   # round(): half to even
            sc[c][a] += int(rgb[v][a])
    qs = [[0] * 10 for _ in range(nc)]
    for fa in faces:
        pa, pb, pc = ([float(x) for x in xyz[k]] for k in fa)
        d1 = [pb[a] - pa[a] for a in range(3)]
        d2 = [pc[a] - pa[a] for a in range(3)]
        nn = [d1[1] * d2[2] - d1[2] * d2[1], d1[2] * d2[0] - d1[0] * d2[2], d1[0] * d2[1] - d1[1] * d2[0]]
        l2 = (nn[0] * nn[0] + nn[1] * nn[1]) + nn[2] * nn[2]
        if l2 == 0:
            continue
        l = math.sqrt(l2)
        u = [x / l for x in nn]
        w = (l * 0.5) / (H * H)
        for k in fa:
            fr = frac[k]
            e = (u[0] * fr[0] + u[1] * fr[1]) + u[2] * fr[2]
            c = [u[0] * u[0], u[0] * u[1], u[0] * u[2], u[1] * u[1], u[1] * u[2], u[2] * u[2], u[0] * e, u[1] * e,
                 u[2] * e, e * e]
            for j in range(10):
                qs[cl[k]][j] += int(round((w * c[j]) * SCALE))
    out_xyz, out_nrm, out_rgb, fallbacks = [], [], [], 0
    for c in range(nc):
        a = [float(x) * 2.0 ** -40 for x in qs[c][:9]]
        ybar = [float(sq[c][k]) / (Q * n[c]) for k in range(3)]
        y = ybar
        tr = (a[0] + a[3]) + a[5]
        if tr != 0:
            mu = DAMPING * (tr / 3.0)
            M = [[a[0] + mu, a[1], a[2]], [a[1], a[3] + mu, a[4]], [a[2], a[4], a[5] + mu]]
            L, D, ok = [[0.0] * 3 for _ in range(3)], [0.0] * 3, mu > 0 and math.isfinite(mu)
            for j in range(3):
                d = M[j][j]
                for k in range(j):
                    d = d - (L[j][k] * L[j][k]) * D[k]
                ok = ok and d > mu * 0.5
                if not ok:
                    break
                D[j] = d
                for i in range(j + 1, 3):
                    v = M[j][i]
                    for k in range(j):
                        v = v - (L[i][k] * L[j][k]) * D[k]
                    L[i][j] = v / d
            if ok:
                z = [0.0] * 3
                for i in range(3):
                    v = a[6 + i] + mu * ybar[i]
                    for k in range(i):
                        v = v - L[i][k] * z[k]
                    z[i] = v
                x = [0.0] * 3
                for i in (2, 1, 0):
                    v = z[i] / D[i]
                    for k in range(i + 1, 3):
                        v = v - L[k][i] * x[k]
                    x[i] = v
                ok = all(0.0 <= v <= 1.0 for v in x)
            if ok:
                y = x
            else:
                fallbacks += 1
        out_xyz.append([F32((ijk[c][k] + y[k]) * H) for k in range(3)])
        X = [float(v) for v in sm[c]]
        l2 = (X[0] * X[0] + X[1] * X[1]) + X[2] * X[2]
        out_nrm.append([F32(v / math.sqrt(l2)) if l2 != 0 else F32(0) for v in X])
        out_rgb.append([(sc[c][k] + n[c] // 2) // n[c] for k in range(3)])
    seen, out_f, col, dup = set(), [], 0, 0
    for fa in faces:
        t = [cl[k] for k in fa]
        if t[0] == t[1] or t[1] == t[2] or t[0] == t[2]:
            col += 1
            continue
        k = t.index(min(t))
        canon = tuple(t[k:] + t[:k])
        if canon in seen:
            dup += 1
            continue
        seen.add(canon)
        out_f.append(t)
    return (np.array(out_xyz, F32).reshape(-1, 3), np.array(out_nrm, F32).reshape(-1, 3),
            np.array(out_rgb, np.uint8).reshape(-1, 3), np.array(out_f, np.int32).reshape(-1, 3), col, dup, fallbacks)


def same_decimation(a, b):
    for x, y in zip(a[:4], b[:4]):
        assert x.shape == y.shape and x.dtype == y.dtype
        assert np.array_equal(x.view(np.uint8), y.view(np.uint8))
    assert tuple(a[4:7]) == tuple(b[4:7])


def nets_mesh(rng, m, s):
    """a surface-nets mesh of a random slab model (test_surface_math_host)"""
    mxyz, mnrm, mrgb, ijk = random_model(rng, m, s)
    return extract_ref(mxyz, mnrm, mrgb, ijk, s, F32(2 * s))[:4]


@pytest.mark.parametrize("seed", [0, 1, 2])
def test_reference_matches_the_loop_on_surface_nets_meshes(seed):
    rng = np.random.default_rng(seed)
    s = F32(0.25)
    mesh = nets_mesh(rng, 300, s)
    assert len(mesh[3]) > 50
    for ratio in (1, 2, 3.5, 8, 256):
        want = decimate_loop(mesh, s, F32(ratio * s))
        got = decimate_ref(mesh, s, F32(ratio * s))
        same_decimation(got, want)
        assert len(got[3]) + got[4] + got[5] == len(mesh[3])


def test_reference_matches_the_loop_on_a_sphere():
    s = F32(0.2)
    p, n, c, ijk = sphere_model(s, 1.2)
    mesh = extract_ref(p, n, c, ijk, s, F32(2 * s))[:4]
    for ratio in (2, 4):
        got = decimate_ref(mesh, s, F32(ratio * s))
        same_decimation(got, decimate_loop(mesh, s, F32(ratio * s)))
        assert got[4] > 0 and len(got[3]) < len(mesh[3]) // 2


def test_faces_rules_on_a_hand_made_mesh():
    """collapsed faces, a duplicate in another rotation, an opposite winding, a degenerate face and an unused
    cluster"""
    H = 1.0
    xyz = np.array([[0.1, 0.1, 0.1], [0.2, 0.3, 0.1], [1.5, 0.2, 0.2], [0.3, 1.6, 0.4], [1.2, 0.3, 0.1],
                    [0.4, 1.4, 0.6], [5.5, 5.5, 5.5]], F32)
    nrm = np.tile(np.array([[0, 0, 1]], F32), (len(xyz), 1))
    rgb = np.arange(len(xyz) * 3, dtype=np.uint8).reshape(-1, 3)
    # clusters by first vertex: 0 = {0, 1}, 1 = {2, 4}, 2 = {3, 5}, 3 = {6}
    faces = np.array([[0, 1, 2],          # collapsed (0, 0, 1)
                      [0, 2, 3],          # (0, 1, 2) kept
                      [4, 5, 1],          # (1, 2, 0): the same canonical triple, a duplicate
                      [0, 3, 2],          # (0, 2, 1): the opposite winding, kept
                      [2, 3, 0],          # (1, 2, 0) again: a duplicate
                      [3, 5, 5]], np.int32)   # collapsed and degenerate
    mesh = (xyz, nrm, rgb, faces)
    got = decimate_ref(mesh, 1.0, H)
    same_decimation(got, decimate_loop(mesh, 1.0, H))
    assert got[3].tolist() == [[0, 1, 2], [0, 2, 1]]
    assert got[4:7] == (2, 2, got[6]) and len(got[0]) == 4
    assert np.array_equal(got[2][3], rgb[6]) and np.array_equal(got[0][3], got[7]["mean"][3])


def test_empty_mesh():
    z = np.zeros((0, 3))
    got = decimate_ref((z.astype(F32), z.astype(F32), z.astype(np.uint8), z.astype(np.int32)), 1.0, 2.0)
    assert [len(a) for a in got[:4]] == [0, 0, 0, 0] and got[4:7] == (0, 0, 0)
