"""The numpy reference of the coherent orientation and the measures (scan3d_voxel_surface_orient, scan3d_mesh_orient_dev,
scan3d_voxel_surface_measure, scan3d_mesh_measure_dev), as include/scan3d.h states them: patches across edges of
count 2, the 2-colouring of each patch (scipy's csgraph over the nodes 2 f and 2 f + 1), the outward rule for closed
patches by the exact fixed-point volume and the fewest-flips rule otherwise, and the area, volume, bounding box and
topology.  The plain-Python loop it is checked against floods each patch from its smallest face.  CPU checks: random
flips of a closed sphere, a sphere turned inside out, an open hemisphere, the tie, a Moebius strip, a torus, pinched
spheres, a book, a bowtie, degenerate faces and an empty mesh; an exact cube; a second orientation that flips nothing;
the edge kinds equal to the repair's; and a fill that closes a hole only after the orientation.
tests/test_gpu_orient.py compares the GPU with orient_ref and measure_ref."""
import math

import numpy as np
import pytest
from scipy.sparse import coo_matrix
from scipy.sparse.csgraph import connected_components

from test_fill_ref import fill_ref, triangle_ref
from test_repair_ref import FACES, VERTICES, book, bowtie, odd, pinched_spheres, repair_ref
from test_smooth_ref import grid_mesh, icosphere

F32, F64, U32, U64 = np.float32, np.float64, np.uint32, np.uint64
P, E_MIN = 59, -149
ORIENT_FIELDS = ("vertices", "faces", "degenerate_faces", "patches", "closed_patches", "nonorientable_patches",
                 "flipped_faces", "flipped_normals", "inconsistent_edges_before", "inconsistent_edges")
MEASURE_FIELDS = ("vertices", "faces", "degenerate_faces", "patches", "closed_patches", "nonorientable_patches",
                  "unreferenced_vertices", "edges", "boundary_edges", "nonmanifold_edges", "inconsistent_edges",
                  "euler_characteristic", "watertight", "area", "volume", "bbox_min", "bbox_max")


class OrientError(Exception):
    pass


# ---- the arithmetic (common/scan3d_orient_math.h) ------------------------------------------------------------------
def order_key(x):
    b = np.asarray(x, F32).view(U32)
    return np.where(b & U32(0x80000000), ~b, b | U32(0x80000000)).astype(U32)


def key_float(k):
    k = np.asarray(k, U32)
    return np.where(k & U32(0x80000000), k & U32(0x7FFFFFFF), ~k).astype(U32).view(F32)


def centre_ref(lo, hi):
    return ((np.asarray(lo, F32).astype(F64) + np.asarray(hi, F32).astype(F64)) * 0.5).astype(F32)


def exponent_ref(x, c):
    """E of the referenced vertices x [m][3] about the centre c"""
    if len(x) == 0:
        return E_MIN
    d = np.asarray(x, F32).astype(F64) - np.asarray(c, F32).astype(F64)
    field = int(((d.view(U64) >> U64(52)) & U64(0x7FF)).max())
    return max(field - 1022, E_MIN)


def volume_terms_ref(pa, pb, pq, c, E):
    a, b, q = (np.asarray(p, F32).astype(F64) - np.asarray(c, F32).astype(F64) for p in (pa, pb, pq))
    x = np.stack([b[..., 1] * q[..., 2] - b[..., 2] * q[..., 1],
                  b[..., 2] * q[..., 0] - b[..., 0] * q[..., 2],
                  b[..., 0] * q[..., 1] - b[..., 1] * q[..., 0]], -1)
    D = (a[..., 0] * x[..., 0] + a[..., 1] * x[..., 1]) + a[..., 2] * x[..., 2]
    return np.rint(D * math.ldexp(1.0, P - 3 * E)).astype(np.int64)


def area_terms_ref(pa, pb, pq, E):
    return np.rint(triangle_ref(pa, pb, pq)[2] * math.ldexp(1.0, P - 2 * E)).astype(np.int64)


def exact_sums(terms, groups, n):
    """the exact sums of int64 terms per group in [0, n), as Python ints"""
    t = np.asarray(terms, np.int64)
    hi, lo = np.zeros(n, np.int64), np.zeros(n, np.int64)
    np.add.at(hi, groups, t >> 31)
    np.add.at(lo, groups, t & ((1 << 31) - 1))
    return [(int(h) << 31) + int(l) for h, l in zip(hi, lo)]


def volume_of(s, E):
    return math.ldexp(float(s), 3 * E - P) / 6.0


def area_of(s, E):
    return math.ldexp(float(s), 2 * E - P)


# ---- the reference -------------------------------------------------------------------------------------------------
def _check(xyz, faces):
    x = np.asarray(xyz, F32).reshape(-1, 3)
    f = np.asarray(faces, np.int64).reshape(-1, 3)
    if not np.isfinite(x).all() or ((f < 0) | (f >= len(x))).any():
        raise OrientError("a coordinate that is not finite or a face index outside [0, n_vertices)")
    return x, f


def analyse(xyz, faces):
    """everything both calls need: a dict of per-face, per-patch and per-mesh arrays and counts"""
    x, f = _check(xyz, faces)
    n, nf = len(x), len(f)
    deg = (f[:, 0] == f[:, 1]) | (f[:, 1] == f[:, 2]) | (f[:, 0] == f[:, 2])
    act = ~deg
    fid = np.repeat(np.arange(nf), 3)
    a, c = f.reshape(-1), f[:, [1, 2, 0]].reshape(-1)
    live = act[fid]
    a, c, fid = a[live], c[live], fid[live]
    keys, inv, cnt = np.unique(np.minimum(a, c) << 32 | np.maximum(a, c), return_inverse=True, return_counts=True)
    inv = inv.reshape(-1)
    face_open = np.zeros(nf, bool)
    face_open[fid[cnt[inv] != 2]] = True
    two = cnt[inv] == 2
    order = np.argsort(inv[two], kind="stable")
    pa, pf = a[two][order].reshape(-1, 2), fid[two][order].reshape(-1, 2)
    same = (pa[:, 0] == pa[:, 1]).astype(np.int64)      # the two sides have the same tail: they run the same way
    N = 2 * nf
    u = np.concatenate([2 * pf[:, 0], 2 * pf[:, 0] + 1])
    w = np.concatenate([2 * pf[:, 1] + same, 2 * pf[:, 1] + 1 - same])
    if N:
        _, lab = connected_components(coo_matrix((np.ones(len(u)), (u, w)), shape=(N, N)), directed=False)
        root_of = np.full(lab.max() + 1, N, np.int64)
        np.minimum.at(root_of, lab, np.arange(N))
        root = root_of[lab]
    else:
        root = np.zeros(0, np.int64)
    r, r1 = root[0::2], root[1::2]
    f0 = r >> 1
    pos = r % 2 == 0
    nonor_p = np.zeros(nf, bool)
    nonor_p[f0[act & (r == r1)]] = True
    open_p = np.zeros(nf, bool)
    open_p[f0[act & face_open]] = True
    ref = np.zeros(n, bool)
    ref[f[act].reshape(-1)] = True
    if ref.any():
        lo = key_float(order_key(x[ref]).min(0))
        hi = key_float(order_key(x[ref]).max(0))
    else:
        lo = hi = np.zeros(3, F32)
    cen = centre_ref(lo, hi)
    E = exponent_ref(x[ref], cen)
    fa = f[act]
    D = np.zeros(nf, np.int64)
    A = np.zeros(nf, np.int64)
    D[act] = volume_terms_ref(x[fa[:, 0]], x[fa[:, 1]], x[fa[:, 2]], cen, E)
    A[act] = area_terms_ref(x[fa[:, 0]], x[fa[:, 1]], x[fa[:, 2]], E)
    ia = np.flatnonzero(act)
    size = np.bincount(f0[ia], minlength=nf)
    npos = np.bincount(f0[ia[pos[ia]]], minlength=nf)
    V0 = exact_sums(np.where(pos, D, -D)[ia], f0[ia], nf)
    is_root = act & (r == 2 * np.arange(nf))
    return dict(x=x, f=f, n=n, nf=nf, deg=deg, act=act, cnt=cnt, pf=pf, same=same.astype(bool), r=r, f0=f0,
                nonor_p=nonor_p, open_p=open_p, ref=ref, lo=lo, hi=hi, E=E, D=D, A=A, size=size, npos=npos, V0=V0,
                is_root=is_root)


def _patch_counts(m):
    roots = np.flatnonzero(m["is_root"])
    return dict(patches=len(roots), closed_patches=int((~m["open_p"][roots]).sum()),
                nonorientable_patches=int(m["nonor_p"][roots].sum()))


def orient_ref(xyz, faces, normals=None):
    """(faces int32 [f][3], normals float32 [v][3] or None, info dict with the fields of scan3d_orient_result)"""
    m = analyse(xyz, faces)
    f, nf, act, r, f0 = m["f"], m["nf"], m["act"], m["r"], m["f0"]
    keep = np.array([(m["V0"][g] > 0) if (not m["open_p"][g] and m["V0"][g] != 0)
                     else 2 * m["npos"][g] >= m["size"][g] for g in range(nf)], bool)
    flip = act & ~m["nonor_p"][f0] & ((r & 1).astype(bool) == keep[f0]) if nf else np.zeros(0, bool)
    kept = np.zeros(m["n"], bool)
    kept[f[act & ~flip].reshape(-1)] = True
    turned = m["ref"] & ~kept
    out = f.copy()
    out[flip] = out[flip][:, [0, 2, 1]]
    nrm = None
    if normals is not None:
        nrm = np.array(normals, F32).reshape(-1, 3).copy()
        nrm.view(U32)[turned] ^= U32(0x80000000)
    left = int((m["same"] & m["nonor_p"][f0[m["pf"][:, 0]]]).sum()) if len(m["pf"]) else 0
    info = dict(vertices=m["n"], faces=nf, degenerate_faces=int(m["deg"].sum()), **_patch_counts(m),
                flipped_faces=int(flip.sum()), flipped_normals=int(turned.sum()),
                inconsistent_edges_before=int(m["same"].sum()), inconsistent_edges=left)
    return out.astype(np.int32), nrm, info


def measure_ref(xyz, faces):
    """the dict of scan3d_measure_result"""
    m = analyse(xyz, faces)
    cnt, live = m["cnt"], int(m["act"].sum())
    boundary, nonmanifold, inconsistent = int((cnt == 1).sum()), int((cnt > 2).sum()), int(m["same"].sum())
    referenced = int(m["ref"].sum())
    return dict(vertices=m["n"], faces=m["nf"], degenerate_faces=int(m["deg"].sum()), **_patch_counts(m),
                unreferenced_vertices=m["n"] - referenced, edges=len(cnt), boundary_edges=boundary,
                nonmanifold_edges=nonmanifold, inconsistent_edges=inconsistent,
                euler_characteristic=referenced - len(cnt) + live,
                watertight=live > 0 and boundary == nonmanifold == inconsistent == 0,
                area=area_of(sum(int(t) for t in m["A"]), m["E"]), volume=volume_of(sum(int(t) for t in m["D"]), m["E"]),
                bbox_min=tuple(float(v) for v in m["lo"]), bbox_max=tuple(float(v) for v in m["hi"]))


# ---- an independent plain-Python loop ------------------------------------------------------------------------------
def orient_loop(xyz, faces):
    """(faces, flipped count, patches, non-orientable patches): each patch flooded from its smallest face"""
    m = analyse(xyz, faces)                               # only its fixed-point volume terms are used
    F = [tuple(int(v) for v in t) for t in np.asarray(faces).reshape(-1, 3)]
    sides = {}
    for i, (a, b, c) in enumerate(F):
        if len({a, b, c}) < 3:
            continue
        for s, t in ((a, b), (b, c), (c, a)):
            sides.setdefault((min(s, t), max(s, t)), []).append((i, s))
    sign = {}
    flips, patches, nonor = [False] * len(F), 0, 0
    for start in range(len(F)):
        if start in sign or len(set(F[start])) < 3:
            continue
        patches += 1
        sign[start], stack, members, ok, closed = 1, [start], [start], True, True
        while stack:
            i = stack.pop()
            a, b, c = F[i]
            for s, t in ((a, b), (b, c), (c, a)):
                on = sides[(min(s, t), max(s, t))]
                if len(on) != 2:
                    closed = False
                    continue
                (j, tj), = [(g, tg) for g, tg in on if g != i] or [on[0]]
                want = -sign[i] if tj == s else sign[i]  # the same tail: the neighbour runs the edge the same way
                if j not in sign:
                    sign[j] = want
                    members.append(j)
                    stack.append(j)
                elif sign[j] != want:
                    ok = False
        if not ok:
            nonor += 1
            continue
        V0 = sum(sign[g] * int(m["D"][g]) for g in members)
        npos = sum(sign[g] > 0 for g in members)
        keep = V0 > 0 if closed and V0 != 0 else 2 * npos >= len(members)
        for g in members:
            flips[g] = (sign[g] > 0) != keep
    out = [(a, c, b) if fl else (a, b, c) for (a, b, c), fl in zip(F, flips)]
    return np.array(out, np.int32).reshape(-1, 3), sum(flips), patches, nonor


def _same(a, b):
    a, b = np.asarray(a), np.asarray(b)
    assert a.shape == b.shape and a.dtype == b.dtype and np.array_equal(a, b)


def check(xyz, faces, normals=None):
    out, nrm, info = orient_ref(xyz, faces, normals)
    lf, flips, patches, nonor = orient_loop(xyz, faces)
    _same(out, lf)
    assert (info["flipped_faces"], info["patches"], info["nonorientable_patches"]) == (flips, patches, nonor)
    # a second orientation flips nothing
    again, _, info2 = orient_ref(xyz, out)
    _same(again, out)
    assert info2["flipped_faces"] == 0 and info2["inconsistent_edges_before"] == info["inconsistent_edges"]
    return out, nrm, info


# ---- constructed meshes --------------------------------------------------------------------------------------------
def sphere(level=2, r=2.0):
    u, f = icosphere(level)
    return (u * r).astype(F32), f


def flipped(faces, which):
    f = np.array(faces, np.int32)
    f[which] = f[which][:, [0, 2, 1]]
    return f


def moebius(n=12):
    t = np.arange(n) * 2 * np.pi / n
    xyz = []
    for s in (-0.3, 0.3):
        xyz.append(np.stack([(1 + s * np.cos(t / 2)) * np.cos(t), (1 + s * np.cos(t / 2)) * np.sin(t),
                             s * np.sin(t / 2)], -1))
    xyz = np.concatenate(xyz).astype(F32)                # top i = i, bottom i = n + i
    faces = []
    for i in range(n):
        ti, bi = i, n + i
        tj, bj = (i + 1, n + i + 1) if i + 1 < n else (n, 0)   # the half twist swaps the sides
        faces += [(ti, bi, tj), (bi, bj, tj)]
    return xyz, np.array(faces, np.int32)


def torus(nu=8, nv=6, R=2.0, r=0.5):
    u, v = np.meshgrid(np.arange(nu) * 2 * np.pi / nu, np.arange(nv) * 2 * np.pi / nv, indexing="ij")
    xyz = np.stack([(R + r * np.cos(v)) * np.cos(u), (R + r * np.cos(v)) * np.sin(u), r * np.sin(v)], -1)
    idx = np.arange(nu * nv).reshape(nu, nv)
    faces = []
    for i in range(nu):
        for j in range(nv):
            a, b, c, d = idx[i, j], idx[(i + 1) % nu, j], idx[i, (j + 1) % nv], idx[(i + 1) % nu, (j + 1) % nv]
            faces += [(a, b, d), (a, d, c)]
    return xyz.reshape(-1, 3).astype(F32), np.array(faces, np.int32)


def cube(s=2.0, t=(0.0, 0.0, 0.0)):
    h = s / 2
    xyz = np.array([[x, y, z] for x in (-h, h) for y in (-h, h) for z in (-h, h)], F64) + np.array(t)
    faces = np.array([[0, 1, 3], [0, 3, 2], [4, 6, 7], [4, 7, 5], [0, 4, 5], [0, 5, 1], [2, 3, 7], [2, 7, 6],
                      [0, 2, 6], [0, 6, 4], [1, 5, 7], [1, 7, 3]], np.int32)
    return xyz.astype(F32), faces


def hemisphere(level=2):
    xyz, f = sphere(level)
    up = xyz[f].mean(1)[:, 2] > 0.1
    return xyz, f[up]


def rim_hole_mesh():
    """a 6 x 6 grid with cell (2, 2) removed and one rim face of the hole flipped"""
    xyz, faces = grid_mesh(6, 6)
    cell = np.concatenate([np.arange(25), np.arange(25)])
    faces = faces[cell != 2 * 5 + 2]
    cell = cell[cell != 2 * 5 + 2]
    # the face of the cell right of the hole that holds the hole's right side, grid vertices 15 and 21
    rim = int(np.flatnonzero((cell == 2 * 5 + 3) & (np.isin(faces, [15, 21]).sum(1) == 2))[0])
    return xyz, flipped(faces, [rim])


# ---- the checks ----------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("seed", range(4))
def test_random_flips_of_a_closed_sphere_are_undone(seed):
    xyz, f = sphere()
    rng = np.random.default_rng(seed)
    which = rng.random(len(f)) < 0.3 + 0.15 * seed
    out, _, info = check(xyz, flipped(f, which))
    _same(out, f)
    assert info["flipped_faces"] == which.sum() and info["closed_patches"] == 1 and info["inconsistent_edges"] == 0
    assert measure_ref(xyz, out)["volume"] > 0


def test_a_sphere_turned_inside_out_is_turned_back():
    xyz, f = sphere()
    inside = flipped(f, slice(None))
    assert measure_ref(xyz, inside)["volume"] < 0
    nrm = xyz / np.linalg.norm(xyz, axis=1, keepdims=True)
    out, n2, info = check(xyz, inside, -nrm)
    _same(out, f)
    assert info["flipped_faces"] == len(f) and info["flipped_normals"] == len(xyz)
    np.testing.assert_array_equal(n2, nrm.astype(F32))
    mr = measure_ref(xyz, out)
    assert mr["volume"] > 0 and mr["watertight"] and mr["euler_characteristic"] == 2
    assert abs(mr["volume"] - 4 / 3 * math.pi * 8) < 0.1 * 4 / 3 * math.pi * 8


def test_an_open_hemisphere_keeps_its_majority():
    xyz, f = hemisphere()
    which = np.zeros(len(f), bool)
    which[1::5] = True
    out, _, info = check(xyz, flipped(f, which))
    _same(out, f)
    assert info["closed_patches"] == 0 and info["flipped_faces"] == which.sum()


def test_the_tie_keeps_the_smallest_face():
    xyz = np.array([[0, 0, 0], [1, 0, 0], [0, 1, 0], [0, -1, 0]], F32)
    faces = np.array([[0, 1, 2], [0, 1, 3]], np.int32)     # both run 0 -> 1: one must flip
    out, _, info = check(xyz, faces)
    _same(out, np.array([[0, 1, 2], [0, 3, 1]], np.int32))
    assert info["flipped_faces"] == 1 and info["inconsistent_edges_before"] == 1 and info["inconsistent_edges"] == 0


def test_a_moebius_strip_is_left_alone_and_counted():
    xyz, f = moebius()
    out, _, info = check(xyz, f)
    _same(out, f)
    assert info["nonorientable_patches"] == 1 and info["flipped_faces"] == 0
    assert info["inconsistent_edges"] == info["inconsistent_edges_before"] >= 1


def test_a_torus_has_euler_characteristic_zero():
    xyz, f = torus()
    out, _, info = check(xyz, flipped(f, [3, 7, 11]))
    _same(out, f)
    mr = measure_ref(xyz, out)
    assert mr["euler_characteristic"] == 0 and mr["watertight"] and mr["patches"] == 1
    assert mr["patches"] - mr["euler_characteristic"] // 2 == 1   # genus 1


def test_pinched_spheres_book_and_bowtie():
    xyz, f = pinched_spheres(2)
    h = len(f) // 2
    out, _, info = check(xyz, flipped(f, slice(h, None)))          # the second sphere inside out
    _same(out, f)
    assert info["patches"] == info["closed_patches"] == 2
    mr = measure_ref(xyz, out)
    assert mr["watertight"] and mr["euler_characteristic"] == 3     # a shared vertex: no genus follows
    xyz, f = book(4, [1.0, 3.0, 0.5, 2.0], [1, 1, -1, 1])
    out, _, info = check(xyz, f)
    assert info["patches"] == 4 and info["flipped_faces"] == 0
    assert measure_ref(xyz, f)["nonmanifold_edges"] == 1
    xyz, f = bowtie()
    out, _, info = check(xyz, f)
    _same(out, f)
    assert info["patches"] == 2 and measure_ref(xyz, f)["boundary_edges"] == 6


def test_degenerate_faces_take_no_part_and_the_empty_mesh():
    xyz, f = sphere(1)
    deg = np.array([[0, 0, 1], [2, 3, 2], [5, 5, 5]], np.int32)
    faces = np.concatenate([flipped(f, [0, 4]), deg])
    out, _, info = check(xyz, faces)
    _same(out[-3:], deg)
    _same(out[:-3], f)
    assert info["degenerate_faces"] == 3
    assert measure_ref(xyz, out) == dict(measure_ref(xyz, out[:-3]), faces=len(faces), degenerate_faces=3)
    for x in (np.zeros((0, 3), F32), np.ones((5, 3), F32)):
        out, _, info = check(x, np.zeros((0, 3), np.int32))
        assert out.shape == (0, 3)
        assert info == dict(dict.fromkeys(ORIENT_FIELDS, 0), vertices=len(x))
        mr = measure_ref(x, np.zeros((0, 3), np.int32))
        assert mr["unreferenced_vertices"] == len(x) and not mr["watertight"] and mr["area"] == mr["volume"] == 0.0
        assert mr["bbox_min"] == mr["bbox_max"] == (0.0, 0.0, 0.0)


@pytest.mark.parametrize("t", [(0.0, 0.0, 0.0), (3.0, -5.0, 7.25), (1024.0, 0.5, -96.0)])
def test_an_exact_cube_has_area_six_s2_and_volume_s3(t):
    for s in (2.0, 0.375, 48.0):
        xyz, f = cube(s, t)
        mr = measure_ref(xyz, f)
        assert mr["area"] == 6 * s * s and mr["volume"] == s ** 3, (s, t, mr)
        assert mr["watertight"] and mr["euler_characteristic"] == 2
        out, _, info = check(xyz, flipped(f, [1, 2, 3, 5, 8]))
        _same(out, f)


@pytest.mark.parametrize("seed", range(6))
def test_the_edge_kinds_equal_the_repairs(seed):
    xyz, f = odd(seed, 40 + 20 * seed, 100 + 60 * seed)
    mr = measure_ref(xyz, f)
    info = repair_ref(xyz, f, VERTICES)[2]                 # no face dropped: the same faces
    assert (mr["nonmanifold_edges"], mr["boundary_edges"], mr["inconsistent_edges"]) == (
        info["nonmanifold_edges"], info["boundary_edges"], info["inconsistent_edges"])
    out, _, info = repair_ref(xyz, f, FACES)
    mr = measure_ref(xyz, out)
    assert (mr["nonmanifold_edges"], mr["boundary_edges"], mr["inconsistent_edges"]) == (
        0, info["boundary_edges"], info["inconsistent_edges"])
    o2, _, oi = check(xyz, out)
    assert oi["inconsistent_edges_before"] == info["inconsistent_edges"]
    assert measure_ref(xyz, o2)["inconsistent_edges"] == oi["inconsistent_edges"]


def test_a_fill_closes_the_hole_only_after_the_orientation():
    xyz, f = rim_hole_mesh()
    before = fill_ref(xyz, f, 22)[1]
    out, _, info = check(xyz, f)
    assert info["flipped_faces"] == 1
    after = fill_ref(xyz, out, 22)[1]
    assert after["open_edges"] < before["open_edges"] and after["filled"] > before["filled"]
    assert after["open_edges"] == 0
