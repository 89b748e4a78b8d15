"""The numpy reference of the non-manifold repair (scan3d_voxel_surface_repair, scan3d_mesh_repair_dev), as
include/scan3d.h states it: degenerate and duplicate faces, the per-edge keep rule of non-manifold edges by area key,
and the split of non-manifold vertices into fans.  The reference finds the fans as the connected components of the
corner graph (scipy's csgraph); the plain-Python loop it is checked against walks the faces around each vertex.  CPU
checks: the reference against the loop on random odd meshes and constructed cases, the manifold promise by an
independent checker, copies on their sources, a second repair that changes nothing, and two holes sharing a vertex
that the fill closes only after the repair.  tests/test_gpu_repair.py compares the GPU with repair_ref."""
import numpy as np
import pytest
from scipy.sparse import coo_matrix
from scipy.sparse.csgraph import connected_components

from test_fill_ref import _tri_loop, edge_counts, fill_ref, triangle_ref
from test_smooth_ref import grid_mesh, icosphere, odd_mesh

F32, F64 = np.float32, np.float64
FACES, VERTICES = 1, 2
FLAGS = (FACES, VERTICES, FACES | VERTICES)
FIELDS = ("vertices", "faces", "degenerate_faces", "duplicate_faces", "nonmanifold_edges", "nonmanifold_faces",
          "split_vertices", "vertices_added", "boundary_edges", "inconsistent_edges")


class RepairError(Exception):
    pass


def face_key_ref(xyz, faces):
    """K(f) = (float_bits((float)area_f) << 32) | (2^32 - 1 - f), uint64 [f]"""
    f = np.asarray(faces, np.int64).reshape(-1, 3)
    x = np.asarray(xyz, F32)
    area = triangle_ref(x[f[:, 0]], x[f[:, 1]], x[f[:, 2]])[2]
    with np.errstate(over="ignore"):                    # an area beyond the float range is +inf, as on the GPU
        bits = area.astype(F32).view(np.uint32).astype(np.uint64)
    return bits << np.uint64(32) | (np.uint64(0xFFFFFFFF) - np.arange(len(f), dtype=np.uint64))


def kept_on_edge_ref(k, m0, m1, second):
    """the edge rule, elementwise over uint64 arrays"""
    f1 = np.maximum(m0, m1)
    opposite = np.minimum(m0, m1)
    f2 = np.where(opposite != 0, opposite, second)
    return (k == f1) | (k == f2)


def _check(xyz, faces):
    x = np.asarray(xyz, F32).reshape(-1, 3)
    f = np.asarray(faces, np.int64).reshape(-1, 3)
    if not np.isfinite(x).all() or ((f < 0) | (f >= len(x))).any():
        raise RepairError("a coordinate that is not finite or a face index outside [0, n_vertices)")
    return x, f


def repair_ref(xyz, faces, flags):
    """(faces int32 [m][3], source int32 [added], info dict with the fields of scan3d_repair_result)"""
    x, f = _check(xyz, faces)
    n, nf = len(x), len(f)
    degenerate = (f[:, 0] == f[:, 1]) | (f[:, 1] == f[:, 2]) | (f[:, 0] == f[:, 2])
    alive = ~degenerate
    dup = np.zeros(nf, bool)
    if flags & FACES and alive.any():
        idx = np.flatnonzero(alive)
        _, first = np.unique(np.sort(f[idx], 1), axis=0, return_index=True)
        dup[idx] = True
        dup[idx[first]] = False
    alive &= ~dup
    K = face_key_ref(x, f)
    # the surviving faces' sides: tail a, head c, edge key, direction (a > c)
    fid = np.repeat(np.arange(nf), 3)
    a, c = f.reshape(-1), f[:, [1, 2, 0]].reshape(-1)
    live = alive[fid]
    a, c, fid = a[live], c[live], fid[live]
    ekey = np.minimum(a, c) << 32 | np.maximum(a, c)
    keys, inv, cnt = np.unique(ekey, return_inverse=True, return_counts=True)
    inv = inv.reshape(-1)
    dropped = np.zeros(nf, bool)
    if flags & FACES:
        m = np.zeros((len(keys), 2), np.uint64)
        np.maximum.at(m, (inv, (a > c).astype(np.int64)), K[fid])
        f1 = m.max(1)
        second = np.zeros(len(keys), np.uint64)
        other = K[fid] != f1[inv]
        np.maximum.at(second, inv[other], K[fid][other])
        bad_side = (cnt[inv] > 2) & ~kept_on_edge_ref(K[fid], m[inv, 0], m[inv, 1], second[inv])
        dropped[fid[bad_side]] = True
    kept = alive & ~dropped
    ks = kept[fid]
    ka, kc, kf, kinv = a[ks], c[ks], fid[ks], inv[ks]
    kcnt = np.bincount(kinv, minlength=len(keys))
    # edges in two kept faces: their two sides
    two = kcnt[kinv] == 2
    order = np.argsort(kinv[two], kind="stable")
    pa, pc, pf = ka[two][order].reshape(-1, 2), kc[two][order].reshape(-1, 2), kf[two][order].reshape(-1, 2)
    inconsistent = int((pa[:, 0] == pa[:, 1]).sum())
    corner = f.copy()
    split = 0
    src = np.zeros(0, np.int64)
    if flags & VERTICES and kept.any():
        def corner_of(face, v):
            return 3 * face + np.argmax(f[face] == v[:, None], 1)
        u = np.concatenate([corner_of(pf[:, 0], pa[:, 0]), corner_of(pf[:, 0], pc[:, 0])])
        w = np.concatenate([corner_of(pf[:, 1], pa[:, 0]), corner_of(pf[:, 1], pc[:, 0])])
        N = 3 * nf
        g = coo_matrix((np.ones(len(u)), (u, w)), shape=(N, N))
        _, lab = connected_components(g, directed=False)
        root_of = np.full(lab.max() + 1, N, np.int64)
        kc_all = np.flatnonzero(np.repeat(kept, 3))
        np.minimum.at(root_of, lab[kc_all], kc_all)
        root = root_of[lab]
        vert = f.reshape(-1)
        first = np.full(n + 1, N, np.int64)
        np.minimum.at(first, vert[kc_all], kc_all)
        roots = np.unique(root[kc_all])
        fresh = roots[roots != first[vert[roots]]]        # ascending
        new_id = np.zeros(N + 1, np.int64)                # N: the root of a corner of a face that is not kept
        new_id[fresh] = n + np.arange(len(fresh))
        src = vert[fresh]
        split = len(np.unique(src))
        rc = root.reshape(-1, 3)
        corner = np.where(rc != first[f], new_id[rc], f)
    out = corner[kept].astype(np.int32)
    info = dict(vertices=n + len(src), faces=int(kept.sum()), degenerate_faces=int(degenerate.sum()),
                duplicate_faces=int(dup.sum()), nonmanifold_edges=int((cnt > 2).sum()),
                nonmanifold_faces=int(dropped.sum()), split_vertices=split, vertices_added=len(src),
                boundary_edges=int((kcnt == 1).sum()), inconsistent_edges=inconsistent)
    return out, src.astype(np.int32), info


def apply_source(xyz, src):
    """the vertex array extended by the copies"""
    return np.concatenate([np.asarray(xyz, F32).reshape(-1, 3), np.asarray(xyz, F32).reshape(-1, 3)[src]])


# ---- an independent plain-Python loop ------------------------------------------------------------------------------
def fans_loop(faces, n):
    """{v: [fans, each a sorted list of corners 3 f + k]} of the faces (None rows skipped), fans by walking the faces
    around each vertex across the edges in exactly two faces, in ascending order of their smallest corner"""
    count, at = {}, {}
    for fi, t in enumerate(faces):
        if t is None:
            continue
        for k in range(3):
            e = (min(t[k], t[(k + 1) % 3]), max(t[k], t[(k + 1) % 3]))
            count.setdefault(e, []).append(fi)
            at.setdefault(t[k], []).append(3 * fi + k)
    out = {}
    for v in sorted(at):
        left, fans = sorted(at[v]), []
        while left:
            fan, todo = [], [left[0]]
            while todo:
                c = todo.pop()
                if c in fan:
                    continue
                fan.append(c)
                t = faces[c // 3]
                for w in (t[(c % 3 + 1) % 3], t[(c % 3 + 2) % 3]):
                    on = count[(min(v, w), max(v, w))]
                    if len(on) == 2:
                        g = on[0] if on[1] == c // 3 else on[1]
                        todo.append(3 * g + faces[g].index(v))
            fans.append(sorted(fan))
            left = [c for c in left if c not in fan]
        out[v] = sorted(fans)
    return out, count


def repair_loop(xyz, faces, flags):
    x = np.asarray(xyz, F32)
    F = [tuple(int(v) for v in t) for t in np.asarray(faces).reshape(-1, 3)]
    n = len(x)
    info = dict.fromkeys(FIELDS, 0)
    alive, seen = [], {}
    for fi, t in enumerate(F):
        if len(set(t)) < 3:
            info["degenerate_faces"] += 1
            alive.append(False)
        elif flags & FACES and tuple(sorted(t)) in seen:
            info["duplicate_faces"] += 1
            alive.append(False)
        else:
            seen.setdefault(tuple(sorted(t)), fi)
            alive.append(True)

    def key(fi):
        t = F[fi]
        area = _tri_loop(x[t[0]], x[t[1]], x[t[2]])[1]
        return int(np.float32(area).view(np.uint32)) << 32 | (0xFFFFFFFF - fi)

    on = {}
    for fi, t in enumerate(F):
        if alive[fi]:
            for k in range(3):
                a, c = t[k], t[(k + 1) % 3]
                on.setdefault((min(a, c), max(a, c)), []).append((fi, a > c))
    drop = set()
    for e, sides in on.items():
        if len(sides) <= 2:
            continue
        info["nonmanifold_edges"] += 1
        if not flags & FACES:
            continue
        f1, d1 = max(sides, key=lambda s: key(s[0]))
        opp = [s for s in sides if s[1] != d1]
        f2 = max(opp or [s for s in sides if s[0] != f1], key=lambda s: key(s[0]))[0]
        drop |= {s[0] for s in sides if s[0] not in (f1, f2)}
    info["nonmanifold_faces"] = len(drop)
    K = [t if alive[fi] and fi not in drop else None for fi, t in enumerate(F)]
    fans, count = fans_loop(K, n)
    for e, fs in count.items():
        if len(fs) == 1:
            info["boundary_edges"] += 1
        elif len(fs) == 2:
            a, b = fs
            ta, tb = K[a], K[b]
            info["inconsistent_edges"] += (ta[(ta.index(e[0]) + 1) % 3] == e[1]) == (tb[(tb.index(e[0]) + 1) % 3] == e[1])
    corner = {}
    src = []
    if flags & VERTICES:
        extra = sorted((fan[0], v) for v, fs in fans.items() for fan in fs[1:])
        info["split_vertices"] = len({v for v, fs in fans.items() if len(fs) > 1})
        for r, v in extra:
            fan = next(fan for fan in fans[v] if fan[0] == r)
            for c in fan:
                corner[c] = n + len(src)
            src.append(v)
    out = [[corner.get(3 * fi + k, t[k]) for k in range(3)] for fi, t in enumerate(K) if t is not None]
    info.update(vertices=n + len(src), faces=len(out), vertices_added=len(src))
    return np.array(out, np.int32).reshape(-1, 3), np.array(src, np.int32), info


def defects_loop(faces, n):
    """(edges in more than 2 faces, vertices whose faces form more than one fan), checked independently of the
    repair"""
    F = [tuple(int(v) for v in t) for t in np.asarray(faces).reshape(-1, 3)]
    fans, count = fans_loop(F, n)
    return sum(len(fs) > 2 for fs in count.values()), sum(len(fs) > 1 for fs in fans.values())


def _same(a, b):
    a, b = np.asarray(a), np.asarray(b)
    assert a.shape == b.shape and a.dtype == b.dtype and np.array_equal(a, b)


def check_against_loop(xyz, faces, flags):
    got = repair_ref(xyz, faces, flags)
    want = repair_loop(xyz, faces, flags)
    _same(got[0], want[0])
    _same(got[1], want[1])
    assert got[2] == want[2]
    return got


# ---- constructed meshes --------------------------------------------------------------------------------------------
def bowtie():
    xyz = np.array([[0, 0, 0], [1, 0, 0], [1, 1, 0], [-1, 0, 0], [-1, -1, 0]], F32)
    return xyz, np.array([[0, 1, 2], [0, 3, 4]], np.int32)


def pinched_spheres(level=1):
    """two closed icospheres touching at one vertex: vertex 0 of the second is vertex 0 of the first"""
    u, f = icosphere(level)
    a = u.astype(F32)
    b = (u + (u[0] * -2.0)).astype(F32)[1:]              # the second sphere shifted to touch at u[0]
    fb = f.astype(np.int64) + len(a) - 1
    fb[f == 0] = 0
    return np.concatenate([a, b]), np.concatenate([f, fb]).astype(np.int32)


def book(pages, widths, windings):
    """faces on the edge (0, 1): page p is (0, 1, 2 + p) when its winding is +1 else (1, 0, 2 + p), at distance
    widths[p] from the spine"""
    xyz = [[0, 0, 0], [0, 0, 1]]
    faces = []
    for p in range(pages):
        ang = 2 * np.pi * p / pages
        xyz.append([widths[p] * np.cos(ang), widths[p] * np.sin(ang), 0.5])
        faces.append((0, 1, 2 + p) if windings[p] > 0 else (1, 0, 2 + p))
    return np.array(xyz, F32), np.array(faces, np.int32)


def odd(seed, n=60, f=150):
    return odd_mesh(np.random.default_rng(seed), n, f)[0::2]


# ---- the checks ----------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("seed", range(6))
@pytest.mark.parametrize("flags", FLAGS)
def test_reference_matches_the_loop_on_odd_meshes(seed, flags):
    xyz, faces = odd(seed, 40 + 20 * seed, 100 + 60 * seed)
    out, src, info = check_against_loop(xyz, faces, flags)
    if flags == FACES | VERTICES:
        assert defects_loop(out, info["vertices"]) == (0, 0)


def test_bowtie_splits_once():
    xyz, faces = bowtie()
    for flags in FLAGS:
        out, src, info = check_against_loop(xyz, faces, flags)
        if flags & VERTICES:
            _same(out, np.array([[0, 1, 2], [5, 3, 4]], np.int32))
            _same(src, np.array([0], np.int32))
            assert info["split_vertices"] == 1 and info["vertices_added"] == 1 and info["boundary_edges"] == 6
        else:
            _same(out, faces)


def test_pinched_spheres_split_into_two_closed_pieces():
    xyz, faces = pinched_spheres()
    out, src, info = check_against_loop(xyz, faces, FACES | VERTICES)
    assert info["vertices_added"] == 1 and info["split_vertices"] == 1 and info["boundary_edges"] == 0
    assert info["nonmanifold_edges"] == 0 and info["inconsistent_edges"] == 0
    und, directed = edge_counts(out)
    assert (und == 2).all() and (directed == 1).all()     # both copies interior, both pieces closed
    assert defects_loop(out, info["vertices"]) == (0, 0)
    assert defects_loop(faces, len(xyz)) == (0, 1)


def test_fin_and_book_keep_the_two_largest_preferring_opposite_windings():
    # a fin of 3: the largest (page 1) and the largest running opposite to it (page 2, smaller than page 0)
    xyz, faces = book(3, [1.0, 3.0, 0.5], [+1, +1, -1])
    out, _, info = check_against_loop(xyz, faces, FACES | VERTICES)
    _same(out, faces[[1, 2]])
    assert info["nonmanifold_edges"] == 1 and info["nonmanifold_faces"] == 1 and info["inconsistent_edges"] == 0
    # no face runs opposite: the two largest
    xyz, faces = book(4, [1.0, 3.0, 0.5, 2.0], [+1, +1, +1, +1])
    out, _, info = check_against_loop(xyz, faces, FACES)
    _same(out, faces[[1, 3]])
    assert info["nonmanifold_faces"] == 2 and info["inconsistent_edges"] == 1
    # a book of 4 with equal areas: ties go to the smaller index, then the opposite winding is preferred
    xyz, faces = book(4, [1.0] * 4, [+1, +1, -1, -1])
    a = face_key_ref(xyz, faces) >> np.uint64(32)
    assert (a == a[0]).all()
    out, _, info = check_against_loop(xyz, faces, FACES | VERTICES)
    _same(out, faces[[0, 2]])
    # without FACES the edge is only counted, and it joins no corners: each page gets its own copies of the spine
    out, _, info = check_against_loop(xyz, faces, VERTICES)
    _same(out, np.array([[0, 1, 2], [6, 7, 3], [8, 9, 4], [10, 11, 5]], np.int32))
    assert info["nonmanifold_edges"] == 1 and info["nonmanifold_faces"] == 0 and info["vertices_added"] == 6


def test_duplicates_in_both_windings_and_degenerate_faces():
    xyz = np.array([[0, 0, 0], [1, 0, 0], [0, 1, 0], [1, 1, 0]], F32)
    faces = np.array([[0, 1, 2], [1, 2, 0], [2, 1, 0], [0, 0, 1], [3, 3, 3], [1, 3, 2], [2, 3, 1]], np.int32)
    out, _, info = check_against_loop(xyz, faces, FACES | VERTICES)
    _same(out, faces[[0, 5]])
    assert info["duplicate_faces"] == 3 and info["degenerate_faces"] == 2 and info["nonmanifold_edges"] == 0
    # without FACES the duplicates stay and make the edges non-manifold; the degenerate faces still go
    out, _, info = check_against_loop(xyz, faces, VERTICES)
    assert len(out) == 5
    assert info["duplicate_faces"] == 0 and info["degenerate_faces"] == 2 and info["nonmanifold_edges"] == 3


def test_empty_mesh_and_vertices_without_faces():
    for xyz in (np.zeros((0, 3), F32), np.ones((5, 3), F32)):
        for flags in FLAGS:
            out, src, info = check_against_loop(xyz, np.zeros((0, 3), np.int32), flags)
            assert out.shape == (0, 3) and len(src) == 0
            assert info == dict(dict.fromkeys(FIELDS, 0), vertices=len(xyz))


@pytest.mark.parametrize("seed", range(4))
def test_copies_sit_on_their_sources_and_a_second_repair_changes_nothing(seed):
    xyz, faces = odd(10 + seed, 80, 300)
    out, src, info = repair_ref(xyz, faces, FACES | VERTICES)
    assert info["vertices_added"] > 0
    x2 = apply_source(xyz, src)
    assert np.array_equal(x2[len(xyz):].view(np.uint32), xyz[src].view(np.uint32))
    out2, src2, info2 = check_against_loop(x2, out, FACES | VERTICES)
    _same(out2, out)
    assert len(src2) == 0
    assert info2["degenerate_faces"] == info2["duplicate_faces"] == info2["nonmanifold_faces"] == 0
    assert info2["split_vertices"] == 0 and info2["nonmanifold_edges"] == 0
    assert (info2["boundary_edges"], info2["inconsistent_edges"]) == (info["boundary_edges"],
                                                                      info["inconsistent_edges"])


def test_two_holes_sharing_a_vertex_are_filled_after_the_repair():
    xyz, faces = grid_mesh(6, 6)
    # cells (1, 1) and (2, 2) of the 5 x 5 cells removed: two square holes that share the vertex at (2, 2)
    cell = np.concatenate([np.arange(25), np.arange(25)])
    faces = faces[~np.isin(cell, [1 * 5 + 1, 2 * 5 + 2])]
    add, info = fill_ref(xyz, faces, 22)
    assert info["filled"] == 1 and info["open_edges"] == 8    # only the rim; both holes stay open
    out, src, rinfo = repair_ref(xyz, faces, FACES | VERTICES)
    assert rinfo["split_vertices"] == 1 and rinfo["vertices_added"] == 1
    # each fan of the shared vertex touches both holes, so after the split the two squares are one loop of 8 edges
    add, info = fill_ref(apply_source(xyz, src), out, 22)
    assert info["holes"] == 2 and info["filled"] == 2 and info["open_edges"] == 0
