"""GPU checks of the connected components (scan3d_mesh_components_dev, scan3d_voxel_surface_components,
scan3d_get_surface_components): labels equal to scipy's, canonicalised to the header's id rule, on random meshes and
the worst cases for union depth and CAS contention, on the camera-grid mesh and on voxel surfaces; the compaction
bit for bit equal to the numpy expression of the header; the state rules, errors and launch counts; and the pieces of
the noise-free multi-view scene."""
import ctypes as C
import math

import numpy as np
import pytest

from gpu_common import s3
from test_components_ref import compact_ref, keep_ref, labels_ref, random_mesh
from test_gpu_align import CENTRE, SMALL, _ctx, _torch
from test_gpu_mesh import _edge_lengths
from test_gpu_mesh import _scene as _mesh_scene
from test_gpu_surface import _edges, _merge, _same, _surface
from test_gpu_voxel import C1, _read_ply, _voxel_size
from test_gpu_voxel import _scene as _voxel_scene

pytestmark = pytest.mark.gpu

F32 = np.float32
DEV_LAUNCHES = 7
CTX_LAUNCHES = 16


def _dev_labels(ctx, faces, n):
    """labels of the _dev entry, run twice: byte-identical, and equal to the reference"""
    t = _torch(np.ascontiguousarray(faces, np.int32).reshape(-1, 3))
    before = ctx.launch_count()
    a, ca = ctx.mesh_components_dev(t, n)
    assert ctx.launch_count() == before + DEV_LAUNCHES
    b, cb = ctx.mesh_components_dev(t, n)
    a, b = a.cpu().numpy(), b.cpu().numpy()
    assert ca == cb and a.tobytes() == b.tobytes()
    want, cw = labels_ref(faces, n)
    assert ca == cw and np.array_equal(a, want)
    return a, ca


def test_dev_labels_random_meshes():
    ctx = _ctx()
    rng = np.random.default_rng(0)
    for n, groups, per, iso in ((50, 3, 5, 4), (20000, 17, 300, 100), (300000, 1000, 50, 3000), (1 << 20, 1, 2000000, 0)):
        faces, free = random_mesh(rng, n, groups, per, iso)
        lab, c = _dev_labels(ctx, faces, n)
        assert c == groups + iso
    ctx.close()


def test_dev_labels_worst_cases():
    ctx = _ctx()
    rng = np.random.default_rng(1)
    # a long path over randomly permuted indices: the deepest union-find trees
    n = 1 << 22
    p = rng.permutation(n).astype(np.int32)
    path = np.stack([p[:-1], p[1:], p[1:]], 1)
    lab, c = _dev_labels(ctx, path[rng.permutation(len(path))], n)
    assert c == 1
    # a star: one vertex in every face, every union contends for the same root
    n, centre = 1 << 20, 777
    others = np.delete(np.arange(n, dtype=np.int32), centre)
    m = len(others) // 2
    star = np.stack([np.full(m, centre, np.int32), others[0:2 * m:2], others[1:2 * m:2]], 1)
    lab, c = _dev_labels(ctx, star, n + 5)                    # others[-1] and 5 more vertices are in no face
    assert c == 1 + 1 + 5
    # a 2000 x 2000 grid of two triangles per cell
    g = np.arange(2000 * 2000, dtype=np.int32).reshape(2000, 2000)
    a, b, cc, d = g[:-1, :-1].ravel(), g[:-1, 1:].ravel(), g[1:, :-1].ravel(), g[1:, 1:].ravel()
    grid = np.concatenate([np.stack([a, b, d], 1), np.stack([a, d, cc], 1)])
    lab, c = _dev_labels(ctx, grid, 2000 * 2000)
    assert c == 1
    # no faces; no vertices
    lab, c = _dev_labels(ctx, np.zeros((0, 3), np.int32), 1000)
    assert c == 1000 and np.array_equal(lab, np.arange(1000))
    lab, c = _dev_labels(ctx, np.zeros((0, 3), np.int32), 0)
    assert c == 0 and len(lab) == 0
    ctx.close()


def test_dev_labels_of_the_camera_grid_mesh():
    cfg, cal, _, stack, roi = _mesh_scene(SMALL)
    ctx = s3.Scan3D(cfg, 0, cal)
    n = ctx.reconstruct(stack, roi)
    ctx.build_mesh(math.inf)
    faces, _ = ctx.mesh()
    cut = 5.0 * float(np.median(_edge_lengths(ctx.points(), faces)))
    ctx.build_mesh(cut)
    faces, _ = ctx.mesh()
    lab, c = _dev_labels(ctx, faces, n)
    print(f"camera-grid mesh 640x480, max_edge {cut:.4f}: {n} points, {len(faces)} faces, {c} components")
    assert 0 < c < n
    ctx.close()


def _sphere(s, r, c):
    k = np.arange(int(400 * (r / s) ** 2)) + 0.5
    phi = np.arccos(1 - 2 * k / len(k))
    th = np.pi * (1 + 5 ** 0.5) * k
    u = np.stack([np.cos(th) * np.sin(phi), np.sin(th) * np.sin(phi), np.cos(phi)], 1)
    return (c + r * u).astype(F32), u.astype(F32), np.full(u.shape, 128, np.uint8)


S, RADIUS, CEN = F32(0.05), 2.0, np.array([0.3, -0.2, 0.1])
ISLANDS = np.array([[3.5, 0.0, 0.0], [0.0, 3.6, 0.2], [-3.4, -0.5, 0.0], [0.4, 0.3, 3.7]])


def _sphere_and_islands(ctx, islands=True):
    """the closed sphere of test_gpu_surface, plus single far-away voxels that each give a small patch"""
    p, n, c = _sphere(S, RADIUS, CEN)
    if islands:
        q = (CEN + ISLANDS).astype(F32)
        nq = np.array([[0, 0, 1.0], [1.0, 0, 0], [0, 0.6, 0.8], [0, 1.0, 0]], F32)
        p, n, c = np.concatenate([p, q]), np.concatenate([n, nq]), np.concatenate([c, np.full((4, 3), 9, np.uint8)])
    _merge(ctx, S, [(p, n, c)])
    return _surface(ctx)[1]


def _closed(mesh):
    xyz, _, _, faces = mesh
    e = _edges(faces)
    und, cnt = np.unique(np.sort(e, axis=1), axis=0, return_counts=True)
    assert (cnt == 2).all()
    assert len(xyz) - len(und) + len(faces) == 2


def _components(ctx, min_faces=0, max_components=0):
    before = ctx.launch_count()
    res = ctx.surface_components(min_faces, max_components)
    assert ctx.launch_count() == before + CTX_LAUNCHES
    return res, ctx.voxel_surface_mesh()


def test_closed_sphere_is_one_component():
    ctx = _ctx()
    raw = _sphere_and_islands(ctx, islands=False)
    _closed(raw)
    res, mesh = _components(ctx, 1, 0)
    assert res == dict(components=1, kept=1, vertices=len(raw[0]), faces=len(raw[3]), largest_faces=len(raw[3]))
    _same(mesh, raw)
    ctx.close()


def test_sphere_with_islands():
    ctx = _ctx()
    raw = _sphere_and_islands(ctx)
    xyz, _, _, faces = raw
    lab, c = _dev_labels(ctx, faces, len(xyz))
    vcount, fcount, _ = keep_ref(lab, faces, c, 0, 0)
    big = int(np.argmax(fcount))
    island_faces = np.delete(fcount, big)
    print(f"sphere + islands: {len(xyz)} vertices, {len(faces)} faces, {c} components; faces per component {fcount}")
    assert 1 < c <= 1 + 8 * len(ISLANDS) and fcount[big] > 10 * island_faces.max()
    for rule in ((0, 1), (int(island_faces.max()) + 1, 0)):
        res, mesh = _components(ctx, *rule)
        _, _, kept = keep_ref(lab, faces, c, *rule)
        assert kept.tolist() == [k == big for k in range(c)]
        want = compact_ref(raw, lab, kept)
        _same(mesh, want)
        _closed(mesh)
        assert res == dict(components=c, kept=1, vertices=len(want[0]), faces=len(want[3]), largest_faces=fcount[big])
        v, f, k = ctx.surface_component_table()
        assert np.array_equal(v, vcount) and np.array_equal(f, fcount) and np.array_equal(k, kept)
        _same(_surface(ctx)[1], raw)                     # a re-extraction brings the raw surface back
    # every rule against the reference, on the raw surface each time
    for rule in ((0, 0), (1, 0), (0, 2), (0, 3), (0, 100), (int(island_faces.min()), 2), (10 ** 12, 0)):
        _same(_surface(ctx)[1], raw)
        res, mesh = _components(ctx, *rule)
        _, _, kept = keep_ref(lab, faces, c, *rule)
        _same(mesh, compact_ref(raw, lab, kept))
        assert res["kept"] == kept.sum() and np.array_equal(ctx.surface_component_table()[2], kept)
    ctx.close()


def test_rules_state_errors_and_launch_counts(tmp_path):
    ctx = _ctx()
    L, h = ctx.L, ctx.h
    prm, out = s3.ComponentsParams(0, 0), s3.ComponentsResultC()
    vbuf, fbuf, kbuf = np.zeros(8, np.int64), np.zeros(8, np.int64), np.zeros(8, np.uint8)

    def run(p=prm):
        return L.scan3d_voxel_surface_components(h, C.byref(p), C.byref(out))

    def table():
        return L.scan3d_get_surface_components(h, vbuf.ctypes.data_as(C.c_void_p), fbuf.ctypes.data_as(C.c_void_p),
                                               kbuf.ctypes.data_as(C.c_void_p), 8)

    before = ctx.launch_count()
    assert run() == -3 and table() == -3                           # before any surface
    assert ctx.launch_count() == before
    raw = _sphere_and_islands(ctx)
    acc = b"".join(a.tobytes() for a in ctx.voxels())
    src = _torch((_sphere(S, RADIUS, CEN)[0][::5] + F32(0.01)).astype(F32))
    kw = dict(max_iterations=3, apply=False, stop_rotation=0.0, stop_translation=0.0)
    r1 = ctx.align_dev(src, 0.2, **kw)
    # (0, 0): every launch, the same bytes; then idempotence of (0, 1)
    res, mesh = _components(ctx)
    _same(mesh, raw)
    assert res["components"] == res["kept"] > 1 and table() == 0
    a = _components(ctx, 0, 1)
    b = _components(ctx, 0, 1)
    assert b[0] == dict(a[0], components=1)
    _same(b[1], a[1])
    # the PLY writer writes the cleaned surface
    path = str(tmp_path / "clean.ply")
    ctx.write_voxel_surface_ply(path, binary=True)
    head, body = _read_ply(path)
    nv, nf = len(a[1][0]), len(a[1][3])
    assert f"element vertex {nv}" in head and f"element face {nf}" in head
    vt = np.dtype([("xyz", "<f4", 3), ("n", "<f4", 3), ("rgb", "u1", 3)])
    ft = np.dtype([("k", "u1"), ("v", "<i4", 3)])
    v = np.frombuffer(body, vt, nv)
    f = np.frombuffer(body, ft, nf, offset=nv * vt.itemsize)
    _same((v["xyz"].copy(), v["n"].copy(), v["rgb"].copy(), f["v"].copy()), a[1])
    # the accumulator is unchanged and an align gives what it gave before
    assert b"".join(x.tobytes() for x in ctx.voxels()) == acc
    r2 = ctx.align_dev(src, 0.2, **kw)
    assert r1.T.tobytes() == r2.T.tobytes() and (r1.pairs_first, r1.rms_last) == (r2.pairs_first, r2.rms_last)
    assert table() == 0                                            # an align keeps the table ...
    _same(ctx.voxel_surface_mesh(), a[1])                          # ... and the surface
    # argument errors: nothing launched, the surface and the table stay
    before = ctx.launch_count()
    assert L.scan3d_voxel_surface_components(h, None, C.byref(out)) == -4
    assert L.scan3d_voxel_surface_components(h, C.byref(prm), None) == -4
    for bad in ((-1, 0), (0, -1), (-(2 ** 63), 5)):
        assert run(s3.ComponentsParams(*bad)) == -4, bad
    n = C.c_int64()
    t = _torch(np.array([[0, 1, 2]], np.int32))
    lab = _torch(np.zeros(4, np.int32))
    fp, lp = C.c_void_p(t.data_ptr()), C.c_void_p(lab.data_ptr())
    for args in ((fp, 1, 3, lp, None), (None, 1, 3, lp, C.byref(n)), (fp, 1, 3, None, C.byref(n)),
                 (fp, -1, 3, lp, C.byref(n)), (fp, 1, -1, lp, C.byref(n)), (fp, 1 << 31, 3, lp, C.byref(n)),
                 (fp, 1, 1 << 31, lp, C.byref(n)), (C.c_void_p(t.data_ptr() + 2), 1, 3, lp, C.byref(n)),
                 (fp, 1, 3, C.c_void_p(lab.data_ptr() + 1), C.byref(n))):
        assert L.scan3d_mesh_components_dev(h, *args) == -4, args
    assert ctx.launch_count() == before
    assert L.scan3d_mesh_components_dev(h, None, 0, 0, None, C.byref(n)) == 0 and n.value == 0
    assert table() == 0
    _same(ctx.voxel_surface_mesh(), a[1])
    # an index outside [0, n_vertices) is found on the device
    for bad in ([[0, 1, 3]], [[-1, 0, 1]], [[0, 0, 2 ** 31 - 1]]):
        tb = _torch(np.array(bad, np.int32))
        assert L.scan3d_mesh_components_dev(h, C.c_void_p(tb.data_ptr()), 1, 3, lp, C.byref(n)) == -4, bad
        assert b"outside" in L.scan3d_last_error(h)
    assert L.scan3d_mesh_components_dev(h, fp, 1, 3, lp, C.byref(n)) == 0 and n.value == 1
    assert table() == 0                                            # the _dev entry leaves the table alone
    # staleness: a re-extraction, then begin, add and finish
    _surface(ctx)
    assert table() == -3
    assert run() == 0 and table() == 0
    p, nn, c = _sphere(S, RADIUS, CEN)
    tp, tn, tc = _torch(p), _torch(nn), _torch(c)
    ctx.voxel_begin(S, len(p))
    assert table() == -3 and run() == -3                           # the surface went stale with the table
    ctx.voxel_add_dev(tp, tn, tc)
    ctx.voxel_finish()
    _surface(ctx)
    assert run() == 0 and table() == 0
    ctx.voxel_add_dev(tp, tn, tc)
    assert table() == -3 and run() == -3
    ctx.voxel_finish()
    _surface(ctx)
    assert run() == 0 and table() == 0
    ctx.voxel_finish()
    assert table() == -3 and run() == -3
    del src, t, lab, tp, tn, tc
    ctx.close()


def test_pieces_of_the_noise_free_scene():
    """The surface of eight merged views of the sphere alone (test_gpu_surface's scene): labels and compaction
    against the reference, and what keeping the largest component does to the distance from the sphere."""
    params = s3.default_synth_params(noise_sigma=0.0)
    cfg, cal, _, stack, roi, truth = _voxel_scene(C1, params=params, want_truth=True)
    centre = np.array(CENTRE)
    on_sphere = np.abs(np.linalg.norm(truth.astype(np.float64) - centre, axis=2) - 25.0) < 1e-3
    roi = (roi * on_sphere).astype(np.uint8)
    ctx = s3.Scan3D(cfg, 0, cal)
    s = None
    for k in range(8):
        ctx.set_registration(True, 45.0 * k, *CENTRE)
        n = ctx.reconstruct(stack, roi)
        ctx.build_mesh(math.inf)
        if s is None:
            s = _voxel_size(ctx.points())
            ctx.voxel_begin(s, 8 * n)
        ctx.voxel_add()
    ctx.voxel_finish()
    raw = _surface(ctx)[1]
    xyz, _, _, faces = raw
    lab, c = _dev_labels(ctx, faces, len(xyz))
    vcount, fcount, kept = keep_ref(lab, faces, c, 0, 1)
    res, mesh = _components(ctx, 0, 1)
    _same(mesh, compact_ref(raw, lab, kept))
    assert res["components"] == c and res["largest_faces"] == fcount.max()
    v, f, k = ctx.surface_component_table()
    assert np.array_equal(v, vcount) and np.array_equal(f, fcount) and np.array_equal(k, kept)

    def off(m):
        return float(np.abs(np.linalg.norm(m[0].astype(np.float64) - centre, axis=1) - 25.0).max())
    print(f"voxel {s:.4f}: {len(xyz)} vertices, {len(faces)} faces, {c} components; the largest holds "
          f"{fcount.max() / max(len(faces), 1):.5f} of the faces and {vcount[np.argmax(fcount)]} vertices; "
          f"max |r - 25| {off(raw):.4f} before, {off(mesh):.4f} after keeping it")
    # measured on a B200 (1000 W power limit): voxel 0.1318, 581 124 vertices, 1 121 566 faces, 8 919 components; the
    # largest holds 0.98899 of the faces and 557 592 vertices; max |r - 25| 2.2338 before, 0.4808 after keeping it.
    # The pieces cut loose from the sphere carry the silhouette's worst outliers.
    ctx.close()
