"""GPU checks of the surface extraction (scan3d_voxel_surface): bit parity with the restatement of
tests/test_surface_math_host.py on device-added clouds, a dense sphere and the ctx route; a closed, oriented sphere;
the invariances the contract promises; edge cases; state rules, errors, launch counts and overflow; PLY files; and
the geometry of the noise-free multi-view scene."""
import ctypes as C
import math

import numpy as np
import pytest

from gpu_common import s3
from test_gpu_align import CENTRE, SMALL, _ctx, _scene, _spacing, _torch
from test_gpu_voxel import C1, _read_ply, _voxel_size
from test_gpu_voxel import _scene as _voxel_scene
from test_surface_math_host import extract_ref, model_ijk, sphere_model

pytestmark = pytest.mark.gpu

F32 = np.float32
LAUNCHES = 3 + 8 + 1


def _surface(ctx, **kw):
    res = ctx.voxel_surface(**kw)
    return res, ctx.voxel_surface_mesh()


def _same(got, want):
    for x, y in zip(got, want):
        assert x.shape == y.shape and x.dtype == y.dtype
        assert np.array_equal(x.view(np.uint8), y.view(np.uint8))


def _check_parity(ctx, added, s, R):
    """the ctx's surface against the restatement, the model's merge indices computed from the added points"""
    mxyz, mnrm, mrgb, _ = ctx.voxels()
    # a voxel's 27 cells have 64 corners: 64 per voxel always suffices
    res, mesh = _surface(ctx, max_distance=R, max_points=max(64 * len(mxyz), 1))
    ijk = model_ijk(added, s)
    assert len(ijk) == len(mxyz)
    want = extract_ref(mxyz, mnrm, mrgb, ijk, s, R)
    _same(mesh, want[:4])
    assert (res["vertices"], res["faces"], res["lattice_points"], res["undefined_points"]) == \
        (len(want[0]), len(want[3]), want[4], want[5])
    return res, mesh


def _cloud(rng, n, r=3.0, noise=0.02):
    u = rng.normal(size=(n, 3))
    u /= np.linalg.norm(u, axis=1, keepdims=True)
    p = (np.array([0.4, -0.3, 0.2]) + (r + noise * rng.normal(size=(n, 1))) * u).astype(F32)
    nrm = (u + 0.1 * rng.normal(size=u.shape)).astype(F32)
    nrm[rng.random(n) < 0.02] = 0
    return p, nrm, rng.integers(0, 256, (n, 3), dtype=np.uint8)


def _merge(ctx, s, parts, max_voxels=None):
    ctx.voxel_begin(s, max_voxels or sum(len(p[0]) for p in parts))
    keep = []
    for p in parts:
        keep.append([_torch(a) for a in p])
        ctx.voxel_add_dev(*keep[-1])
    ctx.voxel_finish()
    ctx.sync()


@pytest.mark.parametrize("seed", [0, 1])
def test_parity_random_clouds(seed):
    rng = np.random.default_rng(seed)
    ctx = _ctx()
    s = F32(0.2)
    p, n, c = _cloud(rng, 40000)
    _merge(ctx, s, [(p, n, c)])
    for R in (F32(2 * s), F32(3.3 * s)):
        res, _ = _check_parity(ctx, p, s, R)
        assert res["faces"] > 1000
    ctx.close()


def test_parity_dense_sphere():
    ctx = _ctx()
    s = F32(0.1)
    p, n, c, _ = sphere_model(s, 2.5)
    _merge(ctx, s, [(p, n, c)])
    _check_parity(ctx, p, s, F32(2 * s))
    ctx.close()


def test_parity_ctx_route_640x480():
    cfg, cal, stack, roi = _scene(SMALL)
    ctx = s3.Scan3D(cfg, 0, cal)
    ctx.set_texture(np.random.default_rng(5).integers(0, 256, (cfg.H, cfg.W, 3), dtype=np.uint8))
    added = []
    for k, theta in enumerate((0.0, 20.0, 40.0)):
        ctx.set_registration(True, theta, *CENTRE)
        n = ctx.reconstruct(stack, roi)
        ctx.build_mesh(math.inf)
        if k == 0:
            s = F32(2.0 * _spacing(ctx))
            ctx.voxel_begin(s, 3 * n)
        added.append(ctx.points())
        ctx.voxel_add()
    ctx.voxel_finish()
    res, _ = _check_parity(ctx, np.concatenate(added), s, F32(2 * s))
    assert res["faces"] > 1000
    ctx.close()


def _edges(faces):
    e = np.concatenate([faces[:, [0, 1]], faces[:, [1, 2]], faces[:, [2, 0]]])
    return e


def test_closed_and_oriented_sphere():
    ctx = _ctx()
    s, r, c = F32(0.05), 2.0, np.array([0.3, -0.2, 0.1])
    k = np.arange(int(400 * (r / s) ** 2)) + 0.5
    phi = np.arccos(1 - 2 * k / len(k))
    th = np.pi * (1 + 5 ** 0.5) * k
    u = np.stack([np.cos(th) * np.sin(phi), np.sin(th) * np.sin(phi), np.cos(phi)], 1)
    _merge(ctx, s, [((c + r * u).astype(F32), u.astype(F32), np.full(u.shape, 128, np.uint8))])
    res, (xyz, nrm, rgb, faces) = _surface(ctx)                  # R = 2 s, the default max_points
    V, Fn = len(xyz), len(faces)
    e = _edges(faces)
    und, cnt = np.unique(np.sort(e, axis=1), axis=0, return_counts=True)
    assert (cnt == 2).all()                                        # every edge in exactly two faces ...
    assert len(np.unique(e, axis=0)) == len(e)                     # ... used once in each direction
    assert np.array_equal(np.unique(faces), np.arange(V))          # every vertex used
    assert V - len(und) + Fn == 2
    # one component: union-find over the edges
    parent = np.arange(V)

    def find(a):
        while parent[a] != a:
            parent[a] = parent[parent[a]]
            a = parent[a]
        return a
    for a, b in und:
        ra, rb = find(a), find(b)
        if ra != rb:
            parent[ra] = rb
    assert len({find(a) for a in range(V)}) == 1
    x = xyz.astype(np.float64)
    fn = np.cross(x[faces[:, 1]] - x[faces[:, 0]], x[faces[:, 2]] - x[faces[:, 0]])
    assert ((fn * (x[faces].mean(1) - c)).sum(1) > 0).all()
    assert ((nrm.astype(np.float64) * (x - c)).sum(1) > 0).all()
    dev = np.abs(np.linalg.norm(x - c, axis=1) - r)
    print(f"sphere r {r} s {s}: {V} vertices, {Fn} faces, {res['lattice_points']} lattice points; "
          f"max | |v - c| - r | = {dev.max():.3g}")
    # the voxel centroids lie within ~s^2 / (8 r) of the sphere and the corner values are exact plane distances to
    # them, so the vertices stay within a small fraction of the voxel (measured on a B200: 4.46e-4 = 0.009 s)
    assert dev.max() < 0.1 * s
    ctx.close()


def test_invariances():
    import torch
    rng = np.random.default_rng(7)
    s, R = F32(0.2), F32(0.4)
    p, n, c = _cloud(rng, 30000)
    ctx = _ctx()
    _merge(ctx, s, [(p, n, c)])
    before = b"".join(a.tobytes() for a in ctx.voxels())
    a = _surface(ctx, max_distance=R)
    b = _surface(ctx, max_distance=R)
    assert a[0] == b[0]
    _same(b[1], a[1])
    assert b"".join(x.tobytes() for x in ctx.voxels()) == before    # the extraction never changes the accumulator
    fresh = _ctx()
    _merge(fresh, s, [(p, n, c)])
    _same(_surface(fresh, max_distance=R)[1], a[1])
    # chunks: the same merge, so the same bytes
    _merge(fresh, s, [(p[:7000], n[:7000], c[:7000]), (p[7000:], n[7000:], c[7000:])], max_voxels=len(p))
    _same(_surface(fresh, max_distance=R)[1], a[1])
    # another add order: the same vertex and face sets, in another order
    perm = rng.permutation(len(p))
    _merge(fresh, s, [(p[perm], n[perm], c[perm])])
    mo = _surface(fresh, max_distance=R)[1]

    def canon(mesh):
        xyz, nrm, rgb, faces = mesh
        verts = [tuple(xyz[i].view(np.uint32)) + tuple(nrm[i].view(np.uint32)) + tuple(rgb[i]) for i in range(len(xyz))]
        tris = set()
        for f in faces:
            t = [verts[i] for i in f]
            k = int(np.argmin([hash(v) for v in t]))
            tris.add(tuple(t[k:] + t[:k]))
        return sorted(verts), tris
    ca, cb = canon(a[1]), canon(mo)
    assert ca[0] == cb[0] and ca[1] == cb[1]
    fresh.close()
    # an align after an extraction gives the result it gives without one
    src = _torch((p[::3] + F32(0.05)).astype(F32))
    kw = dict(max_iterations=4, apply=False, stop_rotation=0.0, stop_translation=0.0)
    r1 = ctx.align_dev(src, 1.0, **kw)
    _surface(ctx, max_distance=R)
    r2 = ctx.align_dev(src, 1.0, **kw)
    assert r1.T.tobytes() == r2.T.tobytes() and (r1.pairs_first, r1.rms_last) == (r2.pairs_first, r2.rms_last)
    # ... and leaves the surface in place
    _same(ctx.voxel_surface_mesh(), a[1])
    del src
    torch.cuda.synchronize()
    ctx.close()


def test_edge_cases():
    ctx = _ctx()
    rng = np.random.default_rng(3)
    s = F32(0.2)
    p, n, c = _cloud(rng, 20000)
    # a normal-free model: no surface
    _merge(ctx, s, [(p, np.zeros_like(n), c)])
    res, mesh = _surface(ctx, max_distance=F32(0.4))
    assert res == dict(vertices=0, faces=0, lattice_points=0, undefined_points=0)
    assert all(len(a) == 0 for a in mesh)
    # a single model voxel: a patch of its plane that ends within R
    q = np.array([[0.25, 0.31, 0.27]], F32)
    _merge(ctx, s, [(q, np.array([[0, 0, 1.0]], F32), np.array([[1, 2, 3]], np.uint8))])
    res, (xyz, _, rgb, faces) = _surface(ctx, max_distance=F32(0.5), max_points=64)
    assert res["vertices"] > 0 and res["faces"] > 0 and (rgb == [[1, 2, 3]]).all()
    assert (np.linalg.norm(xyz.astype(np.float64) - q, axis=1) <= 0.5 + math.sqrt(3) * s).all()
    _check_parity(ctx, q, s, F32(0.5))
    # too small an R: undefined corners, and no face through one (parity with the restatement)
    _merge(ctx, s, [(p, n, c)])
    res, _ = _check_parity(ctx, p, s, F32(0.6 * s))
    assert res["undefined_points"] > 0
    ctx.close()


def test_rules_errors_launch_counts_and_overflow():
    ctx = _ctx()
    L, h = ctx.L, ctx.h
    prm, out = s3.SurfaceParams(0.4, 1 << 20), s3.SurfaceResultC()
    xyz = np.zeros((4, 3), F32)

    def run(p=prm):
        return L.scan3d_voxel_surface(h, C.byref(p), C.byref(out))

    def get():
        return L.scan3d_get_voxel_surface(h, xyz.ctypes.data_as(C.c_void_p), None, None, None, 4, 0)

    assert run() == -3                                             # before begin
    rng = np.random.default_rng(4)
    p, n, c = _cloud(rng, 20000)
    tp, tn, tc = _torch(p), _torch(n), _torch(c)
    ctx.voxel_begin(0.2, 100000)
    assert run() == -3                                             # before the first finish
    assert get() == -3 and L.scan3d_write_voxel_surface_ply(h, b"/nonexistent/x.ply", 0) == -3
    ctx.voxel_add_dev(tp, tn, tc)
    ctx.voxel_finish()
    before = ctx.launch_count()
    assert run() == 0 and out.faces > 0
    assert ctx.launch_count() == before + LAUNCHES
    assert get() == 0
    # argument errors
    assert L.scan3d_voxel_surface(h, None, C.byref(out)) == -4
    assert L.scan3d_voxel_surface(h, C.byref(prm), None) == -4
    for bad in ((0.0, 100), (-1.0, 100), (math.nan, 100), (math.inf, 100), (0.4, 0), (0.4, 1 << 31), (0.4, -5)):
        assert run(s3.SurfaceParams(*bad)) == -4, bad
    assert L.scan3d_write_voxel_surface_ply(h, None, 0) == -4
    assert get() == 0                                              # an argument error keeps the surface
    # staleness: add, finish, begin; an align does not
    ctx.align_dev(tp, 1.0, max_iterations=2, apply=False)
    assert get() == 0
    ctx.voxel_add_dev(tp, tn, tc)
    assert get() == -3 and run() == -3                             # an add since the last finish
    ctx.voxel_finish()
    assert get() == -3
    assert run() == 0 and get() == 0
    ctx.voxel_finish()
    assert get() == -3
    assert run() == 0
    ctx.voxel_begin(0.2, 100000)
    assert get() == -3
    ctx.voxel_add_dev(tp, tn, tc)
    ctx.voxel_finish()
    # max_points overflow: reported, no surface, the same launches; a larger max_points recovers
    assert run() == 0
    want = ctx.voxel_surface_mesh()
    lattice = out.lattice_points
    before = ctx.launch_count()
    assert run(s3.SurfaceParams(0.4, lattice - 1)) == -1
    assert b"max_points" in L.scan3d_last_error(h)
    assert ctx.launch_count() == before + LAUNCHES - 1
    assert get() == -3
    for small in (1, 100):
        assert run(s3.SurfaceParams(0.4, small)) == -1
    assert run(s3.SurfaceParams(0.4, lattice)) == 0 and out.lattice_points == lattice
    _same(ctx.voxel_surface_mesh(), want)
    # an overflowed accumulator
    ctx.voxel_begin(0.2, 10)
    ctx.voxel_add_dev(tp, tn, tc)
    ctx.voxel_finish()
    assert run() == -1 and b"max_voxels" in L.scan3d_last_error(h)
    assert get() == -3
    # an empty model after a begin with nothing added
    ctx.voxel_begin(0.2, 10)
    ctx.voxel_finish()
    assert run() == 0 and (out.vertices, out.faces) == (0, 0)
    ctx.close()


def test_ply_files(tmp_path):
    ctx = _ctx()
    rng = np.random.default_rng(6)
    p, n, c = _cloud(rng, 20000)
    _merge(ctx, F32(0.2), [(p, n, c)])
    _surface(ctx)
    xyz, nrm, rgb, faces = ctx.voxel_surface_mesh()
    nv, nf = len(xyz), len(faces)
    assert nf > 0
    for binary in (0, 1):
        path = str(tmp_path / f"surface{binary}.ply")
        ctx.write_voxel_surface_ply(path, binary=bool(binary))
        head, body = _read_ply(path)
        assert head == ["ply", "format %s 1.0" % ("binary_little_endian" if binary else "ascii"), "comment scan3d-b200",
                        f"element vertex {nv}", "property float x", "property float y", "property float z",
                        "property float nx", "property float ny", "property float nz", "property uchar red",
                        "property uchar green", "property uchar blue", f"element face {nf}",
                        "property list uchar int vertex_indices"]
        if binary:
            vt = np.dtype([("xyz", "<f4", 3), ("n", "<f4", 3), ("rgb", "u1", 3)])
            ft = np.dtype([("k", "u1"), ("v", "<i4", 3)])
            assert len(body) == nv * vt.itemsize + nf * ft.itemsize
            v = np.frombuffer(body, vt, nv)
            f = np.frombuffer(body, ft, nf, offset=nv * vt.itemsize)
            px, pn, pc, pf = v["xyz"], v["n"], v["rgb"], f["v"]
            assert (f["k"] == 3).all()
        else:
            lines = body.decode().split("\n")
            assert lines[-1] == "" and len(lines) == nv + nf + 1
            v = np.array([ln.split() for ln in lines[:nv]])
            px, pn = v[:, :3].astype(np.float64).astype(F32), v[:, 3:6].astype(np.float64).astype(F32)
            pc = v[:, 6:].astype(np.int64)
            f = np.array([ln.split() for ln in lines[nv:nv + nf]]).astype(np.int64)
            assert (f[:, 0] == 3).all()
            pf = f[:, 1:]
        assert np.array_equal(px.view(np.uint32), xyz.view(np.uint32))
        assert np.array_equal(pn.view(np.uint32), nrm.view(np.uint32))
        assert np.array_equal(pc, rgb) and np.array_equal(pf, faces)
    ctx.close()


def test_geometry_of_the_noise_free_scene():
    """The surface of eight merged views of the sphere alone (the voxel test's scene) lies on the sphere within the
    merge's own bound and faces outward."""
    params = s3.default_synth_params(noise_sigma=0.0)
    cfg, cal, _, stack, roi, truth = _voxel_scene(C1, params=params, want_truth=True)
    centre = np.array(CENTRE)
    on_sphere = np.abs(np.linalg.norm(truth.astype(np.float64) - centre, axis=2) - 25.0) < 1e-3
    roi = (roi * on_sphere).astype(np.uint8)
    ctx = s3.Scan3D(cfg, 0, cal)
    err, s = 0.0, None
    for k in range(8):
        ctx.set_registration(True, 45.0 * k, *CENTRE)
        n = ctx.reconstruct(stack, roi)
        ctx.build_mesh(math.inf)
        pts = ctx.points().astype(np.float64)
        err = max(err, float(np.abs(np.linalg.norm(pts - centre, axis=1) - 25.0).max()))
        if s is None:
            s = _voxel_size(ctx.points())
            ctx.voxel_begin(s, 8 * n)
        ctx.voxel_add()
    ctx.voxel_finish()
    res, (xyz, nrm, _, faces) = _surface(ctx)
    x = xyz.astype(np.float64)
    off = float(np.abs(np.linalg.norm(x - centre, axis=1) - 25.0).max())
    outward = float(((nrm.astype(np.float64) * (x - centre)).sum(1) > 0).mean())
    fn = np.cross(x[faces[:, 1]] - x[faces[:, 0]], x[faces[:, 2]] - x[faces[:, 0]])
    face_out = float(((fn * (x[faces].mean(1) - centre)).sum(1) > 0).mean())
    band = np.abs(np.linalg.norm(x - centre, axis=1) - 25.0) <= math.sqrt(3) * s
    out_band = float(((nrm[band].astype(np.float64) * (x[band] - centre)).sum(1) > 0).mean())
    print(f"voxel {s:.4f}: {res}; max |r - 25| {off:.4f} (single-view points {err:.4f}); outward vertex normals "
          f"{outward:.5f} ({out_band:.5f} of the {band.mean():.4f} within sqrt(3) s of the sphere), faces "
          f"{face_out:.5f}; lattice points per voxel {res['lattice_points'] / ctx.voxel_count()[0]:.3f}")
    # measured on a B200: voxel 0.1318, 581 124 vertices, 1 121 566 faces; max |r - 25| 2.2338 against 2.1888 for the
    # single-view points; outward vertex normals 0.98960, faces 0.99310.  The inward ones sit on the silhouette's
    # c_p_map staircase (the points up to 2.19 off the sphere), where the merged normals themselves turn away.
    assert off <= math.sqrt(3) * s + err
    assert outward > 0.985 and face_out > 0.99
    assert out_band > 0.99
    ctx.close()
