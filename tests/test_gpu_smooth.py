"""GPU checks of the surface smoothing (scan3d_voxel_surface_smooth, scan3d_mesh_smooth_dev): bit parity with smooth_ref
of tests/test_smooth_ref.py at iterations 0, 1 and 10 with mu = -0.53 and 0, on surfaces of random clouds and the
dense sphere, after components, after decimation and through the 640x480 ctx route; the dev route on the ctx's own
camera-grid mesh and on hand-made meshes (degenerate and non-manifold faces, isolated vertices, a star); every call
twice, byte-identical.  Also the state rules, every argument error, errors found on the device, the launch count and
the normals of a smoothed sphere.  The ABI check needs no GPU."""
import ctypes as C
import importlib
import math

import numpy as np
import pytest

from test_gpu_align import CENTRE, SMALL, _ctx, _scene, _spacing, _torch
from test_gpu_components import CEN, RADIUS, S, _sphere, _sphere_and_islands
from test_gpu_mesh import _scene as _mesh_scene
from test_gpu_surface import _cloud, _merge, _same, _surface
from test_gpu_voxel import _read_ply
from test_smooth_ref import SmoothError, grid_mesh, noisy_sphere, odd_mesh, passes_of, smooth_ref
from test_surface_math_host import sphere_model

s3 = importlib.import_module("3dscan_b200")
gpu = pytest.mark.gpu

F32 = np.float32
BUILD, END = 7, 2
CASES = [(0, -0.53), (1, -0.53), (10, -0.53), (0, 0.0), (1, 0.0), (10, 0.0)]
ARG, STATE, CONFIG = -4, -3, -1


def launches(iterations, mu):
    return BUILD + passes_of(iterations, mu) + END


def test_abi_symbols_resolve():
    L = C.CDLL(s3.cuda_lib()._name)
    for name in ("scan3d_voxel_surface_smooth", "scan3d_mesh_smooth_dev"):
        assert getattr(L, name)
    assert C.sizeof(s3.SmoothParams) == 12 and C.sizeof(s3.SmoothResultC) == 48
    assert s3.SmoothResultC.max_displacement.offset == 40


def _want(raw, it, mu, lam=0.5):
    xyz, nrm, info = smooth_ref(raw[0], raw[1], raw[3], it, lam, mu)
    return (xyz, nrm, raw[2], raw[3]), info


def _smooth(ctx, it, mu, lam=0.5):
    before = ctx.launch_count()
    res = ctx.surface_smooth(it, lam, mu)
    assert ctx.launch_count() == before + launches(it, mu)
    return res, ctx.voxel_surface_mesh()


def _check(ctx, raw, extract, cases=CASES):
    """for each case: extract again, smooth, compare with the reference; the last case twice"""
    out = None
    for it, mu in cases + cases[-1:]:
        _same(extract(), raw)
        res, mesh = _smooth(ctx, it, mu)
        want, info = _want(raw, it, mu)
        _same(mesh, want)
        assert res == info, (it, mu)
        if out is not None and (it, mu) == out[0]:
            _same(mesh, out[1])
        out = ((it, mu), mesh)
        print(f"iterations {it}, mu {mu}: {res}")


@gpu
@pytest.mark.parametrize("seed", [0, 1])
def test_parity_random_clouds(seed):
    rng = np.random.default_rng(seed)
    ctx = _ctx()
    s = F32(0.2)
    p, n, c = _cloud(rng, 40000)
    _merge(ctx, s, [(p, n, c)])
    raw = _surface(ctx, max_distance=F32(2 * s))[1]
    assert len(raw[3]) > 1000
    _check(ctx, raw, lambda: _surface(ctx, max_distance=F32(2 * s))[1])
    ctx.close()


@gpu
def test_parity_dense_sphere():
    ctx = _ctx()
    s = F32(0.1)
    p, n, c, _ = sphere_model(s, 2.5)
    _merge(ctx, s, [(p, n, c)])
    raw = _surface(ctx)[1]
    _check(ctx, raw, lambda: _surface(ctx)[1])
    ctx.close()


@gpu
def test_parity_ctx_route_640x480():
    cfg, cal, stack, roi = _scene(SMALL)
    ctx = s3.Scan3D(cfg, 0, cal)
    ctx.set_texture(np.random.default_rng(5).integers(0, 256, (cfg.H, cfg.W, 3), dtype=np.uint8))
    for k, theta in enumerate((0.0, 20.0, 40.0)):
        ctx.set_registration(True, theta, *CENTRE)
        n = ctx.reconstruct(stack, roi)
        ctx.build_mesh(math.inf)
        if k == 0:
            s = F32(2.0 * _spacing(ctx))
            ctx.voxel_begin(s, 3 * n)
        ctx.voxel_add()
    ctx.voxel_finish()
    raw = _surface(ctx)[1]
    assert len(raw[3]) > 1000
    _check(ctx, raw, lambda: _surface(ctx)[1])
    ctx.close()


@gpu
def test_parity_after_components_and_after_decimation():
    ctx = _ctx()
    _sphere_and_islands(ctx)

    def largest():
        _surface(ctx)
        ctx.surface_components(0, 1)
        return ctx.voxel_surface_mesh()

    def simplified():
        _surface(ctx)
        ctx.surface_decimate(F32(4 * S))
        return ctx.voxel_surface_mesh()
    for extract in (largest, simplified):
        raw = extract()
        _check(ctx, raw, extract, [(1, -0.53), (10, 0.0), (10, -0.53)])
    # smoothing twice is smoothing the smoothed surface
    raw = largest()
    ctx.surface_smooth(3)
    once = ctx.voxel_surface_mesh()
    _same(once, _want(raw, 3, -0.53)[0])
    ctx.surface_smooth(2, 0.3, 0.0)
    _same(ctx.voxel_surface_mesh(), _want(once, 2, 0.0, 0.3)[0])
    ctx.close()


def _dev(ctx, xyz, nrm, faces, it=10, lam=0.5, mu=-0.53):
    """the dev route on copies of the arrays, twice; returns (xyz, nrm, result) after the first"""
    outs = []
    for _ in range(2):
        tx, tf = _torch(xyz), _torch(np.ascontiguousarray(faces, np.int32).reshape(-1, 3))
        tn = None if nrm is None else _torch(nrm)
        before = ctx.launch_count()
        res = ctx.mesh_smooth_dev(tx, tf, tn, it, lam, mu)
        assert ctx.launch_count() == before + launches(it, mu)
        outs.append((tx.cpu().numpy(), None if tn is None else tn.cpu().numpy(), res))
        assert np.array_equal(tf.cpu().numpy(), np.asarray(faces, np.int32).reshape(-1, 3))
    for a, b in zip(outs[0][:2], outs[1][:2]):
        if a is not None:
            _same((a,), (b,))
    assert outs[0][2] == outs[1][2]
    return outs[0]


def _dev_check(ctx, xyz, nrm, faces, cases=CASES):
    for it, mu in cases:
        gx, gn, res = _dev(ctx, xyz, nrm, faces, it, 0.5, mu)
        wx, wn, info = smooth_ref(xyz, nrm, faces, it, 0.5, mu)
        _same((gx,), (wx,))
        if nrm is not None:
            _same((gn,), (wn,))
        assert res == info, (it, mu)


@gpu
def test_dev_route_hand_made_meshes():
    ctx = _ctx()
    rng = np.random.default_rng(9)
    xyz, nrm, faces = odd_mesh(rng, 3000, 7000)
    _dev_check(ctx, xyz, nrm, faces)
    _dev_check(ctx, xyz, None, faces, [(10, -0.53)])
    gx, gf = grid_mesh(300, 200, 0.01, rng.normal(size=(200, 300)) * 1e-3)
    _dev_check(ctx, gx, np.zeros_like(gx), gf, [(10, -0.53), (50, 0.0)])
    sx, su, sf = noisy_sphere(5, 20.0, (100.0, -50.0, 7.0), 0.05, 1)
    _dev_check(ctx, sx, su, sf, [(10, -0.53), (30, -0.53)])
    # an empty mesh, and vertices without faces
    _dev_check(ctx, np.zeros((0, 3), F32), np.zeros((0, 3), F32), np.zeros((0, 3), np.int32), [(10, -0.53)])
    _dev_check(ctx, xyz[:100], nrm[:100], np.zeros((0, 3), np.int32), [(10, -0.53)])
    ctx.close()


@gpu
def test_dev_route_star_and_hubs():
    """test_gpu_components' star (one vertex in 524 287 faces whose spokes are each in one face, so it is held), and a
    closed fan of as many faces around one free centre, whose row the warp sums together"""
    ctx = _ctx()
    rng = np.random.default_rng(2)
    n, centre = 1 << 20, 777
    others = np.delete(np.arange(n, dtype=np.int32), centre)
    m = len(others) // 2
    star = np.stack([np.full(m, centre, np.int32), others[0:2 * m:2], others[1:2 * m:2]], 1)
    ring = others[:m]
    fan = np.stack([np.full(m, centre, np.int32), ring, np.roll(ring, -1)], 1)
    xyz = rng.normal(size=(n, 3)).astype(F32)
    nrm = rng.normal(size=(n, 3)).astype(F32)
    for faces, centre_held in ((star, True), (fan, False)):
        gx, gn, res = _dev(ctx, xyz, nrm, faces, 2)
        wx, wn, info = smooth_ref(xyz, nrm, faces, 2)
        _same((gx, gn), (wx, wn))
        assert res == info
        assert np.array_equal(gx[centre], xyz[centre]) == centre_held
    assert info["held_vertices"] == m
    ctx.close()


@gpu
def test_dev_route_camera_grid_mesh_in_place(tmp_path):
    """the ctx's own camera-grid mesh smoothed on its own buffers, read back through write_mesh_ply"""
    cfg, cal, _, stack, roi = _mesh_scene(SMALL)
    ctx = s3.Scan3D(cfg, 0, cal)
    ctx.set_texture(np.random.default_rng(5).integers(0, 256, (cfg.H, cfg.W, 3), dtype=np.uint8))
    L, h = ctx.L, ctx.h
    vt = np.dtype([("xyz", "<f4", 3), ("n", "<f4", 3), ("rgb", "u1", 3)])
    ft = np.dtype([("k", "u1"), ("i", "<i4", 3)])
    results = []
    for run in range(2):
        n = ctx.reconstruct(stack, roi)
        ctx.build_mesh(math.inf)
        pts, rgb = ctx.points(want_rgb=True)
        faces, nrm = ctx.mesh()
        p = s3.SmoothParams(10, 0.5, -0.53)
        r = s3.SmoothResultC()
        before = ctx.launch_count()
        assert L.scan3d_mesh_smooth_dev(h, L.scan3d_device_points(h), L.scan3d_device_point_normals(h), n,
                                        L.scan3d_device_mesh_faces(h), len(faces), C.byref(p), C.byref(r)) == 0
        assert ctx.launch_count() == before + launches(10, -0.53)
        path = str(tmp_path / f"smoothed{run}.ply")
        ctx.write_mesh_ply(path, binary=True)
        head, body = _read_ply(path)
        assert f"element vertex {n}" in head and f"element face {len(faces)}" in head
        v = np.frombuffer(body, vt, n)
        f = np.frombuffer(body, ft, len(faces), offset=n * vt.itemsize)
        wx, wn, info = smooth_ref(pts, nrm, faces, 10)
        _same((v["xyz"].copy(), v["n"].copy(), v["rgb"].copy(), f["i"].copy()), (wx, wn, rgb, faces))
        res = s3.Scan3D._smooth_result(r)
        assert res == info
        results.append(body)
        print(f"camera-grid mesh 640x480: {n} points, {len(faces)} faces, {res}")
    assert results[0] == results[1]
    assert info["held_vertices"] > 0
    ctx.close()


@gpu
def test_normals_of_a_smoothed_sphere_are_closer_to_radial():
    """the face normals of a noisy sphere's surface (iterations = 0 only recomputes them) against those after 10"""
    ctx = _ctx()
    rng = np.random.default_rng(4)
    p, n, c = _sphere(S, RADIUS, CEN)
    p = (p + rng.normal(size=p.shape) * 0.3 * S).astype(F32)
    _merge(ctx, S, [(p, n, c)])

    def radial_cos(it):
        _surface(ctx)
        ctx.surface_smooth(it)
        x, nn, _, _ = ctx.voxel_surface_mesh()
        r = x.astype(np.float64) - CEN
        return float(np.mean(np.sum(nn * r, 1) / np.linalg.norm(r, axis=1)))
    before, after = radial_cos(0), radial_cos(10)
    print(f"noisy sphere: mean cos(face normal, radial) {before:.5f} unsmoothed, {after:.5f} after 10 iterations")
    assert after > before
    ctx.close()


@gpu
def test_rules_state_errors_and_launch_count():
    ctx = _ctx()
    L, h = ctx.L, ctx.h
    out = s3.SmoothResultC()

    def run(it=10, lam=0.5, mu=-0.53, res=out):
        p = s3.SmoothParams(it, lam, mu)
        return L.scan3d_voxel_surface_smooth(h, C.byref(p), C.byref(res) if res is not None else None)

    before = ctx.launch_count()
    assert run() == STATE                                          # before any surface
    assert ctx.launch_count() == before
    raw = _sphere_and_islands(ctx)
    acc = b"".join(a.tobytes() for a in ctx.voxels())
    # argument errors: nothing launched, the surface stays byte-identical
    bad = [dict(it=-1), dict(it=4097), dict(lam=0.0), dict(lam=-0.5), dict(lam=1.0001), dict(lam=math.nan),
           dict(lam=math.inf), dict(mu=0.01), dict(mu=-1.001), dict(mu=math.nan), dict(mu=-math.inf)]
    before = ctx.launch_count()
    for kw in bad:
        assert run(**kw) == ARG, kw
    assert L.scan3d_voxel_surface_smooth(None, C.byref(s3.SmoothParams(1, 0.5, 0.0)), C.byref(out)) == ARG
    assert L.scan3d_voxel_surface_smooth(h, None, C.byref(out)) == ARG
    assert run(res=None) == ARG
    assert ctx.launch_count() == before
    _same(ctx.voxel_surface_mesh(), raw)
    # the limits of the range are accepted
    for kw in (dict(it=0), dict(lam=1.0, mu=-1.0), dict(it=1, lam=1e-30, mu=-0.0)):
        _surface(ctx)
        assert run(**kw) == 0, kw
    # the component table stays valid; decimation is refused until a new extraction
    _surface(ctx)
    comp = ctx.surface_components(0, 0)
    table = ctx.surface_component_table()
    res, mesh = _smooth(ctx, 10, -0.53)
    _same(mesh, _want(raw, 10, -0.53)[0])
    for a, b in zip(ctx.surface_component_table(), table):
        assert np.array_equal(a, b)
    before = ctx.launch_count()
    assert L.scan3d_voxel_surface_decimate(h, F32(4 * S), C.byref(s3.DecimateResultC())) == STATE
    assert b"smoothed" in L.scan3d_last_error(h) and ctx.launch_count() == before
    _same(ctx.voxel_surface_mesh(), mesh)
    comp2 = ctx.surface_components(0, 0)                           # components after smoothing keep the refusal
    assert comp2 == comp
    assert L.scan3d_voxel_surface_decimate(h, F32(4 * S), C.byref(s3.DecimateResultC())) == STATE
    _surface(ctx)
    ctx.surface_decimate(F32(4 * S))                               # a new extraction clears it
    # the accumulator is unchanged
    assert b"".join(x.tobytes() for x in ctx.voxels()) == acc
    # the launch count is the formula, an empty surface included
    for it, mu in ((0, -0.53), (3, 0.0), (3, -0.5), (17, -0.53)):
        _surface(ctx)
        _smooth(ctx, it, mu)
    ctx.voxel_begin(S, 16)
    far = _torch(np.array([[1.0, 1.0, 1.0]], F32))
    ctx.voxel_add_dev(far, None, None)
    ctx.voxel_finish()
    assert _surface(ctx)[0]["faces"] == 0
    res, mesh = _smooth(ctx, 10, -0.53)
    assert res == dict(vertices=0, faces=0, held_vertices=0, isolated_vertices=0, passes=20, max_displacement=0.0)
    # begin, add and finish make the smoothed surface stale
    p, nn, c = _sphere(S, RADIUS, CEN)
    tp, tn, tc = _torch(p), _torch(nn), _torch(c)
    for step in ("begin", "add", "finish"):
        ctx.voxel_begin(S, len(p))
        ctx.voxel_add_dev(tp, tn, tc)
        ctx.voxel_finish()
        _surface(ctx)
        assert run() == 0
        if step == "begin":
            ctx.voxel_begin(S, len(p))
        elif step == "add":
            ctx.voxel_add_dev(tp, tn, tc)
        else:
            ctx.voxel_finish()
        assert L.scan3d_get_voxel_surface(h, None, None, None, None, 0, 0) == STATE, step
        assert run() == STATE, step
    del far, tp, tn, tc
    ctx.close()


@gpu
def test_dev_route_errors():
    ctx = _ctx()
    L, h = ctx.L, ctx.h
    rng = np.random.default_rng(8)
    xyz, u, faces = noisy_sphere(2, 1.9, (0, 0, 0), 0.4, 0)
    tx, tn, tf = _torch(xyz), _torch(u), _torch(faces)
    x0, n0 = tx.cpu().numpy().copy(), tn.cpu().numpy().copy()
    out = s3.SmoothResultC()
    good = s3.SmoothParams(10, 0.5, -0.53)

    def call(x=tx, n=tn, nv=len(xyz), f=tf, nf=len(faces), p=good, r=out):
        ptr = lambda t: t if t is None or isinstance(t, int) else t.data_ptr()
        return L.scan3d_mesh_smooth_dev(h, ptr(x), ptr(n), nv, ptr(f), nf, C.byref(p) if p else None,
                                        C.byref(r) if r else None)

    def unchanged():
        assert np.array_equal(tx.cpu().numpy().view(np.uint32), x0.view(np.uint32))
        assert np.array_equal(tn.cpu().numpy().view(np.uint32), n0.view(np.uint32))

    before = ctx.launch_count()
    assert L.scan3d_mesh_smooth_dev(None, tx.data_ptr(), None, 1, tf.data_ptr(), 1, C.byref(good), C.byref(out)) == ARG
    for kw in (dict(p=None), dict(r=None), dict(p=s3.SmoothParams(4097, 0.5, 0.0)), dict(p=s3.SmoothParams(1, 2.0, 0.0)),
               dict(p=s3.SmoothParams(1, 0.5, 0.5)), dict(nv=-1), dict(nv=1 << 31), dict(nf=-1), dict(nf=1 << 31),
               dict(x=None), dict(f=None), dict(x=tx.data_ptr() + 2), dict(n=tn.data_ptr() + 1),
               dict(f=tf.data_ptr() + 2)):
        assert call(**kw) == ARG, kw
    assert ctx.launch_count() == before
    unchanged()
    # found on the device: a face index out of range, a coordinate that is not finite, an overflow
    bad_f = _torch(np.concatenate([faces, [[0, 1, len(xyz)]]]).astype(np.int32))
    assert call(f=bad_f, nf=len(faces) + 1) == ARG and b"face index" in L.scan3d_last_error(h)
    unchanged()
    xn = xyz.copy()
    xn[5, 1] = np.inf
    t_inf = _torch(xn)
    assert call(x=t_inf) == ARG
    assert np.array_equal(t_inf.cpu().numpy().view(np.uint32), xn.view(np.uint32))
    with pytest.raises(SmoothError):
        smooth_ref(xyz, u, faces, 100, 1.0, -1.0)
    before = ctx.launch_count()
    assert call(p=s3.SmoothParams(100, 1.0, -1.0)) == CONFIG
    assert ctx.launch_count() == before + launches(100, -1.0)
    unchanged()
    # the Python wrapper checks shapes and types
    with pytest.raises(s3.Scan3DError):
        ctx.mesh_smooth_dev(tx, tf.long())
    with pytest.raises(s3.Scan3DError):
        ctx.mesh_smooth_dev(tx, tf, tn[:5])
    # the error did not disturb a later call
    gx, gn, res = _dev(ctx, xyz, u, faces, 10)
    wx, wn, info = smooth_ref(xyz, u, faces, 10)
    _same((gx, gn), (wx, wn))
    del tx, tn, tf, bad_f, t_inf
    ctx.close()
