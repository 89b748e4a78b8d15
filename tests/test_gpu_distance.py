"""GPU checks of the sample-to-surface distances (scan3d_voxel_surface_distance, scan3d_voxel_surface_distance_dev,
scan3d_mesh_distance_dev): byte parity of the per-sample distances and faces and of every field of the result with
distance_ref of tests/test_distance_ref.py through all three routes, every call twice with the stated launch count, on
constructed and random meshes, faces spanning many cells and empty inputs; the surface route after extraction,
decimation, smoothing and filling, with the held surface, the component table and the decimation unchanged; a view's
device points; the camera-grid mesh as the target; every argument, state and configuration error with nothing
written; and the invariances under permutation and a change of R that keeps the matches, and what a dyadic
translation keeps."""
import ctypes as C
import importlib
import math

import numpy as np
import pytest

from test_decimate_ref import decimate_ref
from test_distance_ref import cube, distance_ref, icosphere, random_mesh, random_samples
from test_gpu_align import SMALL, _ctx, _torch
from test_gpu_components import S
from test_gpu_mesh import _scene as _mesh_scene
from test_gpu_repair import _shell_and_touching_spheres
from test_gpu_surface import _same, _surface

s3 = importlib.import_module("3dscan_b200")
gpu = pytest.mark.gpu

F32 = np.float32
LAUNCHES, ERROR_LAUNCHES = 7, 2
ARG, STATE, CONFIG = -4, -3, -1


def test_abi_symbols_resolve():
    L = C.CDLL(s3.cuda_lib()._name)
    for name in ("scan3d_voxel_surface_distance", "scan3d_voxel_surface_distance_dev", "scan3d_mesh_distance_dev"):
        assert getattr(L, name)
    assert C.sizeof(s3.DistanceParams) == 4
    assert C.sizeof(s3.DistanceResultC) == 80 and s3.DistanceResultC.max.offset == 40
    assert s3.DistanceResultC.min_signed.offset == 64 and s3.DistanceResultC.entries.offset == 72


def _check(got, want):
    dist, face, res = got
    wd, wf, wres = want
    _same((dist.cpu().numpy(), face.cpu().numpy()), (wd, wf))
    assert set(res) == set(wres)
    for k in res:
        if isinstance(wres[k], float):
            assert np.float64(res[k]).tobytes() == np.float64(wres[k]).tobytes(), (k, res[k], wres[k])
        else:
            assert res[k] == wres[k], (k, res[k], wres[k])


def _mesh_call(ctx, samples, xyz, faces, R, want=None):
    want = want or distance_ref(samples, xyz, faces, R)
    ts, tx, tf = _torch(np.asarray(samples, F32).reshape(-1, 3)), _torch(np.asarray(xyz, F32).reshape(-1, 3)), \
        _torch(np.asarray(faces, np.int32).reshape(-1, 3))
    for _ in range(2):
        before = ctx.launch_count()
        got = ctx.mesh_distance_dev(ts, tx, tf, R)
        assert ctx.launch_count() == before + LAUNCHES
        _check(got, want)
    return want


def _cases():
    out = []
    xyz, f = cube(2.0, (3.0, -5.0, 7.25))
    s = np.concatenate([random_samples(1, 500, 2.0) + F32([4.0, -4.0, 8.25]), xyz[f].mean(1), xyz])
    out += [(s, xyz, f, R) for R in (0.5, 1.5, 20.0)]
    xyz, f = icosphere(2, 3.0)
    out += [(random_samples(2, 2000, 3.0), xyz, f, R) for R in (0.1, 1.0)]
    for seed in range(3):
        xyz, f = random_mesh(seed)
        out += [(random_samples(seed + 5, 3000), xyz, f, R) for R in (0.3, 2.0, 25.0)]
    # a fill-like fan: long thin faces spanning many cells
    ring = np.array([[10 * math.cos(t), 10 * math.sin(t), 0.1 * k] for k, t in enumerate(np.linspace(0, 6.2, 40))], F32)
    xyz = np.concatenate([[[0, 0, 2]], ring]).astype(F32)
    f = np.array([[0, k, k + 1] for k in range(1, 40)], np.int32)
    out.append((random_samples(9, 2000, 6.0), xyz, f, 0.2))
    z = np.zeros((0, 3), F32)
    out += [(z, xyz, f, 1.0), (random_samples(3, 50), z, np.zeros((0, 3), np.int32), 1.0),
            (random_samples(4, 50), np.ones((5, 3), F32), np.zeros((0, 3), np.int32), 1.0), (z, z, np.zeros((0, 3), np.int32), 1.0)]
    return out


@gpu
def test_mesh_route_parity():
    ctx = _ctx()
    for samples, xyz, faces, R in _cases():
        want = _mesh_call(ctx, samples, xyz, faces, R)
        print(f"{len(samples)} samples, {len(faces)} faces, R {R}: {want[2]}")
    ctx.close()


@gpu
def test_invariances():
    ctx = _ctx()
    xyz, faces = random_mesh(11)
    xyz = (np.round(xyz * 64) / 64).astype(F32)                        # one dyadic grid
    samples = (np.round(random_samples(12, 4000) * 64) / 64).astype(F32)
    samples[~np.isfinite(samples)] = 0
    R = 2.0
    base = _mesh_call(ctx, samples, xyz, faces, R)
    perm = np.random.default_rng(0).permutation(len(samples))
    d, f, r = ctx.mesh_distance_dev(_torch(samples[perm]), _torch(xyz), _torch(faces), R)
    _same((d.cpu().numpy(), f.cpu().numpy()), (base[0][perm], base[1][perm]))
    assert (r["matched"], r["inside"], r["max"]) == (base[2]["matched"], base[2]["inside"], base[2]["max"])
    # a dyadic translation keeps every difference of coordinates exact, but a
    # closest point on an edge or inside a face is a + t (b - a), rounded at the translated magnitude, so there the
    # distance moves by rounding only, and a face tied within rounding may give way to its neighbour
    off = F32([256.0, -512.0, 128.0])
    d, f, _ = ctx.mesh_distance_dev(_torch(samples + off), _torch(xyz + off), _torch(faces), R)
    d, f = d.cpu().numpy(), f.cpu().numpy()
    want = distance_ref(samples + off, xyz + off, faces, R)
    _same((d, f), want[:2])
    assert np.array_equal(np.isnan(d), np.isnan(base[0]))
    np.testing.assert_allclose(np.abs(d), np.abs(base[0]), rtol=0, atol=1e-4)
    same = f == base[1]
    np.testing.assert_allclose(d[same], base[0][same], rtol=0, atol=1e-4)    # the sign is the nearest face's
    assert same.mean() > 0.99
    print(f"translated: {(f == base[1]).mean():.4f} of the faces kept, largest change {np.nanmax(np.abs(d - base[0]))}")
    # every sample within 1e6 of the mesh: a larger R keeps the same matches
    d, f, _ = ctx.mesh_distance_dev(_torch(samples), _torch(xyz), _torch(faces), 1e6)
    big = ctx.mesh_distance_dev(_torch(samples), _torch(xyz), _torch(faces), 2e6)
    _same((d.cpu().numpy(), f.cpu().numpy()), (big[0].cpu().numpy(), big[1].cpu().numpy()))
    ctx.close()


def _surface_call(ctx, R):
    mxyz, mnrm, _, _ = ctx.voxels()
    sxyz, _, _, sf = ctx.voxel_surface_mesh()
    want = distance_ref(mxyz, sxyz, sf, R, is_sample=(mnrm != 0).any(1))
    for _ in range(2):
        before = ctx.launch_count()
        got = ctx.surface_distance(R, per_sample=True)
        assert ctx.launch_count() == before + LAUNCHES
        _check(got, want)
        assert ctx.surface_distance(R) == got[2]
    return want


@gpu
def test_surface_route_after_each_stage():
    ctx = _ctx()
    _shell_and_touching_spheres(ctx)
    R = float(2 * S)
    for stage in ("raw", "decimated", "smoothed", "filled"):
        _surface(ctx)
        if stage == "decimated":
            ctx.surface_decimate(F32(4 * S))
        elif stage == "smoothed":
            ctx.surface_smooth(10)
        elif stage == "filled":
            ctx.surface_fill_holes(22)
        want = _surface_call(ctx, R)
        print(f"model -> {stage}: {want[2]}")
        assert want[2]["matched"] > 0
    # a view's points through the dev route
    _surface(ctx)
    pts = ctx.voxels()[0][::3].copy()
    got = ctx.surface_distance_dev(_torch(pts), R)
    sxyz, _, _, sf = ctx.voxel_surface_mesh()
    _check(got, distance_ref(pts, sxyz, sf, R))
    ctx.close()


@gpu
def test_surface_route_changes_nothing():
    ctx = _ctx()
    _shell_and_touching_spheres(ctx)
    _surface(ctx)
    ctx.surface_components(0, 0)
    mesh = ctx.voxel_surface_mesh()
    table = ctx.surface_component_table()
    vox = ctx.voxels()
    ctx.surface_distance(float(2 * S), per_sample=True)
    ctx.surface_distance_dev(_torch(vox[0]), float(S))
    ctx.mesh_distance_dev(_torch(vox[0]), _torch(mesh[0]), _torch(mesh[3]), float(S))
    _same(ctx.voxel_surface_mesh(), mesh)
    _same(ctx.surface_component_table(), table)
    _same(ctx.voxels(), vox)
    assert ctx.L.scan3d_get_surface_components(ctx.h, None, None, None, 0) == 0
    # the decimation behaves as without the calls
    ctx.surface_decimate(F32(4 * S))
    _same(ctx.voxel_surface_mesh()[:4], decimate_ref(mesh, S, F32(4 * S))[:4])
    ctx.close()


@gpu
def test_camera_grid_mesh_as_target():
    cfg, cal, _, stack, roi = _mesh_scene(SMALL)
    ctx = s3.Scan3D(cfg, 0, cal)
    L, h = ctx.L, ctx.h
    n = ctx.reconstruct(stack, roi)
    ctx.build_mesh(8.0)                     # without an edge limit, faces across the background span too many cells
    pts = ctx.points()
    faces, _ = ctx.mesh()
    assert len(faces) > 0
    samples = (pts[::7] + F32([0.01, -0.02, 0.03])).astype(F32)
    ts = _torch(samples)
    dist, face = _torch(np.zeros(len(samples), F32)), _torch(np.zeros(len(samples), np.int32))
    r = s3.DistanceResultC()
    p = s3.DistanceParams(2.0)
    before = ctx.launch_count()
    assert L.scan3d_mesh_distance_dev(h, ts.data_ptr(), len(samples), L.scan3d_device_points(h), n,
                                      L.scan3d_device_mesh_faces(h), len(faces), C.byref(p), dist.data_ptr(),
                                      face.data_ptr(), C.byref(r)) == 0
    assert ctx.launch_count() == before + LAUNCHES
    want = distance_ref(samples, pts, faces, 2.0)
    _check((dist, face, s3.Scan3D._distance_result(r)), want)
    print(f"camera-grid mesh: {len(faces)} faces, {want[2]}")
    ctx.close()


@gpu
def test_errors_write_nothing():
    ctx = _ctx()
    L, h = ctx.L, ctx.h
    xyz, faces = random_mesh(3)
    samples = random_samples(4, 100)
    ts, tx, tf = _torch(samples), _torch(xyz), _torch(faces)
    fill_d, fill_f = np.full(100, 7.5, F32), np.full(100, 99, np.int32)
    td, tfo = _torch(fill_d), _torch(fill_f)
    r = s3.DistanceResultC()
    p = s3.DistanceParams(1.0)
    ptr = lambda t: t if t is None or isinstance(t, int) else t.data_ptr()

    def mesh(s=ts, n=100, x=tx, nv=len(xyz), f=tf, nf=len(faces), prm=p, d=td, fo=tfo, out=r, c=h):
        return L.scan3d_mesh_distance_dev(c, ptr(s), n, ptr(x), nv, ptr(f), nf, C.byref(prm) if prm else None,
                                          ptr(d), ptr(fo), C.byref(out) if out else None)

    def untouched():
        _same((td.cpu().numpy(), tfo.cpu().numpy()), (fill_d, fill_f))

    before = ctx.launch_count()
    for kw in (dict(c=None), dict(prm=None), dict(out=None), dict(prm=s3.DistanceParams(0.0)),
               dict(prm=s3.DistanceParams(-1.0)), dict(prm=s3.DistanceParams(math.inf)),
               dict(prm=s3.DistanceParams(math.nan)), dict(n=-1), dict(n=1 << 31), dict(nv=-1), dict(nv=1 << 31),
               dict(nf=-1), dict(nf=1 << 31), dict(s=None), dict(x=None), dict(f=None), dict(s=ts.data_ptr() + 2),
               dict(x=tx.data_ptr() + 1), dict(f=tf.data_ptr() + 2), dict(d=td.data_ptr() + 2),
               dict(fo=tfo.data_ptr() + 1)):
        assert mesh(**kw) == ARG, kw
    for kw in (dict(s=None, n=0), dict(x=None, nv=0, f=None, nf=0, d=None, fo=None), dict(d=None, fo=None)):
        assert mesh(**kw) == 0, kw
    assert ctx.launch_count() == before + 3 * LAUNCHES
    # without a held surface
    before = ctx.launch_count()
    assert L.scan3d_voxel_surface_distance(h, C.byref(p), None, None, C.byref(r)) == STATE
    assert L.scan3d_voxel_surface_distance_dev(h, ts.data_ptr(), 100, C.byref(p), None, None, C.byref(r)) == STATE
    assert L.scan3d_voxel_surface_distance(h, None, None, None, C.byref(r)) == ARG
    assert L.scan3d_voxel_surface_distance_dev(h, None, 5, C.byref(p), None, None, C.byref(r)) == ARG
    assert ctx.launch_count() == before
    untouched()
    # found on the device: a face index out of range, a coordinate that is not finite; the limits
    cases = [(ARG, xyz, np.concatenate([faces, [[0, 1, len(xyz)]]]), 1.0),
             (ARG, xyz, np.concatenate([faces, [[0, -1, 2]]]), 1.0)]
    xn = xyz.copy()
    xn[len(xyz) - 1, 2] = np.inf                                        # a vertex no face uses
    cases.append((ARG, xn, faces, 1.0))
    far = np.concatenate([xyz, [[2.0 ** 21, 0, 0]]]).astype(F32)
    cases.append((CONFIG, far, np.concatenate([faces, [[0, 1, len(xyz)]]]), 1.0))        # the key range
    big = np.array([[-1e5, -1e5, -1e5], [1e5, 1e5, 1e5], [0, 1e5, 0]], F32)
    cases.append((CONFIG, big, np.array([[0, 1, 2]], np.int32), 0.15))                    # 2^32 entries
    for code, x, f, R in cases:
        before = ctx.launch_count()
        assert mesh(x=_torch(x), nv=len(x), f=_torch(np.asarray(f, np.int32)), nf=len(f),
                    prm=s3.DistanceParams(R)) == code, (code, R)
        assert ctx.launch_count() == before + ERROR_LAUNCHES
        untouched()
    with pytest.raises(s3.Scan3DError):
        ctx.mesh_distance_dev(ts.double(), tx, tf, 1.0)
    with pytest.raises(s3.Scan3DError):
        ctx.mesh_distance_dev(ts, tx, tf.long(), 1.0)
    ctx.close()
