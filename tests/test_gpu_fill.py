"""GPU checks of the hole filling (scan3d_voxel_surface_fill_holes, scan3d_mesh_fill_holes_dev): bit parity with
fill_ref of tests/test_fill_ref.py on random holed meshes, a sphere merged without its polar cap (raw, after
decimation at 4 s and after smoothing), the 640x480 ctx route, the camera-grid mesh with ROI holes through the dev
route and an empty mesh; every call twice, byte-identical.  Also the state rules, every argument error, errors found
on the device, the capacity error, the launch count, a second fill that adds nothing, decimation after a raw fill, and
the largest piece of the noise-free multi-view scene after smoothing.  The ABI check needs no GPU.

A hole of n edges costs the numpy DP about n^3 / 6 candidate triangles (44 s for n = 1000), so holes of more than
NUMPY_EDGES edges are triangulated for the reference by the header compiled for the host, which
tests/test_fill_math_host.py compares bit for bit with the numpy DP."""
import ctypes as C
import importlib
import math

import numpy as np
import pytest

from test_decimate_ref import decimate_ref
from test_fill_math_host import build_host_lib, host_polygon
from test_fill_ref import (annulus, cube_without_a_face, edge_counts, fill_ref, holes_ref, polygon_faces_ref,
                           punched_sphere)
from test_gpu_align import CENTRE, SMALL, _ctx, _scene, _spacing, _torch
from test_gpu_components import CEN, RADIUS, S, _sphere, _sphere_and_islands
from test_gpu_mesh import _scene as _mesh_scene
from test_gpu_surface import _merge, _same, _surface
from test_gpu_voxel import C1, _voxel_size
from test_gpu_voxel import _scene as _voxel_scene
from test_smooth_ref import grid_mesh, odd_mesh

s3 = importlib.import_module("3dscan_b200")
gpu = pytest.mark.gpu

F32 = np.float32
LAUNCHES, LAUNCHES_BAD = 10, 6
ARG, STATE, CONFIG = -4, -3, -1
NUMPY_EDGES = 64
_HOST = []


@pytest.fixture(scope="module", autouse=True)
def _host_lib(tmp_path_factory):
    _HOST.append(build_host_lib(tmp_path_factory.mktemp("fillhost")))
    yield
    _HOST.clear()


def _polygon(p, rims, exists):
    if len(p) <= NUMPY_EDGES:
        return polygon_faces_ref(p, rims, exists)
    return host_polygon(_HOST[0], p, rims, exists)[0]


def _ref(xyz, faces, max_edges):
    return fill_ref(xyz, faces, max_edges, _polygon)


def test_abi_symbols_resolve():
    L = C.CDLL(s3.cuda_lib()._name)
    for name in ("scan3d_voxel_surface_fill_holes", "scan3d_mesh_fill_holes_dev"):
        assert getattr(L, name)
    assert C.sizeof(s3.FillResultC) == 56 and s3.FillResultC.open_edges.offset == 48
    assert (s3.FILL_NETS_MAX_EDGES, s3.FILL_MAX_EDGES) == (22, 1024)


def _fill(ctx, max_edges=None):
    before = ctx.launch_count()
    res = ctx.surface_fill_holes(max_edges)
    assert ctx.launch_count() == before + LAUNCHES
    return res, ctx.voxel_surface_mesh()


def _check_surface(ctx, raw, max_edges):
    """fill the held surface raw; compare with the reference; returns the filled mesh"""
    res, mesh = _fill(ctx, max_edges)
    add, info = _ref(raw[0], raw[3], max_edges)
    _same(mesh, (raw[0], raw[1], raw[2], np.concatenate([raw[3], add])))
    assert res == info
    print(f"max_edges {max_edges}: {res}")
    return mesh, res


def _dev(ctx, xyz, faces, max_edges):
    """the dev route on copies of the arrays, twice, against the reference; returns (added faces, result)"""
    outs = []
    for _ in range(2):
        tx = _torch(np.ascontiguousarray(xyz, F32).reshape(-1, 3))
        tf = _torch(np.ascontiguousarray(faces, np.int32).reshape(-1, 3))
        before = ctx.launch_count()
        add, res = ctx.mesh_fill_holes_dev(tx, tf, max_edges)
        assert ctx.launch_count() == before + LAUNCHES       # n_faces rows always suffice here
        outs.append((add.cpu().numpy(), res))
        assert np.array_equal(tf.cpu().numpy(), np.asarray(faces, np.int32).reshape(-1, 3))
    want, info = _ref(xyz, faces, max_edges)
    for add, res in outs:
        _same((add,), (want,))
        assert res == info
    return outs[0]


@gpu
def test_dev_route_random_holed_meshes():
    ctx = _ctx()
    rng = np.random.default_rng(3)
    for seed in range(3):
        xyz, faces = punched_sphere(3, 20, seed, sigma=0.03 * seed)
        for m in (3, 8, 22, 1024):
            _dev(ctx, xyz, faces, m)
    for _ in range(3):
        xyz, _, faces = odd_mesh(rng, 300, 500)
        _dev(ctx, xyz, faces, 1024)
    xyz, faces = grid_mesh(60, 40, 0.1, rng.normal(size=(40, 60)) * 0.01)
    add, res = _dev(ctx, xyz, faces, 1024)                  # the rim: one loop of 196 edges
    assert res["filled"] == 1 and len(add) == 194
    for mesh, m in ((cube_without_a_face(), 4), (annulus(300), 300), (annulus(600), 1024)):
        add, res = _dev(ctx, *mesh, m)
        assert res["filled"] == 1
    # an empty mesh, and vertices without faces
    add, res = _dev(ctx, np.zeros((0, 3), F32), np.zeros((0, 3), np.int32), 22)
    assert len(add) == 0 and res == dict(vertices=0, faces=0, boundary_edges=0, holes=0, filled=0, faces_added=0,
                                         open_edges=0)
    _dev(ctx, xyz[:100], np.zeros((0, 3), np.int32), 22)
    ctx.close()


def _capless_sphere(ctx):
    """the closed sphere of test_gpu_components without the points above z = 0.9 R: a hole at the pole"""
    p, n, c = _sphere(S, RADIUS, CEN)
    keep = p[:, 2] - CEN[2] < 0.9 * RADIUS
    _merge(ctx, S, [(p[keep], n[keep], c[keep])])
    return _surface(ctx)[1]


@gpu
def test_sphere_without_a_polar_cap_raw_decimated_and_smoothed():
    ctx = _ctx()
    raw = _capless_sphere(ctx)
    filled, res = _check_surface(ctx, raw, 22)
    # a second fill adds nothing, and the held surface stays byte-identical
    res2, again = _fill(ctx, 22)
    _same(again, filled)
    assert res2["faces_added"] == 0 and res2["boundary_edges"] == res["open_edges"]
    # the polar hole is longer than the unrefined surface's cap; it closes on a decimated surface (cap 1024) and on a
    # smoothed one
    for refine in (lambda: ctx.surface_decimate(F32(4 * S)), lambda: ctx.surface_smooth(10)):
        _surface(ctx)
        refine()
        before = ctx.voxel_surface_mesh()
        mesh, res = _check_surface(ctx, before, 1024)
        assert res["filled"] >= 1 and res["open_edges"] < res["boundary_edges"]
        if res["open_edges"] == 0:
            und, directed = edge_counts(mesh[3])
            assert (und == 2).all() and (directed == 1).all()
        res2, again = _fill(ctx, 1024)
        _same(again, mesh)
        assert res2["faces_added"] == 0
    ctx.close()


@gpu
def test_ctx_route_640x480():
    cfg, cal, stack, roi = _scene(SMALL)
    ctx = s3.Scan3D(cfg, 0, cal)
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
    _check_surface(ctx, raw, 22)
    _surface(ctx)
    ctx.surface_smooth(10)
    _check_surface(ctx, ctx.voxel_surface_mesh(), 1024)
    ctx.close()


@gpu
def test_dev_route_camera_grid_mesh_with_roi_holes():
    cfg, cal, _, stack, roi = _mesh_scene(SMALL)
    roi = roi.copy()
    roi[100:140, 200:260] = 0                                          # test_gpu_mesh's holes
    roi[300:340, 100:300] = 0
    roi[300:340:3, 100:300:3] = 1
    roi[200, ::2] = 0
    ctx = s3.Scan3D(cfg, 0, cal)
    L, h = ctx.L, ctx.h
    n = ctx.reconstruct(stack, roi)
    ctx.build_mesh(math.inf)
    pts = ctx.points()
    faces, _ = ctx.mesh()
    out = []
    for _ in range(2):
        dst = _torch(np.full((len(faces), 3), -7, np.int32))
        r = s3.FillResultC()
        before = ctx.launch_count()
        assert L.scan3d_mesh_fill_holes_dev(h, L.scan3d_device_points(h), n, L.scan3d_device_mesh_faces(h),
                                            len(faces), 1024, dst.data_ptr(), len(faces), C.byref(r)) == 0
        assert ctx.launch_count() == before + LAUNCHES
        res = s3.Scan3D._fill_result(r)
        out.append((dst.cpu().numpy()[:res["faces_added"]], res))
    want, info = _ref(pts, faces, 1024)
    for add, res in out:
        _same((add,), (want,))
        assert res == info
    assert np.array_equal(ctx.mesh()[0], faces)
    print(f"camera-grid mesh 640x480 with ROI holes: {n} points, {len(faces)} faces, {info}")
    assert info["filled"] > 0
    ctx.close()


@gpu
def test_rules_state_errors_and_launch_count():
    ctx = _ctx()
    L, h = ctx.L, ctx.h
    out = s3.FillResultC()
    before = ctx.launch_count()
    assert L.scan3d_voxel_surface_fill_holes(h, 22, C.byref(out)) == STATE       # before any surface
    assert ctx.launch_count() == before
    raw = _sphere_and_islands(ctx)
    ctx.surface_components(0, 0)
    # argument errors: nothing launched, the surface and the component table stay
    before = ctx.launch_count()
    for m in (-1, 0, 2, 23, 1024):
        assert L.scan3d_voxel_surface_fill_holes(h, m, C.byref(out)) == ARG, m
    assert L.scan3d_voxel_surface_fill_holes(None, 22, C.byref(out)) == ARG
    assert L.scan3d_voxel_surface_fill_holes(h, 22, None) == ARG
    assert ctx.launch_count() == before
    _same(ctx.voxel_surface_mesh(), raw)
    assert L.scan3d_get_surface_components(h, None, None, None, 0) == 0
    # a fill makes the component table stale; the islands' patches have short rims
    filled, res = _check_surface(ctx, raw, 22)
    assert res["filled"] >= 1
    assert L.scan3d_get_surface_components(h, None, None, None, 0) == STATE
    # a raw surface stays decimatable: decimation after the fill is the decimation of the filled mesh
    ctx.surface_decimate(F32(4 * S))
    _same(ctx.voxel_surface_mesh(), decimate_ref(filled, S, F32(4 * S))[:4])
    # after decimation or smoothing the cap is 1024
    for refine in (lambda: ctx.surface_decimate(F32(4 * S)), lambda: ctx.surface_smooth(1)):
        _surface(ctx)
        refine()
        assert L.scan3d_voxel_surface_fill_holes(h, 1025, C.byref(out)) == ARG
        assert L.scan3d_voxel_surface_fill_holes(h, 1024, C.byref(out)) == 0
    # the launch count is fixed, an empty surface included
    ctx.voxel_begin(S, 16)
    far = _torch(np.array([[1.0, 1.0, 1.0]], F32))
    ctx.voxel_add_dev(far, None, None)
    ctx.voxel_finish()
    assert _surface(ctx)[0]["faces"] == 0
    res, mesh = _fill(ctx, 3)
    assert res == dict(vertices=0, faces=0, boundary_edges=0, holes=0, filled=0, faces_added=0, open_edges=0)
    # begin, add and finish make the filled surface stale
    p, nn, c = _sphere(S, RADIUS, CEN)
    tp, tn, tc = _torch(p), _torch(nn), _torch(c)
    for step in ("begin", "add", "finish"):
        ctx.voxel_begin(S, len(p))
        ctx.voxel_add_dev(tp, tn, tc)
        ctx.voxel_finish()
        _surface(ctx)
        assert L.scan3d_voxel_surface_fill_holes(h, 22, C.byref(out)) == 0
        getattr(ctx, {"begin": "voxel_begin", "add": "voxel_add_dev", "finish": "voxel_finish"}[step])(
            *{"begin": (S, len(p)), "add": (tp, tn, tc), "finish": ()}[step])
        assert L.scan3d_voxel_surface_fill_holes(h, 22, C.byref(out)) == STATE, step
    del far, tp, tn, tc
    ctx.close()


@gpu
def test_dev_route_errors_and_capacity():
    ctx = _ctx()
    L, h = ctx.L, ctx.h
    xyz, faces = punched_sphere(3, 10, 4)
    tx, tf = _torch(xyz), _torch(faces)
    dst = _torch(np.full((len(faces), 3), -7, np.int32))
    out = s3.FillResultC()

    def call(x=tx, nv=len(xyz), f=tf, nf=len(faces), m=1024, o=dst, cap=len(faces), r=out):
        ptr = lambda t: t if t is None or isinstance(t, int) else t.data_ptr()
        return L.scan3d_mesh_fill_holes_dev(h, ptr(x), nv, ptr(f), nf, m, ptr(o), cap, C.byref(r) if r else None)

    def untouched():
        assert (dst.cpu().numpy() == -7).all()

    before = ctx.launch_count()
    assert L.scan3d_mesh_fill_holes_dev(None, tx.data_ptr(), len(xyz), tf.data_ptr(), len(faces), 22, dst.data_ptr(),
                                        len(faces), C.byref(out)) == ARG
    for kw in (dict(r=None), dict(m=2), dict(m=1025), dict(nv=-1), dict(nv=1 << 31), dict(nf=-1), dict(nf=1 << 31),
               dict(cap=-1), dict(cap=1 << 31), dict(x=None), dict(f=None), dict(o=None),
               dict(x=tx.data_ptr() + 2), dict(f=tf.data_ptr() + 1), dict(o=dst.data_ptr() + 2)):
        assert call(**kw) == ARG, kw
    assert ctx.launch_count() == before
    untouched()
    # found on the device: a face index out of range, a coordinate that is not finite
    bad_f = _torch(np.concatenate([faces, [[0, 1, len(xyz)]]]).astype(np.int32))
    assert call(f=bad_f, nf=len(faces) + 1) == ARG and b"face index" in L.scan3d_last_error(h)
    assert ctx.launch_count() == before + LAUNCHES_BAD
    xn = xyz.copy()
    xn[5, 1] = np.nan
    assert call(x=_torch(xn)) == ARG
    untouched()
    # too small an output: nothing written, faces_added reported; the wrapper retries once with that size
    want, info = _ref(xyz, faces, 1024)
    assert len(want) > 1
    before = ctx.launch_count()
    assert call(cap=len(want) - 1) == CONFIG and b"max_faces_out" in L.scan3d_last_error(h)
    assert ctx.launch_count() == before + LAUNCHES
    untouched()
    res = s3.Scan3D._fill_result(out)
    assert res == dict(info, faces=len(faces), open_edges=info["boundary_edges"])
    assert call(cap=len(want)) == 0
    _same((dst.cpu().numpy()[:len(want)],), (want,))
    assert (dst.cpu().numpy()[len(want):] == -7).all()
    # the wrapper checks shapes and types
    with pytest.raises(s3.Scan3DError):
        ctx.mesh_fill_holes_dev(tx, tf.long())
    with pytest.raises(s3.Scan3DError):
        ctx.mesh_fill_holes_dev(tx[:, :2], tf)
    del tx, tf, dst, bad_f
    ctx.close()


@gpu
def test_largest_piece_of_the_noise_free_scene_after_smoothing():
    """The largest component of eight merged views of the sphere alone (test_gpu_decimate's scene), smoothed with
    MeshLab's defaults, then filled at max_edges = 1024: against the reference, and what stays open and why."""
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
    _surface(ctx)
    ctx.surface_components(0, 1)
    ctx.surface_smooth(10)
    big = ctx.voxel_surface_mesh()
    mesh, res = _check_surface(ctx, big, 1024)
    # why the rest stays open: loops longer than 1024 edges, unfillable loops, and chains through vertices that are
    # not regular
    loops = holes_ref(len(big[0]), big[3], 10 ** 9)[0]
    in_long = sum(len(x) for x in loops if len(x) > 1024)
    unfillable = sum(len(x) for x in loops if len(x) <= 1024) - (res["faces_added"] + 2 * res["filled"])
    chains = res["open_edges"] - in_long - unfillable
    print(f"largest piece after smoothing: {len(big[0])} vertices, {len(big[3])} faces; {res['boundary_edges']} "
          f"boundary edges, {res['holes']} holes, {res['filled']} filled ({res['faces_added']} faces); "
          f"{res['open_edges']} open: {in_long} in loops over 1024 edges, {unfillable} in "
          f"{res['holes'] - res['filled']} unfillable loops, {chains} on chains through vertices that are not regular")
    assert res["open_edges"] < res["boundary_edges"] and res["filled"] > 0
    ctx.close()
