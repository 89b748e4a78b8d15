"""GPU checks of the coherent orientation and the measures (scan3d_voxel_surface_orient, scan3d_mesh_orient_dev,
scan3d_voxel_surface_measure, scan3d_mesh_measure_dev): byte parity of the faces, the normals and both result structs
with orient_ref and measure_ref of tests/test_orient_ref.py through the dev route on the constructed meshes and through
the surface route on a thin shell and two touching spheres, every call twice with the stated launch count; the
measure's edge kinds against the repair's; a fill that closes a hole only after the orientation; the camera-grid mesh;
the state rules (the component table stays current, decimation after orienting a raw surface, the decimation refusing a
surface filled after flips); every argument error and the errors found on the device.  The ABI check needs no GPU."""
import ctypes as C
import importlib
import math

import numpy as np
import pytest

from test_decimate_ref import decimate_ref
from test_gpu_align import SMALL, _ctx, _torch
from test_gpu_components import S
from test_gpu_mesh import _scene as _mesh_scene
from test_gpu_repair import _shell_and_touching_spheres
from test_gpu_surface import _same, _surface
from test_orient_ref import (bowtie, book, cube, flipped, hemisphere, measure_ref, moebius, odd, orient_ref,
                             pinched_spheres, rim_hole_mesh, sphere, torus)

s3 = importlib.import_module("3dscan_b200")
gpu = pytest.mark.gpu

F32 = np.float32
ORIENT_LAUNCHES, MEASURE_LAUNCHES = 8, 7
ARG, STATE, CONFIG = -4, -3, -1


def test_abi_symbols_resolve():
    L = C.CDLL(s3.cuda_lib()._name)
    for name in ("scan3d_voxel_surface_orient", "scan3d_mesh_orient_dev", "scan3d_voxel_surface_measure",
                 "scan3d_mesh_measure_dev"):
        assert getattr(L, name)
    assert C.sizeof(s3.OrientResultC) == 80 and s3.OrientResultC.inconsistent_edges.offset == 72
    assert C.sizeof(s3.MeasureResultC) == 144 and s3.MeasureResultC.area.offset == 104
    assert s3.MeasureResultC.bbox_max.offset == 132


def _meshes():
    xyz, f = sphere()
    rng = np.random.default_rng(5)
    out = [(xyz, flipped(f, rng.random(len(f)) < 0.4)), (xyz, flipped(f, slice(None))), hemisphere(),
           (np.array([[0, 0, 0], [1, 0, 0], [0, 1, 0], [0, -1, 0]], F32), np.array([[0, 1, 2], [0, 1, 3]], np.int32)),
           moebius(), torus(), pinched_spheres(2), book(4, [1.0, 3.0, 0.5, 2.0], [1, 1, -1, 1]), bowtie(),
           cube(2.0, (3.0, -5.0, 7.25)), rim_hole_mesh()]
    s1, f1 = sphere(1)
    out.append((s1, np.concatenate([flipped(f1, [0, 4]), [[0, 0, 1], [2, 3, 2], [5, 5, 5]]]).astype(np.int32)))
    out += [odd(seed, 300, 900) for seed in range(3)]
    out += [(np.zeros((0, 3), F32), np.zeros((0, 3), np.int32)), (np.ones((7, 3), F32), np.zeros((0, 3), np.int32))]
    return out


def _dev(ctx, xyz, faces):
    """both dev routes on copies of the arrays, twice each, against the references; returns the oriented faces"""
    xyz = np.ascontiguousarray(xyz, F32).reshape(-1, 3)
    nrm = np.random.default_rng(len(faces)).normal(size=xyz.shape).astype(F32)
    want_f, want_n, info = orient_ref(xyz, faces, nrm)
    mwant = measure_ref(xyz, faces)
    for _ in range(2):
        tx, tn = _torch(xyz), _torch(nrm)
        tf = _torch(np.ascontiguousarray(faces, np.int32).reshape(-1, 3))
        before = ctx.launch_count()
        assert ctx.mesh_measure_dev(tx, tf) == mwant
        assert ctx.launch_count() == before + MEASURE_LAUNCHES
        res = ctx.mesh_orient_dev(tx, tf, tn)
        assert ctx.launch_count() == before + MEASURE_LAUNCHES + ORIENT_LAUNCHES
        assert res == info
        _same((tf.cpu().numpy(), tn.cpu().numpy(), tx.cpu().numpy()), (want_f, want_n, xyz))
    tf = _torch(np.ascontiguousarray(faces, np.int32).reshape(-1, 3))
    assert ctx.mesh_orient_dev(_torch(xyz), tf) == info                       # without normals
    _same((tf.cpu().numpy(),), (want_f,))
    return want_f, info


@gpu
def test_dev_route_constructed_and_random_meshes():
    ctx = _ctx()
    for xyz, faces in _meshes():
        out, info = _dev(ctx, xyz, faces)
        again = ctx.mesh_orient_dev(_torch(np.asarray(xyz, F32).reshape(-1, 3)), _torch(out))
        assert again["flipped_faces"] == 0
    ctx.close()


@gpu
def test_a_fill_after_orienting_closes_the_rim_hole():
    ctx = _ctx()
    xyz, faces = rim_hole_mesh()
    tx = _torch(xyz)
    _, before = ctx.mesh_fill_holes_dev(tx, _torch(faces), 22)
    tf = _torch(faces)
    assert ctx.mesh_orient_dev(tx, tf)["flipped_faces"] == 1
    _, after = ctx.mesh_fill_holes_dev(tx, tf, 22)
    print(f"rim hole: open edges {before['open_edges']} without orienting, {after['open_edges']} after")
    assert before["open_edges"] > 0 and after["open_edges"] == 0
    ctx.close()


@gpu
def test_dev_route_camera_grid_mesh():
    cfg, cal, _, stack, roi = _mesh_scene(SMALL)
    ctx = s3.Scan3D(cfg, 0, cal)
    L, h = ctx.L, ctx.h
    n = ctx.reconstruct(stack, roi)
    ctx.build_mesh(math.inf)
    pts = ctx.points()
    faces, _ = ctx.mesh()
    r = s3.MeasureResultC()
    before = ctx.launch_count()
    assert L.scan3d_mesh_measure_dev(h, L.scan3d_device_points(h), n, L.scan3d_device_mesh_faces(h), len(faces),
                                     C.byref(r)) == 0
    assert ctx.launch_count() == before + MEASURE_LAUNCHES
    mwant = measure_ref(pts, faces)
    assert s3.Scan3D._measure_result(r) == mwant
    o = s3.OrientResultC()
    assert L.scan3d_mesh_orient_dev(h, L.scan3d_device_points(h), None, n, L.scan3d_device_mesh_faces(h), len(faces),
                                    C.byref(o)) == 0
    info = s3.Scan3D._orient_result(o)
    assert info == orient_ref(pts, faces)[2] and info["flipped_faces"] == 0
    assert np.array_equal(ctx.mesh()[0], faces)
    print(f"camera-grid mesh 640x480: {n} points, {len(faces)} faces, area {mwant['area']}, {info}")
    ctx.close()


def _orient_surface(ctx):
    before = ctx.launch_count()
    res = ctx.surface_orient()
    assert ctx.launch_count() == before + ORIENT_LAUNCHES
    return res, ctx.voxel_surface_mesh()


def _measure_surface(ctx):
    before = ctx.launch_count()
    res = ctx.surface_measure()
    assert ctx.launch_count() == before + MEASURE_LAUNCHES
    return res


@gpu
def test_surface_route_shell_and_touching_spheres():
    ctx = _ctx()
    _shell_and_touching_spheres(ctx)
    raw = _surface(ctx)[1]
    want_f, want_n, info = orient_ref(raw[0], raw[3], raw[1])
    for _ in range(2):
        _surface(ctx)
        assert _measure_surface(ctx) == measure_ref(raw[0], raw[3])
        res, mesh = _orient_surface(ctx)
        assert res == info
        _same(mesh, (raw[0], want_n, raw[2], want_f))
    print(f"raw surface: {len(raw[0])} vertices, {len(raw[3])} faces, {info}")
    # after a repair with FACES the measure's edge kinds are the repair's, and after orienting none is inconsistent
    # outside a non-orientable patch
    _surface(ctx)
    rr = ctx.surface_repair(True, False)
    m = _measure_surface(ctx)
    assert (m["boundary_edges"], m["inconsistent_edges"], m["nonmanifold_edges"]) == (
        rr["boundary_edges"], rr["inconsistent_edges"], 0)
    rep = ctx.voxel_surface_mesh()
    want_f, want_n, info = orient_ref(rep[0], rep[3], rep[1])
    res, mesh = _orient_surface(ctx)
    assert res == info
    _same(mesh, (rep[0], want_n, rep[2], want_f))
    m2 = _measure_surface(ctx)
    assert m2 == measure_ref(rep[0], want_f) and m2["inconsistent_edges"] == res["inconsistent_edges"]
    if res["nonorientable_patches"] == 0:
        assert m2["inconsistent_edges"] == 0
    print(f"repaired surface: {rr}; orientation {res}; measure {m2}")
    ctx.close()


@gpu
def test_state_rules():
    ctx = _ctx()
    L, h = ctx.L, ctx.h
    o, m = s3.OrientResultC(), s3.MeasureResultC()
    before = ctx.launch_count()
    assert L.scan3d_voxel_surface_orient(h, C.byref(o)) == STATE                  # before any surface
    assert L.scan3d_voxel_surface_measure(h, C.byref(m)) == STATE
    assert L.scan3d_voxel_surface_orient(None, C.byref(o)) == ARG
    assert L.scan3d_voxel_surface_orient(h, None) == ARG
    assert L.scan3d_voxel_surface_measure(h, None) == ARG
    assert ctx.launch_count() == before
    _shell_and_touching_spheres(ctx)
    raw = _surface(ctx)[1]
    # the component table stays current through an orientation and a measure
    ctx.surface_components(0, 0)
    assert L.scan3d_get_surface_components(h, None, None, None, 0) == 0
    _orient_surface(ctx)
    _measure_surface(ctx)
    assert L.scan3d_get_surface_components(h, None, None, None, 0) == 0
    # an oriented raw surface can still be decimated: the decimation of the oriented mesh
    _surface(ctx)
    res, oriented = _orient_surface(ctx)
    ctx.surface_decimate(F32(4 * S))
    _same(ctx.voxel_surface_mesh(), decimate_ref(oriented, S, F32(4 * S))[:4])
    # flips followed by a fill that adds faces stop the decimation until the next extraction
    dr, fr = s3.DecimateResultC(), s3.FillResultC()
    _surface(ctx)
    tf = _torch(raw[3])
    flips = ctx.mesh_orient_dev(_torch(raw[0]), tf)["flipped_faces"]
    rr = ctx.surface_repair(True, False)
    res, _ = _orient_surface(ctx)
    assert L.scan3d_voxel_surface_fill_holes(h, 22, C.byref(fr)) == 0
    changed = rr["nonmanifold_faces"] + rr["duplicate_faces"] + rr["degenerate_faces"] > 0 or res["flipped_faces"] > 0
    print(f"raw flips {flips}, repair {rr}, flips after it {res['flipped_faces']}, fill added {fr.faces_added}")
    assert L.scan3d_voxel_surface_decimate(h, F32(4 * S), C.byref(dr)) == (STATE if changed and fr.faces_added else 0)
    # an orientation alone: the decimation refuses exactly when it flipped faces and the fill added some
    _surface(ctx)
    res, _ = _orient_surface(ctx)
    assert L.scan3d_voxel_surface_fill_holes(h, 22, C.byref(fr)) == 0
    assert L.scan3d_voxel_surface_decimate(h, F32(4 * S), C.byref(dr)) == (
        STATE if res["flipped_faces"] and fr.faces_added else 0)
    # the launch counts are fixed, an empty surface included
    ctx.voxel_begin(S, 16)
    far = _torch(np.array([[1.0, 1.0, 1.0]], F32))
    ctx.voxel_add_dev(far, None, None)
    ctx.voxel_finish()
    empty = _surface(ctx)[1]
    assert len(empty[3]) == 0
    res, mesh = _orient_surface(ctx)
    assert res == orient_ref(empty[0], empty[3])[2]
    assert _measure_surface(ctx) == measure_ref(empty[0], empty[3])
    del far
    ctx.close()


@gpu
def test_dev_route_errors():
    ctx = _ctx()
    L, h = ctx.L, ctx.h
    xyz, faces = odd(7, 200, 600)
    nrm = np.ones_like(xyz)
    tx, tf, tn = _torch(xyz), _torch(faces), _torch(nrm)
    o, m = s3.OrientResultC(), s3.MeasureResultC()

    def orient(x=tx, n=tn, nv=len(xyz), f=tf, nf=len(faces), r=o):
        ptr = lambda t: t if t is None or isinstance(t, int) else t.data_ptr()
        return L.scan3d_mesh_orient_dev(h, ptr(x), ptr(n), nv, ptr(f), nf, C.byref(r) if r else None)

    def measure(x=tx, nv=len(xyz), f=tf, nf=len(faces), r=m):
        ptr = lambda t: t if t is None or isinstance(t, int) else t.data_ptr()
        return L.scan3d_mesh_measure_dev(h, ptr(x), nv, ptr(f), nf, C.byref(r) if r else None)

    def untouched():
        assert np.array_equal(tf.cpu().numpy(), faces) and np.array_equal(tn.cpu().numpy(), nrm)
        assert np.array_equal(tx.cpu().numpy(), xyz)

    before = ctx.launch_count()
    assert L.scan3d_mesh_orient_dev(None, tx.data_ptr(), tn.data_ptr(), len(xyz), tf.data_ptr(), len(faces),
                                    C.byref(o)) == ARG
    assert L.scan3d_mesh_measure_dev(None, tx.data_ptr(), len(xyz), tf.data_ptr(), len(faces), C.byref(m)) == ARG
    for kw in (dict(r=None), dict(nv=-1), dict(nv=1 << 31), dict(nf=-1), dict(nf=1 << 31), dict(x=None), dict(f=None),
               dict(x=tx.data_ptr() + 2), dict(f=tf.data_ptr() + 1)):
        assert orient(**kw) == ARG, kw
        assert measure(**kw) == ARG, kw
    assert orient(n=tn.data_ptr() + 2) == ARG
    assert orient(nf=(1 << 32) // 6 + 1) == CONFIG and measure(nf=(1 << 32) // 6 + 1) == CONFIG
    assert ctx.launch_count() == before
    untouched()
    # found on the device: a face index out of range, a coordinate that is not finite; nothing written
    bad_f = np.concatenate([faces[::-1], [[0, 1, len(xyz)]]]).astype(np.int32)
    tb = _torch(bad_f)
    assert orient(f=tb, nf=len(bad_f)) == ARG and b"face index" in L.scan3d_last_error(h)
    assert ctx.launch_count() == before + ORIENT_LAUNCHES
    assert np.array_equal(tb.cpu().numpy(), bad_f)
    assert measure(f=tb, nf=len(bad_f)) == ARG
    assert ctx.launch_count() == before + ORIENT_LAUNCHES + MEASURE_LAUNCHES
    xn = xyz.copy()
    xn[5, 1] = np.nan
    assert orient(x=_torch(xn)) == ARG and measure(x=_torch(xn)) == ARG
    untouched()
    with pytest.raises(s3.Scan3DError):
        ctx.mesh_orient_dev(tx, tf.long())
    with pytest.raises(s3.Scan3DError):
        ctx.mesh_orient_dev(tx, tf, tn[:5])
    with pytest.raises(s3.Scan3DError):
        ctx.mesh_measure_dev(tx[:, :2], tf)
    del tx, tf, tn, tb
    ctx.close()
