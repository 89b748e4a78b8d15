"""GPU checks of the non-manifold repair (scan3d_voxel_surface_repair, scan3d_mesh_repair_dev): byte parity with
repair_ref of tests/test_repair_ref.py for every flag combination on random odd meshes and constructed cases through
the dev route, the camera-grid mesh with ROI holes, a surface extracted from a thin shell and two touching spheres
(raw and after decimation) and an empty mesh; every call twice, byte-identical, with the stated launch count.  Also the
state rules (no surface, the stale component table, pinched spheres that become two components, decimation after a
raw repair, the decimation refusing a surface filled after a repair), every argument error, the errors found on the
device and the capacity error.  The ABI check needs no GPU."""
import ctypes as C
import importlib
import math

import numpy as np
import pytest

from test_decimate_ref import decimate_ref
from test_gpu_align import SMALL, _ctx, _torch
from test_gpu_components import CEN, S, _sphere
from test_gpu_mesh import _scene as _mesh_scene
from test_gpu_surface import _merge, _same, _surface
from test_repair_ref import FACES, FLAGS, VERTICES, apply_source, book, bowtie, odd, pinched_spheres, repair_ref

s3 = importlib.import_module("3dscan_b200")
gpu = pytest.mark.gpu

F32 = np.float32
LAUNCHES, LAUNCHES_BAD = 12, 10
ARG, STATE, CONFIG = -4, -3, -1
BOTH = FACES | VERTICES


def test_abi_symbols_resolve():
    L = C.CDLL(s3.cuda_lib()._name)
    for name in ("scan3d_voxel_surface_repair", "scan3d_mesh_repair_dev"):
        assert getattr(L, name)
    assert C.sizeof(s3.RepairResultC) == 80 and s3.RepairResultC.inconsistent_edges.offset == 72
    assert (s3.REPAIR_FACES, s3.REPAIR_VERTICES) == (1, 2)


def _flags_kw(flags):
    return dict(repair_faces=bool(flags & FACES), vertices=bool(flags & VERTICES))


def _dev(ctx, xyz, faces, flags):
    """the dev route on copies of the arrays, twice, against the reference; returns (faces, source, result)"""
    outs = []
    for _ in range(2):
        tx = _torch(np.ascontiguousarray(xyz, F32).reshape(-1, 3))
        tf = _torch(np.ascontiguousarray(faces, np.int32).reshape(-1, 3))
        before = ctx.launch_count()
        f, src, res = ctx.mesh_repair_dev(tx, tf, **_flags_kw(flags))
        assert ctx.launch_count() == before + LAUNCHES
        outs.append((f.cpu().numpy(), src.cpu().numpy(), res))
        assert np.array_equal(tf.cpu().numpy(), np.asarray(faces, np.int32).reshape(-1, 3))
    want, wsrc, info = repair_ref(xyz, faces, flags)
    for f, src, res in outs:
        _same((f, src), (want, wsrc))
        assert res == info
    return outs[0]


@gpu
def test_dev_route_random_and_constructed_meshes():
    ctx = _ctx()
    for flags in FLAGS:
        for seed in range(4):
            _dev(ctx, *odd(seed, 300, 900), flags)
        for mesh in (bowtie(), pinched_spheres(2), book(3, [1.0, 3.0, 0.5], [1, 1, -1]),
                     book(4, [1.0] * 4, [1, 1, -1, -1])):
            _dev(ctx, *mesh, flags)
        f, src, res = _dev(ctx, np.zeros((0, 3), F32), np.zeros((0, 3), np.int32), flags)
        assert len(f) == 0 and len(src) == 0 and res["vertices"] == 0
        _dev(ctx, np.ones((7, 3), F32), np.zeros((0, 3), np.int32), flags)
    ctx.close()


@gpu
def test_pinched_spheres_become_two_components():
    ctx = _ctx()
    xyz, faces = pinched_spheres(2)
    _, before = ctx.mesh_components_dev(_torch(faces), len(xyz))
    f, src, res = _dev(ctx, xyz, faces, BOTH)
    _, after = ctx.mesh_components_dev(_torch(f), res["vertices"])
    assert (before, after) == (1, 2) and res["boundary_edges"] == 0
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
    for flags in FLAGS:
        out = []
        for _ in range(2):
            dst = _torch(np.full((len(faces), 3), -7, np.int32))
            src = _torch(np.full(3 * len(faces), -7, np.int32))
            r = s3.RepairResultC()
            before = ctx.launch_count()
            assert L.scan3d_mesh_repair_dev(h, L.scan3d_device_points(h), n, L.scan3d_device_mesh_faces(h),
                                            len(faces), flags, dst.data_ptr(), src.data_ptr(), 3 * len(faces),
                                            C.byref(r)) == 0
            assert ctx.launch_count() == before + LAUNCHES
            res = s3.Scan3D._repair_result(r)
            out.append((dst.cpu().numpy()[:res["faces"]], src.cpu().numpy()[:res["vertices_added"]], res))
        want, wsrc, info = repair_ref(pts, faces, flags)
        for f, s, res in out:
            _same((f, s), (want, wsrc))
            assert res == info
        print(f"camera-grid mesh 640x480 with ROI holes, flags {flags}: {n} points, {len(faces)} faces, {info}")
    assert info["split_vertices"] > 0
    assert np.array_equal(ctx.mesh()[0], faces)
    ctx.close()


def _shell_and_touching_spheres(ctx):
    """a thin shell (two concentric spheres 0.6 voxel apart, the inner one facing in) and two spheres that touch"""
    parts = []
    p, n, c = _sphere(S, 1.0, CEN)
    q, m, d = _sphere(S, 1.0 - 0.6 * S, CEN)
    parts += [(p, n, c), (q, -m, d)]
    for k in (-1, 1):
        p, n, c = _sphere(S, 0.6, CEN + np.array([4.0 + k * 0.6, 0, 0]))
        parts.append((p, n, c))
    _merge(ctx, S, [tuple(np.concatenate(x) for x in zip(*parts))])


def _expected(raw, flags):
    out, src, info = repair_ref(raw[0], raw[3], flags)
    return (apply_source(raw[0], src), apply_source(raw[1], src), np.concatenate([raw[2], raw[2][src]]), out), info


def _repair(ctx, flags):
    before = ctx.launch_count()
    res = ctx.surface_repair(bool(flags & FACES), bool(flags & VERTICES))
    assert ctx.launch_count() == before + LAUNCHES
    return res, ctx.voxel_surface_mesh()


@gpu
def test_surface_route_shell_and_touching_spheres_raw_and_decimated():
    ctx = _ctx()
    _shell_and_touching_spheres(ctx)
    raw = _surface(ctx)[1]
    info = repair_ref(raw[0], raw[3], BOTH)[2]
    print(f"raw surface: {len(raw[0])} vertices, {len(raw[3])} faces, {info}")
    assert info["nonmanifold_edges"] > 0 and info["split_vertices"] > 0
    for flags in FLAGS:
        got = []
        for _ in range(2):
            _surface(ctx)
            got.append(_repair(ctx, flags))
        want, info = _expected(raw, flags)
        for res, mesh in got:
            _same(mesh, want)
            assert res == info
    # after decimation, which joins sheets in a cluster
    _surface(ctx)
    ctx.surface_decimate(F32(4 * S))
    dec = ctx.voxel_surface_mesh()
    want, info = _expected(dec, BOTH)
    print(f"decimated surface: {len(dec[0])} vertices, {len(dec[3])} faces, {info}")
    res, mesh = _repair(ctx, BOTH)
    _same(mesh, want)
    assert res == info
    # a second repair changes nothing
    res2, again = _repair(ctx, BOTH)
    _same(again, mesh)
    assert res2["vertices_added"] == res2["nonmanifold_faces"] == res2["duplicate_faces"] == 0
    ctx.close()


@gpu
def test_state_rules_and_the_decimation_after_a_repair():
    ctx = _ctx()
    L, h = ctx.L, ctx.h
    out = s3.RepairResultC()
    before = ctx.launch_count()
    assert L.scan3d_voxel_surface_repair(h, BOTH, C.byref(out)) == STATE          # before any surface
    assert ctx.launch_count() == before
    _shell_and_touching_spheres(ctx)
    raw = _surface(ctx)[1]
    ctx.surface_components(0, 0)
    # argument errors: nothing launched, the surface and the component table stay
    before = ctx.launch_count()
    for flags in (0, 4, -1, 3 | 8):
        assert L.scan3d_voxel_surface_repair(h, flags, C.byref(out)) == ARG, flags
    assert L.scan3d_voxel_surface_repair(None, BOTH, C.byref(out)) == ARG
    assert L.scan3d_voxel_surface_repair(h, BOTH, None) == ARG
    assert ctx.launch_count() == before
    _same(ctx.voxel_surface_mesh(), raw)
    assert L.scan3d_get_surface_components(h, None, None, None, 0) == 0
    # a repair makes the component table stale
    res, repaired = _repair(ctx, BOTH)
    assert res["vertices_added"] > 0
    assert L.scan3d_get_surface_components(h, None, None, None, 0) == STATE
    # a raw repaired surface stays decimatable: the decimation of the repaired mesh
    ctx.surface_decimate(F32(4 * S))
    _same(ctx.voxel_surface_mesh(), decimate_ref(repaired, S, F32(4 * S))[:4])
    # a fill after a repair that changed the surface stops the decimation until the next extraction; the cap stays 22
    _surface(ctx)
    ctx.surface_repair()
    fr = s3.FillResultC()
    assert L.scan3d_voxel_surface_fill_holes(h, 23, C.byref(fr)) == ARG
    assert L.scan3d_voxel_surface_fill_holes(h, 22, C.byref(fr)) == 0 and fr.faces_added > 0
    dr = s3.DecimateResultC()
    assert L.scan3d_voxel_surface_decimate(h, F32(4 * S), C.byref(dr)) == STATE
    assert b"filled after a repair" in L.scan3d_last_error(h)
    _surface(ctx)
    assert L.scan3d_voxel_surface_decimate(h, F32(4 * S), C.byref(dr)) == 0
    # a fill before the repair leaves it decimatable; a repair that changes nothing does not undo an earlier one
    _surface(ctx)
    ctx.surface_fill_holes(22)
    ctx.surface_repair()
    assert L.scan3d_voxel_surface_decimate(h, F32(4 * S), C.byref(dr)) == 0
    _surface(ctx)
    ctx.surface_repair()
    assert ctx.surface_repair()["vertices_added"] == 0
    ctx.surface_fill_holes(22)
    assert L.scan3d_voxel_surface_decimate(h, F32(4 * S), C.byref(dr)) == STATE   # the first repair changed it
    # the launch count is fixed, an empty surface included
    ctx.voxel_begin(S, 16)
    far = _torch(np.array([[1.0, 1.0, 1.0]], F32))
    ctx.voxel_add_dev(far, None, None)
    ctx.voxel_finish()
    empty = _surface(ctx)[1]
    assert len(empty[3]) == 0
    res, mesh = _repair(ctx, BOTH)
    assert res == repair_ref(empty[0], empty[3], BOTH)[2]
    _same(mesh, empty)
    del far
    ctx.close()


@gpu
def test_dev_route_errors_and_capacity():
    ctx = _ctx()
    L, h = ctx.L, ctx.h
    xyz, faces = odd(7, 200, 600)
    tx, tf = _torch(xyz), _torch(faces)
    dst = _torch(np.full((len(faces), 3), -7, np.int32))
    src = _torch(np.full(3 * len(faces), -7, np.int32))
    out = s3.RepairResultC()

    def call(x=tx, nv=len(xyz), f=tf, nf=len(faces), fl=BOTH, o=dst, s=src, cap=3 * len(faces), r=out):
        ptr = lambda t: t if t is None or isinstance(t, int) else t.data_ptr()
        return L.scan3d_mesh_repair_dev(h, ptr(x), nv, ptr(f), nf, fl, ptr(o), ptr(s), cap, C.byref(r) if r else None)

    def untouched():
        assert (dst.cpu().numpy() == -7).all() and (src.cpu().numpy() == -7).all()
        assert np.array_equal(tf.cpu().numpy(), faces) and np.array_equal(tx.cpu().numpy(), xyz)

    before = ctx.launch_count()
    assert L.scan3d_mesh_repair_dev(None, tx.data_ptr(), len(xyz), tf.data_ptr(), len(faces), BOTH, dst.data_ptr(),
                                    src.data_ptr(), len(faces), C.byref(out)) == ARG
    for kw in (dict(r=None), dict(fl=0), dict(fl=4), dict(nv=-1), dict(nv=1 << 31), dict(nf=-1), dict(nf=1 << 31),
               dict(cap=-1), dict(cap=1 << 31), dict(x=None), dict(f=None), dict(o=None), dict(s=None),
               dict(x=tx.data_ptr() + 2), dict(f=tf.data_ptr() + 1), dict(o=dst.data_ptr() + 2),
               dict(s=src.data_ptr() + 1), dict(o=tf)):
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
    # too small a source output: nothing written, *out filled; the wrapper retries once with that size
    want, wsrc, info = repair_ref(xyz, faces, BOTH)
    assert len(wsrc) > 1
    before = ctx.launch_count()
    assert call(cap=len(wsrc) - 1) == CONFIG and b"max_source_out" in L.scan3d_last_error(h)
    assert ctx.launch_count() == before + LAUNCHES_BAD
    untouched()
    assert s3.Scan3D._repair_result(out) == info
    assert call(cap=len(wsrc)) == 0
    _same((dst.cpu().numpy()[:len(want)], src.cpu().numpy()[:len(wsrc)]), (want, wsrc))
    bx, bf = book(4, [1.0] * 4, [1, 1, -1, -1])                     # more added vertices than faces
    f, s, res = ctx.mesh_repair_dev(_torch(bx), _torch(bf), repair_faces=False)
    _same((f.cpu().numpy(), s.cpu().numpy()), repair_ref(bx, bf, VERTICES)[:2])
    assert res["vertices_added"] == 6
    with pytest.raises(s3.Scan3DError):
        ctx.mesh_repair_dev(tx, tf.long())
    with pytest.raises(s3.Scan3DError):
        ctx.mesh_repair_dev(tx[:, :2], tf)
    del tx, tf, dst, src, bad_f
    ctx.close()
