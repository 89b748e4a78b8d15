"""GPU checks of the scan-to-model alignment (scan3d_align_to_voxels*): one iteration against the restatement of
tests/test_align_math_host.py, recovery of a known rigid offset, the ctx route on synthetic scans with a texture and a
mesh, degenerate models, the invariances the contract promises (repetition, stride, ctx vs device route, apply),
state rules, errors, launch counts and overflow."""
import ctypes as C
import math

import numpy as np
import pytest
from scipy.spatial.transform import Rotation

from gpu_common import calibs, s3
from test_align_math_host import (compose_ref, pairs_ref, products_ref, rodrigues_ref, rows_ref, solve_ref,
                                  transform_ref)

pytestmark = pytest.mark.gpu

C1 = (1600, 1200, 1280, 720, 3, 6, 5, 32, 32)
SMALL = (640, 480, 512, 288, 3, 7, 6, 4, 5)
CENTRE = (60.0, 40.0, -30.0)
F32 = np.float32


def _torch(a):
    import torch
    t = torch.from_numpy(np.ascontiguousarray(a)).cuda()
    torch.cuda.synchronize()      # the ctx works on its own stream
    return t


def _field(x, y):
    """a non-symmetric height field (mm) and its unit normals: every rigid DOF is constrained"""
    z = 3 * np.sin(x / 8) + 2 * np.cos(y / 10 + 0.4) + 0.005 * x * x + 0.003 * x * y
    fx = 3 / 8 * np.cos(x / 8) + 0.01 * x + 0.003 * y
    fy = -0.2 * np.sin(y / 10 + 0.4) + 0.003 * x
    n = np.stack([-fx, -fy, np.ones_like(x)], -1)
    return np.stack([x, y, z], -1), n / np.linalg.norm(n, axis=-1, keepdims=True)


def _rigid(deg, axis, t):
    T = np.eye(4)
    a = np.asarray(axis, float)
    T[:3, :3] = Rotation.from_rotvec(np.deg2rad(deg) * a / np.linalg.norm(a)).as_matrix()
    T[:3, 3] = t
    return T


S_FIELD = 0.2                                          # voxel of the height-field model (mm)


def _field_model(ctx):
    """voxel model of the height field sampled every 0.05 mm over [-20, 20)^2, added from device memory"""
    g = np.arange(-20, 20, 0.05)
    gx, gy = np.meshgrid(g, g)
    p, n = _field(gx.reshape(-1), gy.reshape(-1))
    ctx.voxel_begin(S_FIELD, p.shape[0])
    keep = [_torch(p.astype(F32)), _torch(n.astype(F32))]
    ctx.voxel_add_dev(*keep)
    ctx.voxel_finish()
    xyz, nrm, _, _ = ctx.voxels()
    return xyz, nrm


def _field_source(T_true, n=60000, seed=0):
    """surface samples at random (x, y), moved so that T_true maps them back onto the surface"""
    rng = np.random.default_rng(seed)
    p, _ = _field(rng.uniform(-15, 15, n), rng.uniform(-15, 15, n))
    Ti = np.linalg.inv(T_true)
    return (p @ Ti[:3, :3].T + Ti[:3, 3]).astype(F32)


def _ctx():
    W, H = 320, 240
    cal, _, _ = calibs(W / 1600.0, 256 / 1280.0)
    return s3.Scan3D(s3.make_config(W, H, 256, 144, 3, 6, 5, 8, 8, 2), 0, cal)


def _bits(r):
    return (r.T.tobytes(), r.iterations, r.status, r.pairs_first, r.pairs_last,
            np.float64(r.rms_first).tobytes(), np.float64(r.rms_last).tobytes())


def test_one_iteration_matches_the_restatement():
    ctx = _ctx()
    mxyz, mnrm = _field_model(ctx)
    T_true = _rigid(1.0, (0.3, -0.5, 0.8), (0.4, -0.3, 0.25))
    src = _field_source(T_true)
    T0 = _rigid(0.2, (1, 1, 0), (0.05, 0, -0.02))
    md = 2.0
    t = _torch(src)
    for stride in (1, 5):
        got = ctx.align_dev(t, md, max_iterations=1, stride=stride, T_init=T0, apply=False, stop_rotation=0.0,
                            stop_translation=0.0)
        x = src[::stride]
        p = transform_ref(T0, x)
        si, oi, _ = pairs_ref(p, mxyz, mnrm, md)
        J, r = rows_ref(p[si], mxyz[oi], mnrm[oi])
        assert got.pairs_first == got.pairs_last == si.size > 0.9 * x.shape[0]
        want_rms = math.sqrt(float(np.sum(r * r)) / si.size)
        assert abs(got.rms_first - want_rms) <= 1e-12 * want_rms
        ok, w = solve_ref(np.sum(products_ref(J, r), axis=0))
        assert ok
        _, dR, _ = rodrigues_ref(w[:3])
        want_T = compose_ref(dR, w[3:], T0)
        # the GPU's sums are reduced in another order than np.sum: T agrees to float64 rounding of ~1e4-term sums
        assert np.abs(got.T[:3].reshape(-1) - want_T).max() < 1e-9
        assert got.iterations == 1 and got.status == 1 and np.array_equal(got.T[3], [0, 0, 0, 1])
    ctx.close()


def test_coarse_then_fine_recovers_a_known_offset():
    """The model points are voxel centroids of a surface whose curvature is below 0.05 / mm: they lie within
    kappa s^2 / 8 = 2.5e-4 mm of it (s = 0.2 mm), and their normals average exact ones.  The source samples lie on the
    surface exactly, so the alignment error is bounded by that model error, far below the 1e-3 degree and 1e-2 s =
    2e-3 mm asserted (a B200 run and the host build both recover T to ~2e-5 degree and ~1e-5 mm)."""
    ctx = _ctx()
    _field_model(ctx)
    T_true = _rigid(1.0, (0.3, -0.5, 0.8), (0.4, -0.3, 0.25))    # about 1 degree and 2.8 voxels
    t = _torch(_field_source(T_true))
    coarse = ctx.align_dev(t, 2.0, stride=4, stop_translation=2e-4)
    fine = ctx.align_dev(t, 0.5, T_init=np.eye(4))
    E = fine.T @ coarse.T @ np.linalg.inv(T_true)
    rot = math.degrees(np.linalg.norm(Rotation.from_matrix(E[:3, :3]).as_rotvec()))
    print(coarse, fine, f"rotation error {rot:.3g} deg, translation error {np.linalg.norm(E[:3, 3]):.3g} mm")
    assert coarse.status == 0 and fine.status == 0
    assert rot < 1e-3 and np.linalg.norm(E[:3, 3]) < 1e-2 * S_FIELD
    assert fine.rms_last < 1e-3 < coarse.rms_first
    ctx.close()


def _scene(shape, params=None):
    W, H, PW, PH, N, Mv, Mh, fv, fh = shape
    cal, _, _ = calibs(W / 1600.0, PW / 1280.0)
    cfg = s3.make_config(W, H, PW, PH, N, Mv, Mh, fv, fh, 2)
    stack, roi = s3.synth_stack(cfg, cal, params)
    return cfg, cal, stack, roi


def _spacing(ctx):
    """median distance between the points of horizontally adjacent valid pixels"""
    pix = np.flatnonzero(ctx.plane(s3.PLANE_VALID).reshape(-1))
    p = ctx.points().astype(np.float64)
    adj = (pix[1:] == pix[:-1] + 1) & (pix[1:] % ctx.cfg.W != 0)
    d = np.linalg.norm(p[1:][adj] - p[:-1][adj], axis=1)
    return float(np.median(d[d > 0]))


def _rms_to_model(xyz, mxyz, mnrm, md):
    p = transform_ref(np.eye(4), xyz)
    si, oi, _ = pairs_ref(p, mxyz, mnrm, md)
    _, r = rows_ref(p[si], mxyz[oi], mnrm[oi])
    return math.sqrt(float(np.sum(r * r)) / si.size), si.size


def _view_model(ctx, stack, roi, s):
    """the model: the view at turntable angle 0 about CENTRE, with its mesh"""
    ctx.set_registration(True, 0.0, *CENTRE)
    n = ctx.reconstruct(stack, roi)
    ctx.build_mesh(math.inf)
    ctx.voxel_begin(s, n)
    ctx.voxel_add()
    ctx.voxel_finish()
    return ctx.points(), n


@pytest.mark.parametrize("shape", [SMALL, C1], ids=["640x480", "c1"])
def test_ctx_route_end_to_end(shape):
    cfg, cal, stack, roi = _scene(shape)
    ctx = s3.Scan3D(cfg, 0, cal)
    ctx.set_texture(np.random.default_rng(5).integers(0, 256, (cfg.H, cfg.W, 3), dtype=np.uint8))
    ctx.set_registration(True, 0.0, *CENTRE)
    ctx.reconstruct(stack, roi)
    s = 2.0 * _spacing(ctx)
    view0, _ = _view_model(ctx, stack, roi, s)
    mxyz, mnrm, mrgb, mcnt = ctx.voxels()
    before = b"".join(a.tobytes() for a in (mxyz, mnrm, mrgb, mcnt))
    fine_md = 4.0 * s
    rms0, _ = _rms_to_model(view0, mxyz, mnrm, fine_md)
    # the same stack, registered with a perturbed angle and pivot
    ctx.set_registration(True, 0.6, CENTRE[0] + 0.3, CENTRE[1], CENTRE[2] - 0.2)
    ctx.reconstruct(stack, roi)
    ctx.build_mesh(math.inf)
    perturbed = ctx.points()
    L, h = ctx.L, ctx.h
    nf = C.c_int64()
    launches = ctx.launch_count()
    coarse = ctx.align(max(10 * s, 2.0), stride=4, max_iterations=20)
    assert ctx.launch_count() == launches + 3 + 2 * 20 + 1
    assert L.scan3d_mesh_face_count(h, C.byref(nf)) == -3             # the points moved: the mesh is stale
    fine = ctx.align(fine_md, T_init=np.eye(4))
    aligned = ctx.points()
    rms_after, pairs = _rms_to_model(aligned, mxyz, mnrm, fine_md)
    rms_before, _ = _rms_to_model(perturbed, mxyz, mnrm, fine_md)
    print(f"voxel {s:.4f}: rms {rms_before:.4g} -> {rms_after:.4g} (view 0 against its own merge {rms0:.4g}); "
          f"coarse {coarse}, fine {fine}")
    assert fine.status in (0, 1) and coarse.status in (0, 1)
    assert abs(rms_after - fine.rms_last) <= 0.02 * fine.rms_last + 1e-6 * s
    assert rms_after <= 1.5 * rms0 + 1e-3 * s and rms_after < 0.5 * rms_before
    assert pairs >= 0.9 * aligned.shape[0]
    # the merge is untouched, the mesh is stale until rebuilt
    got = ctx.voxels()
    assert b"".join(a.tobytes() for a in got) == before
    assert L.scan3d_mesh_face_count(h, C.byref(nf)) == -3
    ctx.build_mesh(math.inf)
    assert L.scan3d_mesh_face_count(h, C.byref(nf)) == 0 and nf.value > 0
    ctx.close()


def test_plane_alone_and_a_model_without_normals():
    cfg, cal, stack, roi = _scene(SMALL, s3.default_synth_params(sphere_r=0.0))
    ctx = s3.Scan3D(cfg, 0, cal)
    ctx.set_registration(True, 0.0, *CENTRE)
    ctx.reconstruct(stack, roi)
    s = 2.0 * _spacing(ctx)
    view0, _ = _view_model(ctx, stack, roi, s)
    mxyz, mnrm, _, _ = ctx.voxels()
    rms0, _ = _rms_to_model(view0, mxyz, mnrm, 4 * s)
    ctx.set_registration(True, 0.4, CENTRE[0] + 0.2, CENTRE[1], CENTRE[2])
    ctx.reconstruct(stack, roi)
    res = ctx.align(4 * s, max_iterations=30)
    rms_after, _ = _rms_to_model(ctx.points(), mxyz, mnrm, 4 * s)
    print(res, rms0, rms_after)
    assert np.isfinite(res.T).all() and res.status in (0, 1)
    assert rms_after <= 1.5 * rms0 + 1e-3 * s
    # a model whose view had no mesh: every normal is zero, so there is no pair and T stays T_init
    ctx.set_registration(True, 0.0, *CENTRE)
    ctx.reconstruct(stack, roi)
    ctx.voxel_begin(s, cfg.W * cfg.H)
    ctx.voxel_add()
    ctx.voxel_finish()
    assert not ctx.voxels()[1].any()
    T0 = _rigid(0.5, (0, 1, 0), (0.1, 0.2, 0.3))
    res = ctx.align(4 * s, T_init=T0, apply=False)
    assert (res.status, res.iterations, res.pairs_first, res.pairs_last, res.rms_first) == (2, 0, 0, 0, 0.0)
    assert np.array_equal(res.T, T0)
    ctx.close()


def test_invariances():
    import torch
    cfg, cal, stack, roi = _scene(SMALL)
    ctx = s3.Scan3D(cfg, 0, cal)
    ctx.set_registration(True, 0.0, *CENTRE)
    ctx.reconstruct(stack, roi)
    s = 2.0 * _spacing(ctx)
    _view_model(ctx, stack, roi, s)
    ctx.set_registration(True, 0.5, *CENTRE)
    n = ctx.reconstruct(stack, roi)
    xyz = ctx.points()
    md = 3.0
    kw = dict(max_iterations=6, apply=False, stop_rotation=0.0, stop_translation=0.0)
    # the ctx route and the device route agree bit for bit; two runs too
    a = ctx.align(md, **kw)
    t = _torch(xyz)
    b = ctx.align_dev(t, md, **kw)
    c = ctx.align_dev(t, md, **kw)
    assert _bits(a) == _bits(b) == _bits(c) and a.iterations == 6 and a.pairs_first > 0.9 * n
    # stride k is the device route on xyz[::k]
    for k in (2, 7):
        sk = ctx.align_dev(t, md, stride=k, **kw)
        dk = ctx.align_dev(_torch(xyz[::k]), md, **kw)
        assert _bits(sk) == _bits(dk) and sk.pairs_first < a.pairs_first
    # apply: register_point's float order with R = (float)T and a zero pivot
    res = ctx.align_dev(t, md, max_iterations=6, apply=True)
    ctx.sync()
    R = res.T.astype(F32)
    x = xyz.astype(F32)
    want = np.empty_like(x)
    for i in range(3):
        acc = R[i, 0] * (x[:, 0] - F32(0))
        acc = acc + R[i, 1] * (x[:, 1] - F32(0))
        acc = acc + R[i, 2] * (x[:, 2] - F32(0))
        acc = acc + R[i, 3] * F32(1)
        want[:, i] = acc + F32(0)
    assert np.array_equal(t.cpu().numpy().view(np.uint32), want.view(np.uint32))
    # the ctx route applies the same
    ctx.align(md, max_iterations=6, apply=True)
    assert np.array_equal(ctx.points().view(np.uint32), want.view(np.uint32))
    del t
    torch.cuda.synchronize()
    ctx.close()


def test_state_errors_launch_counts_and_overflow():
    import torch
    ctx = _ctx()
    L, h = ctx.L, ctx.h
    buf = torch.zeros((1000, 3), dtype=torch.float32, device="cuda")
    ptr = buf.data_ptr()
    r = s3.AlignResultC()

    def params(**kw):
        a = dict(max_distance=1.0, max_iterations=5, stride=1, T_init=None, apply=False, stop_rotation=0.0,
                 stop_translation=0.0)
        a.update(kw)
        return s3.Scan3D._align_params(**a)

    def dev(p, n=1000, x=ptr):
        return L.scan3d_align_to_voxels_dev(h, C.c_void_p(x), n, C.byref(p), C.byref(r))

    ok = params()
    assert dev(ok) == -3                                           # before begin
    ctx.voxel_begin(0.2, 100000)
    assert dev(ok) == -3                                           # before the first finish
    g = np.arange(-5, 5, 0.05)
    gx, gy = np.meshgrid(g, g)
    p, n = _field(gx.reshape(-1), gy.reshape(-1))
    tp, tn = _torch(p.astype(F32)), _torch(n.astype(F32))
    ctx.voxel_add_dev(tp, tn)
    ctx.voxel_finish()
    assert dev(ok) == 0
    assert L.scan3d_align_to_voxels(h, C.byref(ok), C.byref(r)) == -3    # the ctx has no points
    assert b"points" in L.scan3d_last_error(h)
    ctx.voxel_add_dev(tp, tn)
    assert dev(ok) == -3                                           # stale: an add after the finish
    ctx.voxel_finish()
    # argument errors
    assert L.scan3d_align_to_voxels_dev(h, C.c_void_p(ptr), 10, None, C.byref(r)) == -4
    assert L.scan3d_align_to_voxels_dev(h, C.c_void_p(ptr), 10, C.byref(ok), None) == -4
    assert L.scan3d_align_to_voxels(h, None, C.byref(r)) == -4
    for bad in (dict(max_distance=0.0), dict(max_distance=-1.0), dict(max_distance=math.nan),
                dict(max_distance=math.inf), dict(max_iterations=0), dict(max_iterations=65), dict(stride=0),
                dict(stop_rotation=-1.0), dict(stop_translation=math.nan),
                dict(T_init=np.diag([1.01, 1, 1, 1])), dict(T_init=np.diag([1.0, 1, -1, 1])),
                dict(T_init=np.array([[1, 0, 0, 0], [0, 1, 0, 0], [0, 0, 1, 0], [0, 0, 1e-3, 1.0]])),
                dict(T_init=np.array([[1, 0, 0, math.nan], [0, 1, 0, 0], [0, 0, 1, 0], [0, 0, 0, 1.0]]))):
        assert dev(params(**bad)) == -4, bad
    assert dev(ok, n=-1) == -4
    assert dev(ok, x=ptr + 2) == -4
    assert dev(ok, n=5, x=0) == -4
    assert dev(ok, n=0, x=0) == 0                                  # an empty source: no pairs
    assert r.status == 2 and r.pairs_first == 0
    assert dev(params(T_init=_rigid(30, (1, 2, 3), (1, 2, 3)), max_iterations=64)) == 0    # a rotation within 1e-6
    # launch counts: fixed, whatever the run does
    for iters, apply, extra in ((5, False, 0), (5, True, 1), (64, False, 0), (1, True, 1)):
        before = ctx.launch_count()
        assert dev(params(max_iterations=iters, apply=apply, stop_rotation=1e-3, stop_translation=1e-3)) == 0
        assert ctx.launch_count() == before + 3 + 2 * iters + extra
    before = ctx.launch_count()
    assert dev(params(apply=True), n=0, x=0) == 0
    assert ctx.launch_count() == before + 3 + 2 * 5                # nothing to apply
    # an overflowed accumulator is reported after the run, nothing is applied
    ctx.voxel_begin(0.2, 10)
    ctx.voxel_add_dev(tp, tn)
    ctx.voxel_finish()
    keep = buf.clone()
    assert dev(params(apply=True)) == -1
    assert b"max_voxels" in L.scan3d_last_error(h)
    torch.cuda.synchronize()
    assert torch.equal(buf, keep)
    ctx.close()
    # one direction only: no point cloud to align
    W, H = 320, 240
    one = s3.Scan3D(s3.make_config(W, H, 256, 144, 3, 6, 5, 8, 8, 1), 0)
    one.voxel_begin(0.2, 100000)
    one.voxel_add_dev(tp, tn)
    one.voxel_finish()
    assert L.scan3d_align_to_voxels(one.h, C.byref(ok), C.byref(r)) == -3
    assert L.scan3d_align_to_voxels_dev(one.h, C.c_void_p(ptr), 1000, C.byref(ok), C.byref(r)) == 0
    one.close()
    del buf
