"""GPU parity of the steps either side of the path (SURVEY.md 8 f2 / f4) through the C ABI:
cvUndistort2 (capture side), image_scissor's region fill, register_point_clouds' transform.
Bit-exact against the oracle (oracle/scan3d_oracle_f4.c) and the committed cv2 known answers."""
import ctypes as C
import os

import numpy as np
import pytest

import oracle_ffi as o
from gpu_common import calibs, s3
from helpers import GOLDEN

pytestmark = pytest.mark.gpu
LIBDIR = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "3dscan_b200", "lib")


def _ctx(W, H, PW, PH, cal):
    return s3.Scan3D(s3.make_config(W, H, PW, PH, 3, 4, 4, 8, 8, 2), 0, cal)


@pytest.mark.parametrize("W,H,dscale", [(640, 480, 1.0), (1600, 1200, 1.0), (1000, 37, 6.0), (333, 250, 3.0), (4096, 64, 1.0)])
def test_undistort_frames_match_oracle(W, H, dscale):
    cal, _, c = calibs(W / 1600.0, 0.5, dc=None)
    c["dc"] = c["dc"] * dscale
    cal = s3.make_calib(*[c[k] for k in ("Kc", "dc", "Kp", "dp", "rc", "tc", "rp", "tp")])
    ctx = _ctx(W, H, 640, 360, cal)
    xy, fr = ctx.undistort_map(0)
    oxy, ofr = o.undistort_map(c["Kc"], c["dc"], W, H)
    assert np.array_equal(xy, oxy) and np.array_equal(fr, ofr)
    frames = np.random.default_rng(W + H).integers(0, 256, (5, H, W), dtype=np.uint8)
    before = ctx.launch_count()
    out = ctx.undistort_frames(frames, 0)
    assert ctx.launch_count() == before + 1                    # the map is reused, one launch for all frames
    assert np.array_equal(out, o.undistort_frames(frames, c["Kc"], c["dc"]))
    # projector patterns go through the same call with (Kp, dp) (2/project_pattern.cpp:372): the reference's
    # projector has no distortion, so this must be the identity
    pat = np.random.default_rng(1).integers(0, 256, (2, 360, 640), dtype=np.uint8)
    assert np.array_equal(ctx.undistort_frames(pat, 1), pat)
    # a new calibration invalidates the cached map
    c2 = dict(c)
    c2["dc"] = np.array([-0.2, 0.05, 0.001, -0.002, 0.01])
    ctx.set_calibration(s3.make_calib(*[c2[k] for k in ("Kc", "dc", "Kp", "dp", "rc", "tc", "rp", "tp")]))
    assert np.array_equal(ctx.undistort_frames(frames[:1], 0), o.undistort_frames(frames[:1], c2["Kc"], c2["dc"]))
    ctx.close()


@pytest.mark.parametrize("W,H,dscale,frames", [(640, 480, 5.0, 20), (2048, 104, 1.0, 14), (256, 8, 2.0, 13), (1024, 61, -3.0, 7)])
def test_undistort_stack_longer_than_the_staging_ring(W, H, dscale, frames):
    """k_remap_tiled's ring of staged boxes is 6 frames deep: stacks longer than that reuse every stage (both phases
    of its mbarriers), with boxes that reach outside the image (strong distortion of either sign), partial tiles
    (W % 256 != 0, H % 8 != 0) and a single-tile image."""
    cal, _, c = calibs(W / 1600.0, 0.5, dc=None)
    c["dc"] = c["dc"] * dscale
    cal = s3.make_calib(*[c[k] for k in ("Kc", "dc", "Kp", "dp", "rc", "tc", "rp", "tp")])
    ctx = _ctx(W, H, 640, 360, cal)
    stack = np.random.default_rng(W * H + frames).integers(0, 256, (frames, H, W), dtype=np.uint8)
    want = o.undistort_frames(stack, c["Kc"], c["dc"])
    for _ in range(2):                                         # twice: the second launch starts from used barriers' memory
        assert np.array_equal(ctx.undistort_frames(stack, 0), want)
    ctx.close()


def test_undistort_frames_match_cv2_golden():
    g = np.load(os.path.join(GOLDEN, "f4_kat.npz"))
    _, _, c = calibs()
    for i in range(int(g["n_undistort"])):
        K, d, src, dst = g[f"und_K{i}"], g[f"und_d{i}"], g[f"und_src{i}"], g[f"und_dst{i}"]
        H, W = src.shape
        cal = s3.make_calib(K, d, c["Kp"], c["dp"], c["rc"], c["tc"], c["rp"], c["tp"])
        ctx = _ctx(W, H, 64, 64, cal)
        assert np.array_equal(ctx.undistort_frames(src[None], 0)[0], dst), i      # == cv2.undistort, bit for bit
        ctx.close()


def test_undistort_argument_checks():
    cal, _, _ = calibs(0.2, 0.2)
    ctx = s3.Scan3D(s3.make_config(320, 240, 256, 144, 3, 4, 4, 8, 8, 2), 0)
    img = np.zeros((1, 240, 320), np.uint8)
    with pytest.raises(s3.Scan3DError):
        ctx.undistort_frames(img, 0)                             # calibration missing
    ctx.set_calibration(cal)
    with pytest.raises(s3.Scan3DError):
        ctx.undistort_frames(img, 2)                             # bad device kind
    with pytest.raises(s3.Scan3DError):
        ctx.undistort_frames(np.zeros((1, 10, 10), np.uint8), 0)
    assert ctx.undistort_frames(img[:0], 0).shape == (0, 240, 320)
    ctx.close()


@pytest.mark.parametrize("W,H", [(320, 240), (1600, 1200), (97, 40), (4096, 16)])
def test_roi_fill_matches_reference_loop(W, H):
    rng = np.random.default_rng(W * 7 + H)
    outline = np.zeros((H, W), np.uint8)
    # a closed lasso (ellipse outline, concave on purpose via a second one) plus stray pixels
    yy, xx = np.mgrid[0:H, 0:W]
    e = ((xx - W * 0.45) / (W * 0.3)) ** 2 + ((yy - H * 0.5) / (H * 0.35)) ** 2
    outline[np.abs(e - 1.0) < 0.03] = 255
    e2 = ((xx - W * 0.8) / (W * 0.1)) ** 2 + ((yy - H * 0.4) / (H * 0.2)) ** 2
    outline[np.abs(e2 - 1.0) < 0.06] = 200
    outline[rng.random((H, W)) < 0.0005] = 1
    outline[0, :] = 0
    outline[H - 1, :] = 0
    outline[H - 1, W // 3] = 9                                   # a single pixel selects nothing
    ctx = s3.Scan3D(s3.make_config(W, H, 64, 64, 3, 4, 4, 8, 8, 2), 0)
    roi, filled = ctx.roi_fill(outline)
    oroi, ofilled = o.roi_fill(outline)
    assert np.array_equal(roi, oroi) and np.array_equal(filled, ofilled)
    assert roi[0].sum() == 0 and roi[H - 1].sum() == 0 and roi.sum() > 0
    ctx.close()


def test_register_points_match_oracle_and_cv2():
    g = np.load(os.path.join(GOLDEN, "f4_kat.npz"))
    pts, exp = g["reg_pts"], g["reg_out"]
    theta, t = float(g["reg_theta"]), [float(v) for v in g["reg_t"]]
    ctx = s3.Scan3D(s3.make_config(64, 64, 64, 64, 3, 4, 4, 8, 8, 2), 0)
    got = ctx.register_points(pts, theta, *t)
    assert np.array_equal(got.view(np.uint32), exp.view(np.uint32))           # == the cv2.gemm chain
    assert np.array_equal(s3.register_rotation(theta), g["reg_R"])
    big = (np.random.default_rng(4).normal(size=(1_000_003, 3)) * 500).astype(np.float32)
    for th in (0.0, 10.0, 180.0, 350.0):
        a = ctx.register_points(big, th, 1.5, -2.0, 880.0)
        b = o.register_points(big, th, 1.5, -2.0, 880.0)
        assert np.array_equal(a.view(np.uint32), b.view(np.uint32)), th
    assert ctx.register_points(big[:0], 10.0, 0, 0, 0).shape == (0, 3)
    ctx.close()


def test_register_point_clouds_call(tmp_path):
    """The reference's register_point_clouds(num, tx, ty, tz, rot_step) (m_tech_project_console.cpp:408) through
    libscan3d_compat.so: reads point_cloud_<i>.ply, writes registered_point_cloud.ply."""
    root = str(tmp_path / "M_tech_project_console")
    os.makedirs(f"{root}/Point_cloud")
    rng = np.random.default_rng(8)
    H = s3.host_lib()
    H.scan3d_write_ply_points.argtypes = [C.c_char_p, C.c_void_p, C.c_void_p, C.c_int64, C.c_int]
    clouds = []
    for i, n in enumerate((1000, 1, 2500)):
        xyz = (rng.normal(size=(n, 3)) * 50).astype(np.float32)
        rgb = rng.integers(0, 256, (n, 3), dtype=np.uint8)
        assert H.scan3d_write_ply_points(f"{root}/Point_cloud/point_cloud_{i}.ply".encode(), xyz.ctypes.data_as(C.c_void_p),
                                         rgb.ctypes.data_as(C.c_void_p), n, i % 2) == 0   # ascii and binary inputs
        clouds.append((xyz, rgb))
    s3.cuda_lib()
    L = C.CDLL(os.path.join(LIBDIR, "libscan3d_compat.so"))
    init = getattr(L, "_Z18scan3d_compat_initPKciiiii")
    init.argtypes = [C.c_char_p, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int]
    assert init(root.encode(), 320, 240, 256, 144, 0) == 0
    reg = getattr(L, "_Z21register_point_cloudsjffff")
    reg.argtypes = [C.c_uint, C.c_float, C.c_float, C.c_float, C.c_float]
    reg(3, 2.5, -1.0, 30.0, 36.0)
    body = open(f"{root}/Point_cloud/registered_point_cloud.ply").read().split("end_header\n")[1]
    rows = np.loadtxt(body.splitlines())
    assert rows.shape == (3501, 6)
    theta = np.float32(0.0)
    exp = []
    for xyz, _ in clouds:
        # the ascii round trip (%.9g) is exact for floats, so the oracle sees the same inputs
        exp.append(o.register_points(xyz, float(theta), 2.5, -1.0, 30.0))
        theta = np.float32(theta + np.float32(36.0))
    assert np.array_equal(rows[:, :3].astype(np.float32), np.concatenate(exp))
    assert np.array_equal(rows[:, 3:].astype(np.uint8), np.concatenate([r for _, r in clouds]))
    # image_scissor()'s fill through the same library: outline image in, selected_region global + i1.bmp out
    outline = np.zeros((240, 320), np.uint8)
    outline[40:200, 60] = 255
    outline[40:200, 250] = 255
    outline[120, 100] = 255
    fill = getattr(L, "_Z18image_scissor_fillPKh")
    fill.argtypes = [C.c_void_p]
    fill(outline.ctypes.data_as(C.c_void_p))
    oroi, ofilled = o.roi_fill(outline)
    sel = np.ctypeslib.as_array(C.cast(C.c_void_p.in_dll(L, "selected_region").value, C.POINTER(C.c_int)), shape=(320, 240))
    assert np.array_equal(sel.T, oroi.astype(np.int32))          # the reference's [col][row] layout
    assert np.array_equal(s3.read_bmp8(f"{root}/i1.bmp"), ofilled)
    getattr(L, "_Z22scan3d_compat_shutdownv")()


@pytest.mark.parametrize("shape", [(640, 480, 512, 288, 3, 7, 6, 4, 5), (1000, 40, 512, 288, 3, 7, 6, 4, 5),
                                   (256, 64, 8192, 8192, 8, 14, 14, 1, 1)])
def test_raw_entry_and_folded_registration_equal_the_separate_calls(shape):
    """SURVEY 8 f4: scan3d_reconstruct_raw (capture-side cvUndistort2 of every frame + the single-pass kernel, one call)
    with scan3d_set_registration (register_point_clouds' transform in the kernel's point store) gives, bit for bit,
    what scan3d_undistort_frames -> scan3d_reconstruct -> scan3d_register_points give (2/project_pattern.cpp:220-234,
    9/register_point_clouds.cpp:83-148).  The second shape takes the shape-generic stage route (W % 16 != 0); the
    third one's 72 frames take the single-pass kernel's launch shape with 2 CTAs per SM."""
    W, H, PW, PH, N, Mv, Mh, fwv, fwh = shape
    cal, ocal, _ = calibs(W / 1600.0, PW / 1280.0)
    cfg = s3.make_config(W, H, PW, PH, N, Mv, Mh, fwv, fwh, 2)
    raw, roi = s3.synth_stack(cfg, cal)
    theta, t = 36.0, (12.5, -3.25, 903.1)
    a = s3.Scan3D(cfg, 0, cal)
    und = a.undistort_frames(raw)
    n = a.reconstruct(und, roi)
    want = a.register_points(a.points(), theta, *t)
    cp = a.plane(s3.PLANE_CPMAP)
    a.close()
    b = s3.Scan3D(cfg, 0, cal)
    b.set_registration(True, theta, *t)
    n2 = b.reconstruct_raw(raw, roi)
    assert n2 == n and n > 1000
    assert np.array_equal(b.plane(s3.PLANE_CPMAP), cp)
    assert np.array_equal(b.points().view(np.uint32), want.view(np.uint32))
    b.set_registration(False)
    b.reconstruct_raw(raw, roi)
    assert not np.array_equal(b.points().view(np.uint32), want.view(np.uint32))
    b.close()
    # ... and the oracle's chain of the same three reference steps (exact triangulation order by default)
    from gpu_common import run_oracle
    _, _, c = calibs(W / 1600.0, PW / 1280.0)
    ref = run_oracle(cfg, ocal, o.undistort_frames(raw, c["Kc"], c["dc"]), roi)
    assert ref.count == n
    assert np.array_equal(o.register_points(ref.pts, theta, *t).view(np.uint32), want.view(np.uint32))
