"""Pins the CPU oracle against everything the reference tree holds for the path
(SURVEY.md 8c): the stored wrapped / unwrapped phase images of its own scan (bit-for-bit),
the Relative_geometry XML (Rodrigues + composition), and cv2 4.13 known answers for the
OpenCV arithmetic (undistort, Rodrigues, gemm/invert triangulation chain)."""
import os

import numpy as np
import pytest

import oracle_ffi as o
from helpers import GOLDEN, load_c1_crop, load_c1_full, load_calib_c1, scaled_calib


def _stage34(fr, g, gi, gw, direction):
    valid = (gw != 0).astype(np.int32)          # post-recurrence mask stored by the reference
    w, dbg = o.wrapped_phase(fr, valid)
    code = o.decode_gray(g, gi, valid)
    w2, unw = o.unwrap(direction, w, code, valid)
    return valid, w, dbg, code, w2, unw


@pytest.mark.parametrize("key,direction,codes", [("v", 0, 40), ("h", 1, 23)])
def test_c1_crop_matches_reference_images(key, direction, codes):
    d = load_c1_crop()
    valid, w, dbg, code, w2, unw = _stage34(d[f"fringe_{key}"], d[f"gray_{key}"], d[f"inv_{key}"],
                                            d[f"golden_wrapped_{key}"], direction)
    assert valid.sum() > 50000
    m = valid == 1
    assert np.array_equal(dbg[m], d[f"golden_wrapped_{key}"][m])
    img = o.unwrapped_image(unw, valid, codes)
    # the crop's first/last column (vertical) or row (horizontal) is skipped by unwrap()
    inner = m.copy()
    if direction == 0:
        inner[:, 0] = inner[:, -1] = False
    else:
        inner[0, :] = inner[-1, :] = False
    assert np.array_equal(img[inner], d[f"golden_unwrapped_{key}"][inner])
    assert (code[~m] == -1).all() and (code[m] >= 0).all()


@pytest.mark.parametrize("name,M,direction,codes", [("Vertical", 6, 0, 40), ("Horizontal", 5, 1, 23)])
def test_full_frame_matches_reference_images(name, M, direction, codes):
    """The reference's whole 1600x1200 scan and its stored stage-3/4 images (tests/golden/c1_full.npz)."""
    d = load_c1_full()
    key = name[0].lower()
    fr, g, gi = d[f"fringe_{key}"], d[f"gray_{key}"], d[f"inv_{key}"]
    assert len(g) == len(gi) == M
    gw, gu = d[f"golden_wrapped_{key}"], d[f"golden_unwrapped_{key}"]
    valid, w, dbg, code, w2, unw = _stage34(fr, g, gi, gw, direction)
    assert int(valid.sum()) == 358580
    m = valid == 1
    assert np.array_equal(dbg[m], gw[m])
    img = o.unwrapped_image(unw, valid, codes)
    assert np.array_equal(img[m], gu[m])
    assert (gu[~m] == 0).all()


def test_relative_geometry_kat():
    c = load_calib_c1()
    R, T = o.compose_relative(c["rc"], c["tc"], c["rp"], c["tp"])
    assert np.abs(R - c["rel_R"].reshape(3, 3)).max() <= 1e-15
    assert np.abs(T - c["rel_T"]).max() <= 1e-13


def test_opencv_known_answers_bit_exact():
    k = np.load(os.path.join(GOLDEN, "opencv_kat.npz"))
    for dist, want in zip(k["und_dists"], k["und_out"]):
        got = o.undistort_points(k["und_pts"], k["und_K"], dist)
        assert np.array_equal(got, want)
    for r, want in zip(k["rod_in"], k["rod_out"]):
        assert np.array_equal(o.rodrigues(r), want)
    c = load_calib_c1()
    Ac = o.compute_A(c["Kc"], c["rc"], c["tc"])
    Ap = o.compute_A(c["Kp"], c["rp"], c["tp"])
    assert np.array_equal(Ac, k["A_cam"]) and np.array_equal(Ap, k["A_proj"])
    for (uc, vc, up, vp), want in zip(k["tri_in"][:1024], k["tri_out"][:1024]):
        assert np.array_equal(o.triangulate_point(Ac, Ap, uc, vc, up, vp), want)


def test_undistort_lut_matches_pointwise():
    c = load_calib_c1()
    W, H = 64, 48
    lut = o.undistort_lut(c["Kc"], c["dc"], W, H)
    yy, xx = np.mgrid[0:H, 0:W]
    pts = np.stack([xx.ravel(), yy.ravel()], 1).astype(np.float64)
    n = o.undistort_points(pts, c["Kc"], c["dc"])
    K = c["Kc"].reshape(3, 3)
    u = (K[0, 0] * n[:, 0] + K[0, 1] * n[:, 1]) + K[0, 2]
    v = (K[1, 0] * n[:, 0] + K[1, 1] * n[:, 1]) + K[1, 2]
    assert np.array_equal(lut[0].ravel(), u) and np.array_equal(lut[1].ravel(), v)
    # zero distortion: identity up to the (x-cx)*ifx*fx+cx round trip
    lutp = o.undistort_lut(c["Kp"], c["dp"], W, H)
    assert np.abs(lutp[0] - xx).max() < 1e-9 and np.abs(lutp[1] - yy).max() < 1e-9


@pytest.mark.parametrize("seed", range(6))
def test_mask_closed_form_equals_sequential(seed):
    rng = np.random.default_rng(seed)
    H, W = int(rng.integers(3, 40)), int(rng.integers(3, 40))
    p = [0.5, 0.8, 0.95, 0.99, 0.2, 1.0][seed]
    v0 = (rng.random((H, W)) < p).astype(np.int32)
    assert np.array_equal(o.mask_recurrence(v0), o.mask_closed_form(v0))


def test_mask_edge_shapes():
    for H, W in ((1, 1), (1, 7), (7, 1), (2, 2), (3, 3), (2, 9)):
        v0 = np.ones((H, W), np.int32)
        v0.flat[0] = 0
        assert np.array_equal(o.mask_recurrence(v0), o.mask_closed_form(v0))


def test_quirks():
    # tie in Gray threshold decodes as 1; bit 0 is the MSB; code is not range-limited
    g = np.array([[[7]], [[9]], [[3]]], np.uint8)
    gi = np.array([[[7]], [[9]], [[200]]], np.uint8)
    code = o.decode_gray(g, gi, np.ones((1, 1), np.int32))
    # G = 1,1,0 -> B = 1,0,0 -> code = 4
    assert code[0, 0] == 4
    assert o.decode_gray(g, gi, np.zeros((1, 1), np.int32))[0, 0] == -1
    # unwrap: Pi is 22/7 and is stored back into the wrapped plane; border col skipped
    w = np.full((3, 4), 0.5, np.float32)
    c = np.full((3, 4), 3, np.int32)
    w2, u = o.unwrap(0, w, c, np.ones((3, 4), np.int32))
    want_w = np.float32(np.float64(np.float32(0.5)) + 22.0 / 7.0)
    want_u = np.float32(np.float64(want_w) + 3 * 2.0 * 22.0 / 7.0)
    assert (w2[:, 1:3] == want_w).all() and (u[:, 1:3] == want_u).all()
    assert (w2[:, [0, 3]] == np.float32(0.5)).all() and (u[:, [0, 3]] == 0).all()
    w2, u = o.unwrap(1, w, c, np.ones((3, 4), np.int32))
    assert (u[1, :] == want_u).all() and (u[[0, 2], :] == 0).all()
    # lrint half-to-even + bounds reject keeps the computed value
    unw = np.array([[np.float32(0.5 * 44.0 / 7.0 / 1.0)]], np.float32)
    cp, valid = o.compute_c_p_map(unw * 0 + np.float32(2.5 * (44.0 / 7.0)), unw * 0, np.ones((1, 1), np.int32),
                                  np.ones((1, 1), np.int32), 1, 1, 10, 10)
    assert cp[0, 0] in (2, 3) and valid[0, 0] == 1
    cp, valid = o.compute_c_p_map(unw * 0 + 1000.0, unw * 0, np.ones((1, 1), np.int32),
                                  np.ones((1, 1), np.int32), 4, 4, 10, 10)
    assert valid[0, 0] == 0 and cp[0, 0] == int(np.rint(4 * (1000.0 / (44.0 / 7.0))))


def test_fdlibm_atan2f_restatement_equals_libm():
    """the 5-step formula calls float atan2f (3/wrapped_phase.cpp:220); the CUDA path mirrors
    glibc's fdlibm operation sequence, pinned here against this machine's libm on every
    (t1, t2) the 5-step formula can produce."""
    import ctypes
    L = o.lib()
    L.o3d_atan2f_restated_mismatches.restype = ctypes.c_long
    assert L.o3d_atan2f_restated_mismatches() == 0


def test_modulation_criterion_restatement_all_triples():
    """The commented-out criterion of check_I_mod_criteria (3/wrapped_phase.cpp:84-104) over every
    (I0, I1, I2) triple, against a literal numpy transcription of the expression's C types."""
    v = np.arange(256, dtype=np.int64)
    i0, i1, i2 = np.meshgrid(v, v, v, indexing="ij")
    fr = np.stack([i0, i1, i2]).astype(np.uint8).reshape(3, 4096, 4096)
    roi = np.ones((4096, 4096), np.uint8)
    got = o.check_I_mod_criteria(fr, roi)
    a, b, c = (fr[k].astype(np.float64) for k in range(3))
    t1 = np.sqrt((3.0 * (a - c) ** 2 + (2.0 * b - a - c) ** 2).astype(np.float32))   # sqrtf(float arg)
    t2 = (a + b + c).astype(np.float32)
    with np.errstate(divide="ignore", invalid="ignore"):
        t3 = (t1 / t2).astype(np.float32)                                            # float division
        want = (t3.astype(np.float64) > 0.01).astype(np.int32)                      # NaN (0/0) -> 0
    assert t1.dtype == np.float32 and np.array_equal(got, want)
    assert got[0, 0] == 0 and 0 < got.sum() < got.size            # black pixel rejected; both outcomes occur
    roi[:, ::2] = 0
    assert np.array_equal(o.check_I_mod_criteria(fr, roi), want * (roi != 0))


def test_quirk_check_I_mod_criteria_as_committed():
    """3/wrapped_phase.cpp:106-127: the valid map is filled from selected_region == 1 only for N == 3 or 4; the 5-step
    block is commented out.  o3d_check_roi_strict is that literal form, o3d_check_roi the default (documented)
    extension: any non-zero byte, every N."""
    import ctypes as C
    roi = np.array([[0, 1, 2, 255, 1, 0, 1, 1]], np.uint8)
    out = np.empty(roi.shape, np.int32)
    L = o.lib()
    for N, want in ((3, [0, 1, 0, 0, 1, 0, 1, 1]), (4, [0, 1, 0, 0, 1, 0, 1, 1]), (5, [0] * 8), (8, [0] * 8)):
        L.o3d_check_roi_strict(roi.ctypes.data_as(C.c_void_p), N, roi.shape[1], roi.shape[0], out.ctypes.data_as(C.c_void_p))
        assert out.ravel().tolist() == want, N
    assert o.check_roi(roi).ravel().tolist() == [0, 1, 1, 1, 1, 0, 1, 1]


def test_colrow_layout_leg_equals_the_row_major_oracle():
    """o3d_reconstruct_colrow (BASELINE.md section 3: the reference's [col][row] planes, row-outer loops, one thread)
    produces exactly the planes, c_p_map and points of o3d_reconstruct -- the layout changes the memory traffic of the
    timed CPU leg, not a single value."""
    import importlib
    s3 = importlib.import_module("3dscan_b200")
    W, H, PW, PH = 336, 200, 256, 160
    c = scaled_calib(load_calib_c1(), W / 1600.0, PW / 1280.0)
    args = [c[k] for k in ("Kc", "dc", "Kp", "dp", "rc", "tc", "rp", "tp")]
    ocal = o.make_calib(*args)
    for N, M in ((3, 6), (8, 7)):
        cfg = s3.make_config(W, H, PW, PH, N, M, M, 4, 4, 2)
        stack, roi = s3.synth_stack(cfg, s3.make_calib(*args))
        d = s3.split_stack(cfg, stack)
        cd = {k: getattr(cfg, k) for k in ("W", "H", "PW", "PH", "N", "M_v", "M_h", "fw_v", "fw_h", "dirs")}
        inp = (d["fringe_v"], d["gray_v"], d["inv_v"], d["fringe_h"], d["gray_h"], d["inv_h"], roi)
        a = o.reconstruct(cd, ocal, *inp, threads=2)
        b = o.reconstruct(cd, ocal, *inp, colrow=True)
        assert a.count == b.count > 1000
        for name in ("valid_v", "valid_h", "valid", "code_v", "code_h"):
            assert np.array_equal(getattr(a, name), getattr(b, name)), name
        for name in ("wrapped_v", "wrapped_h", "unwrapped_v", "unwrapped_h"):
            assert np.array_equal(getattr(a, name).view(np.uint32), getattr(b, name).view(np.uint32)), name
        assert np.array_equal(a.cpmap, b.cpmap) and np.array_equal(a.pix, b.pix)
        assert np.array_equal(a.pts.view(np.uint32), b.pts.view(np.uint32))
        m = a.valid == 1
        assert np.array_equal(a.xyz[m], b.xyz[m])
