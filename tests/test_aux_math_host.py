"""CPU checks of the arithmetic the auxiliary CUDA kernels evaluate (SURVEY.md 8 f2 / f4): the shared
header 3dscan_b200/common/scan3d_aux_math.h is compiled for the host and compared with the oracle
(oracle/scan3d_oracle_f4.c) and with the committed cv2 known answers (tests/golden/f4_kat.npz)."""
import ctypes as C
import os
import subprocess

import numpy as np
import pytest

import oracle_ffi as o
from helpers import GOLDEN, load_calib_c1

HERE = os.path.dirname(os.path.abspath(__file__))


@pytest.fixture(scope="module")
def shim(tmp_path_factory):
    so = str(tmp_path_factory.mktemp("auxhost") / "libaux_math_host.so")
    subprocess.check_call(["/usr/bin/g++", "-O2", "-std=c++17", "-fPIC", "-shared", "-Wall", "-ffp-contract=off",
                           "-o", so, os.path.join(HERE, "aux_math_host.cpp")])
    return C.CDLL(so)


def _p(a):
    return a.ctypes.data_as(C.c_void_p)


def _cases():
    c = load_calib_c1()
    rng = np.random.default_rng(11)
    out = [(640, 480, c["Kc"].reshape(3, 3) * np.array([[0.4], [0.4], [1.0]]), c["dc"]),
           (1600, 64, c["Kc"].reshape(3, 3), c["dc"] * 4)]
    for W, H, skew in ((333, 250, 0.0), (800, 37, 0.7), (4096, 8, 0.0), (5000, 6, 0.0)):
        K = np.array([[W * 0.9 + rng.normal() * 10, skew, W / 2 + rng.normal() * 20],
                      [0, W * 0.92 + rng.normal() * 10, H / 2 + rng.normal() * 20], [0, 0, 1]])
        d = np.array([rng.normal() * 0.2, rng.normal() * 0.2, rng.normal() * 0.01, rng.normal() * 0.01, rng.normal() * 0.1])
        out.append((W, H, K, d))
    return out


def _host_map(shim, K, d, W, H):
    K = np.ascontiguousarray(K, np.float64)
    d = np.ascontiguousarray(d, np.float64)
    xy = np.empty((H, W, 2), np.int16)
    fr = np.empty((H, W), np.uint16)
    shim.s3a_host_undistort_map(_p(K), _p(d), W, H, _p(xy), _p(fr))
    return xy, fr


def _host_remap(shim, img, xy, fr):
    img = np.ascontiguousarray(img, np.uint8)
    H, W = img.shape
    out = np.empty_like(img)
    shim.s3a_host_remap(_p(img), W, H, _p(xy), _p(fr), _p(out))
    return out


def test_undistort_map_and_remap_match_oracle(shim):
    rng = np.random.default_rng(5)
    for W, H, K, d in _cases():
        xy, fr = _host_map(shim, K, d, W, H)
        oxy, ofr = o.undistort_map(K, d, W, H)
        assert np.array_equal(xy, oxy) and np.array_equal(fr, ofr), (W, H)
        img = rng.integers(0, 256, (H, W), dtype=np.uint8)
        assert np.array_equal(_host_remap(shim, img, xy, fr), o.undistort_frames(img[None], K, d)[0]), (W, H)


def test_tiled_remap_arithmetic_matches_oracle(shim):
    """k_remap_tiled's arithmetic on the host (the tile's source box staged row by row in a buffer with the kernel's
    pitch, the taps of a pixel pair cut out of two words per row by one byte permute, doubled weight pairs, two-way
    dot products, byte 2 of the accumulators packed) gives the oracle's pixels; with the reference's calibration
    almost every tile qualifies for staging, and the strongly distorted cases exercise the pairs that do not
    qualify for the shared window."""
    shim.s3a_host_remap_tiled.restype = C.c_longlong
    rng = np.random.default_rng(7)
    c = load_calib_c1()
    K12 = c["Kc"].reshape(3, 3) * np.array([[2.56], [2.56], [1.0]])
    cases = [(1600, 1200, c["Kc"].reshape(3, 3), c["dc"], 0.99), (4096, 64, K12, c["dc"], 0.9),
             (640, 480, c["Kc"].reshape(3, 3) * np.array([[0.4], [0.4], [1.0]]), c["dc"] * 8, 0.0),
             (800, 48, np.array([[700.0, 0.7, 400.0], [0, 705.0, 20.0], [0, 0, 1]]), np.array([-0.3, 0.1, 0.01, -0.01, 0.0]), 0.0),
             (1280, 720, c["Kp"].reshape(3, 3), c["dp"], 0.95)]
    seen_irregular = 0
    for W, H, K, d, min_staged in cases:
        xy, fr = _host_map(shim, K, d, W, H)
        img = rng.integers(0, 256, (H, W), dtype=np.uint8)
        out = np.zeros_like(img)
        irregular = C.c_longlong(0)
        staged = shim.s3a_host_remap_tiled(_p(img), W, H, _p(xy), _p(fr), _p(out), C.byref(irregular))
        assert np.array_equal(out, o.undistort_frames(img[None], K, d)[0]), (W, H)
        tiles = -(-W // 256) * -(-H // 8)
        assert staged >= min_staged * tiles, (W, H, staged, tiles)
        seen_irregular += irregular.value
    assert seen_irregular > 100                          # the fix-up path is covered


def test_doubled_weights_give_the_reference_byte(shim):
    """bilinear_weight_pairs_x2 (weights doubled so that the result is a whole byte of the accumulator, the one weight
    that overflows 16 bits saturated) == bilinear_u8 for every fraction, on extreme and random taps."""
    rng = np.random.default_rng(11)
    taps = [(0, 0, 0, 0), (255, 255, 255, 255), (255, 0, 0, 0), (0, 255, 0, 0), (0, 0, 255, 0), (0, 0, 0, 255),
            (255, 0, 255, 0), (1, 254, 127, 128)] + [tuple(int(v) for v in rng.integers(0, 256, 4)) for _ in range(300)]
    for t in taps:
        assert shim.s3a_host_blend_x2_equals_reference(*t) == 0, t


def test_oracle_undistort_matches_cv2_golden(shim):
    g = np.load(os.path.join(GOLDEN, "f4_kat.npz"))
    for i in range(int(g["n_undistort"])):
        K, d, src, dst = g[f"und_K{i}"], g[f"und_d{i}"], g[f"und_src{i}"], g[f"und_dst{i}"]
        assert np.array_equal(o.undistort_frames(src[None], K, d)[0], dst), i   # oracle == cv2.undistort, bit for bit
        H, W = src.shape
        xy, fr = _host_map(shim, K, d, W, H)
        assert np.array_equal(_host_remap(shim, src, xy, fr), dst), i           # kernel arithmetic == cv2.undistort


def test_zero_distortion_is_the_identity():
    # the reference's projector has no distortion (proj_dist_vect = 0): cvUndistort2 must copy
    c = load_calib_c1()
    img = np.random.default_rng(3).integers(0, 256, (1, 720, 1280), dtype=np.uint8)
    assert np.array_equal(o.undistort_frames(img, c["Kp"], c["dp"]), img)


def test_register_points_match_oracle_and_cv2(shim):
    g = np.load(os.path.join(GOLDEN, "f4_kat.npz"))
    pts, exp = g["reg_pts"], g["reg_out"]
    theta, t = float(g["reg_theta"]), g["reg_t"]
    got = o.register_points(pts, theta, *[float(v) for v in t])
    assert np.array_equal(got.view(np.uint32), exp.view(np.uint32))          # oracle == cv2.gemm chain
    mine = np.ascontiguousarray(pts, np.float32).copy()
    shim.s3a_host_register_points(_p(mine), C.c_longlong(len(mine)), C.c_float(theta), C.c_float(t[0]), C.c_float(t[1]),
                                  C.c_float(t[2]))
    assert np.array_equal(mine.view(np.uint32), exp.view(np.uint32))         # kernel arithmetic == cv2
    R = np.empty(16, np.float32)
    shim.s3a_host_register_rotation(C.c_float(theta), _p(R))
    assert np.array_equal(R.reshape(4, 4), o.register_rotation(theta))
    assert np.array_equal(R.reshape(4, 4), g["reg_R"])
    # the reference's Pi is 22/7: a "180 degree" turn is not exactly a half turn
    assert o.register_rotation(180.0)[0, 0] == np.float32(np.cos(180.0 * 22.0 / 7.0 / 180.0))
    assert o.register_rotation(180.0)[2, 0] != 0.0


def test_roi_fill_closed_form_equals_the_reference_loop(shim):
    rng = np.random.default_rng(9)
    for W, H, density in ((97, 40, 0.02), (256, 64, 0.2), (31, 9, 0.0), (64, 16, 1.0), (500, 30, 0.004)):
        outline = (rng.random((H, W)) < density).astype(np.uint8) * 255
        outline[0, :] = 0
        outline[2, :] = 0
        outline[2, W // 2] = 7                  # a single outline pixel selects nothing
        outline[3, :] = 0
        outline[3, 0] = outline[3, W - 1] = 1   # first and last column: everything between
        roi, filled = o.roi_fill(outline)
        r2 = np.empty_like(roi)
        f2 = np.empty_like(roi)
        shim.s3a_host_roi_fill(_p(np.ascontiguousarray(outline)), W, H, _p(r2), _p(f2))
        assert np.array_equal(roi, r2) and np.array_equal(filled, f2), (W, H)
        assert roi[0].sum() == 0 and roi[2].sum() == 0 and roi[3].sum() == W - 2


def test_roi_fill_pinned_by_the_reference_i1_rows():
    # the reference's stored i1.jpg is internal_image AFTER the fill: with the loop's "restart at the end
    # pixel" every row must be one single run (JPEG, so thresholded); committed as per-row first/last/count
    g = np.load(os.path.join(GOLDEN, "f4_kat.npz"))
    first, last, count = g["i1_first"].astype(np.int64), g["i1_last"].astype(np.int64), g["i1_count"].astype(np.int64)
    rows = count > 0
    assert rows.sum() > 500
    assert np.array_equal(count[rows], (last - first + 1)[rows])
    # rebuild an outline with the same extent per row, fill it, and get the stored image's rows back
    H, W = int(g["i1_shape"][0]), int(g["i1_shape"][1])
    outline = np.zeros((H, W), np.uint8)
    ys = np.nonzero(rows)[0]
    outline[ys, first[ys]] = 255
    outline[ys, last[ys]] = 255
    roi, filled = o.roi_fill(outline)
    assert np.array_equal((filled != 0).sum(1), count)
    assert np.array_equal(roi.sum(1)[ys], np.maximum(count[ys] - 2, 0))
