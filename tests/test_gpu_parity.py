"""GPU parity tests proper: the CUDA path (through the C ABI) against the CPU oracle on the
same seeded inputs.  Bar (BASELINE.json north_star): Gray codes / fringe orders / validity
bit-exact; unwrapped phase within 1e-4 rad; 3-D points within 1e-5 relative."""
import os

import numpy as np
import pytest

import oracle_ffi as o
from gpu_common import calibs, compare, run_oracle, s3
from helpers import load_c1_crop, load_c1_full

pytestmark = pytest.mark.gpu


def _ctx(cfg, cal):
    return s3.Scan3D(cfg, 0, cal)


# ---------------------------------------------------------------------------- atan2 numerics
def test_wrapped_phase_exhaustive_3step():
    """Every (I0,I1,I2) triple: 2^24 pixels through scan3d_compute_wrapped_phase vs libm."""
    v = np.arange(256, dtype=np.uint8)
    fr = np.empty((3, 4096, 4096), np.uint8)
    fr[0] = np.repeat(v, 16)[:, None]                      # I0 = row // 16
    fr[1] = (np.arange(4096) % 256).astype(np.uint8)[None, :]   # I1 = col % 256
    fr[2] = ((np.arange(4096)[:, None] % 16) * 16 + (np.arange(4096)[None, :] // 256)).astype(np.uint8)
    roi = np.ones((4096, 4096), np.uint8)
    cfg = s3.make_config(4096, 4096, N=3, M_v=1, dirs=1)
    ctx = s3.Scan3D(cfg, 0)
    ctx.compute_wrapped_phase(0, fr, roi)
    got = ctx.plane(s3.PLANE_WRAPPED_V)
    want, _ = o.wrapped_phase(fr, np.ones((4096, 4096), np.int32), threads=0, want_dbg=False)
    bad = int((got.view(np.uint32) != want.view(np.uint32)).sum())
    print("3-step exhaustive: non-identical wrapped-phase floats:", bad, "of", got.size)
    assert bad == 0
    ctx.close()


@pytest.mark.parametrize("N", [4, 5, 8, 6])
def test_wrapped_phase_random(N):
    rng = np.random.default_rng(N)
    H, W = 2048, 2048
    fr = rng.integers(0, 256, (N, H, W), dtype=np.uint8)
    roi = np.ones((H, W), np.uint8)
    cfg = s3.make_config(W, H, N=N, M_v=1, dirs=1)
    ctx = s3.Scan3D(cfg, 0)
    ctx.compute_wrapped_phase(0, fr, roi)
    got = ctx.plane(s3.PLANE_WRAPPED_V)
    want, _ = o.wrapped_phase(fr, np.ones((H, W), np.int32), threads=0, want_dbg=False)
    bad = int((got.view(np.uint32) != want.view(np.uint32)).sum())
    print(f"N={N}: non-identical wrapped-phase floats: {bad} of {got.size}")
    assert np.abs(got.astype(np.float64) - want).max() <= 4e-7
    assert bad <= 2
    ctx.close()


def test_debug_atan2_modes_agree_with_libm():
    rng = np.random.default_rng(7)
    y = rng.integers(-510, 511, 1 << 20).astype(np.float64)
    x = rng.integers(-1020, 1021, 1 << 20).astype(np.float64)
    y[:8] = [0, 0, 0, 1, -1, 5, -5, 0]
    x[:8] = [0, 5, -5, 0, 0, 5, -5, 1]
    cfg = s3.make_config(16, 16, N=3, M_v=1, dirs=1)
    ctx = s3.Scan3D(cfg, 0)
    import math
    want = np.fromiter((math.atan2(a, b) for a, b in zip(y, x)), np.float64, y.size).astype(np.float32)
    for mode in (0, 1):
        got = ctx.debug_atan2(y, x, mode)
        bad = int((got.view(np.uint32) != want.view(np.uint32)).sum())
        print("atan2 mode", mode, "non-identical:", bad)
        assert bad == 0
    ctx.close()


def test_exact_quotient_shortcut_equals_ieee_division_on_every_float():
    ctx = s3.Scan3D(s3.make_config(16, 16, N=3, M_v=1, dirs=1), 0)
    assert ctx.debug_divcheck() == 0
    ctx.close()


# ---------------------------------------------------------------------------- stage by stage
@pytest.mark.parametrize("W,H,N,Mv,Mh,fw", [(200, 150, 3, 6, 5, 4), (333, 77, 4, 7, 6, 3), (64, 40, 5, 5, 4, 4),
                                            (640, 480, 8, 9, 8, 2), (97, 33, 6, 6, 5, 2)])
def test_stage_entries_match_oracle(W, H, N, Mv, Mh, fw):
    PW, PH = fw * (1 << Mv) // 2 + 37, fw * (1 << Mh) // 2 + 11
    cal, ocal, _ = calibs(W / 1600.0, PW / 1280.0)
    cfg = s3.make_config(W, H, PW, PH, N, Mv, Mh, fw, fw, 2)
    stack, roi = s3.synth_stack(cfg, cal, s3.default_synth_params(seed=W * 7 + H))
    ref = run_oracle(cfg, ocal, stack, roi)
    d = s3.split_stack(cfg, stack)
    ctx = _ctx(cfg, cal)
    for k, key in enumerate(("v", "h")):
        ctx.compute_wrapped_phase(k, d["fringe_" + key], roi)
        ctx.unwrap_phase(k, d["gray_" + key], d["inv_" + key])
    # wrapped plane after unwrap's in-place += Pi
    wv = ctx.plane(s3.PLANE_WRAPPED_V)
    assert np.abs(wv.astype(np.float64) - ref.wrapped_v).max() <= 4e-7
    assert np.array_equal(ctx.plane(s3.PLANE_MASK).astype(np.int32), ref.valid_v)
    assert np.array_equal(ctx.plane(s3.PLANE_MASK_H).astype(np.int32), ref.valid_h)
    ctx.compute_c_p_map()
    ctx.triangulate()
    n = ctx.compact_points()
    st = compare(cfg, ref, ctx, fused=False)
    if st["unw_v_nonidentical"] == 0 and st["unw_h_nonidentical"] == 0:
        xyz = ctx.plane(s3.PLANE_XYZ)
        m = ref.valid == 1
        assert np.array_equal(xyz[m], ref.xyz[m]), "dense XYZ not bit-identical"
        assert n == ref.count
    print(st)
    ctx.close()


# ---------------------------------------------------------------------------- fused kernel
FUSED_CASES = [
    # W, H, PW, PH, N, Mv, Mh, fw_v, fw_h, dirs
    (1600, 1200, 1280, 720, 3, 6, 5, 32, 32, 2),     # C1 geometry
    (1920, 1080, 1920, 1080, 3, 8, 8, 8, 8, 1),      # C2: vertical stage only
    (1040, 64, 1024, 768, 8, 10, 10, 1, 1, 2),       # partial tile at the row end
    (2048, 96, 2048, 1500, 8, 10, 10, 2, 2, 2),
    (512, 300, 640, 480, 4, 7, 6, 5, 8, 2),
    (256, 128, 512, 512, 5, 6, 6, 8, 8, 2),
    (16, 3, 64, 64, 3, 4, 4, 4, 4, 2),               # degenerate tiny frame
    (256, 64, 2048, 2048, 8, 12, 12, 1, 1, 2),       # 64 frames: launch shape (9 consumer warps, 2 CTAs per SM)
    (256, 64, 8192, 8192, 8, 14, 14, 1, 1, 2),       # 72 frames: launch shape (7, 2)
]


@pytest.mark.parametrize("case", FUSED_CASES)
def test_fused_matches_oracle(case):
    W, H, PW, PH, N, Mv, Mh, fwv, fwh, dirs = case
    cal, ocal, _ = calibs(W / 1600.0, PW / 1280.0)
    cfg = s3.make_config(W, H, PW, PH, N, Mv, Mh, fwv, fwh, dirs, flags=s3.FLAG_POINT_PIXELS)
    stack, roi = s3.synth_stack(cfg, cal, s3.default_synth_params(seed=W + 31 * H))
    ref = run_oracle(cfg, ocal, stack, roi)
    ctx = _ctx(cfg, cal)
    n = ctx.reconstruct(stack, roi)
    st = compare(cfg, ref, ctx, fused=True)
    if dirs == 2 and st.get("pts_nonidentical") is not None:
        assert n == ref.count
        _, pix = ctx.points(want_pix=True)
        assert np.array_equal(pix, ref.pix)
    # a second scan on the same ctx (epoch-tagged look-back state, reused buffers)
    stack2, roi2 = s3.synth_stack(cfg, cal, s3.default_synth_params(seed=W + 31 * H + 1, roi_fraction=0.4))
    ref2 = run_oracle(cfg, ocal, stack2, roi2)
    ctx.reconstruct(stack2, roi2)
    compare(cfg, ref2, ctx, fused=True)
    print(case, st)
    ctx.close()


@pytest.mark.parametrize("case", FUSED_CASES[:1] + FUSED_CASES[2:5] + FUSED_CASES[7:8])
def test_fused_fast_triangulation_within_tolerance(case):
    """SCAN3D_FLAG_FAST_TRIANGULATION: everything up to c_p_map stays bit-exact; the points are
    the same least-squares solution with a different rounding order (bar: 1e-5 relative)."""
    W, H, PW, PH, N, Mv, Mh, fwv, fwh, dirs = case
    cal, ocal, _ = calibs(W / 1600.0, PW / 1280.0)
    cfg = s3.make_config(W, H, PW, PH, N, Mv, Mh, fwv, fwh, dirs, flags=s3.FLAG_FAST_TRIANGULATION)
    stack, roi = s3.synth_stack(cfg, cal, s3.default_synth_params(seed=W + 31 * H))
    ref = run_oracle(cfg, ocal, stack, roi)
    ctx = _ctx(cfg, cal)
    ctx.reconstruct(stack, roi)
    st = compare(cfg, ref, ctx, fused=True)
    assert st["cpmap_mismatch"] == 0 and st["valid_mismatch"] == 0
    assert st["pts_max_rel"] <= 1e-6
    print(case, st)
    ctx.close()


def test_full_size_c3_matches_oracle_and_round_trips():
    """BASELINE configs[2] at its full size (4096x3000, V+H, 8-step, 10-bit): the bench kernel (fast
    triangulation) against the oracle on every pixel, the reference-order kernel bit for bit on the
    points, a second run byte-identical (the look-back state is reused across launches), and the
    size-independent round trip: a noise-free rendered scene comes back within 0.5 mm wherever the
    projector reaches."""
    W, H, PW, PH, N, M, fw = 4096, 3000, 4096, 3000, 8, 10, 4
    cal, ocal, _ = calibs(W / 1600.0, PW / 1280.0)
    p = s3.default_synth_params(seed=0x3D5CA9, noise_sigma=0.0, ambient_max=0.0, albedo_lo=1.0)
    cfg = s3.make_config(W, H, PW, PH, N, M, M, fw, fw, 2, flags=s3.FLAG_FAST_TRIANGULATION | s3.FLAG_POINT_PIXELS)
    stack, roi, truth = s3.synth_stack(cfg, cal, p, want_truth=True)
    ref = run_oracle(cfg, ocal, stack, roi)
    assert ref.count > 5_000_000
    ctx = _ctx(cfg, cal)
    n = ctx.reconstruct(stack, roi)
    st = compare(cfg, ref, ctx, fused=True)
    assert n == ref.count and st["cpmap_mismatch"] == 0 and st["valid_mismatch"] == 0 and st["pts_max_rel"] <= 1e-6
    pts, pix = ctx.points(want_pix=True)
    assert np.array_equal(pix, ref.pix)
    # round trip on the pixels the projector reaches (the ROI also holds unlit pixels, which the
    # reference's ROI-only validity keeps: all their Gray ties decode to one constant code)
    lit = (stack[:N].max(0) > stack[:N].min(0)).reshape(-1)[pix]
    err = np.linalg.norm(pts.astype(np.float64) - truth.reshape(-1, 3)[pix], axis=1)[lit]
    assert 0.7 < lit.mean() < 0.85 and np.median(err) < 0.05 and err.max() < 0.5, (lit.mean(), np.median(err), err.max())
    ctx.reconstruct(stack, roi)                                   # same scan again on the same context
    pts2, pix2 = ctx.points(want_pix=True)
    assert np.array_equal(pts2.view(np.uint32), pts.view(np.uint32)) and np.array_equal(pix2, pix)
    ctx.close()
    exact = _ctx(s3.make_config(W, H, PW, PH, N, M, M, fw, fw, 2), cal)       # reference operation order
    assert exact.reconstruct(stack, roi) == ref.count
    assert np.array_equal(exact.points().view(np.uint32), ref.pts.view(np.uint32))
    exact.close()


def test_fused_distorted_projector_and_tangential_camera():
    W, H, PW, PH = 1024, 256, 1024, 768
    cal, ocal, _ = calibs(W / 1600.0, PW / 1280.0, dc=[0.0813, -0.1102, 0.0013, -0.0007, 0.021],
                          dp=[-0.05, 0.02, 0.001, -0.0005, 0.0])
    cfg = s3.make_config(W, H, PW, PH, 8, 10, 10, 1, 1, 2)
    stack, roi = s3.synth_stack(cfg, cal)
    ref = run_oracle(cfg, ocal, stack, roi)
    ctx = _ctx(cfg, cal)
    ctx.reconstruct(stack, roi)
    print(compare(cfg, ref, ctx))
    ctx.close()


def test_fused_undistorted_camera():
    W, H, PW, PH = 1024, 128, 1024, 768
    cal, ocal, _ = calibs(W / 1600.0, PW / 1280.0, dc=[0, 0, 0, 0, 0])
    cfg = s3.make_config(W, H, PW, PH, 3, 10, 10, 1, 1, 2)
    stack, roi = s3.synth_stack(cfg, cal)
    ref = run_oracle(cfg, ocal, stack, roi)
    ctx = _ctx(cfg, cal)
    ctx.reconstruct(stack, roi)
    print(compare(cfg, ref, ctx))
    ctx.close()


def test_fused_skewed_intrinsics_without_distortion():
    """Zero distortion but an intrinsic matrix outside the standard form (skew on both devices): the re-projection
    of 7/triangulation.cpp:262-307 then is a full 3x3 product with a division (the oracle does it per pixel); the
    library routes that case through the undistortion tables.  Points stay bit-identical in the exact mode."""
    W, H, PW, PH = 1024, 128, 1024, 768
    _, _, c = calibs(W / 1600.0, PW / 1280.0, dc=[0, 0, 0, 0, 0])
    c["Kc"] = c["Kc"].copy(); c["Kp"] = c["Kp"].copy()
    c["Kc"][1] = 0.75                   # K[0][1]: skew
    c["Kp"][1] = -0.4
    args = [c[k] for k in ("Kc", "dc", "Kp", "dp", "rc", "tc", "rp", "tp")]
    cal, ocal = s3.make_calib(*args), o.make_calib(*args)
    cfg = s3.make_config(W, H, PW, PH, 3, 10, 10, 1, 1, 2)
    stack, roi = s3.synth_stack(cfg, cal)
    ref = run_oracle(cfg, ocal, stack, roi)
    assert ref.count > 10000
    ctx = _ctx(cfg, cal)
    ctx.reconstruct(stack, roi)
    st = compare(cfg, ref, ctx)
    assert st["pts_nonidentical"] == 0
    ctx.close()


@pytest.mark.parametrize("kind", ["empty", "full", "random", "border"])
def test_fused_roi_edge_cases(kind):
    W, H, PW, PH = 1056, 40, 1024, 768
    cal, ocal, _ = calibs(W / 1600.0, PW / 1280.0)
    cfg = s3.make_config(W, H, PW, PH, 3, 10, 10, 1, 1, 2)
    stack, roi = s3.synth_stack(cfg, cal)
    rng = np.random.default_rng(3)
    if kind == "empty":
        roi[:] = 0
    elif kind == "full":
        roi[:] = 1          # includes the image border: exercises the uninitialised-border policy
    elif kind == "random":
        roi[:] = (rng.random(roi.shape) < 0.93)
    else:
        roi[:] = 0
        roi[:3, :] = 1; roi[-2:, :] = 1; roi[:, :3] = 7; roi[:, -3:] = 255
    ref = run_oracle(cfg, ocal, stack, roi)
    ctx = _ctx(cfg, cal)
    n = ctx.reconstruct(stack, roi)
    st = compare(cfg, ref, ctx)
    if kind == "empty":
        assert n == 0
    print(kind, st)
    ctx.close()


@pytest.mark.parametrize("kind", ["bottom_band", "top_band", "sparse", "all_zero", "left_column"])
def test_fused_long_runs_without_roi(kind):
    """Thousands of consecutive work units without a single ROI pixel (the single-pass kernel hands them out from a
    global counter and resolves their place in the raster order later): every launch of a series gives the oracle's
    result, whatever the interleaving of the warps was."""
    W, H, PW, PH = 2048, 1200, 1024, 768
    cal, ocal, _ = calibs(W / 1600.0, PW / 1280.0)
    cfg = s3.make_config(W, H, PW, PH, 3, 8, 8, 4, 4, 2, flags=s3.FLAG_POINT_PIXELS)
    stack, roi = s3.synth_stack(cfg, cal)
    keep = np.zeros_like(roi)
    if kind == "bottom_band":
        keep[-40:] = 1
    elif kind == "top_band":
        keep[:25] = 1
    elif kind == "sparse":
        keep.reshape(-1)[::2999] = 1
        keep[600, 100:1900] = 1
    elif kind == "left_column":
        keep[:, :130] = 1
    roi[:] = roi * keep if kind != "sparse" else keep
    ref = run_oracle(cfg, ocal, stack, roi)
    ctx = _ctx(cfg, cal)
    first = None
    for rep in range(12):
        n = ctx.reconstruct(stack, roi)
        pts, pix = ctx.points(want_pix=True)
        cur = (n, pts.tobytes(), pix.tobytes(), ctx.plane(s3.PLANE_CPMAP).tobytes())
        if first is None:
            first = cur
            st = compare(cfg, ref, ctx)
            assert np.array_equal(pix, ref.pix)
            assert n == ref.count
            if kind == "all_zero":
                assert n == 0
        else:
            assert cur == first, "launch %d differs from launch 0" % rep
    ctx.close()


@pytest.mark.parametrize("N", [3, 5])
def test_quirk_strict_reference_validity(N):
    """check_I_mod_criteria as committed (3/wrapped_phase.cpp:106,117-127): the ROI is read as `== 1`, and only for
    N == 3 or 4 -- the 5-step block is commented out, so the reference's own 5-step run ends with an all-zero valid map
    and an empty cloud.  Default: every non-zero ROI byte selects, for every N (documented extension);
    SCAN3D_FLAG_STRICT_REFERENCE: the committed behaviour.  Both against the oracle's two restatements."""
    W, H, PW, PH = 640, 96, 512, 288
    cal, ocal, _ = calibs(W / 1600.0, PW / 1280.0)
    base = s3.make_config(W, H, PW, PH, N, 7, 6, 4, 5, 2)
    stack, roi = s3.synth_stack(base, cal)
    roi[20:40, 100:300] *= 7            # selected, but not with the value 1
    for strict in (False, True):
        cfg = s3.make_config(W, H, PW, PH, N, 7, 6, 4, 5, 2, flags=s3.FLAG_STRICT_REFERENCE if strict else 0)
        ref = run_oracle(cfg, ocal, stack, roi, strict=strict)
        ctx = _ctx(cfg, cal)
        n = ctx.reconstruct(stack, roi)
        compare(cfg, ref, ctx)
        assert n == ref.count
        v = ctx.plane(s3.PLANE_VALID)
        if strict and N == 5:
            assert n == 0 and not v.any()                 # the reference as committed: nothing survives a 5-step run
        elif strict:
            assert n > 0 and not v[20:40, 100:300].any()  # ROI bytes != 1 are not selected
        else:
            assert n > 0 and v[22:38, 110:290].any()
        # the stage entries follow the same rule
        d = s3.split_stack(cfg, stack)
        ctx.compute_wrapped_phase(0, d["fringe_v"], roi)
        m = ctx.plane(s3.PLANE_MASK)
        assert np.array_equal(m.astype(np.int32), ref.valid_v)
        ctx.close()


def test_planes_nothing_has_written_are_not_handed_out():
    """scan3d_get_plane / scan3d_device_plane refuse planes no compute entry has produced (after the single-pass
    entry: the wrapped phases and per-direction masks, which it keeps in registers)."""
    W, H, PW, PH = 640, 64, 512, 288
    cal, ocal, _ = calibs(W / 1600.0, PW / 1280.0)
    cfg = s3.make_config(W, H, PW, PH, 3, 7, 6, 4, 5, 2)
    stack, roi = s3.synth_stack(cfg, cal)
    ctx = _ctx(cfg, cal)
    for which in (s3.PLANE_UNWRAPPED_V, s3.PLANE_VALID, s3.PLANE_CPMAP, s3.PLANE_MASK, s3.PLANE_WRAPPED_V, s3.PLANE_XYZ):
        with pytest.raises(RuntimeError):
            ctx.plane(which)
        assert not ctx.device_plane(which)
    ctx.reconstruct(stack, roi)
    ctx.plane(s3.PLANE_UNWRAPPED_H); ctx.plane(s3.PLANE_VALID); ctx.plane(s3.PLANE_CPMAP)
    for which in (s3.PLANE_MASK, s3.PLANE_WRAPPED_V, s3.PLANE_XYZ):
        with pytest.raises(RuntimeError):
            ctx.plane(which)
    d = s3.split_stack(cfg, stack)
    ctx.compute_wrapped_phase(0, d["fringe_v"], roi)
    ctx.plane(s3.PLANE_MASK); ctx.plane(s3.PLANE_WRAPPED_V)
    with pytest.raises(RuntimeError):
        ctx.plane(s3.PLANE_VALID)         # the inputs changed: the old final map no longer belongs to them
    ctx.close()


def test_c5_size_single_rank_matches_oracle():
    """BASELINE.json configs[4] at its own size on ONE rank: 8192 x 6144 (50 MP), 8-step + 10-bit Gray code, both
    directions -- every contract output against the oracle (multi-threaded, a few seconds), points bit for bit."""
    W, H, PW, PH = 8192, 6144, 8192, 6144
    cal, ocal, _ = calibs(W / 1600.0, PW / 1280.0)
    cfg = s3.make_config(W, H, PW, PH, 8, 10, 10, 8, 8, 2, flags=s3.FLAG_POINT_PIXELS)
    stack, roi = s3.synth_stack(cfg, cal)
    ref = run_oracle(cfg, ocal, stack, roi, threads=0)
    ctx = _ctx(cfg, cal)
    n = ctx.reconstruct(stack, roi)
    st = compare(cfg, ref, ctx)
    assert st["unw_v_nonidentical"] == 0 and st["unw_h_nonidentical"] == 0 and st["pts_nonidentical"] == 0
    pts, pix = ctx.points(want_pix=True)
    assert np.array_equal(pix, ref.pix) and n == ref.count and n > 25_000_000
    print(st)
    ctx.close()


def test_modulation_mask_flag_matches_oracle():
    """SCAN3D_FLAG_MODULATION_MASK = the reference's commented-out criterion (3/wrapped_phase.cpp:84-104):
    every (I0,I1,I2) triple through scan3d_compute_wrapped_phase, then a whole scan with flat and
    nearly flat patches inside the ROI (V and H masks then differ) against the oracle."""
    v = np.arange(256, dtype=np.int64)
    i0, i1, i2 = np.meshgrid(v, v, v, indexing="ij")
    fr = np.stack([i0, i1, i2]).astype(np.uint8).reshape(3, 4096, 4096)
    roi = np.ones((4096, 4096), np.uint8)
    roi[7::13, :] = 0
    cfg = s3.make_config(4096, 4096, 1, 1, 3, 1, 1, 8, 8, 1, flags=s3.FLAG_MODULATION_MASK)
    ctx = s3.Scan3D(cfg, 0, None)
    ctx.compute_wrapped_phase(0, fr, roi)
    valid0 = o.check_I_mod_criteria(fr, roi)
    want = o.mask_recurrence(valid0)
    assert np.array_equal(ctx.plane(s3.PLANE_MASK).astype(np.int32), want)
    ctx.close()

    W, H, PW, PH = 640, 480, 1024, 768
    cal, ocal, _ = calibs(W / 1600.0, PW / 1280.0)
    cfg = s3.make_config(W, H, PW, PH, 3, 7, 7, 8, 8, 2, flags=s3.FLAG_MODULATION_MASK)
    stack, roi = s3.synth_stack(cfg, cal)
    stack = stack.copy()
    rng = np.random.default_rng(5)
    stack[0:3, 100:160, 200:300] = 90                                                   # flat in V only
    stack[17:20, 300:340, 100:220] = rng.integers(118, 122, (3, 40, 120), dtype=np.uint8)   # around the threshold, H only
    stack[0:3, 200:230, 400:470] = 0                                                    # black: 0/0
    ctx = _ctx(cfg, cal)
    l0 = ctx.launch_count()
    n = ctx.reconstruct(stack, roi)
    # the single-pass kernel, not the stage chain: 2 pre-pass launches (one effective ROI plane per direction),
    # the 2 work-list launches and the persistent kernel (the stage chain takes 13)
    assert ctx.launch_count() - l0 == 5
    ref = run_oracle(cfg, ocal, stack, roi, modulation=True)
    assert (ref.valid_v != ref.valid_h).any() and 0 < ref.count == n
    st = compare(cfg, ref, ctx, fused=True)
    assert st["pts_nonidentical"] == 0
    # 54 frames (12 + 12 Gray bits): the variant at launch shape (7 consumer warps, 2 CTAs per SM)
    cfg54 = s3.make_config(256, 64, 2048, 2048, 3, 12, 12, 1, 1, 2, flags=s3.FLAG_MODULATION_MASK)
    cal54, ocal54, _ = calibs(256 / 1600.0, 2048 / 1280.0)
    stack54, roi54 = s3.synth_stack(cfg54, cal54)
    stack54 = stack54.copy()
    stack54[0:3, 20:40, 80:160] = 90                                                    # flat in V only
    ctx54 = _ctx(cfg54, cal54)
    l0 = ctx54.launch_count()
    n54 = ctx54.reconstruct(stack54, roi54)
    assert ctx54.launch_count() - l0 == 5
    ref54 = run_oracle(cfg54, ocal54, stack54, roi54, modulation=True)
    assert (ref54.valid_v != ref54.valid_h).any() and 0 < ref54.count == n54
    assert compare(cfg54, ref54, ctx54, fused=True)["pts_nonidentical"] == 0
    ctx54.close()
    # fast triangulation + one direction through the same variant
    cfg1 = s3.make_config(W, H, PW, PH, 3, 7, 7, 8, 8, 1, flags=s3.FLAG_MODULATION_MASK)
    ctx1 = _ctx(cfg1, cal)
    ctx1.reconstruct(stack[:17], roi)
    ref1 = run_oracle(cfg1, ocal, stack[:17], roi, modulation=True)
    compare(cfg1, ref1, ctx1, fused=True)
    ctx1.close()
    plain = run_oracle(cfg, ocal, stack, roi)
    assert plain.count > ref.count                                                      # the criterion removed pixels
    ctx.close()
    with pytest.raises(RuntimeError):
        s3.Scan3D(s3.make_config(W, H, PW, PH, 4, 7, 7, 8, 8, 2, flags=s3.FLAG_MODULATION_MASK), 0, cal)


def test_concurrent_contexts_with_cta_limit_equal_serial():
    """bench.py's default schedule: four contexts on four streams, each limited to one CTA slot per SM
    (scan3d_set_cta_limit), reconstruct DIFFERENT scans at the same time.  Every context's planes and point cloud
    must equal what an unrestricted context produces for the same scan alone, over several rounds."""
    import torch
    W, H, PW, PH = 1024, 611, 1024, 768
    cal, ocal, _ = calibs(W / 1600.0, PW / 1280.0)
    cfg = s3.make_config(W, H, PW, PH, 8, 10, 10, 2, 2, 2)
    NCTX, ROUNDS = 4, 3
    scans = [s3.synth_stack(cfg, cal, s3.default_synth_params(seed=0xC0FFEE + k, roi_fraction=0.9 - 0.1 * (k % 5)))
             for k in range(NCTX * ROUNDS)]
    solo = _ctx(cfg, cal)
    want = []
    for stack, roi in scans:
        solo.reconstruct(stack, roi)
        want.append((solo.points().copy(), solo.plane(s3.PLANE_VALID).copy(), solo.code_i32(0).copy(),
                     solo.plane(s3.PLANE_UNWRAPPED_V).copy()))
    solo.close()
    ref = run_oracle(cfg, ocal, *scans[0])
    assert np.array_equal(want[0][0].view(np.uint32), ref.pts.view(np.uint32))
    streams = [torch.cuda.Stream() for _ in range(NCTX)]
    ctxs = [s3.Scan3D(cfg, 0, cal, stream=st.cuda_stream) for st in streams]
    for c in ctxs:
        c.set_cta_limit(1)
    d_stacks = [torch.from_numpy(st).cuda() for st, _ in scans]
    d_rois = [torch.from_numpy(r).cuda() for _, r in scans]
    torch.cuda.synchronize()
    for r in range(ROUNDS):
        for i, c in enumerate(ctxs):                      # enqueue all four without waiting in between
            k = r * NCTX + i
            c.reconstruct_dev(d_stacks[k].data_ptr(), d_rois[k].data_ptr())
        for i, c in enumerate(ctxs):
            k = r * NCTX + i
            pts, valid, code, unw = want[k]
            assert c.point_count() == len(pts), (r, i)
            assert np.array_equal(c.points().view(np.uint32), pts.view(np.uint32)), (r, i)
            assert np.array_equal(c.plane(s3.PLANE_VALID), valid), (r, i)
            assert np.array_equal(c.code_i32(0), code), (r, i)
            assert np.array_equal(c.plane(s3.PLANE_UNWRAPPED_V).view(np.uint32), unw.view(np.uint32)), (r, i)
    for c in ctxs:
        c.close()


def test_fused_row_shards_concatenate_to_full_frame():
    W, H, PW, PH = 1024, 90, 1024, 768
    cal, ocal, _ = calibs(W / 1600.0, PW / 1280.0)
    full = s3.make_config(W, H, PW, PH, 8, 10, 10, 1, 1, 2, flags=s3.FLAG_POINT_PIXELS)
    stack, roi = s3.synth_stack(full, cal)
    ref = run_oracle(full, ocal, stack, roi)
    pts, pix = [], []
    for r0, r1 in ((0, 31), (31, 32), (32, 90)):
        cfg = s3.make_config(W, r1 - r0, PW, PH, 8, 10, 10, 1, 1, 2, row0=r0, H_total=H, flags=s3.FLAG_POINT_PIXELS)
        ctx = _ctx(cfg, cal)
        ctx.reconstruct(np.ascontiguousarray(stack[:, r0:r1]), roi)
        p, q = ctx.points(want_pix=True)
        pts.append(p); pix.append(q)
        assert np.array_equal(ctx.code_i32(0), ref.code_v[r0:r1])
        assert np.array_equal(ctx.plane(s3.PLANE_VALID).astype(np.int32), ref.valid[r0:r1])
        ctx.close()
    pts, pix = np.concatenate(pts), np.concatenate(pix)
    assert np.array_equal(pix, ref.pix)
    assert np.array_equal(pts.view(np.uint32), ref.pts.view(np.uint32))


# ---------------------------------------------------------------------------- golden data
def test_c1_crop_through_gpu_matches_reference_images():
    d = load_c1_crop()
    H, W = d["golden_wrapped_v"].shape
    cal, ocal, _ = calibs()
    cfg = s3.make_config(W, H, 1280, 720, 3, 6, 5, 32, 32, 2)
    ctx = _ctx(cfg, cal)
    roi = (d["golden_wrapped_v"] != 0).astype(np.uint8)   # the reference's post-recurrence mask
    for k, key, codes in ((0, "v", 40), (1, "h", 23)):
        ctx.compute_wrapped_phase(k, d["fringe_" + key], roi)
        w = ctx.plane(s3.PLANE_WRAPPED_V + k)
        m = roi == 1
        dbg = (128.0 + 127.0 * (w.astype(np.float64) / (22.0 / 7.0))).astype(np.float32).astype(np.int32).astype(np.uint8)
        assert np.array_equal(dbg[m], d["golden_wrapped_" + key][m])
    # full path on the crop against the oracle (real captured data)
    stack = np.concatenate([d["fringe_v"], d["gray_v"], d["inv_v"], d["fringe_h"], d["gray_h"], d["inv_h"]])
    ref = run_oracle(cfg, ocal, stack, roi)
    ctx.reconstruct(stack, roi)
    st = compare(cfg, ref, ctx)
    unw = ctx.plane(s3.PLANE_UNWRAPPED_V)
    m = ref.valid_v == 1
    m[:, 0] = m[:, -1] = False
    img = o.unwrapped_image(unw, m.astype(np.int32), 40)
    assert np.array_equal(img[m], d["golden_unwrapped_v"][m])
    print(st)
    ctx.close()


def test_c1_full_capture_through_gpu_matches_reference_images():
    """BASELINE.json configs[0] at its own size: the reference's whole 1600x1200 captured scan (28 frames,
    tests/golden/c1_full.npz) through scan3d_reconstruct -- both stored unwrapped-phase images and the
    wrapped-phase image come out bit for bit, everything else equals the oracle on the same input."""
    d = load_c1_full()
    H, W = d["golden_wrapped_v"].shape
    assert (W, H) == (1600, 1200)
    cal, ocal, _ = calibs()
    cfg = s3.make_config(W, H, 1280, 720, 3, 6, 5, 32, 32, 2)
    ctx = _ctx(cfg, cal)
    roi = (d["golden_wrapped_v"] != 0).astype(np.uint8)   # the reference's post-recurrence mask
    stack = np.concatenate([d["fringe_v"], d["gray_v"], d["inv_v"], d["fringe_h"], d["gray_h"], d["inv_h"]])
    ref = run_oracle(cfg, ocal, stack, roi)
    l0 = ctx.launch_count()
    n = ctx.reconstruct(stack, roi)
    assert ctx.launch_count() - l0 == 3           # the single-pass kernel and its two work-list launches, not the stage chain
    st = compare(cfg, ref, ctx)
    assert st["unw_v_nonidentical"] == 0 and st["unw_h_nonidentical"] == 0 and st["pts_nonidentical"] == 0
    assert n == ref.count and n > 300000
    for k, key, codes in ((0, "v", 40), (1, "h", 23)):
        unw = ctx.plane(s3.PLANE_UNWRAPPED_V + k)
        m = (ref.valid_v if k == 0 else ref.valid_h) == 1
        if k == 0:
            m[:, 0] = m[:, -1] = False
        else:
            m[0, :] = m[-1, :] = False
        img = o.unwrapped_image(unw, m.astype(np.int32), codes)
        assert np.array_equal(img[m], d["golden_unwrapped_" + key][m]), key
    # stage entry on the full frame: the stored wrapped-phase image
    for k, key in ((0, "v"), (1, "h")):
        ctx.compute_wrapped_phase(k, d["fringe_" + key], roi)
        w = ctx.plane(s3.PLANE_WRAPPED_V + k)
        m = roi == 1
        dbg = (128.0 + 127.0 * (w.astype(np.float64) / (22.0 / 7.0))).astype(np.float32).astype(np.int32).astype(np.uint8)
        assert np.array_equal(dbg[m], d["golden_wrapped_" + key][m])
    print(st)
    ctx.close()


@pytest.mark.parametrize("N,Mv,Mh,fw,PW,PH", [(3, 6, 5, 32, 1280, 720), (4, 7, 7, 8, 1024, 768), (5, 8, 8, 8, 1920, 1080), (8, 10, 10, 4, 4096, 3000)])
def test_device_pattern_generator(N, Mv, Mh, fw, PW, PH):
    """scan3d_generate_patterns (stage 1 on the GPU) against the host profiles of the same expressions,
    and for the reference's own configuration against its stored Generated_patterns images."""
    cfg = s3.make_config(64, 16, PW, PH, N, Mv, Mh, fw, fw, 2)
    ctx = s3.Scan3D(cfg, 0, None)
    for d, (M, length) in enumerate(((Mv, PW), (Mh, PH))):
        got = ctx.generate_patterns(d)
        assert got.shape == (N + 2 * M, PH, PW)
        rows = [s3.synth_pattern_row(0, N, fw, k, length) for k in range(N)]
        rows += [s3.synth_pattern_row(1, M, fw, k, length) for k in range(M)]
        rows += [s3.synth_pattern_row(2, M, fw, k, length) for k in range(M)]
        for p, r in enumerate(rows):
            want = np.broadcast_to(r[None, :] if d == 0 else r[:, None], (PH, PW))
            assert np.array_equal(got[p], want), (d, p)
    if (N, fw, PW, PH) == (3, 32, 1280, 720):
        import os
        from helpers import GOLDEN
        k = np.load(os.path.join(GOLDEN, "pattern_kat.npz"))          # rows/columns of the reference's pattern images
        gv, gh = ctx.generate_patterns(0), ctx.generate_patterns(1)
        for i in range(3):
            assert np.array_equal(gv[i, 0], k["fringe_v_row0"][i]) and np.array_equal(gh[i, :, 0], k["fringe_h_col0"][i])
        for i in range(6):
            assert np.array_equal(gv[3 + i, 0], k["gray_v_row0"][i]) and np.array_equal(gv[9 + i, 0], k["inv_v_row0"][i])
        for i in range(5):
            assert np.array_equal(gh[3 + i, :, 0], k["gray_h_col0"][i]) and np.array_equal(gh[8 + i, :, 0], k["inv_h_col0"][i])
    ctx.close()


def test_device_pattern_generator_4_and_5_step_reference_images():
    """The reference tree also keeps one 4-step (k=3, fw 16) and one 5-step (k=4, fw 32) image of a
    1024x768 projector: the device generator reproduces their first row / column."""
    import os
    from helpers import GOLDEN
    k = np.load(os.path.join(GOLDEN, "pattern_kat.npz"))
    for N, fw, idx, key in ((4, 16, 3, "fringe4_k3"), (5, 32, 4, "fringe5_k4")):
        ctx = s3.Scan3D(s3.make_config(64, 16, 1024, 768, N, 6, 5, fw, fw, 2), 0, None)
        assert np.array_equal(ctx.generate_patterns(0)[idx, 0], k[key + "_v_row0"])
        assert np.array_equal(ctx.generate_patterns(1)[idx, :, 0], k[key + "_h_col0"])
        ctx.close()


def test_ply_writer(tmp_path):
    W, H, PW, PH = 256, 64, 512, 512
    cal, ocal, _ = calibs(W / 1600.0, PW / 1280.0)
    cfg = s3.make_config(W, H, PW, PH, 3, 6, 6, 8, 8, 2)
    stack, roi = s3.synth_stack(cfg, cal)
    ctx = _ctx(cfg, cal)
    tex = np.random.default_rng(0).integers(0, 256, (H, W, 3), dtype=np.uint8)
    ctx.set_texture(tex)
    n = ctx.reconstruct(stack, roi)
    xyz, rgb = ctx.points(want_rgb=True)
    valid = ctx.plane(s3.PLANE_VALID).astype(bool)
    assert np.array_equal(rgb, tex[valid][:, ::-1])
    for binary in (False, True):
        path = str(tmp_path / f"cloud_{int(binary)}.ply")
        ctx.write_ply(path, binary)
        raw = open(path, "rb").read()
        head, body = raw.split(b"end_header\n", 1)
        assert f"element vertex {n}".encode() in head
        if binary:
            rec = np.frombuffer(body, np.dtype([("p", "<f4", 3), ("c", "u1", 3)]))
            assert np.array_equal(rec["p"], xyz) and np.array_equal(rec["c"], rgb)
        else:
            rows = np.loadtxt(body.decode().splitlines()) if n else np.empty((0, 6))
            assert np.array_equal(rows[:, :3].astype(np.float32), xyz)
    # savePCDFileASCII layout (8/save_point_cloud.cpp:212): x y z rgb, 8 significant digits
    path = str(tmp_path / "cloud.pcd")
    ctx.write_pcd(path)
    lines = open(path).read().splitlines()
    assert lines[2] == "FIELDS x y z rgb" and lines[9] == f"POINTS {n}" and len(lines) == 11 + n
    rows = np.array([[float(v) for v in ln.split()] for ln in lines[11:]]).reshape(n, 4)
    assert np.allclose(rows[:, :3], xyz, rtol=5e-8, atol=0)
    packed = (rgb[:, 0].astype(np.uint32) << 16) | (rgb[:, 1].astype(np.uint32) << 8) | rgb[:, 2]
    assert np.allclose(rows[:, 3], packed.view(np.float32).astype(np.float64), rtol=5e-8, atol=0)
    ctx.close()


def test_points_carry_the_colours_of_the_texture_they_were_computed_with():
    """A texture set after the points were computed does not colour them: with texture A, a reconstruct, no texture, a
    reconstruct, then texture B, the points and the voxels merged from them read zeros, not A's colours."""
    W, H, PW, PH = 256, 64, 512, 512
    cal, _, _ = calibs(W / 1600.0, PW / 1280.0)
    cfg = s3.make_config(W, H, PW, PH, 3, 6, 6, 8, 8, 2)
    stack, roi = s3.synth_stack(cfg, cal)
    ctx = _ctx(cfg, cal)
    rng = np.random.default_rng(3)
    tex_a, tex_b = (rng.integers(1, 256, (H, W, 3), dtype=np.uint8) for _ in range(2))
    ctx.set_texture(tex_a)
    ctx.reconstruct(stack, roi)
    _, rgb = ctx.points(want_rgb=True)
    valid = ctx.plane(s3.PLANE_VALID).astype(bool)
    assert np.array_equal(rgb, tex_a[valid][:, ::-1]) and rgb.all()
    ctx.set_texture(None)
    n = ctx.reconstruct(stack, roi)
    ctx.set_texture(tex_b)
    xyz, rgb = ctx.points(want_rgb=True)
    assert n > 1000 and not rgb.any()
    ctx.voxel_begin(float(np.ptp(xyz, axis=0).max()) / 64, n)
    ctx.voxel_add()
    ctx.voxel_finish()
    assert not ctx.voxels()[2].any()
    # the next reconstruct is computed with B
    ctx.reconstruct(stack, roi)
    assert np.array_equal(ctx.points(want_rgb=True)[1], tex_b[valid][:, ::-1])
    ctx.close()
