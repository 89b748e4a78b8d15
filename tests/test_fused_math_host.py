"""The fused kernels' arithmetic on the CPU: the product's own device headers (scan3d_math.cuh,
scan3d_fused_math.cuh: SWAR decode, table-driven atan2, exact quotients, correspondence, triangulation) are
compiled for the host (tests/fused_math_host.cpp + tests/cuda_host_shim.h) and run on whole scans against the
oracle and the reference's golden images.  The kernels' pipeline itself is covered by the GPU tests."""
import ctypes as C
import os
import subprocess

import numpy as np
import pytest

import oracle_ffi as o
from gpu_common import calibs, run_oracle, s3
from helpers import load_c1_crop, load_c1_full, load_calib_c1

HERE = os.path.dirname(os.path.abspath(__file__))
CUDA_INC = "/usr/local/cuda/include"

pytestmark = pytest.mark.skipif(not os.path.exists(os.path.join(CUDA_INC, "cuda_runtime.h")),
                                reason="CUDA headers not installed")


@pytest.fixture(scope="module")
def shim(tmp_path_factory):
    so = str(tmp_path_factory.mktemp("fusedhost") / "libfused_math_host.so")
    # S3D_HOST_DEFS="-DS3D_VAR_ROWSEL_RCP=1 ...": the same checks for an experimental variant (tools/build_variants.py)
    defs = [d for d in os.environ.get("S3D_HOST_DEFS", "").split() if d.startswith("-D")]
    subprocess.check_call(["/usr/bin/g++", "-O2", "-std=c++17", "-fPIC", "-shared", "-Wall", "-Wno-unknown-pragmas",
                           "-Wno-unused-function", "-ffp-contract=off", "-I", CUDA_INC] + defs +
                          ["-o", so, os.path.join(HERE, "fused_math_host.cpp")])
    return C.CDLL(so)


def _p(a):
    return a.ctypes.data_as(C.c_void_p)


class Out:
    pass


def run_host(shim, cfg, c, stack, roi, exact=True, mask_is_final=False):
    W, H = cfg["W"], cfg["H"]
    arr = np.array([cfg[k] for k in ("W", "H", "PW", "PH", "N", "M_v", "M_h", "fw_v", "fw_h", "dirs")] +
                   [int(exact), int(mask_is_final)], np.int32)
    Ac = np.ascontiguousarray(o.compute_A(c["Kc"], c["rc"], c["tc"]))
    Ap = np.ascontiguousarray(o.compute_A(c["Kp"], c["rp"], c["tp"]))
    r = Out()
    r.unw_v = np.zeros((H, W), np.float32); r.unw_h = np.zeros((H, W), np.float32)
    r.code_v = np.zeros((H, W), np.int16); r.code_h = np.zeros((H, W), np.int16)
    r.valid = np.zeros((H, W), np.uint8)
    r.cpmap = np.zeros((H * W, 2), np.int32)
    pts = np.zeros((H * W, 3), np.float32)
    n = C.c_int64()
    f64 = lambda k: np.ascontiguousarray(c[k], np.float64)
    keep = [f64(k) for k in ("Kc", "dc", "Kp", "dp")]
    stack = np.ascontiguousarray(stack, np.uint8)
    roi = np.ascontiguousarray(roi, np.uint8)
    rc = shim.s3d_host_fused_math(_p(arr), *[_p(k) for k in keep], _p(Ac), _p(Ap), _p(stack), _p(roi), _p(r.unw_v),
                                  _p(r.unw_h), _p(r.code_v), _p(r.code_h), _p(r.valid), _p(r.cpmap), _p(pts), C.byref(n))
    assert rc == 0
    r.count = n.value
    r.pts = pts[:r.count]
    return r


def test_c1_golden_crop_through_the_kernel_arithmetic(shim):
    """The reference's own captured scan (320x384 crop) through the kernels' arithmetic: the unwrapped-phase images
    the reference stored come out bit for bit, and every plane equals the oracle's."""
    d = load_c1_crop()
    c = load_calib_c1()
    gw = d["golden_wrapped_v"]
    assert np.array_equal(gw != 0, d["golden_wrapped_h"] != 0)        # V and H masks are the same plane
    H, W = gw.shape
    cfg = dict(W=W, H=H, PW=1280, PH=720, N=3, M_v=6, M_h=5, fw_v=32, fw_h=32, dirs=2)
    stack = np.concatenate([d["fringe_v"], d["gray_v"], d["inv_v"], d["fringe_h"], d["gray_h"], d["inv_h"]])
    roi = (gw != 0).astype(np.uint8)
    r = run_host(shim, cfg, c, stack, roi, mask_is_final=True)
    valid = roi.astype(np.int32)
    m = valid == 1
    for key, direction, codes, unw, code in (("v", 0, 40, r.unw_v, r.code_v), ("h", 1, 23, r.unw_h, r.code_h)):
        w, _ = o.wrapped_phase(d[f"fringe_{key}"], valid)
        ocode = o.decode_gray(d[f"gray_{key}"], d[f"inv_{key}"], valid)
        _, ounw = o.unwrap(direction, w, ocode, valid)
        assert np.array_equal(code.astype(np.int32), ocode)
        assert np.array_equal(unw.view(np.uint32), ounw.view(np.uint32))
        inner = m.copy()
        if direction == 0:
            inner[:, 0] = inner[:, -1] = False
        else:
            inner[0, :] = inner[-1, :] = False
        img = o.unwrapped_image(unw, valid, codes)
        assert np.array_equal(img[inner], d[f"golden_unwrapped_{key}"][inner])      # the reference's stored image


@pytest.mark.parametrize("N,Mv,Mh,fw,W,H,dist", [(3, 6, 5, 8, 256, 192, True), (4, 5, 5, 8, 256, 160, False),
                                                   (5, 6, 6, 4, 192, 128, True), (8, 7, 6, 4, 320, 200, True)])
def test_synthetic_scan_matches_oracle(shim, N, Mv, Mh, fw, W, H, dist):
    PW, PH = fw << Mv if (fw << Mv) <= 1024 else 512, 288
    PW = min(PW, 512)
    cal, ocal, c = calibs(W / 1600.0, PW / 1280.0, dc=None if dist else np.zeros(5))
    cfg = s3.make_config(W, H, PW, PH, N, Mv, Mh, fw, fw, 2)
    stack, roi = s3.synth_stack(cfg, cal)
    ref = run_oracle(cfg, ocal, stack, roi)
    cfgd = dict(W=W, H=H, PW=PW, PH=PH, N=N, M_v=Mv, M_h=Mh, fw_v=fw, fw_h=fw, dirs=2)
    r = run_host(shim, cfgd, c, stack, roi, exact=True)
    assert ref.count > 1000
    assert np.array_equal(r.code_v.astype(np.int32), ref.code_v) and np.array_equal(r.code_h.astype(np.int32), ref.code_h)
    assert np.array_equal(r.unw_v.view(np.uint32), ref.unwrapped_v.view(np.uint32))
    assert np.array_equal(r.unw_h.view(np.uint32), ref.unwrapped_h.view(np.uint32))
    assert np.array_equal(r.valid.astype(np.int32), ref.valid)
    assert np.array_equal(r.cpmap.astype(np.int64)[ref.valid.ravel() == 1], ref.cpmap[ref.valid.ravel() == 1])
    assert r.count == ref.count
    assert np.array_equal(r.pts.view(np.uint32), ref.pts.view(np.uint32))          # reference operation order: bit-identical
    fast = run_host(shim, cfgd, c, stack, roi, exact=False)
    assert fast.count == ref.count
    scale = np.maximum(np.abs(ref.pts).max(axis=1, keepdims=True), 1e-30)
    assert (np.abs(fast.pts - ref.pts) / scale).max() <= 1e-6                      # FMA mode, bar is 1e-5


def test_atan2_on_every_3_and_4_step_argument_pair(shim):
    """(float)atan2(t1, t2) for every (t1, t2) the 3-step (|t1| <= 255, |t2| <= 510) and 4-step formulas can produce,
    against glibc's double atan2 rounded to float (what the reference computes, 3/wrapped_phase.cpp:175,198)."""
    t1, t2 = np.meshgrid(np.arange(-255, 256, dtype=np.float64), np.arange(-510, 511, dtype=np.float64), indexing="ij")
    y = np.ascontiguousarray(t1.ravel())
    x = np.ascontiguousarray(t2.ravel())
    out = np.empty(y.size, np.float32)
    shim.s3d_host_atan2_to_float(_p(y), _p(x), y.size, _p(out))
    want = np.arctan2(y, x).astype(np.float32)
    assert np.array_equal(out.view(np.uint32), want.view(np.uint32))


def test_reference_scan_full_frame_through_the_kernel_arithmetic(shim):
    """configs[0]: the reference's own 1600x1200 capture (3-step, 6/5 Gray bits, fw 32, its calibration files),
    whole frame (tests/golden/c1_full.npz): the stored wrapped-phase image gives the mask, the stored unwrapped-phase
    images must come out of the kernel arithmetic bit for bit (358 580 pixels x 2 directions), and c_p_map /
    validity / points equal the oracle."""
    d = load_c1_full()
    planes = []
    gold = {}
    for name, M in (("Vertical", 6), ("Horizontal", 5)):
        key = name[0].lower()
        assert len(d[f"gray_{key}"]) == len(d[f"inv_{key}"]) == M
        planes += [d[f"fringe_{key}"], d[f"gray_{key}"], d[f"inv_{key}"]]
        gold[name] = (d[f"golden_wrapped_{key}"], d[f"golden_unwrapped_{key}"])
    stack = np.concatenate(planes)
    roi = (gold["Vertical"][0] != 0).astype(np.uint8)
    assert int(roi.sum()) == 358580
    c = load_calib_c1()
    cfg = dict(W=1600, H=1200, PW=1280, PH=720, N=3, M_v=6, M_h=5, fw_v=32, fw_h=32, dirs=2)
    r = run_host(shim, cfg, c, stack, roi, exact=True, mask_is_final=True)
    valid = roi.astype(np.int32)
    m = valid == 1
    assert np.array_equal(o.unwrapped_image(r.unw_v, valid, 40)[m], gold["Vertical"][1][m])
    assert np.array_equal(o.unwrapped_image(r.unw_h, valid, 23)[m], gold["Horizontal"][1][m])
    # stages 5-8 against the oracle on the same planes
    cp, ovalid = o.compute_c_p_map(r.unw_v, r.unw_h, valid, valid, 32, 32, 1280, 720)
    assert np.array_equal(r.valid.astype(np.int32), ovalid)
    assert np.array_equal(r.cpmap.astype(np.int64)[ovalid.ravel() == 1], cp[ovalid.ravel() == 1])
    Ac = o.compute_A(c["Kc"], c["rc"], c["tc"])
    Ap = o.compute_A(c["Kp"], c["rp"], c["tp"])
    xyz = o.triangulate(Ac, Ap, o.undistort_lut(c["Kc"], c["dc"], 1600, 1200), o.undistort_lut(c["Kp"], c["dp"], 1280, 720),
                        cp, ovalid, 1280, 720)
    pts, _, _ = o.compact(xyz, ovalid)
    assert r.count == len(pts) > 300000
    assert np.array_equal(r.pts.view(np.uint32), pts.view(np.uint32))


@pytest.mark.parametrize("N", [3, 4, 5, 6, 7, 8, 12, 16])
def test_stage_kernel_wrapped_phase_all_step_counts(shim, N):
    """k_wrapped's arithmetic (the per-stage path, incl. the generic-N extension) against the oracle on random and
    extreme samples: saturated, black, equal frames (atan2(0, 0)), single bright frame."""
    rng = np.random.default_rng(N)
    n = 200_000
    I = rng.integers(0, 256, (N, n), dtype=np.uint8)
    I[:, :256] = np.arange(256, dtype=np.uint8)[None, :]          # all frames equal: t1 = t2 = 0
    I[:, 256:512] = 0
    I[0, 256:512] = np.arange(256, dtype=np.uint8)               # one bright frame
    I[:, 512:768] = 255
    I[N - 1, 512:768] = np.arange(256, dtype=np.uint8)
    out = np.empty(n, np.float32)
    assert shim.s3d_host_stage_wrapped_phase(_p(np.ascontiguousarray(I)), N, n, _p(out)) == 0
    want, _ = o.wrapped_phase(I.reshape(N, 1, n), np.ones((1, n), np.int32), want_dbg=False)
    assert np.array_equal(out.view(np.uint32), want.ravel().view(np.uint32))
