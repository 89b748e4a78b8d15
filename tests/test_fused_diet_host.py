"""The identities that let the single-pass kernel skip FP64 work, checked on the CPU with the product's own device
header (scan3d_math.cuh, compiled for the host through tests/cuda_host_shim.h):

* the fast triangulation in the camera's frame gives the world-frame fast solve's point, on the golden calibration;
* correspond32's FE_INVALID test always passes on the phases k_fused7 can produce, so correspond32_finite, which
  leaves it out, gives the same correspondences;
* the table of unwrap terms (fill_code_term_table) holds the exact quotient the kernel computed before, for every
  fringe order a configuration can have (M <= 15), and gives the same unwrapped phases."""
import ctypes as C
import os
import subprocess

import numpy as np
import pytest

import oracle_ffi as o
from helpers import load_calib_c1, scaled_calib

HERE = os.path.dirname(os.path.abspath(__file__))
CUDA_INC = "/usr/local/cuda/include"

pytestmark = pytest.mark.skipif(not os.path.exists(os.path.join(CUDA_INC, "cuda_runtime.h")),
                                reason="CUDA headers not installed")


@pytest.fixture(scope="module")
def shim(tmp_path_factory):
    so = str(tmp_path_factory.mktemp("diethost") / "libfused_diet_host.so")
    subprocess.check_call(["/usr/bin/g++", "-O2", "-std=c++17", "-fPIC", "-shared", "-Wall", "-Wno-unknown-pragmas",
                           "-Wno-unused-function", "-ffp-contract=off", "-I", CUDA_INC,
                           "-o", so, os.path.join(HERE, "fused_diet_host.cpp")])
    return C.CDLL(so)


def _p(a):
    return a.ctypes.data_as(C.c_void_p)


def rodrigues(r):
    r = np.asarray(r, np.float64)
    theta = np.linalg.norm(r)
    if theta < 2.2204460492503131e-16:
        return np.eye(3)
    k = r / theta
    K = np.array([[0, -k[2], k[1]], [k[2], 0, -k[0]], [-k[1], k[0], 0]])
    return np.cos(theta) * np.eye(3) + (1 - np.cos(theta)) * np.outer(k, k) + np.sin(theta) * K


def project(A, X):
    h = X @ A[:, :3].T + A[:, 3]
    return h[:, 0] / h[:, 2], h[:, 1] / h[:, 2], h[:, 2]


@pytest.mark.parametrize("scale", [1.0, 0.4, 2.5])
def test_camera_frame_solve_matches_world_frame_fast_solve(shim, scale):
    c = scaled_calib(load_calib_c1(), scale, scale)
    Ac = np.ascontiguousarray(o.compute_A(c["Kc"], c["rc"], c["tc"]))
    Ap = np.ascontiguousarray(o.compute_A(c["Kp"], c["rp"], c["tp"]))
    Rc, Rp = rodrigues(c["rc"]), rodrigues(c["rp"])
    cc, cp = -Rc.T @ c["tc"], -Rp.T @ c["tp"]                       # device centres in the world
    base = np.linalg.norm(cc - cp)
    rng = np.random.default_rng(7)
    # points around the world origin (the calibration target), seen by both devices
    X = rng.uniform(-0.5, 0.5, (200_000, 3)) * base
    uc, vc, zc = project(Ac, X)
    up, vp, zp = project(Ap, X)
    keep = (zc > 0) & (zp > 0)
    assert keep.mean() > 0.9
    n = int(keep.sum())
    # camera pixels from a table are arbitrary doubles; projector pixels are integers without a projector table
    uc = np.ascontiguousarray(uc[keep] + rng.normal(0, 0.3, n))
    vc = np.ascontiguousarray(vc[keep] + rng.normal(0, 0.3, n))
    up = np.ascontiguousarray(np.round(up[keep]))
    vp = np.ascontiguousarray(np.round(vp[keep]))
    xf = np.empty((n, 3))
    xc = np.empty((n, 3))
    Kc = np.ascontiguousarray(c["Kc"], np.float64)
    std = shim.s3d_host_camframe(_p(Kc), _p(np.ascontiguousarray(Rc.ravel())), _p(np.ascontiguousarray(c["tc"])),
                                 _p(Ac), _p(Ap), n, _p(uc), _p(vc), _p(up), _p(vp), _p(xf), _p(xc))
    assert std == 1
    scale_pt = np.abs(xf).max(axis=1)
    rel = np.abs(xc - xf).max(axis=1) / scale_pt
    assert rel.max() <= 1e-9, rel.max()


def test_singular_camera_frame_solve_is_the_world_origin(shim):
    """cvInvert's zero matrix for a singular system: the point is (0, 0, 0) in the world, not the camera centre."""
    c = load_calib_c1()
    Kc = np.ascontiguousarray(c["Kc"], np.float64)
    Ac = np.ascontiguousarray(o.compute_A(c["Kc"], c["rc"], c["tc"]))
    Ap = np.zeros(12)                                              # no projector rows: rank 2 with du = dv = 0
    uc = np.array([Kc[2]]); vc = np.array([Kc[5]]); up = np.array([3.0]); vp = np.array([4.0])
    xf = np.empty(3); xc = np.full(3, np.nan)
    shim.s3d_host_camframe(_p(Kc), _p(np.ascontiguousarray(rodrigues(c["rc"]).ravel())),
                           _p(np.ascontiguousarray(c["tc"])), _p(Ac), _p(Ap), 1, _p(uc), _p(vc), _p(up), _p(vp),
                           _p(xf), _p(xc))
    assert np.array_equal(xc, np.zeros(3))


@pytest.mark.parametrize("fw", [1, 32, 2**31 - 1])
def test_kernel_phases_pass_the_fe_invalid_test(shim, fw):
    """Every fringe order k_fused7 can see (M <= 15 bits) with the extreme and random wrapped phases (atan2 lies in
    [-pi, pi]): the phase is finite, correspond32's |v| < 2^63 test passes, and both give the same correspondence,
    including the saturated ones at fw = 2^31 - 1."""
    codes = np.arange(1 << 15, dtype=np.int32)
    rng = np.random.default_rng(fw)
    ws = [np.float32(-np.pi), np.float32(np.pi), np.float32(0.0)]
    w = np.concatenate([np.full(codes.size, v, np.float32) for v in ws] +
                       [rng.uniform(-np.pi, np.pi, codes.size).astype(np.float32)])
    code = np.ascontiguousarray(np.tile(codes, len(ws) + 1))
    n = w.size
    phi = np.empty(n, np.float32)
    px_old = np.empty(n, np.int32); ok = np.empty(n, np.int32); px_new = np.empty(n, np.int32)
    shim.s3d_host_correspond(_p(np.ascontiguousarray(w)), _p(code), n, C.c_double(float(fw)), _p(phi), _p(px_old),
                             _p(ok), _p(px_new))
    assert np.isfinite(phi).all() and np.abs(phi).max() < 2.0**18
    assert ok.all()
    assert np.array_equal(px_old, px_new)


def test_code_term_table_is_the_exact_quotient_for_every_fringe_order(shim):
    w = np.array([-np.pi, -1.0, 0.0, 1e-3, 2.5, np.pi], np.float32)
    w = np.ascontiguousarray(np.concatenate([w + np.float32(22 / 7), np.float32(22 / 7) * np.ones(1, np.float32)]))
    assert shim.s3d_host_code_term(1 << 15, _p(w), w.size) == 0
