"""CPU checks of the orientation's and the measures' arithmetic (scan3d_voxel_surface_orient, scan3d_mesh_orient_dev,
scan3d_voxel_surface_measure, scan3d_mesh_measure_dev): the shared header 3dscan_b200/common/scan3d_orient_math.h is
compiled for the host and compared bit for bit with the numpy restatement of tests/test_orient_ref.py: the centre and
the exponent, the per-face fixed-point volume and area terms on random, tiny, huge, degenerate and far-off faces, and
the exact int128 sum with its sign and scaling, including sums that need the high word and a carry."""
import ctypes as C
import math
import os
import subprocess

import numpy as np
import pytest

from test_orient_ref import area_terms_ref, centre_ref, exponent_ref, volume_of, area_of, volume_terms_ref

HERE = os.path.dirname(os.path.abspath(__file__))
F32 = np.float32


@pytest.fixture(scope="module")
def L(tmp_path_factory):
    so = os.path.join(str(tmp_path_factory.mktemp("orienthost")), "liborient_math_host.so")
    subprocess.check_call(["/usr/bin/g++", "-O2", "-std=c++17", "-fPIC", "-shared", "-Wall", "-ffp-contract=off",
                           "-o", so, os.path.join(HERE, "orient_math_host.cpp")])
    lib = C.CDLL(so)
    vp, ll = C.c_void_p, C.c_longlong
    lib.s3o_host_frame.argtypes = [vp, vp, vp, ll, vp]
    lib.s3o_host_terms.argtypes = [vp, ll, vp, C.c_int, vp, vp]
    lib.s3o_host_sum.argtypes = [vp, ll, C.c_int, vp, vp]
    return lib


def _p(a):
    return a.ctypes.data_as(C.c_void_p)


@pytest.mark.parametrize("scale", [1.0, 2.0 ** -70, 2.0 ** 60, 1e-3])
def test_frame_and_terms_bit_for_bit(L, scale):
    rng = np.random.default_rng(int(-math.log2(scale)) + 80 if scale != 1e-3 else 3)
    n = 20000
    off = np.array([5.0, -3.0, 1000.0]) * scale
    t = (rng.normal(size=(n, 3, 3)) * scale + off).astype(F32)
    t[: n // 10, 2] = t[: n // 10, 0]                                   # degenerate: D and area 0
    t[n // 10: n // 5] = t[n // 10: n // 5, :, :1]                        # on a line
    pts = np.ascontiguousarray(t.reshape(-1, 3))
    lo, hi = pts.min(0), pts.max(0)
    c = np.zeros(3, F32)
    E = L.s3o_host_frame(_p(lo), _p(hi), _p(pts), len(pts), _p(c))
    np.testing.assert_array_equal(c.view(np.uint32), centre_ref(lo, hi).view(np.uint32))
    assert E == exponent_ref(pts, c)
    vol, area = np.zeros(n, np.int64), np.zeros(n, np.int64)
    L.s3o_host_terms(_p(np.ascontiguousarray(t)), n, _p(c), E, _p(vol), _p(area))
    np.testing.assert_array_equal(vol, volume_terms_ref(t[:, 0], t[:, 1], t[:, 2], c, E))
    np.testing.assert_array_equal(area, area_terms_ref(t[:, 0], t[:, 1], t[:, 2], E))
    assert np.abs(vol).max() < 2 ** 62 and np.abs(area).max() < 2 ** 62 and (area >= 0).all()
    # the bound's worst case: the corners of the box about the centre
    corners = np.array([[[E2 * sx, E2 * sy, E2 * sz] for sx, sy, sz in ((1, -1, -1), (-1, 1, -1), (-1, -1, 1))]
                        for E2 in (0.999 * math.ldexp(1.0, E),)], np.float64) + c
    v2, a2 = np.zeros(1, np.int64), np.zeros(1, np.int64)
    L.s3o_host_terms(_p(np.ascontiguousarray(corners.astype(F32))), 1, _p(c), E, _p(v2), _p(a2))
    assert abs(int(v2[0])) < 2 ** 62 and int(a2[0]) < 2 ** 62


def test_the_int128_sum_bit_for_bit(L):
    rng = np.random.default_rng(7)
    for case in range(12):
        m = int(rng.integers(0, 5000))
        big = case % 3 != 0
        t = rng.integers(-(2 ** 62) + 1, 2 ** 62, m, dtype=np.int64) if big else rng.integers(-1000, 1000, m)
        if case == 1:
            t = np.full(m, 2 ** 62 - 1, np.int64)                       # every add carries into the high word
        if case == 2:
            t = -np.abs(t)
        t = np.ascontiguousarray(t, np.int64)
        E = int(rng.integers(-149, 130))
        lohi = np.zeros(2, np.uint64)
        va = np.zeros(2)
        sign = L.s3o_host_sum(_p(t), len(t), E, _p(lohi), _p(va))
        want = sum(int(x) for x in t)
        got = int(lohi[0]) | (int(lohi[1]) << 64)
        assert got == want % (1 << 128)
        assert sign == (want > 0) - (want < 0)
        assert va[0] == volume_of(want, E) and va[1] == area_of(want, E)
