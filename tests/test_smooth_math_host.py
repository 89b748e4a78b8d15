"""CPU checks of the surface smoothing arithmetic (scan3d_voxel_surface_smooth, scan3d_mesh_smooth_dev): the shared
header 3dscan_b200/common/scan3d_smooth_math.h is compiled for the host and compared bit for bit with the numpy
restatement of tests/test_smooth_ref.py (the exponent and the fixed point, including negative zero, subnormals and
coordinates far below 2^E; the pass update, including rint ties; the face normals and their finish); and the
overflow bound the header derives is checked at its extremes."""
import ctypes as C
import os
import subprocess

import numpy as np
import pytest

from test_smooth_ref import (DEGREE_LIMIT, P, Q_LIMIT, dequantise_ref, displacement_ref, exponent_ref,
                             face_normals_ref, normal_out_ref, quantise_ref, update_ref)

HERE = os.path.dirname(os.path.abspath(__file__))
F32, F64 = np.float32, np.float64


@pytest.fixture(scope="module")
def L(tmp_path_factory):
    so = str(tmp_path_factory.mktemp("smoothhost") / "libsmooth_math_host.so")
    subprocess.check_call(["/usr/bin/g++", "-O2", "-std=c++17", "-fPIC", "-shared", "-Wall", "-ffp-contract=off",
                           "-o", so, os.path.join(HERE, "smooth_math_host.cpp")])
    lib = C.CDLL(so)
    vp, ll, i32, d = C.c_void_p, C.c_longlong, C.c_int, C.c_double
    lib.s3t_host_exponent.argtypes = [vp, ll]
    lib.s3t_host_exponent.restype = i32
    lib.s3t_host_quantise.argtypes = [vp, ll, i32, vp]
    lib.s3t_host_dequantise.argtypes = [vp, ll, i32, vp]
    lib.s3t_host_update.argtypes = [vp, vp, vp, ll, d, vp, vp]
    lib.s3t_host_face_normals.argtypes = [vp, ll, vp, vp]
    lib.s3t_host_normal_out.argtypes = [vp, ll, vp]
    lib.s3t_host_displacement.argtypes = [vp, vp, ll, vp]
    lib.s3t_host_limits.argtypes = [vp]
    return lib


def _p(a):
    return a.ctypes.data_as(C.c_void_p)


def _bits_equal(a, b):
    assert a.shape == b.shape and a.dtype == b.dtype
    assert np.array_equal(a.view(np.uint8), b.view(np.uint8))


def host_exponent(L, x):
    x = np.ascontiguousarray(x, F32).reshape(-1)
    return L.s3t_host_exponent(_p(x), x.size)


def host_quantise(L, x, E):
    x = np.ascontiguousarray(x, F32).reshape(-1)
    q = np.zeros(x.size, np.int64)
    L.s3t_host_quantise(_p(x), x.size, E, _p(q))
    return q


def host_dequantise(L, q, E):
    q = np.ascontiguousarray(q, np.int64).reshape(-1)
    x = np.zeros(q.size, F32)
    L.s3t_host_dequantise(_p(q), q.size, E, _p(x))
    return x


def host_update(L, q, s, d, k):
    q, s = np.ascontiguousarray(q, np.int64), np.ascontiguousarray(s, np.int64)
    d = np.ascontiguousarray(d, np.uint32)
    out, over = np.zeros(q.size, np.int64), np.zeros(q.size, np.uint8)
    L.s3t_host_update(_p(q), _p(s), _p(d), q.size, k, _p(out), _p(over))
    return out, over.astype(bool)


def test_limits(L):
    out = np.zeros(4, np.int64)
    L.s3t_host_limits(_p(out))
    assert list(out) == [P, Q_LIMIT, DEGREE_LIMIT, -126]
    # the neighbour sums of the bound stay below 2^63
    assert DEGREE_LIMIT * Q_LIMIT <= 2 ** 62


def _coords(rng):
    x = rng.normal(size=4000) * np.exp2(rng.integers(-40, 40, 4000))
    specials = [0.0, -0.0, 1e-45, -1e-45, 1.1754942e-38, 1.17549435e-38, 2.0, -2.0, 0.5, 1.0, 3.4028235e38,
                -3.4028235e38, 2.0 ** 127, 1.5 * 2 ** -140]
    return np.concatenate([x, specials]).astype(F32)


def test_exponent(L):
    rng = np.random.default_rng(0)
    x = _coords(rng)
    for part in (x, x[:10], np.zeros(5, F32), -np.zeros(5, F32), np.array([1e-45], F32), np.array([2.0], F32),
                 np.array([1.9999999], F32), np.array([3.4028235e38], F32), np.zeros(0, F32)):
        E = host_exponent(L, part)
        assert E == exponent_ref(part)
        a = np.abs(part.astype(F64))
        assert (a < 2.0 ** E).all() and (part.size == 0 or E == -126 or a.max() >= 2.0 ** (E - 1))


def test_quantise_and_dequantise(L):
    rng = np.random.default_rng(1)
    x = _coords(rng)
    for E in sorted({exponent_ref(x), exponent_ref(x[:4000]), 3, -126, -100, 0}):
        xs = x[np.abs(x.astype(F64)) < 2.0 ** E]
        q = host_quantise(L, xs, E)
        _bits_equal(q, quantise_ref(xs, E))
        assert (np.abs(q) < 2 ** 40).all()
        # exact wherever |x| >= 2^(E - 17); the sign of zero is lost
        back = host_dequantise(L, q, E)
        _bits_equal(back, dequantise_ref(q, E))
        exact = np.abs(xs.astype(F64)) >= 2.0 ** (E - 17)
        assert np.array_equal(back.view(np.uint32)[exact], xs.view(np.uint32)[exact])
        assert (back[xs == 0].view(np.uint32) == 0).all()
    # rint ties go to even: x = (k + 1/2) 2^(E - 40)
    E = 0
    xs = (np.arange(-20, 20) + 0.5) * 2.0 ** (E - P)
    q = host_quantise(L, xs.astype(F32), E)
    assert np.array_equal(q, np.rint(np.arange(-20, 20) + 0.5).astype(np.int64)) and (q % 2 == 0).all()
    # an output coordinate beyond the float range (E = 128, |Q| > 2^40) is +-inf
    big = host_dequantise(L, np.array([2 ** 41, -(2 ** 41), 2 ** 39], np.int64), 128)
    assert np.isinf(big[:2]).all() and np.isfinite(big[2])


def test_update(L):
    rng = np.random.default_rng(2)
    n = 20000
    d = rng.integers(1, 40, n).astype(np.uint32)
    d[:50] = DEGREE_LIMIT
    q = rng.integers(-2 ** 40, 2 ** 40, n)
    s = rng.integers(-2 ** 40, 2 ** 40, n) * d.astype(np.int64)
    s[100:200] = q[100:200] * d[100:200].astype(np.int64) + rng.integers(-3, 4, 100)   # near the vertex itself
    for k in (0.5, float(F32(-0.53)), 1.0, -1.0, float(F32(0.33))):
        got, over = host_update(L, q, s, d, k)
        _bits_equal(got, update_ref(q, s, d, k))
        _bits_equal(over, np.abs(got) > Q_LIMIT)
    # ties: k (m - Q) = j + 1/2 rounds to even
    q = np.zeros(8, np.int64)
    s = np.array([1, 3, 5, 7, -1, -3, -5, -7], np.int64)
    got, _ = host_update(L, q, s, np.ones(8, np.uint32), 0.5)
    assert np.array_equal(got, [0, 2, 2, 4, 0, -2, -2, -4])
    _bits_equal(got, update_ref(q, s, np.ones(8), 0.5))


def test_overflow_bound(L):
    # the extremes the header allows: |Q| = 2^42 at every neighbour of a vertex of 2^20 neighbours, k = +-1
    lim, dl = Q_LIMIT, DEGREE_LIMIT
    q = np.array([lim, -lim, lim, -lim, 0, lim], np.int64)
    s = np.array([-lim * dl, lim * dl, lim * dl, -lim * dl, lim * dl, -lim * dl], np.int64)
    assert (np.abs(s) <= 2 ** 62).all()
    for k in (1.0, -1.0):
        got, over = host_update(L, q, s, np.full(6, dl, np.uint32), k)
        _bits_equal(got, update_ref(q, s, np.full(6, dl), k))
        assert (np.abs(got) < 2 ** 44).all()
        assert np.array_equal(got, q + (k * (s // dl - q)).astype(np.int64))   # exact at these powers of two
    # a mu pass can leave the limit: that is the device's overflow flag
    got, over = host_update(L, np.array([lim], np.int64), np.array([-lim], np.int64), np.ones(1, np.uint32), -1.0)
    assert over[0] and got[0] == 3 * lim
    # the normal sums: fewer than 2^31 faces of |m| <= 2^24
    assert 2 ** 31 * 2 ** 24 <= 2 ** 55


def test_face_normals_and_finish(L):
    rng = np.random.default_rng(3)
    n = 3000
    tri = (rng.normal(size=(n, 3, 3)) * np.exp2(rng.integers(-20, 20, (n, 1, 1)))).astype(F32)
    tri[:50, 1] = tri[:50, 0]                            # zero area
    tri[50:100, 2] = tri[50:100, 0] + 2 * (tri[50:100, 1] - tri[50:100, 0])   # nearly collinear
    tri[100:105] = (rng.uniform(-1, 1, (5, 3, 3)) * 3e38).astype(F32)         # huge: still finite in double
    tri[105:110, 1, 2] = np.inf                                                # not finite: adds nothing
    tri[110:120] = (rng.normal(size=(10, 3, 3)) * 1e-40).astype(F32)          # subnormal corners
    tri[120:130] = np.where(rng.random((10, 3, 3)) < 0.5, F32(-0.0), F32(0.0))
    m, ok = np.zeros((n, 3), np.int64), np.zeros(n, np.uint8)
    flat = np.ascontiguousarray(tri)
    L.s3t_host_face_normals(_p(flat), n, _p(m), _p(ok))
    p = tri.reshape(-1, 3)
    with np.errstate(invalid="ignore"):
        want_ok, want_m = face_normals_ref(p, np.arange(3 * n).reshape(n, 3))
    assert np.array_equal(ok.astype(bool), want_ok)
    assert not want_ok[:50].any() and want_ok[100:105].all() and not want_ok[105:110].any()
    assert want_ok[130:].mean() > 0.99
    assert np.array_equal(m[want_ok], want_m[want_ok])
    assert (np.abs(m) <= 2 ** 24).all()
    # the finish: sums of a few faces per vertex, zeros included
    s = np.concatenate([want_m[130:1130].reshape(-1, 5, 3).sum(1), np.zeros((3, 3), np.int64),
                        [[1, 0, 0], [0, -1, 0], [2 ** 54, -(2 ** 54), 3]]])
    out = np.zeros(s.shape, F32)
    L.s3t_host_normal_out(_p(np.ascontiguousarray(s)), len(s), _p(out))
    _bits_equal(out, normal_out_ref(s))
    a = rng.normal(size=(500, 3)).astype(F32)
    b = (a + rng.normal(size=(500, 3)) * np.exp2(rng.integers(-30, 5, (500, 1)))).astype(F32)
    b[:10] = a[:10]
    got = np.zeros(500)
    L.s3t_host_displacement(_p(a), _p(b), 500, _p(got))
    _bits_equal(got, displacement_ref(a, b))
    assert (got[:10] == 0).all()
