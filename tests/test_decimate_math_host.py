"""CPU checks of the surface simplification arithmetic (scan3d_voxel_surface_decimate): the shared header
3dscan_b200/common/scan3d_decimate_math.h is compiled for the host and compared bit for bit with the numpy
restatement of tests/test_decimate_ref.py (face quadrics, fixed point, the damped solve and its fallbacks, the
canonical rotation); and the overflow bound the header derives is checked against surface-nets meshes."""
import ctypes as C
import itertools
import os
import subprocess

import numpy as np
import pytest

from test_decimate_ref import (DAMPING, canonical_ref, clusters_ref, corner_coeffs_ref, face_planes_ref, nets_mesh,
                               place_ref)

HERE = os.path.dirname(os.path.abspath(__file__))
F32, F64 = np.float32, np.float64
Q = 2.0 ** 24


@pytest.fixture(scope="module")
def L(tmp_path_factory):
    so = str(tmp_path_factory.mktemp("decimatehost") / "libdecimate_math_host.so")
    subprocess.check_call(["/usr/bin/g++", "-O2", "-std=c++17", "-fPIC", "-shared", "-Wall", "-ffp-contract=off",
                           "-o", so, os.path.join(HERE, "decimate_math_host.cpp")])
    lib = C.CDLL(so)
    vp, ll, d = C.c_void_p, C.c_longlong, C.c_double
    lib.s3q_host_face_planes.argtypes = [vp, ll, d, vp, vp, vp]
    lib.s3q_host_corner_coeffs.argtypes = [vp, vp, vp, ll, vp]
    lib.s3q_host_fractions.argtypes = [vp, ll, d, vp]
    lib.s3q_host_to_fixed.argtypes = [vp, ll, vp]
    lib.s3q_host_place.argtypes = [vp, vp, vp, ll, vp, vp]
    lib.s3q_host_coords.argtypes = [vp, vp, ll, d, vp]
    lib.s3q_host_canonical.argtypes = [vp, ll, vp, vp]
    for f in ("s3q_host_face_bound", "s3q_host_sum_bound"):
        getattr(lib, f).argtypes = [d]
        getattr(lib, f).restype = d
    lib.s3q_host_damping.restype = d
    return lib


def _p(a):
    return a.ctypes.data_as(C.c_void_p)


def _bits_equal(a, b):
    assert a.shape == b.shape and a.dtype == b.dtype
    assert np.array_equal(a.view(np.uint8), b.view(np.uint8))


def host_planes(L, tri, H):
    tri = np.ascontiguousarray(tri, F32).reshape(-1, 3, 3)
    n = len(tri)
    u, w, ok = np.zeros((n, 3)), np.zeros(n), np.zeros(n, np.int32)
    L.s3q_host_face_planes(_p(tri), n, H, _p(u), _p(w), _p(ok))
    return u, w, ok.astype(bool)


def host_coeffs(L, u, w, f):
    u, w, f = (np.ascontiguousarray(a, F64) for a in (u, w, f))
    q = np.zeros((len(w), 10), np.int64)
    L.s3q_host_corner_coeffs(_p(u), _p(w), _p(f), len(w), _p(q))
    return q


def host_fractions(L, x, H):
    x = np.ascontiguousarray(x, F32).reshape(-1)
    f = np.zeros(x.shape, F64)
    L.s3q_host_fractions(_p(x), x.size, H, _p(f))
    return f


def host_place(L, qs, sq, cnt):
    qs, sq, cnt = np.ascontiguousarray(qs, np.int64), np.ascontiguousarray(sq, np.uint64), np.ascontiguousarray(cnt, np.uint32)
    y, st = np.zeros((len(cnt), 3)), np.zeros(len(cnt), np.int32)
    L.s3q_host_place(_p(qs), _p(sq), _p(cnt), len(cnt), _p(y), _p(st))
    return y, st


def test_constants(L):
    assert L.s3q_host_p() == 40 and L.s3q_host_damping() == DAMPING


def test_face_quadrics_and_fractions(L):
    rng = np.random.default_rng(0)
    n = 20000
    tri = (rng.normal(size=(n, 3, 3)) * rng.choice([1e-20, 1e-3, 1.0, 1e3, 1e18], size=(n, 1, 1))).astype(F32)
    tri[:500, 1] = tri[:500, 0]                                     # two equal corners
    tri[500:1000, 2] = tri[500:1000, 0] + (tri[500:1000, 1] - tri[500:1000, 0]) * 2   # collinear in float
    tri[1000:1500] = np.abs(tri[1000:1500]) * F32(0)                # signed zeros ...
    tri[1000:1500, :, 1] = -tri[1000:1500, :, 1]
    tri[1500:1600] = np.array([[0.0, 0.0, 0.0], [-0.0, 1.0, 0.0], [0.0, -0.0, 1.0]], F32)
    tri[1600:1700] *= F32(1e-25)                                   # tiny areas
    tri[1700:1800] = tri[1700:1800] * F32(1e-20) + F32(1e20)        # differences that round to 0 in float
    for H in (F64(F32(0.05)), F64(F32(3.7)), F64(F32(256 * 0.05))):
        u, w, ok = host_planes(L, tri, H)
        ru, rw, rok = face_planes_ref(tri.reshape(-1, 3), np.arange(3 * n).reshape(-1, 3), H)
        assert np.array_equal(ok, rok) and ok.sum() > n // 2
        assert (~ok[:500]).all() and (~ok[1000:1500]).all() and ok[1500:1600].all() and (~ok[1700:1800]).all()
        _bits_equal(u[ok], ru[ok])
        _bits_equal(w[ok], rw[ok])
        f = host_fractions(L, tri[:, 0], H).reshape(-1, 3)
        t = tri[:, 0].astype(F64) / H
        _bits_equal(f, t - np.floor(t))
        assert ((f >= 0) & (f <= 1)).all()                          # 1 when a tiny negative t rounds up
        live = ok & (w < 1e6)                                       # 3 w 2^40 fits int64
        _bits_equal(host_coeffs(L, u[live], w[live], f[live]), corner_coeffs_ref(u[live], w[live], f[live]))


def test_fixed_point_rounding(L):
    k = np.arange(-2000, 2000, dtype=F64)
    v = np.concatenate([(k + 0.5) * 2.0 ** -40, (k + 0.25) * 2.0 ** -40, k * 2.0 ** -40, [0.0, -0.0, 3.0, -3.0]])
    q = np.zeros(v.shape, np.int64)
    L.s3q_host_to_fixed(_p(v), v.size, _p(q))
    assert np.array_equal(q, np.rint(v * 2.0 ** 40).astype(np.int64))
    assert q[2000] == 0 and q[2001] == 2 and q[1999] == 0 and q[1998] == -2   # half to even: 0.5, 1.5, -0.5, -1.5


def _sums_of_planes(rng, c, planes=6):
    """quadric sums of random planes through random corners, as int64 [c][10]"""
    u = rng.normal(size=(c * planes, 3))
    u /= np.linalg.norm(u, axis=1, keepdims=True)
    f = rng.random((c * planes, 3))
    w = rng.random(c * planes) * 2
    q = corner_coeffs_ref(u, w, f)
    return q.reshape(c, planes, 10).sum(1)


def test_placement(L):
    rng = np.random.default_rng(1)
    c = 5000
    qs = np.concatenate([_sums_of_planes(rng, c, 6), _sums_of_planes(rng, c, 1), _sums_of_planes(rng, c, 2),
                         np.zeros((10, 10), np.int64)])
    n = rng.integers(1, 40, len(qs)).astype(np.uint32)
    sq = (rng.integers(0, 2 ** 24, (len(qs), 3)) * n[:, None]).astype(np.uint64)
    y, st = host_place(L, qs, sq, n)
    ry, rst = place_ref(qs, sq, n)
    _bits_equal(y, ry)
    assert np.array_equal(st, rst)
    assert (st[-10:] == 1).all() and (st == 0).sum() > 0 and (st == 2).sum() > 0
    print(f"placement: {np.bincount(st, minlength=3)} solved / mean / fallback")
    # coordinates
    ijk = rng.integers(-2 ** 20, 2 ** 20, y.shape).astype(np.int64)
    out = np.zeros(y.shape, F32)
    H = F64(F32(0.37))
    L.s3q_host_coords(_p(ijk), _p(y), len(y), H, _p(out))
    _bits_equal(out, ((ijk.astype(F64) + y) * H).astype(F32))


def _fixed(A, b):
    """int64 [10] sums of the symmetric A and b"""
    v = np.array([A[0, 0], A[0, 1], A[0, 2], A[1, 1], A[1, 2], A[2, 2], b[0], b[1], b[2], 0.0])
    return np.rint(v * 2.0 ** 40).astype(np.int64)


def test_pivot_failures_and_the_faces_of_the_cube(L):
    half = np.array([[Q / 2] * 3], np.uint64)                    # ybar = (0.5, 0.5, 0.5) for one vertex
    cases, want = [], []
    # indefinite matrices fail the pivot test
    for A in (np.array([[1.0, 2, 0], [2, 1, 0], [0, 0, 1]]), np.array([[1.0, 0, 0], [0, 1, 0], [0, 0, -0.5]]),
              np.array([[0.0, 1, 0], [1, 0, 0], [0, 0, 1]])):
        cases.append(_fixed(A, np.array([0.5, 0.5, 0.5])))
        want.append(2)
    # a well-conditioned quadric whose minimum is just outside / on / inside each face of the unit cube
    for axis, side in itertools.product(range(3), (0.0, 1.0)):
        for d, st in ((-0.01, 2), (0.0, 0), (0.01, 0)):
            t = np.full(3, 0.5)
            t[axis] = side + (d if side == 0.0 else -d)
            A = np.eye(3) * 4.0
            # (A + mu I) y = A t + mu ybar with ybar = 0.5: y = t exactly where t = 0.5, and y_axis = (4 t + mu / 2) /
            # (4 + mu), which lies within [0, 1] exactly when t does
            cases.append(_fixed(A, A @ t))
            want.append(st)
    qs = np.array(cases)
    sq = np.repeat(half, len(qs), 0)
    n = np.ones(len(qs), np.uint32)
    y, st = host_place(L, qs, sq, n)
    ry, rst = place_ref(qs, sq, n)
    _bits_equal(y, ry)
    assert np.array_equal(st, rst) and st.tolist() == want
    assert (y[st == 2] == 0.5).all()


def test_canonical_rotation(L):
    t = np.array(list(itertools.permutations([3, 7, 11])) + [[5, 5, 9], [9, 5, 5], [5, 9, 5], [4, 4, 4],
                                                             [-1, 2, 3], [2 ** 31 - 1, 0, 7]], np.int32)
    out, col = np.zeros_like(t), np.zeros(len(t), np.uint8)
    L.s3q_host_canonical(_p(t), len(t), _p(out), _p(col))
    assert col.tolist() == [0] * 6 + [1, 1, 1, 1, 0, 0]
    live = col == 0
    assert np.array_equal(out[live], canonical_ref(t[live]))
    assert out[:6].tolist() == [[3, 7, 11], [3, 11, 7], [3, 11, 7], [3, 7, 11], [3, 7, 11], [3, 11, 7]]


@pytest.mark.parametrize("seed", [0, 1])
def test_overflow_bound_on_surface_nets_meshes(L, seed):
    """the largest rounded corner coefficient, the faces per vertex, the vertices per cluster and the cluster sums of
    random surface-nets meshes against the bounds the header derives, at H = s and H = 256 s"""
    rng = np.random.default_rng(seed)
    s = F32(0.25)
    xyz, _, _, faces = nets_mesh(rng, 400, s)
    assert len(faces) > 100
    faces = faces.astype(np.int64)
    assert np.bincount(faces.ravel()).max() <= 24
    for r in (1.0, 256.0):
        H = F64(F32(r * s))
        u, w, ok = host_planes(L, xyz[faces], H)
        cid, _, _, f = clusters_ref(xyz, H)
        sums = np.zeros((cid.max() + 1, 10), np.int64)
        top = 0
        for k in range(3):
            q = host_coeffs(L, u[ok], w[ok], f[faces[ok, k]])
            top = max(top, int(np.abs(q).max()))
            np.add.at(sums, cid[faces[ok, k]], q)
        bound = L.s3q_host_face_bound(r)
        assert 0 < top <= bound, (r, top, bound)
        assert np.bincount(cid).max() <= (np.floor(r) + 3) ** 3
        assert np.abs(sums).max() <= L.s3q_host_sum_bound(r)
        print(f"H/s {r:g}: largest corner coefficient {top} <= {bound:.6g} ({top / bound:.3f} of the bound)")
    rs = np.concatenate([np.linspace(1, 256, 2551), np.nextafter(np.arange(2, 257), 0)])
    worst = max(L.s3q_host_sum_bound(float(r)) for r in rs)
    assert worst == L.s3q_host_sum_bound(256.0) and worst < 2.0 ** 56.3 < 2.0 ** 63
