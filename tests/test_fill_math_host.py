"""CPU checks of the hole-filling arithmetic (scan3d_voxel_surface_fill_holes, scan3d_mesh_fill_holes_dev): the shared
header 3dscan_b200/common/scan3d_fill_math.h is compiled for the host and compared bit for bit with the numpy
restatement of tests/test_fill_ref.py (the triangle terms, including degenerate triangles and signed zeros; the cos
rule; the whole per-hole DP on random planar and non-planar polygons, with existing edges, and on integer polygons
whose weights tie); and the decimation bound behind SCAN3D_FILL_NETS_MAX_EDGES is checked at 22 and 23."""
import ctypes as C
import os
import subprocess

import numpy as np
import pytest

from test_fill_ref import NETS_MAX_EDGES, MAX_EDGES, cos_ref, polygon_ref, triangle_ref

HERE = os.path.dirname(os.path.abspath(__file__))
F32, F64 = np.float32, np.float64


def build_host_lib(directory):
    """the header compiled for the host (tests/fill_math_host.cpp) into directory, with its argument types"""
    so = os.path.join(str(directory), "libfill_math_host.so")
    subprocess.check_call(["/usr/bin/g++", "-O2", "-std=c++17", "-fPIC", "-shared", "-Wall", "-ffp-contract=off",
                           "-o", so, os.path.join(HERE, "fill_math_host.cpp")])
    lib = C.CDLL(so)
    vp, ll, i32 = C.c_void_p, C.c_longlong, C.c_int
    lib.s3h_host_triangle.argtypes = [vp, ll, vp, vp, vp]
    lib.s3h_host_cos.argtypes = [vp, vp, vp, vp, ll, vp]
    lib.s3h_host_polygon.argtypes = [vp, vp, vp, i32, vp, vp, vp, vp]
    lib.s3h_host_polygon.restype = i32
    lib.s3h_host_limits.argtypes = [vp, vp]
    return lib


@pytest.fixture(scope="module")
def L(tmp_path_factory):
    return build_host_lib(tmp_path_factory.mktemp("fillhost"))


def _p(a):
    return a.ctypes.data_as(C.c_void_p)


def _bits_equal(a, b):
    a, b = np.ascontiguousarray(a), np.ascontiguousarray(b)
    assert a.shape == b.shape and a.dtype == b.dtype
    assert np.array_equal(a.view(np.uint8), b.view(np.uint8))


def host_triangle(L, t):
    t = np.ascontiguousarray(t, F32)
    n = len(t)
    u, a, h = np.zeros((n, 3)), np.zeros(n), np.zeros(n, np.uint8)
    L.s3h_host_triangle(_p(t), n, _p(u), _p(a), _p(h))
    return u, h.astype(bool), a


def host_polygon(L, p, rims, exists):
    p, rims = np.ascontiguousarray(p, F32), np.ascontiguousarray(rims, F32)
    ex = np.ascontiguousarray(exists, np.uint8)
    n = len(p)
    cmin, area, k = np.zeros((n, n)), np.zeros((n, n)), np.zeros((n, n), np.int32)
    faces = np.zeros((max(n - 2, 1), 3), np.int32)
    ok = L.s3h_host_polygon(_p(p), _p(rims), _p(ex), n, _p(cmin), _p(area), _p(k), _p(faces))
    return (faces[:n - 2] if ok else None), cmin, area, k


def _triangles(rng, n):
    t = (rng.normal(size=(n, 3, 3)) * np.exp2(rng.integers(-20, 20, (n, 1, 1)))).astype(F32)
    t[:40, 1] = t[:40, 0]                                                    # two equal corners
    t[40:80, 2] = t[40:80, 0] + 2 * (t[40:80, 1] - t[40:80, 0])              # (nearly) collinear
    t[80:100] = np.where(rng.random((20, 3, 3)) < 0.5, F32(-0.0), F32(0.0))  # signed zeros
    t[100:120, :, 2] = F32(-0.0)                                             # planar, z = -0
    t[120:130] = (rng.uniform(-1, 1, (10, 3, 3)) * 3e38).astype(F32)         # huge: still finite in double
    t[130:140] = (rng.normal(size=(10, 3, 3)) * 1e-40).astype(F32)           # subnormal corners
    t[140:160] = rng.integers(-3, 4, (20, 3, 3)).astype(F32)                 # small integers
    return t


def test_triangle_terms_and_cos(L):
    rng = np.random.default_rng(0)
    t = _triangles(rng, 4000)
    u, has, area = host_triangle(L, t)
    wu, whas, warea = triangle_ref(t[:, 0], t[:, 1], t[:, 2])
    _bits_equal(has, whas)
    _bits_equal(u, wu)
    _bits_equal(area, warea)
    assert not has[:40].any() and (area[:40] == 0).all() and has[160:].mean() > 0.99
    # the cos rule, -1 where either normal is missing, on pairs that include equal and opposite normals
    j = rng.permutation(len(t))
    j[:50] = np.arange(50) + 150
    pairs = [(u, has, u[j], has[j]), (u, has, -u, has), (u, has, u, has)]
    for a, ha, b, hb in pairs:
        a, b = np.ascontiguousarray(a), np.ascontiguousarray(b)
        out = np.zeros(len(a))
        L.s3h_host_cos(_p(a), _p(ha.astype(np.uint8)), _p(b), _p(hb.astype(np.uint8)), len(a), _p(out))
        _bits_equal(out, cos_ref(a, ha, b, hb))
        assert (out[~(ha & hb)] == -1.0).all()


def _rims(rng, p, lift):
    """rim faces of a polygon p: (v_{t+1}, v_t, w_t) with w_t outside, lifted by `lift` off the polygon's plane"""
    n = len(p)
    c = p.astype(F64).mean(0)
    nxt = np.roll(p, -1, 0).astype(F64)
    mid = (p.astype(F64) + nxt) / 2
    w = mid + (mid - c) * 0.5 + lift * rng.normal(size=(n, 3)) * [0, 0, 1]
    return np.stack([nxt, p.astype(F64), w], 1).astype(F32)


def _check_polygon(L, p, rims, exists):
    got = host_polygon(L, p, rims, exists)
    ru, rh, _ = triangle_ref(rims[:, 0], rims[:, 1], rims[:, 2])
    want = polygon_ref(p, ru, rh, exists)
    n = len(p)
    if want[0] is None:
        assert got[0] is None
    else:
        assert got[0] is not None and np.array_equal(got[0], want[0])
    iu = np.triu_indices(n, 2)
    _bits_equal(got[3][iu].astype(np.int64), want[3][iu])
    feas = want[3][iu] >= 0
    _bits_equal(got[1][iu][feas], want[1][iu][feas])
    _bits_equal(got[2][iu][feas], want[2][iu][feas])
    return want


@pytest.mark.parametrize("seed", range(3))
def test_dp_on_random_polygons(L, seed):
    rng = np.random.default_rng(seed)
    for n in (3, 4, 5, 8, 13, 22, 40):
        th = np.sort(rng.uniform(0, 2 * np.pi, n))
        r = 1 + 0.3 * rng.random(n)
        flat = np.stack([r * np.cos(th), r * np.sin(th), np.zeros(n)], 1).astype(F32)
        bumpy = (flat + rng.normal(size=(n, 3)) * [0.05, 0.05, 0.3]).astype(F32)
        for p, lift in ((flat, 0.0), (bumpy, 0.2)):
            ex = np.zeros((n, n), bool)
            _check_polygon(L, p, _rims(rng, p, lift), ex)
            # some diagonals already exist (symmetric), which blocks cells and can leave the hole open
            ex = rng.random((n, n)) < 0.3
            ex = ex | ex.T
            _check_polygon(L, p, _rims(rng, p, lift), ex)
    # every diagonal exists: only the closing cell of a triangle is feasible
    for n in (3, 4, 6):
        p = np.stack([np.cos(np.arange(n)), np.sin(np.arange(n)), np.zeros(n)], 1).astype(F32)
        want = _check_polygon(L, p, _rims(rng, p, 0.0), np.ones((n, n), bool))
        assert (want[0] is not None) == (n == 3)


def test_dp_ties_on_integer_polygons(L):
    """planar integer polygons: every cos is exactly 1 or -1 (collinear vertices give triangles without a normal), so
    cmin ties everywhere, areas tie by symmetry and the smaller k decides"""
    rng = np.random.default_rng(7)
    square = np.array([[0, 0, 0], [1, 0, 0], [2, 0, 0], [2, 1, 0], [2, 2, 0], [1, 2, 0], [0, 2, 0], [0, 1, 0]], F32)
    hexagon = np.array([[2, 0, 0], [1, 2, 0], [-1, 2, 0], [-2, 0, 0], [-1, -2, 0], [1, -2, 0]], F32)
    rect = np.array([[x, 0, 0] for x in range(6)] + [[5, 1, 0]] + [[x, 1, 0] for x in range(4, -1, -1)], F32)
    for p in (square, hexagon, rect, square[::-1].copy()):
        want = _check_polygon(L, p, _rims(rng, p, 0.0), np.zeros((len(p), len(p)), bool))
        iu = np.triu_indices(len(p), 2)
        k = want[3][iu]
        assert (k >= 0).all()
    # a regular polygon's symmetric candidates: equal weights, the smallest k wins
    p = np.array([[1, 0, 0], [0, 1, 0], [-1, 0, 0], [0, -1, 0]], F32)
    faces = _check_polygon(L, p, _rims(rng, p, 0.0), np.zeros((4, 4), bool))[0]
    assert faces.tolist() == [[0, 1, 3], [1, 2, 3]]


def test_decimation_bound_at_the_nets_cap(L):
    out, bound = np.zeros(4, np.int64), np.zeros(256)
    L.s3h_host_limits(_p(out), _p(bound))
    assert list(out) == [NETS_MAX_EDGES, MAX_EDGES, 1, 0]
    area_max, scale = 9 * np.sqrt(3) / 4, 2.0 ** 40

    def sum_bound(m, N):
        face = 3 * area_max / (m * m) * scale + 0.5
        fill = 3 * area_max * (N / 2) ** 2 / (m * m) * scale + 0.5
        return (m + 3.0) ** 3 * (24 * face + (N - 2) * fill)
    m = np.arange(1, 257, dtype=F64)
    assert np.allclose(bound, sum_bound(m, NETS_MAX_EDGES), rtol=1e-15, atol=0)
    assert sum_bound(m, NETS_MAX_EDGES).max() < 2.0 ** 63 <= sum_bound(m, NETS_MAX_EDGES + 1).max()
    assert 62.8 < np.log2(sum_bound(m, 22).max()) < 62.9 and 63.0 < np.log2(sum_bound(m, 23).max()) < 63.1
    # on each [m, m + 1) the bound is largest at r = m: the floor is constant and 1 / r^2 falls
    r = np.linspace(255.0, 255.999, 50)
    c = np.floor(r) + 3
    mid = c ** 3 * (24 * (3 * area_max / r ** 2 * scale + 0.5) + 20 * (3 * area_max * 121 / r ** 2 * scale + 0.5))
    assert (np.diff(mid) < 0).all()
