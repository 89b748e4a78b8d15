"""CPU checks of the sample-to-surface distance arithmetic (scan3d_voxel_surface_distance and its dev routes): the shared
header 3dscan_b200/common/scan3d_distance_math.h is compiled for the host and compared bit for bit with the numpy
restatement of tests/test_distance_ref.py: the closest point, d2 and the side on random triangles, on points in every
Voronoi region, on needle, sliver, collinear and zero-area faces (no NaN), on vertices, edges and face interiors; and
the cell box and entry count of faces at cell boundaries, with the clamp and the key range."""
import ctypes as C
import os
import subprocess

import numpy as np
import pytest

from test_distance_ref import cell_edge, cells_ref, closest_ref, face_boxes

HERE = os.path.dirname(os.path.abspath(__file__))
F32 = np.float32


@pytest.fixture(scope="module")
def L(tmp_path_factory):
    so = os.path.join(str(tmp_path_factory.mktemp("distancehost")), "libdistance_math_host.so")
    subprocess.check_call(["/usr/bin/g++", "-O2", "-std=c++17", "-fPIC", "-shared", "-Wall", "-ffp-contract=off",
                           "-o", so, os.path.join(HERE, "distance_math_host.cpp")])
    lib = C.CDLL(so)
    vp, ll = C.c_void_p, C.c_longlong
    lib.s3p_host_pairs.argtypes = [vp, vp, ll, vp, vp, vp]
    lib.s3p_host_cells.argtypes = [vp, ll, C.c_float, vp, vp, vp, vp]
    return lib


def _p(a):
    return a.ctypes.data_as(C.c_void_p)


def _pairs(L, p, t):
    p, t = np.ascontiguousarray(p, F32), np.ascontiguousarray(t, F32)
    n = len(p)
    d2, s, sd = np.zeros(n), np.zeros(n), np.zeros(n, F32)
    L.s3p_host_pairs(_p(p), _p(t), n, _p(d2), _p(s), _p(sd))
    return d2, s, sd


def _check(L, p, t):
    d2, s, sd = _pairs(L, p, t)
    T = t.astype(np.float64)
    wd2, ws = closest_ref(p.astype(np.float64), T[:, 0], T[:, 1], T[:, 2])
    assert np.array_equal(d2.view(np.uint64), wd2.view(np.uint64))
    assert np.array_equal(s.view(np.uint64), ws.view(np.uint64))
    r = np.sqrt(wd2)
    assert np.array_equal(sd.view(np.uint32), np.where(ws < 0, -r, r).astype(F32).view(np.uint32))
    assert np.isfinite(d2).all() and np.isfinite(s).all()
    return d2, s


def _faces(rng, n, scale):
    t = (rng.normal(size=(n, 3, 3)) * scale + rng.normal(size=(n, 1, 3)) * 10 * scale).astype(F32)
    k = n // 8
    t[:k, 1] = t[:k, 0] + (rng.normal(size=(k, 3)) * 1e-6 * scale).astype(F32)          # needles
    t[k:2 * k, 2] = ((t[k:2 * k, 0].astype(np.float64) + t[k:2 * k, 1]) / 2 +
                     rng.normal(size=(k, 3)) * 1e-5 * scale).astype(F32)                  # slivers
    w = rng.random((k, 1))
    t[2 * k:3 * k, 2] = (t[2 * k:3 * k, 0] * w + t[2 * k:3 * k, 1] * (1 - w)).astype(F32)  # collinear
    t[3 * k:4 * k, 1] = t[3 * k:4 * k, 0]                                                   # zero area
    t[4 * k:5 * k] = t[4 * k:5 * k, :1]                                                     # a point
    return t


@pytest.mark.parametrize("scale", [1.0, 1e-3, 1e4])
def test_pairs_bit_for_bit(L, scale):
    rng = np.random.default_rng(int(np.log10(scale)) + 5)
    n = 40000
    t = _faces(rng, n, scale)
    T = t.astype(np.float64)
    p = np.empty((n, 3), F32)
    m = n // 4
    p[:m] = (T[:m].mean(1) + rng.normal(size=(m, 3)) * 3 * scale).astype(F32)             # every region
    b = rng.dirichlet([1, 1, 1], n - m)
    p[m:] = (np.einsum("ij,ijk->ik", b, T[m:]) + rng.normal(size=(n - m, 1)) * 0.1 * scale *
             rng.normal(size=(n - m, 3))).astype(F32)
    p[m:m + 500] = t[m:m + 500, 0]                                                          # on vertices
    p[m + 500:m + 1000] = ((T[m + 500:m + 1000, 1] + T[m + 500:m + 1000, 2]) / 2).astype(F32)  # on edges
    p[m + 1000:m + 1500] = T[m + 1000:m + 1500].mean(1).astype(F32)                         # inside
    d2, _ = _check(L, p, t)
    assert (d2[m:m + 500] == 0).all()


def test_every_region_and_the_rounding_case(L):
    a, b, c = [0, 0, 0], [4, 0, 0], [0, 4, 0]
    pts = [[-1, -1, 1], [5, -1, 1], [-1, 5, -1], [2, -1, 1], [-1, 2, -1], [3, 3, 2], [1, 1, 1], [1, 1, -1]]
    p = np.array(pts, F32)
    t = np.array([[a, b, c]] * len(pts), F32)
    d2, s = _check(L, p, t)
    assert list(d2) == [3.0, 3.0, 3.0, 2.0, 2.0, 6.0, 1.0, 1.0]
    assert list(np.sign(s)) == [1, 1, -1, 1, -1, 1, 1, -1]
    # d1 = d3 = 0 on a face of non-zero area: the fallback, no NaN
    _check(L, np.array([[1e20, -1e20, 1]], F32), np.array([[[0, 0, 0], [1, 1, 0], [0, 0, 1]]], F32))


def test_cells_bit_for_bit(L):
    rng = np.random.default_rng(2)
    n = 5000
    for R in (0.5, 1.0, 3.0e-3):
        S = cell_edge(R)
        t = (rng.integers(-40, 40, (n, 3, 3)) * S).astype(F32)                             # on cell boundaries
        t[: n // 2] = (t[: n // 2] + rng.normal(size=(n // 2, 3, 3)) * S).astype(F32)
        t[:50] = np.nextafter(t[:50], F32(np.inf))
        t[50:100, 0, 0] = F32(2.0 ** 21 * S)                                               # out of the key range
        lo, hi, ok, ent = np.zeros((n, 3), np.int64), np.zeros((n, 3), np.int64), np.zeros(n, np.int32), \
            np.zeros(n, np.uint64)
        L.s3p_host_cells(_p(np.ascontiguousarray(t)), n, R, _p(lo), _p(hi), _p(ok), _p(ent))
        xyz = t.reshape(-1, 3)
        faces = np.arange(3 * n, dtype=np.int32).reshape(n, 3)
        wlo, whi, wok, went = face_boxes(xyz, faces, S)
        assert np.array_equal(ok.astype(bool), wok) and not wok[50:100].any() and wok[100:].all()
        assert np.array_equal(lo[wok], wlo[wok]) and np.array_equal(hi[wok], whi[wok])
        assert np.array_equal(ent, went)
        c, cok = cells_ref(xyz[:, 0], S)
        assert cok[300:].all() and (np.floor(xyz[300:, 0].astype(np.float64) / S) == c[300:]).all()
