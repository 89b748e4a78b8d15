"""CPU checks of the non-manifold repair's arithmetic (scan3d_voxel_surface_repair, scan3d_mesh_repair_dev): the
shared header 3dscan_b200/common/scan3d_repair_math.h is compiled for the host and compared bit for bit with the numpy
restatement of tests/test_repair_ref.py: the face key on random, degenerate, tiny and huge triangles, and the per-edge
keep rule on random books of faces, including equal areas and books with no opposite winding."""
import ctypes as C
import os
import subprocess

import numpy as np
import pytest

from test_repair_ref import face_key_ref, kept_on_edge_ref

HERE = os.path.dirname(os.path.abspath(__file__))
F32, U64 = np.float32, np.uint64


@pytest.fixture(scope="module")
def L(tmp_path_factory):
    so = os.path.join(str(tmp_path_factory.mktemp("repairhost")), "librepair_math_host.so")
    subprocess.check_call(["/usr/bin/g++", "-O2", "-std=c++17", "-fPIC", "-shared", "-Wall", "-ffp-contract=off",
                           "-o", so, os.path.join(HERE, "repair_math_host.cpp")])
    lib = C.CDLL(so)
    vp, ll = C.c_void_p, C.c_longlong
    lib.s3r_host_face_key.argtypes = [vp, vp, ll, vp]
    lib.s3r_host_kept.argtypes = [vp, vp, vp, vp, ll, vp]
    return lib


def _p(a):
    return a.ctypes.data_as(C.c_void_p)


def test_face_key_bit_for_bit(L):
    rng = np.random.default_rng(1)
    n = 20000
    t = rng.normal(size=(n, 3, 3)).astype(F32)
    t[:n // 8] *= np.exp2(rng.integers(-80, 80, (n // 8, 1, 1))).astype(F32)   # tiny and huge: areas to 0 and inf
    t[n // 8:n // 4, 2] = t[n // 8:n // 4, 0]                                     # degenerate: area 0
    t[n // 4:n // 4 + 100, :, 2] = 0.0                                            # flat, signed zeros
    t[n // 4 + 100:n // 4 + 200] *= -0.0
    xyz = t.reshape(-1, 3)
    faces = np.arange(3 * n).reshape(n, 3)
    want = face_key_ref(xyz, faces)
    got = np.zeros(n, U64)
    L.s3r_host_face_key(_p(np.ascontiguousarray(t)), _p(np.arange(n, dtype=np.uint32)), n, _p(got))
    assert np.array_equal(got, want)
    hi = want >> U64(32)
    assert (hi == 0).any() and (hi == 0x7F800000).any()


def test_edge_rule_bit_for_bit(L):
    rng = np.random.default_rng(2)
    rows = []
    for _ in range(3000):
        m = int(rng.integers(3, 7))
        k = (rng.integers(0, 4, m).astype(U64) << U64(32)) | (U64(0xFFFFFFFF) - rng.permutation(50)[:m].astype(U64))
        d = rng.integers(0, 2, m) if rng.random() < 0.7 else np.zeros(m, np.int64)
        m0 = k[d == 0].max(initial=U64(0))
        m1 = k[d == 1].max(initial=U64(0))
        f1 = max(m0, m1)
        second = k[k != f1].max()
        for x in k:
            rows.append((x, m0, m1, second))
    k, m0, m1, second = (np.ascontiguousarray(c, U64) for c in zip(*rows))
    got = np.zeros(len(k), np.uint8)
    L.s3r_host_kept(_p(k), _p(m0), _p(m1), _p(second), len(k), _p(got))
    want = kept_on_edge_ref(k, m0, m1, second)
    assert np.array_equal(got.astype(bool), want)
    assert want.mean() < 1.0
