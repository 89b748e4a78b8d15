"""CPU checks of the voxel-grid merge arithmetic (scan3d_voxel_*): the shared header
3dscan_b200/common/scan3d_voxel_math.h is compiled for the host, a sequential merge (hash map + first-occurrence list)
is built from its functions and compared bit for bit with voxel_reference below, an independent numpy restatement of
the contract in include/scan3d.h.  tests/test_gpu_voxel.py holds the GPU's merge to the same function."""
import ctypes as C
import os
import subprocess

import numpy as np
import pytest

HERE = os.path.dirname(os.path.abspath(__file__))
F32, F64 = np.float32, np.float64
Q = 2.0 ** 24


def voxel_reference(adds, voxel_size):
    """(xyz f32 [v][3], normals f32 [v][3], rgb u8 [v][3], counts u32 [v], dropped) of the points of `adds`, a list of
    (xyz f32 [n][3], normals f32 [n][3] or None, rgb u8 [n][3] or None), merged in voxels of edge voxel_size.  Voxels
    come in order of their first point over the concatenated adds.  Sums are exact integers (np.add.at on uint64 /
    int64); every float operation is one float64 numpy operation in the contract's order."""
    xyz = np.concatenate([np.asarray(a[0], F32).reshape(-1, 3) for a in adds])
    nrm = np.concatenate([np.zeros((len(a[0]), 3), F32) if a[1] is None else np.asarray(a[1], F32).reshape(-1, 3)
                          for a in adds])
    rgb = np.concatenate([np.zeros((len(a[0]), 3), np.uint8) if a[2] is None else np.asarray(a[2], np.uint8).reshape(-1, 3)
                          for a in adds])
    S = F64(F32(voxel_size))
    with np.errstate(all="ignore"):
        t = xyz.astype(F64) / S
        i = np.floor(t)
        keep = np.isfinite(xyz).all(1) & ((i >= -2.0 ** 20) & (i < 2.0 ** 20)).all(1)
        q = np.minimum(np.floor((t - i) * Q), Q - 1)
    dropped = int((~keep).sum())
    i, q, nk, ck = i[keep].astype(np.int64), q[keep].astype(np.uint64), nrm[keep], rgb[keep]
    with np.errstate(invalid="ignore"):
        m = np.where(np.isfinite(nk).all(1)[:, None], np.rint(np.clip(nk, -1, 1).astype(F64) * Q), 0).astype(np.int64)
    if i.shape[0] == 0:
        z = np.zeros((0, 3))
        return z.astype(F32), z.astype(F32), z.astype(np.uint8), np.zeros(0, np.uint32), dropped
    uniq, first, inv = np.unique(i, axis=0, return_index=True, return_inverse=True)
    order = np.argsort(first)
    rank = np.empty_like(order)
    rank[order] = np.arange(order.size)
    vid = rank[inv.reshape(-1)]
    nv = uniq.shape[0]
    sq, sm, sc = np.zeros((nv, 3), np.uint64), np.zeros((nv, 3), np.int64), np.zeros((nv, 3), np.uint64)
    cnt = np.zeros(nv, np.uint64)
    np.add.at(sq, vid, q)
    np.add.at(sm, vid, m)
    np.add.at(sc, vid, ck.astype(np.uint64))
    np.add.at(cnt, vid, np.uint64(1))
    iv = uniq[order]
    n = cnt.astype(F64)
    coord = ((iv.astype(F64) + sq.astype(F64) / (Q * n)[:, None]) * S).astype(F32)
    X = sm.astype(F64)
    l2 = (X[:, 0] * X[:, 0] + X[:, 1] * X[:, 1]) + X[:, 2] * X[:, 2]
    with np.errstate(invalid="ignore", divide="ignore"):
        normals = np.where((l2 != 0)[:, None], X / np.sqrt(l2)[:, None], 0.0).astype(F32)
    colour = ((sc + (cnt // np.uint64(2))[:, None]) // cnt[:, None]).astype(np.uint8)
    return coord, normals, colour, cnt.astype(np.uint32), dropped


def assert_same_voxels(got, want):
    assert len(got) == len(want) == 5
    assert got[4] == want[4], "dropped"
    assert got[3].shape == want[3].shape and np.array_equal(got[3], want[3]), "counts"
    assert np.array_equal(got[0].view(np.uint32), want[0].view(np.uint32)), "xyz"
    assert np.array_equal(got[1].view(np.uint32), want[1].view(np.uint32)), "normals"
    assert np.array_equal(got[2], want[2]), "rgb"


@pytest.fixture(scope="module")
def shim(tmp_path_factory):
    so = str(tmp_path_factory.mktemp("voxelhost") / "libvoxel_math_host.so")
    subprocess.check_call(["/usr/bin/g++", "-O2", "-std=c++17", "-fPIC", "-shared", "-Wall", "-ffp-contract=off",
                           "-o", so, os.path.join(HERE, "voxel_math_host.cpp")])
    L = C.CDLL(so)
    L.s3v_host_begin.restype = C.c_void_p
    L.s3v_host_begin.argtypes = [C.c_float]
    L.s3v_host_end.argtypes = [C.c_void_p]
    L.s3v_host_add.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_longlong]
    L.s3v_host_count.restype = C.c_longlong
    L.s3v_host_count.argtypes = [C.c_void_p]
    L.s3v_host_finish.restype = C.c_longlong
    L.s3v_host_finish.argtypes = [C.c_void_p] * 5 + [C.POINTER(C.c_longlong)]
    return L


def host_merge(shim, adds, voxel_size):
    p = lambda a: None if a is None else a.ctypes.data_as(C.c_void_p)   # noqa: E731
    h = shim.s3v_host_begin(voxel_size)
    try:
        for xyz, nrm, rgb in adds:
            xyz = np.ascontiguousarray(xyz, F32).reshape(-1, 3)
            nrm = None if nrm is None else np.ascontiguousarray(nrm, F32).reshape(-1, 3)
            rgb = None if rgb is None else np.ascontiguousarray(rgb, np.uint8).reshape(-1, 3)
            shim.s3v_host_add(h, p(xyz), p(nrm), p(rgb), xyz.shape[0])
        v = shim.s3v_host_count(h)
        out = (np.empty((v, 3), F32), np.empty((v, 3), F32), np.empty((v, 3), np.uint8), np.empty(v, np.uint32))
        dropped = C.c_longlong()
        assert shim.s3v_host_finish(h, *[p(a) for a in out], C.byref(dropped)) == v
        return out + (dropped.value,)
    finally:
        shim.s3v_host_end(h)


def random_cloud(rng, n, spread=10.0, centre=(0.0, 0.0, 0.0)):
    xyz = (rng.normal(size=(n, 3)) * spread + np.asarray(centre)).astype(F32)
    nrm = rng.normal(size=(n, 3)).astype(F32)
    nrm /= np.linalg.norm(nrm, axis=1, keepdims=True)
    rgb = rng.integers(0, 256, (n, 3), dtype=np.uint8)
    return xyz, nrm, rgb


def check(shim, adds, voxel_size):
    want = voxel_reference(adds, voxel_size)
    assert_same_voxels(host_merge(shim, adds, voxel_size), want)
    return want


@pytest.mark.parametrize("voxel_size", [0.25, 0.1, 1.7, 3.0])
def test_random_clouds_over_several_adds(shim, voxel_size):
    rng = np.random.default_rng(int(voxel_size * 100))
    adds = []
    for k in range(5):
        xyz, nrm, rgb = random_cloud(rng, 3000 + 700 * k, centre=(k, -2 * k, 5))
        adds.append((xyz, nrm if k != 2 else None, rgb if k != 3 else None))
    adds.append((np.zeros((0, 3), F32), None, None))                  # an empty add changes nothing
    want = check(shim, adds, voxel_size)
    assert want[3].sum() == sum(len(a[0]) for a in adds) and want[4] == 0
    assert (want[3] > 1).any() and (want[3] == 1).any()


def test_negative_coordinates_and_the_clamp(shim):
    """x = -1e-30: t = x / S is a tiny negative number, i = -1 and t - i rounds to 1.0, so floor(f Q) = Q; the clamp
    keeps q = Q - 1 and the voxel's coordinate stays inside it."""
    s = 0.25
    S = F64(F32(s))
    t = F64(F32(-1e-30)) / S
    assert np.floor(t) == -1 and np.floor((t - np.floor(t)) * Q) == Q
    pts = np.array([[-1e-30, 0, 5], [-1e-30, -1e-30, -1e-30], [1e-30, -0.0, 0.0], [-0.0, 0.0, -0.0],
                    [-3.1, -7.9, -0.2], [-0.25, -0.5, -1e-7], [-1e-38, 2.0, -1e-45]], F32)
    want = check(shim, [(pts, None, None)], s)
    # the voxel [-0.25, 0) of -1e-30 averages to just below 0, never to the next voxel's 0.0
    assert want[0][0, 0] < 0 and want[0][0, 0] > -0.25 * 1e-6
    rng = np.random.default_rng(7)
    xyz = (rng.normal(size=(5000, 3)) * 3 - 4).astype(F32)
    check(shim, [(xyz, None, None), (pts, None, None)], 0.3)


@pytest.mark.parametrize("s", [0.25, 0.1, 0.5, 2.0])
def test_exact_multiples_of_the_voxel(shim, s):
    k = np.arange(-40, 41)
    x = (k.astype(F32) * F32(s)).astype(F32)
    pts = np.stack([x, np.roll(x, 7), -x], -1)
    pts = np.concatenate([pts, np.nextafter(pts, F32(np.inf)), np.nextafter(pts, F32(-np.inf))])
    want = check(shim, [(pts, None, None)], s)
    assert want[4] == 0


def test_keys_at_the_range_limits(shim):
    s = 0.5
    lim = 2.0 ** 20
    kept = np.array([[(lim - 1) * s, 0, 0], [-lim * s, 0, 0], [0, (lim - 0.5) * s, 0], [0, 0, -lim * s + 0.1],
                     [(lim - 1) * s, -lim * s, (lim - 1) * s]], F32)
    dropped = np.array([[lim * s, 0, 0], [-lim * s - s / 2, 0, 0], [0, 0, (lim + 1) * s], [0, -1e30, 0],
                        [3e38, 0, 0]], F32)
    want = check(shim, [(kept, None, None), (dropped, None, None)], s)
    assert want[4] == dropped.shape[0] and want[3].size == kept.shape[0]
    # the extreme voxels keep their signed position
    assert want[0][0, 0] == F32(((lim - 1) + 0.0) * s) and want[0][1, 0] == F32(-lim * s)


def test_non_finite_coordinates_are_dropped(shim):
    rng = np.random.default_rng(11)
    xyz, nrm, rgb = random_cloud(rng, 2000)
    xyz[::7, 0] = np.nan
    xyz[3::11, 1] = np.inf
    xyz[5::13, 2] = -np.inf
    want = check(shim, [(xyz, nrm, rgb)], 0.5)
    bad = ~np.isfinite(xyz).all(1)
    assert want[4] == bad.sum() and want[3].sum() == (~bad).sum()


def test_normals_with_nan_large_and_zero_components(shim):
    rng = np.random.default_rng(12)
    xyz = rng.uniform(0, 2, (4000, 3)).astype(F32)
    nrm = rng.normal(size=(4000, 3)).astype(F32)
    nrm[::5] = [1.5, -1.5, 0.25]
    nrm[1::5] = 0
    nrm[2::17, 1] = np.nan
    nrm[3::19, 2] = np.inf
    nrm[4::23] = [-0.0, 1e-9, -1e-9]
    want = check(shim, [(xyz, nrm, None)], 1.0)
    assert np.isfinite(want[1]).all()
    # a voxel whose points all carry zero normals gets (0, 0, 0); a lone (1.5, -1.5, 0.25) normalises the clamped (1, -1, .25)
    z = np.array([[0.5, 0.5, 0.5], [0.6, 0.6, 0.6], [5.5, 5.5, 5.5]], F32)
    zn = np.array([[0, 0, 0], [np.nan, 0, 0], [1.5, -1.5, 0.25]], F32)
    w = check(shim, [(z, zn, None)], 1.0)
    assert not w[1][0].any()
    assert np.allclose(w[1][1], np.array([1, -1, 0.25]) / np.linalg.norm([1, -1, 0.25]), atol=1e-7)


def test_colour_rounds_half_up(shim):
    # n = 2, sum 1 -> 1 (0.5 up); n = 4, sum 2 -> 1; n = 2, sum 509 -> 255 (254.5 up); n = 3, sum 4 -> 1 (1.33)
    groups = [([0, 1], 1), ([0, 0, 1, 1], 1), ([255, 254], 255), ([1, 1, 2], 1), ([3], 3), ([0, 0, 0, 1], 0)]
    xyz, rgb = [], []
    for g, (vals, _) in enumerate(groups):
        for v in vals:
            xyz.append([g * 10 + 0.5, 0.5, 0.5])
            rgb.append([v, 255 - v, v // 2])
    want = check(shim, [(np.array(xyz, F32), None, np.array(rgb, np.uint8))], 1.0)
    assert want[2][:, 0].tolist() == [e for _, e in groups]


def test_single_point_voxels_and_one_voxel_for_everything(shim):
    rng = np.random.default_rng(13)
    xyz, nrm, rgb = random_cloud(rng, 5000, centre=(60, 40, -30))
    tiny = check(shim, [(xyz, nrm, rgb)], 1e-4)
    assert (tiny[3] == 1).all() and tiny[3].size == 5000
    assert np.array_equal(tiny[2], rgb)                       # n = 1: the colour itself
    pos = xyz + F32(200)                                      # every coordinate in [0, 1e6): one voxel
    huge = check(shim, [(pos, nrm, rgb), (pos[::-1], None, rgb[::-1])], 1e6)
    assert huge[3].tolist() == [10000]


def test_add_order_changes_only_the_voxel_order():
    rng = np.random.default_rng(14)
    a, b = random_cloud(rng, 3000), random_cloud(rng, 3000, centre=(5, 5, 5))
    ab, ba = voxel_reference([a, b], 0.7), voxel_reference([b, a], 0.7)

    def as_map(r):
        return {tuple(r[0][k].view(np.uint32)): (tuple(r[1][k].view(np.uint32)), tuple(r[2][k]), r[3][k])
                for k in range(r[3].size)}

    assert as_map(ab) == as_map(ba) and len(as_map(ab)) == ab[3].size
    assert not np.array_equal(ab[0], ba[0])


def test_voxel_entries_reject_null_arguments_without_a_gpu():
    import importlib
    L = importlib.import_module("3dscan_b200").cuda_lib()
    n = C.c_int64()
    assert L.scan3d_voxel_begin(None, 1.0, 10) == -4
    assert L.scan3d_voxel_add_points(None) == -4
    assert L.scan3d_voxel_add_points_dev(None, None, None, None, 0) == -4
    assert L.scan3d_voxel_finish(None) == -4
    assert L.scan3d_voxel_count(None, C.byref(n), None) == -4
    assert L.scan3d_get_voxels(None, None, None, None, None, 0) == -4
    assert L.scan3d_write_voxel_ply(None, b"voxels.ply", 0) == -4
