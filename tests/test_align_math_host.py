"""CPU checks of the scan-to-model alignment arithmetic (scan3d_align_to_voxels*): the shared header
3dscan_b200/common/scan3d_align_math.h is compiled for the host and its functions are compared bit for bit with an
independent restatement below (numpy float64 arrays and Python floats, one IEEE operation each, in the order the
header documents).  A sequential ICP built from the header is compared with a numpy / scipy ICP whose candidates come
from a k-d tree.  tests/test_gpu_align.py holds the GPU to the same restatement."""
import ctypes as C
import importlib
import math
import os
import subprocess

import numpy as np
import pytest
from scipy.spatial import cKDTree
from scipy.spatial.transform import Rotation

HERE = os.path.dirname(os.path.abspath(__file__))
F32, F64 = np.float32, np.float64
CELL_MARGIN = 1.0 + 1.0 / 1048576.0
KEY_LIM = 2.0 ** 20


# ---- the restatement ----------------------------------------------------------------------------------------------
def transform_ref(T, xyz):
    """p' = T p, T the 4x4 (or its first 12 entries), xyz float32 [n][3] -> float64 [n][3]"""
    T = np.asarray(T, F64).reshape(-1)[:12]
    x = np.asarray(xyz, F32).astype(F64)
    with np.errstate(invalid="ignore"):
        return np.stack([((T[4 * i] * x[:, 0] + T[4 * i + 1] * x[:, 1]) + T[4 * i + 2] * x[:, 2]) + T[4 * i + 3]
                         for i in range(3)], 1)


def cells_ref(p, max_distance):
    S = F64(F32(max_distance)) * CELL_MARGIN
    with np.errstate(all="ignore"):
        f = np.floor(p / S)
        ok = np.isfinite(p).all(1) & ((f >= -KEY_LIM) & (f < KEY_LIM)).all(1)
    return np.where(ok[:, None], f, 0).astype(np.int64), ok


def dist2_ref(p, q):
    d = p - np.asarray(q, F32).astype(F64)
    return (d[:, 0] * d[:, 0] + d[:, 1] * d[:, 1]) + d[:, 2] * d[:, 2]


def rows_ref(p, q, n):
    n = np.asarray(n, F32).astype(F64)
    J = np.stack([p[:, 1] * n[:, 2] - p[:, 2] * n[:, 1], p[:, 2] * n[:, 0] - p[:, 0] * n[:, 2],
                  p[:, 0] * n[:, 1] - p[:, 1] * n[:, 0], n[:, 0], n[:, 1], n[:, 2]], 1)
    d = p - np.asarray(q, F32).astype(F64)
    r = (d[:, 0] * n[:, 0] + d[:, 1] * n[:, 1]) + d[:, 2] * n[:, 2]
    return J, r


def products_ref(J, r):
    """[n][28]: J_i J_j (i <= j, row-major), J_i r, r r"""
    cols = [J[:, i] * J[:, j] for i in range(6) for j in range(i, 6)]
    cols += [J[:, i] * r for i in range(6)] + [r * r]
    return np.stack(cols, 1)


def sums_ref(J, r):
    """running sums from +0, one pair after the other (np.cumsum adds sequentially)"""
    if len(r) == 0:
        return np.zeros(28)
    return np.cumsum(np.vstack([np.zeros((1, 28)), products_ref(J, r)]), axis=0)[-1]


def _up(i, j):
    return i * 6 - (i * (i - 1)) // 2 + (j - i)


def solve_ref(s):
    """(ok, x) of (A + mu I) x = -b, LDL^T in the header's order, Python floats"""
    s = [float(v) for v in s]
    tr = s[_up(0, 0)]
    for i in range(1, 6):
        tr = tr + s[_up(i, i)]
    mu = 1e-6 * (tr / 6.0)
    if not (mu > 0.0 and math.isfinite(mu)):
        return False, None
    half = mu * 0.5
    L = [[0.0] * 6 for _ in range(6)]
    D = [0.0] * 6
    for j in range(6):
        d = s[_up(j, j)] + mu
        for k in range(j):
            d = d - (L[j][k] * L[j][k]) * D[k]
        if not d > half:
            return False, None
        D[j] = d
        for i in range(j + 1, 6):
            v = s[_up(j, i)]
            for k in range(j):
                v = v - (L[i][k] * L[j][k]) * D[k]
            L[i][j] = v / d
    y = [0.0] * 6
    for i in range(6):
        v = -s[21 + i]
        for k in range(i):
            v = v - L[i][k] * y[k]
        y[i] = v
    x = [0.0] * 6
    for i in range(5, -1, -1):
        v = y[i] / D[i]
        for k in range(i + 1, 6):
            v = v - L[k][i] * x[k]
        x[i] = v
    if not all(math.isfinite(v) for v in x):
        return False, None
    return True, np.array(x)


def sincos_ref(h):
    t, m = float(h), 0
    while t > 0.125:
        t = t * 0.5
        m += 1
    t2 = t * t
    a = 1.0 - t2 / 110.0
    for c in (72.0, 42.0, 20.0, 6.0):
        a = 1.0 - (t2 / c) * a
    s = t * a
    b = 1.0 - t2 / 90.0
    for c in (56.0, 30.0, 12.0):
        b = 1.0 - (t2 / c) * b
    c = 1.0 - (t2 / 2.0) * b
    for _ in range(m):
        s2 = 2.0 * s
        s, c = s2 * c, 1.0 - s2 * s
    return s, c


def rodrigues_ref(w):
    """(ok, dR [3][3], |w|)"""
    w = [float(v) for v in w]
    th2 = (w[0] * w[0] + w[1] * w[1]) + w[2] * w[2]
    if not math.isfinite(th2):
        return False, None, None
    if th2 == 0.0:
        return True, np.eye(3), 0.0
    t = math.sqrt(th2)
    k = [w[0] / t, w[1] / t, w[2] / t]
    sh, ch = sincos_ref(t * 0.5)
    sh2 = 2.0 * sh
    s, c1 = sh2 * ch, sh2 * sh
    c = 1.0 - c1
    K = [[0.0, -k[2], k[1]], [k[2], 0.0, -k[0]], [-k[1], k[0], 0.0]]
    R = np.array([[((c if i == j else 0.0) + (c1 * k[i]) * k[j]) + s * K[i][j] for j in range(3)] for i in range(3)])
    return True, R, t


def compose_ref(dR, v, T):
    T = np.asarray(T, F64).reshape(-1)[:12]
    o = np.empty(12)
    for i in range(3):
        for j in range(4):
            e = (float(dR[i][0]) * T[j] + float(dR[i][1]) * T[4 + j]) + float(dR[i][2]) * T[8 + j]
            o[4 * i + j] = e + float(v[i]) if j == 3 else e
    return o


def rms_ref(sum_r2, pairs):
    return math.sqrt(sum_r2 / float(pairs)) if pairs > 0 else 0.0


def pairs_ref(p, mxyz, mnrm, max_distance, tree=None, k=8):
    """(source index, model ordinal) of every kept pair: the k nearest model points with a non-zero normal from a k-d
    tree (exact distances, radius slightly above max_distance) are the candidates, and the header's rule (double
    distance <= max_distance^2, smallest, then smallest ordinal) picks the winner among them"""
    mxyz, mnrm = np.asarray(mxyz, F32), np.asarray(mnrm, F32)
    live = np.flatnonzero((mnrm != 0).any(1) & np.isfinite(mxyz).all(1))
    tree = tree or cKDTree(mxyz[live].astype(F64))
    md = F64(F32(max_distance))
    r2 = md * md
    _, ok = cells_ref(p, max_distance)
    src = np.flatnonzero(ok)
    if src.size == 0 or live.size == 0:
        return np.zeros(0, np.int64), np.zeros(0, np.int64), tree
    _, idx = tree.query(p[src], k=k, distance_upper_bound=md * (1 + 1e-9))
    valid = idx < live.size
    ords = live[np.where(valid, idx, 0)]
    q = mxyz[ords].astype(F64)
    d = p[src][:, None, :] - q
    d = (d[..., 0] * d[..., 0] + d[..., 1] * d[..., 1]) + d[..., 2] * d[..., 2]
    valid &= d <= r2
    d = np.where(valid, d, np.inf)
    dmin = d.min(1)
    best = np.where(valid & (d == dmin[:, None]), ords, np.iinfo(np.int64).max).min(1)
    keep = np.isfinite(dmin)
    return src[keep], best[keep], tree


def icp_ref(mxyz, mnrm, src, T_init, max_distance, max_iterations, stride=1, stop_rotation=0.0, stop_translation=0.0):
    """a numpy / scipy point-to-plane ICP with the contract's rules (pairs by pairs_ref, damped normal equations solved
    by numpy, Rodrigues by scipy).  Returns (T 4x4, iterations, status, pairs_first, pairs_last, rms_first, rms_last)."""
    T = np.asarray(T_init, F64).reshape(4, 4).copy()
    x = np.asarray(src, F32)[::stride]
    mxyz, mnrm = np.asarray(mxyz, F32), np.asarray(mnrm, F32)
    tree, first, it, status = None, None, 0, 1
    last = (0, 0.0)
    for _ in range(max_iterations):
        p = transform_ref(T, x)
        si, oi, tree = pairs_ref(p, mxyz, mnrm, max_distance, tree)
        J, r = rows_ref(p[si], mxyz[oi], mnrm[oi])
        npairs = si.size
        rms = float(np.sqrt((r * r).sum() / npairs)) if npairs else 0.0
        first = first or (npairs, rms)
        last = (npairs, rms)
        if npairs < 6:
            status = 2
            break
        A, b = J.T @ J, J.T @ r
        mu = 1e-6 * np.trace(A) / 6
        w = np.linalg.solve(A + mu * np.eye(6), -b)
        dR = Rotation.from_rotvec(w[:3]).as_matrix()
        D = np.eye(4)
        D[:3, :3], D[:3, 3] = dR, w[3:]
        T = D @ T
        it += 1
        if (stop_rotation > 0 or stop_translation > 0) and np.linalg.norm(w[:3]) <= stop_rotation and \
                np.linalg.norm(w[3:]) <= stop_translation:
            status = 0
            break
    return T, it, status, first[0], last[0], first[1], last[1]


# ---- the host build -----------------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def shim(tmp_path_factory):
    so = str(tmp_path_factory.mktemp("alignhost") / "libalign_math_host.so")
    subprocess.check_call(["/usr/bin/g++", "-O2", "-std=c++17", "-fPIC", "-shared", "-Wall", "-ffp-contract=off",
                           "-o", so, os.path.join(HERE, "align_math_host.cpp")])
    L = C.CDLL(so)
    vp, i64, d = C.c_void_p, C.c_longlong, C.c_double
    L.s3l_host_transform.argtypes = [vp, vp, i64, vp]
    L.s3l_host_cells.argtypes = [vp, i64, C.c_float, vp, vp]
    L.s3l_host_dist2.argtypes = [vp, vp, i64, vp]
    L.s3l_host_closer.argtypes = [d, C.c_uint32, d, C.c_uint32]
    L.s3l_host_rows.argtypes = [vp, vp, vp, i64, vp, vp]
    L.s3l_host_sums.argtypes = [vp, vp, i64, vp]
    L.s3l_host_solve.argtypes = [vp, vp]
    L.s3l_host_rodrigues.argtypes = [vp, vp, vp]
    L.s3l_host_sincos.argtypes = [d, vp, vp]
    L.s3l_host_compose.argtypes = [vp, vp, vp]
    L.s3l_host_icp.argtypes = [vp, vp, i64, vp, i64, vp, C.c_float, C.c_int, C.c_int, d, d, vp, vp]
    L.s3l_host_layout.argtypes = [vp]
    return L


def _p(a):
    return a.ctypes.data_as(C.c_void_p)


def host_icp(shim, mxyz, mnrm, src, T_init, max_distance, max_iterations, stride=1, stop_rotation=0.0,
             stop_translation=0.0):
    mxyz, mnrm, src = (np.ascontiguousarray(a, F32).reshape(-1, 3) for a in (mxyz, mnrm, src))
    T = np.ascontiguousarray(np.asarray(T_init, F64).reshape(-1)[:12])
    info, rms = np.zeros(4, np.int64), np.zeros(2)
    shim.s3l_host_icp(_p(mxyz), _p(mnrm), len(mxyz), _p(src), len(src), _p(T), max_distance, max_iterations, stride,
                      stop_rotation, stop_translation, _p(info), _p(rms))
    return np.vstack([T.reshape(3, 4), [0, 0, 0, 1]]), int(info[0]), int(info[1]), int(info[2]), int(info[3]), \
        float(rms[0]), float(rms[1])


def same_bits(a, b):
    a, b = np.asarray(a, F64), np.asarray(b, F64)
    return a.shape == b.shape and np.array_equal(a.view(np.uint64), b.view(np.uint64))


def rigid(rng, deg, shift):
    T = np.eye(4)
    T[:3, :3] = Rotation.from_rotvec(np.deg2rad(deg) * rng.normal(size=3) / math.sqrt(3)).as_matrix()
    T[:3, 3] = rng.normal(size=3) * shift
    return T


def height_field(x, y):
    """a non-symmetric surface (every rigid DOF constrained) and its unit normals"""
    z = 0.3 * np.sin(1.3 * x) + 0.2 * np.cos(0.9 * y + 0.4) + 0.05 * x * x + 0.03 * x * y
    fx = 0.39 * np.cos(1.3 * x) + 0.1 * x + 0.03 * y
    fy = -0.18 * np.sin(0.9 * y + 0.4) + 0.03 * x
    n = np.stack([-fx, -fy, np.ones_like(x)], -1)
    return np.stack([x, y, z], -1), n / np.linalg.norm(n, axis=-1, keepdims=True)


# ---- per-element functions ----------------------------------------------------------------------------------------
def test_transform_and_cells(shim):
    rng = np.random.default_rng(1)
    xyz = (rng.normal(size=(5000, 3)) * 40 + [60, 40, -30]).astype(F32)
    xyz[::97, 0] = np.nan
    xyz[5::101, 1] = np.inf
    xyz[7::103, 2] = 3e37                                   # finite, outside the key range
    for k in range(4):
        T = rigid(rng, 30 * k, 5.0 * k)
        out = np.empty((len(xyz), 3))
        shim.s3l_host_transform(_p(T.reshape(-1).copy()), _p(xyz), len(xyz), _p(out))
        want = transform_ref(T, xyz)
        assert same_bits(np.nan_to_num(out, nan=7.0), np.nan_to_num(want, nan=7.0))
        assert np.array_equal(np.isnan(out), np.isnan(want))
        for md in (0.05, 0.5, 3.0, 1e-5):
            cells, ok = np.empty((len(xyz), 3), np.int64), np.empty(len(xyz), np.uint8)
            shim.s3l_host_cells(_p(out), len(xyz), md, _p(cells), _p(ok))
            wc, wok = cells_ref(want, md)
            assert np.array_equal(ok.astype(bool), wok)
            assert np.array_equal(cells[wok], wc[wok])
            assert (~wok).sum() >= (~np.isfinite(xyz).all(1)).sum()
    # cells at the key range limits
    S = F64(F32(0.5)) * CELL_MARGIN
    p = np.array([[(KEY_LIM - 1) * S, 0, 0], [-KEY_LIM * S, 0, 0], [KEY_LIM * S, 0, 0], [0, -KEY_LIM * S - S, 0]])
    cells, ok = np.empty((4, 3), np.int64), np.empty(4, np.uint8)
    shim.s3l_host_cells(_p(p), 4, 0.5, _p(cells), _p(ok))
    assert ok.tolist() == [1, 1, 0, 0] and cells[0, 0] == KEY_LIM - 1 and cells[1, 0] == -KEY_LIM


def test_the_cell_margin_keeps_every_neighbour_within_one_cell():
    """|q - p| <= max_distance along an axis never puts q two cells away, even with both quotients rounded"""
    rng = np.random.default_rng(2)
    for md in (0.05, 0.3, 1.0, 7.0):
        S = F64(F32(md)) * CELL_MARGIN
        p = rng.uniform(-2e5 * md, 2e5 * md, 200000)
        q = p + rng.choice([-1, 1], p.size) * F64(F32(md)) * rng.uniform(0.999999, 1.0, p.size)
        assert np.abs(np.floor(q / S) - np.floor(p / S)).max() <= 1


def test_distances_ties_and_the_radius(shim):
    rng = np.random.default_rng(3)
    p = rng.normal(size=(4000, 3)) * 10
    q = (p + rng.normal(size=p.shape)).astype(F32)
    out = np.empty(len(p))
    shim.s3l_host_dist2(_p(p), _p(q), len(p), _p(out))
    assert same_bits(out, dist2_ref(p, q))
    # the rule: smaller distance, then smaller ordinal; equal candidates never replace the best
    assert shim.s3l_host_closer(1.0, 9, 2.0, 1) and not shim.s3l_host_closer(2.0, 1, 1.0, 9)
    assert shim.s3l_host_closer(1.0, 3, 1.0, 4) and not shim.s3l_host_closer(1.0, 4, 1.0, 3)
    assert not shim.s3l_host_closer(1.0, 4, 1.0, 4)
    # an exact tie between two model points resolves to the smaller ordinal: the residual tells which was taken
    md = 1.0
    src = np.zeros((1, 3), F32)
    a, na = [0.0, 0.5, 0.0], [0.0, 1.0, 0.0]              # r = -0.5
    b, nb = [0.5, 0.0, 0.0], [0.6, 0.8, 0.0]              # r = -0.3
    for model, nrm, want in (([a, b], [na, nb], 0.5), ([b, a], [nb, na], F64(F32(0.6)) * 0.5)):
        res = host_icp(shim, model, nrm, src, np.eye(4), md, 1)
        assert res[3] == 1 and res[2] == 2 and res[5] == want
    # exactly at the radius a point pairs; one float step further out it does not
    md = F32(0.75)
    ring = np.array([[md, 0, 0], [0, -md, 0], [0, 0, md], [-md, 0, 0]], F32)
    out_ = np.array([[np.nextafter(md, F32(2)), 0, 0], [0, 0, -np.nextafter(md, F32(2))]], F32)
    model = np.vstack([ring, out_])
    nrm = np.tile(np.array([[0, 0, 1]], F32), (len(model), 1))
    res = host_icp(shim, model, nrm, np.zeros((1, 3), F32), np.eye(4), float(md), 1)
    assert res[3] == 1 and res[5] == 0.0                   # paired with ring[0] (ordinal 0), r = 0
    dist = dist2_ref(np.zeros((len(model), 3)), model)
    assert (dist[:4] == F64(md) * F64(md)).all() and (dist[4:] > F64(md) * F64(md)).all()
    res = host_icp(shim, out_, nrm[:2], np.zeros((1, 3), F32), np.eye(4), float(md), 1)
    assert res[3] == 0 and res[2] == 2


def test_rows_and_sums(shim):
    rng = np.random.default_rng(4)
    p = rng.normal(size=(3000, 3)) * 30
    q = (p + rng.normal(size=p.shape) * 0.1).astype(F32)
    n = rng.normal(size=p.shape).astype(F32)
    J, r = np.empty((len(p), 6)), np.empty(len(p))
    shim.s3l_host_rows(_p(p), _p(q), _p(n), len(p), _p(J), _p(r))
    wJ, wr = rows_ref(p, q, n)
    assert same_bits(J, wJ) and same_bits(r, wr)
    s = np.empty(28)
    shim.s3l_host_sums(_p(J), _p(r), len(p), _p(s))
    assert same_bits(s, sums_ref(wJ, wr))
    shim.s3l_host_sums(_p(J), _p(r), 0, _p(s))
    assert same_bits(s, np.zeros(28))


def _solve(shim, s):
    s = np.ascontiguousarray(s, F64)
    x = np.zeros(6)
    ok = shim.s3l_host_solve(_p(s), _p(x))
    return bool(ok), x


def _sums_of(A, b, r2=1.0):
    return np.array([A[i, j] for i in range(6) for j in range(i, 6)] + list(b) + [r2])


def test_damped_solve(shim):
    rng = np.random.default_rng(5)
    for k in range(200):
        M = rng.normal(size=(8, 6)) * rng.uniform(0.1, 100, 6)
        A = M.T @ M
        b = rng.normal(size=6) * 10
        ok, x = _solve(shim, _sums_of(A, b))
        wok, wx = solve_ref(_sums_of(A, b))
        assert ok and wok and same_bits(x, wx)
        mu = 1e-6 * np.trace(A) / 6
        assert np.allclose(x, np.linalg.solve(A + mu * np.eye(6), -b), rtol=1e-7, atol=1e-9 * np.abs(x).max())
    # a plane alone: A has rank 3 (rotation about the normal and the two in-plane translations are free)
    p = np.column_stack([rng.uniform(-20, 20, 500), rng.uniform(-20, 20, 500), np.full(500, 5.0)])
    nrm = np.tile([0.0, 0.0, 1.0], (500, 1)).astype(F32)
    J, r = rows_ref(p, (p - [0, 0, 0.01]).astype(F32), nrm)
    s = sums_ref(J, r)
    ok, x = _solve(shim, s)
    wok, wx = solve_ref(s)
    assert ok and wok and same_bits(x, wx) and np.isfinite(x).all()
    assert abs(x[5] + 0.01) < 1e-6 and np.abs(x[[0, 1, 2, 3, 4]]).max() < 1e-6
    # singular / invalid systems fail their pivot test
    for bad in (np.zeros(28), np.full(28, np.nan), _sums_of(-np.eye(6), np.ones(6)),
                _sums_of(np.diag([1.0, 1, 1, 1, 1, -1e3]), np.ones(6)), _sums_of(np.where(np.eye(6) > 0, np.inf, 0.0), np.ones(6))):
        ok, _ = _solve(shim, bad)
        wok, _ = solve_ref(bad)
        assert not ok and not wok


def test_rodrigues_update(shim):
    rng = np.random.default_rng(6)
    ws = [np.zeros(3), np.array([1e-20, 0, 0]), np.array([0, -3e-9, 1e-9]), np.array([1e-160, 1e-160, 0]),
          np.array([0, 0, 0.125]), np.array([0, 0, 0.25]), np.array([3.0, 0, 0]), np.array([0, 10.0, 0]),
          np.array([50.0, -20, 7])]
    ws += [rng.normal(size=3) * sc for sc in (1e-6, 1e-3, 0.05, 0.5, 2.0) for _ in range(20)]
    for w in ws:
        w = np.ascontiguousarray(w, F64)
        R, th = np.empty(9), C.c_double()
        ok = shim.s3l_host_rodrigues(_p(w), _p(R), C.byref(th))
        wok, wR, wth = rodrigues_ref(w)
        assert ok and wok and same_bits(R, wR.reshape(-1)) and th.value == wth
        assert np.abs(R.reshape(3, 3) - Rotation.from_rotvec(w).as_matrix()).max() < 1e-13 * max(1.0, np.linalg.norm(w))
    R, th = np.empty(9), C.c_double()
    shim.s3l_host_rodrigues(_p(np.zeros(3)), _p(R), C.byref(th))
    assert same_bits(R, np.eye(3).reshape(-1)) and th.value == 0.0
    assert not shim.s3l_host_rodrigues(_p(np.array([1e200, 0, 0])), _p(R), C.byref(th))
    assert not shim.s3l_host_rodrigues(_p(np.array([np.nan, 0, 0])), _p(R), C.byref(th))
    for h in (0.0, 1e-300, 0.1, 0.125, 0.126, 1.0, 3.0, 100.0):
        sn, cs = C.c_double(), C.c_double()
        shim.s3l_host_sincos(h, C.byref(sn), C.byref(cs))
        assert (sn.value, cs.value) == sincos_ref(h)
        assert abs(sn.value - math.sin(h)) < 1e-14 * max(1, h) and abs(cs.value - math.cos(h)) < 1e-14 * max(1, h)


def test_compose(shim):
    rng = np.random.default_rng(7)
    for _ in range(50):
        T = rigid(rng, 40, 20).reshape(-1)[:12].copy()
        _, dR, _ = rodrigues_ref(rng.normal(size=3) * 0.1)
        v = rng.normal(size=3)
        want = compose_ref(dR, v, T)
        shim.s3l_host_compose(_p(np.ascontiguousarray(dR.reshape(-1))), _p(v), _p(T))
        assert same_bits(T, want)


def test_public_struct_layout_matches_the_binding(shim):
    s3 = importlib.import_module("3dscan_b200")
    out = np.zeros(14, np.int64)
    shim.s3l_host_layout(_p(out))
    P, R = s3.AlignParams, s3.AlignResultC
    assert out.tolist() == [C.sizeof(P), P.max_distance.offset, P.max_iterations.offset, P.stride.offset,
                            P.stop_rotation.offset, P.stop_translation.offset, P.apply.offset, C.sizeof(R),
                            R.iterations.offset, R.status.offset, R.pairs_first.offset, R.pairs_last.offset,
                            R.rms_first.offset, R.rms_last.offset]


# ---- the whole run --------------------------------------------------------------------------------------------------
def _surface_pair(rng, T_true, model_step=0.1, src_step=0.13):
    gx, gy = np.meshgrid(np.arange(-3, 3, model_step), np.arange(-3, 3, model_step))
    mxyz, mnrm = height_field(gx.reshape(-1), gy.reshape(-1))
    sx = rng.uniform(-2.5, 2.5, int((5 / src_step) ** 2))
    sy = rng.uniform(-2.5, 2.5, sx.size)
    sp, _ = height_field(sx, sy)
    Ti = np.linalg.inv(T_true)
    src = (sp @ Ti[:3, :3].T + Ti[:3, 3]).astype(F32)       # T_true maps the source onto the surface
    return mxyz.astype(F32), mnrm.astype(F32), src


@pytest.mark.parametrize("stride", [1, 3])
def test_sequential_icp_matches_numpy_scipy(shim, stride):
    rng = np.random.default_rng(8 + stride)
    T_true = rigid(rng, 2.0, 0.05)
    mxyz, mnrm, src = _surface_pair(rng, T_true)
    mnrm[::11] = 0                                          # voxels without a normal are never correspondences
    md = 0.4
    got = host_icp(shim, mxyz, mnrm, src, np.eye(4), md, 12, stride)
    want = icp_ref(mxyz, mnrm, src, np.eye(4), md, 12, stride)
    assert got[1:5] == want[1:5]                            # iterations, status, pairs first / last
    # the summation orders and the solvers differ: T agrees to float64 rounding of ~1e3 pair sums
    assert np.abs(got[0] - want[0]).max() < 1e-10
    assert abs(got[5] - want[5]) <= 1e-12 * want[5] and abs(got[6] - want[6]) <= 1e-9 * want[5]
    assert got[6] < 0.1 * got[5]
    # recovered: the residual transform is tiny (the surface samples are exact, the model is 0.1-spaced)
    E = got[0] @ np.linalg.inv(T_true)
    assert np.linalg.norm(Rotation.from_matrix(E[:3, :3]).as_rotvec()) < 2e-3 and np.linalg.norm(E[:3, 3]) < 5e-3


def test_convergence_and_failure_statuses(shim):
    rng = np.random.default_rng(10)
    T_true = rigid(rng, 1.0, 0.02)
    mxyz, mnrm, src = _surface_pair(rng, T_true)
    T, it, status, pf, pl, rf, rl = host_icp(shim, mxyz, mnrm, src, np.eye(4), 0.4, 64, 1, 1e-7, 1e-6)
    assert status == 0 and 1 <= it < 64 and pl == pf
    wT, wit, wst, *_ = icp_ref(mxyz, mnrm, src, np.eye(4), 0.4, 64, 1, 1e-7, 1e-6)
    assert (it, status) == (wit, wst) and np.abs(T - wT).max() < 1e-10
    # no normals at all: no pairs, T stays T_init
    T0 = rigid(rng, 3.0, 0.1)
    T, it, status, pf, pl, rf, rl = host_icp(shim, mxyz, np.zeros_like(mnrm), src, T0, 0.4, 5)
    assert (it, status, pf, pl, rf, rl) == (0, 2, 0, 0, 0.0, 0.0) and same_bits(T, T0)


def test_align_entries_reject_null_arguments_without_a_gpu():
    s3 = importlib.import_module("3dscan_b200")
    L = s3.cuda_lib()
    p, r = s3.AlignParams(), s3.AlignResultC()
    assert L.scan3d_align_to_voxels(None, C.byref(p), C.byref(r)) == -4
    assert L.scan3d_align_to_voxels_dev(None, None, 0, C.byref(p), C.byref(r)) == -4
