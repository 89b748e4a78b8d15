"""CPU checks of the surface extraction arithmetic (scan3d_voxel_surface): the shared header
3dscan_b200/common/scan3d_surface_math.h is compiled for the host and its functions are compared bit for bit with an
independent restatement below (numpy float64 arrays, one IEEE operation each, in the order the header documents).  A
sequential extraction built from the header (plain loops and a map) is compared with a vectorised numpy / scipy
extraction whose nearest-neighbour candidates come from a k-d tree.  tests/test_gpu_surface.py holds the GPU to the
same restatement."""
import ctypes as C
import importlib
import os
import subprocess

import numpy as np
import pytest
from scipy.spatial import cKDTree

HERE = os.path.dirname(os.path.abspath(__file__))
F32, F64 = np.float32, np.float64
KEY_LIM = 2 ** 20


# ---- the restatement ----------------------------------------------------------------------------------------------
def voxel_ijk(xyz, voxel_size):
    """merge index of each point: floor((double)x / S) per axis"""
    return np.floor(np.asarray(xyz, F32).astype(F64) / F64(F32(voxel_size))).astype(np.int64)


def model_ijk(xyz, voxel_size):
    """merge indices of the voxels of a cloud added in order (finite points): the distinct point voxels in order of
    their first point, which is the merge's output order"""
    ijk = voxel_ijk(xyz, voxel_size)
    _, first = np.unique(ijk, axis=0, return_index=True)
    return ijk[np.sort(first)]


def pack(g):
    g = np.asarray(g, np.int64) + KEY_LIM
    return (g[..., 0] << 42) | (g[..., 1] << 21) | g[..., 2]


def corner_bits():
    """corner number c = a + 2 b + 4 c -> (a, b, c)"""
    return np.array([[c & 1, (c >> 1) & 1, c >> 2] for c in range(8)], np.int64)


def edge_lower(e, m):
    p, q = [x for x in range(3) if x != e]
    return ((m & 1) << p) | ((m >> 1) << q)


def vertex_ref(g, f, S):
    """vertices [n][3] float32 of cells g [n][3] with corner values f [n][8]"""
    s = np.zeros((len(g), 3))
    cnt = np.zeros(len(g))
    for e in range(3):
        for m in range(4):
            u = edge_lower(e, m)
            w = u | (1 << e)
            cross = (f[:, u] < 0) != (f[:, w] < 0)
            with np.errstate(all="ignore"):
                t = f[:, u] / (f[:, u] - f[:, w])
            for x in range(3):
                c = (g[:, e].astype(F64) + t) * S if x == e else (g[:, x] + ((u >> x) & 1)).astype(F64) * S
                s[:, x] = np.where(cross, s[:, x] + c, s[:, x])
            cnt += cross
    with np.errstate(all="ignore"):
        return (s / cnt[:, None]).astype(F32)


def normal_ref(f):
    gr = []
    for e in range(3):
        d = [f[:, edge_lower(e, m) | (1 << e)] - f[:, edge_lower(e, m)] for m in range(4)]
        gr.append((d[0] + d[1]) + (d[2] + d[3]))
    gr = np.stack(gr, 1)
    with np.errstate(all="ignore"):
        l = np.sqrt((gr[:, 0] * gr[:, 0] + gr[:, 1] * gr[:, 1]) + gr[:, 2] * gr[:, 2])
        ok = (l > 0) & np.isfinite(l)
        return np.where(ok[:, None], gr / l[:, None], 0.0).astype(F32)


def mixed_ref(f):
    n = (f < 0).sum(1)
    return (n > 0) & (n < 8)


def quad_ref(a):
    """cell offsets of v0..v3 around lattice edge g -> g + e_a"""
    b, d = (a + 1) % 3, (a + 2) % 3
    off = np.zeros((4, 3), np.int64)
    off[0, b] = off[0, d] = -1
    off[1, d] = -1
    off[3, b] = -1
    return off


def triangles_ref(v, lower_inside):
    return [(v[0], v[1], v[2]), (v[0], v[2], v[3])] if lower_inside else [(v[0], v[2], v[1]), (v[0], v[3], v[2])]


def nearest_ref(x, mxyz, R):
    """(ordinal, f) of the nearest model point (rows of mxyz are the model, with their own ordinals) to each x [n][3]
    within R, -1 when none; candidates from a k-d tree, the exact rule on top"""
    R = F64(F32(R))
    q = mxyz.astype(F64)
    tree = cKDTree(q)
    lists = tree.query_ball_point(x, R * (1 + 1e-9) + 1e-300)
    lens = np.array([len(l) for l in lists])
    xi = np.repeat(np.arange(len(x)), lens)
    oi = np.concatenate([np.asarray(l, np.int64) for l in lists]) if lens.sum() else np.zeros(0, np.int64)
    d = x[xi] - q[oi]
    d2 = (d[:, 0] * d[:, 0] + d[:, 1] * d[:, 1]) + d[:, 2] * d[:, 2]
    keep = d2 <= R * R
    xi, oi, d2 = xi[keep], oi[keep], d2[keep]
    order = np.lexsort((oi, d2, xi))
    xi, oi = xi[order], oi[order]
    first = np.ones(len(xi), bool)
    first[1:] = xi[1:] != xi[:-1]
    best = np.full(len(x), -1, np.int64)
    best[xi[first]] = oi[first]
    return best


def extract_ref(mxyz, mnrm, mrgb, mijk, voxel_size, max_distance):
    """the whole surface: (xyz, normals, rgb, faces, lattice_points, undefined_points)"""
    S = F64(F32(voxel_size))
    mxyz, mnrm = np.asarray(mxyz, F32), np.asarray(mnrm, F32)
    model = np.flatnonzero(np.any(mnrm != 0, axis=1))
    offs = np.array([[dx, dy, dz] for dz in (-1, 0, 1) for dy in (-1, 0, 1) for dx in (-1, 0, 1)], np.int64)
    g = (mijk[model][:, None, :] + offs[None]).reshape(-1, 3)
    key27 = (27 * model[:, None] + np.arange(27)[None]).reshape(-1)
    ok = ((g >= -KEY_LIM) & (g + 1 < KEY_LIM)).all(1)
    g, key27 = g[ok], key27[ok]
    pk = pack(g)
    order = np.lexsort((key27, pk))
    pk, g, key27 = pk[order], g[order], key27[order]
    first = np.ones(len(pk), bool)
    first[1:] = pk[1:] != pk[:-1]
    cells, owner = g[first], key27[first]
    corners = (cells[:, None, :] + corner_bits()[None]).reshape(-1, 3)
    pts_keys, idx = np.unique(pack(corners), return_index=True)
    pts = corners[idx]
    x = pts.astype(F64) * S
    near_m = nearest_ref(x, mxyz[model], max_distance)
    near = np.where(near_m >= 0, model[np.maximum(near_m, 0)], -1)
    qn = np.maximum(near, 0)
    d = x - mxyz[qn].astype(F64)
    n = mnrm[qn].astype(F64)
    fv = (d[:, 0] * n[:, 0] + d[:, 1] * n[:, 1]) + d[:, 2] * n[:, 2]
    ci = np.searchsorted(pts_keys, pack(corners)).reshape(-1, 8)
    defined = (near[ci] >= 0).all(1)
    f8 = fv[ci]
    act = defined & mixed_ref(f8)
    order = np.argsort(owner[act], kind="stable")
    acells, af8, aci = cells[act][order], f8[act][order], ci[act][order]
    V = len(acells)
    vxyz = vertex_ref(acells, af8, S) if V else np.zeros((0, 3), F32)
    vnrm = normal_ref(af8) if V else np.zeros((0, 3), F32)
    csum = mrgb[near[aci]].astype(np.int64).sum(1) if V else np.zeros((0, 3), np.int64)
    vrgb = ((csum + 4) // 8).astype(np.uint8)
    akeys = pack(acells)
    srt = np.argsort(akeys)
    faces = []
    for r in range(V):
        gr = acells[r]
        lower = af8[r, 0] < 0
        for a in range(3):
            up = gr.copy()
            up[a] += 1
            fu = fv[np.searchsorted(pts_keys, pack(up))]
            if (fu < 0) == lower:
                continue
            nb = pack(gr[None] + quad_ref(a))
            pos = np.searchsorted(akeys, nb, sorter=srt)
            pos = np.minimum(pos, V - 1)
            hit = akeys[srt[pos]] == nb
            if not hit.all():
                continue
            faces += triangles_ref(srt[pos], lower)
    faces = np.array(faces, np.int32).reshape(-1, 3)
    return vxyz, vnrm, vrgb, faces, len(pts), int((near < 0).sum())


# ---- the host build -----------------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def shim(tmp_path_factory):
    so = str(tmp_path_factory.mktemp("surfacehost") / "libsurface_math_host.so")
    subprocess.check_call(["/usr/bin/g++", "-O2", "-std=c++17", "-fPIC", "-shared", "-Wall", "-ffp-contract=off",
                           "-o", so, os.path.join(HERE, "surface_math_host.cpp")])
    L = C.CDLL(so)
    vp, i64 = C.c_void_p, C.c_longlong
    L.s3s_host_lattice_pos.argtypes = [vp, i64, C.c_float, vp]
    L.s3s_host_residual.argtypes = [vp, vp, vp, i64, vp]
    L.s3s_host_cells.argtypes = [vp, vp, i64, C.c_float, vp, vp, vp]
    L.s3s_host_colour.argtypes = [vp, i64, vp]
    L.s3s_host_offsets.argtypes = [vp, vp]
    L.s3s_host_quad.argtypes = [C.c_int, C.c_int, vp, vp]
    L.s3s_host_extract.argtypes = [vp, vp, vp, vp, i64, C.c_float, C.c_float, vp, vp, vp, vp, i64, i64, vp]
    L.s3s_host_layout.argtypes = [vp]
    return L


def _p(a):
    return a.ctypes.data_as(C.c_void_p)


def host_extract(L, mxyz, mnrm, mrgb, mijk, voxel_size, max_distance):
    m = len(mxyz)
    cap_v, cap_f = 27 * m + 1, 6 * 27 * m + 1
    mxyz, mnrm = np.ascontiguousarray(mxyz, F32), np.ascontiguousarray(mnrm, F32)
    mrgb, mijk = np.ascontiguousarray(mrgb, np.uint8), np.ascontiguousarray(mijk, np.int64)
    vx, vn = np.zeros((cap_v, 3), F32), np.zeros((cap_v, 3), F32)
    vr, fc = np.zeros((cap_v, 3), np.uint8), np.zeros((cap_f, 3), np.int32)
    cnt = np.zeros(4, np.int64)
    L.s3s_host_extract(_p(mxyz), _p(mnrm), _p(mrgb), _p(mijk), m, voxel_size, max_distance, _p(vx), _p(vn), _p(vr),
                       _p(fc), cap_v, cap_f, _p(cnt))
    V, Fn = int(cnt[0]), int(cnt[1])
    return vx[:V], vn[:V], vr[:V], fc[:Fn], int(cnt[2]), int(cnt[3])


def assert_same_surface(a, b):
    for x, y in zip(a[:4], b[:4]):
        assert x.shape == y.shape and x.dtype == y.dtype
        assert np.array_equal(x.view(np.uint8), y.view(np.uint8))
    assert a[4:] == b[4:]


def random_model(rng, m, s, spread=6):
    """up to m voxels of a rough slab (two voxels thick) over a small block of the lattice, with unit normals
    scattered about +z (some zero) and random colours; the voxel outputs lie inside their voxels"""
    ijk = np.concatenate([rng.integers(-spread, spread, (4 * m, 2)), rng.integers(0, 2, (4 * m, 1))], 1)
    _, first = np.unique(ijk, axis=0, return_index=True)
    ijk = ijk[np.sort(first)][:m]
    xyz = ((ijk + rng.uniform(0.02, 0.98, ijk.shape)) * s).astype(F32)
    n = 0.5 * rng.normal(size=ijk.shape) + [0.0, 0.0, 1.0]
    nrm = (n / np.linalg.norm(n, axis=1, keepdims=True)).astype(F32)
    nrm[rng.random(len(ijk)) < 0.1] = 0
    rgb = rng.integers(0, 256, ijk.shape, dtype=np.uint8)
    return xyz, nrm, rgb, ijk


def sphere_model(s, r, centre=(0.3, -0.2, 0.1)):
    """points sampled densely on a whole sphere with outward normals, merged by the restatement of the voxel merge's
    order (first point) -- one point per voxel is enough for these checks: its coordinate is the point itself"""
    c = np.array(centre)
    n = int(40 * (r / s) ** 2)
    k = np.arange(n) + 0.5
    phi = np.arccos(1 - 2 * k / n)
    th = np.pi * (1 + 5 ** 0.5) * k
    u = np.stack([np.cos(th) * np.sin(phi), np.sin(th) * np.sin(phi), np.cos(phi)], 1)
    p = (c + r * u).astype(F32)
    ijk = voxel_ijk(p, s)
    _, first = np.unique(ijk, axis=0, return_index=True)
    first = np.sort(first)
    return p[first], u[first].astype(F32), np.full((len(first), 3), 200, np.uint8), ijk[first]


# ---- per-function checks ------------------------------------------------------------------------------------------
def test_layout(shim):
    out = np.zeros(6, np.int64)
    shim.s3s_host_layout(_p(out))
    s3 = importlib.import_module("3dscan_b200")
    assert list(out) == [C.sizeof(s3.SurfaceParams), s3.SurfaceParams.max_points.offset, C.sizeof(s3.SurfaceResultC),
                         s3.SurfaceResultC.faces.offset, s3.SurfaceResultC.lattice_points.offset,
                         s3.SurfaceResultC.undefined_points.offset]


def test_lattice_positions_and_corner_values(shim):
    rng = np.random.default_rng(1)
    s = F32(0.137)
    g = np.concatenate([rng.integers(-KEY_LIM, KEY_LIM, (500, 3)), [[-KEY_LIM] * 3, [KEY_LIM - 1] * 3, [0, 0, 0]]])
    x = np.zeros(g.shape)
    shim.s3s_host_lattice_pos(_p(g), len(g), s, _p(x))
    assert np.array_equal(x, g.astype(F64) * F64(s))
    q = (x + rng.normal(size=x.shape)).astype(F32)
    n = rng.normal(size=x.shape).astype(F32)
    r = np.zeros(len(g))
    shim.s3s_host_residual(_p(x), _p(q), _p(n), len(g), _p(r))
    d = x - q.astype(F64)
    nn = n.astype(F64)
    assert np.array_equal(r, (d[:, 0] * nn[:, 0] + d[:, 1] * nn[:, 1]) + d[:, 2] * nn[:, 2])


def test_ties_at_the_radius_and_in_ordinal(shim):
    """a point exactly at R qualifies, one beyond does not; equal distances go to the smaller ordinal"""
    s = F32(1.0)
    ijk = np.array([[0, 0, 0], [1, 0, 0], [-1, 0, 0], [0, 5, 0]])
    xyz = np.array([[0.5, 0.5, 0.5], [1.5, 0.5, 0.5], [-0.5, 0.5, 0.5], [0.5, 5.5, 0.5]], F32)
    nrm = np.array([[1, 0, 0], [0, 1, 0], [0, 0, 1], [1, 0, 0]], F32)
    rgb = np.array([[10, 20, 30], [40, 50, 60], [70, 80, 90], [1, 2, 3]], np.uint8)
    R = F32(np.sqrt(F32(0.75)))            # lattice corners of cell 0 lie at sqrt(0.75) from its point
    R = np.nextafter(R, F32(10)) if F64(R) ** 2 < 0.75 else R
    for md in (R, np.nextafter(R, F32(0)), F32(2.0)):
        assert_same_surface(host_extract(shim, xyz, nrm, rgb, ijk, s, md), extract_ref(xyz, nrm, rgb, ijk, s, md))
    # the lattice point (1, 1, 1) is equidistant from voxels 0 and 1: the ordinal decides
    got = host_extract(shim, xyz, nrm, rgb, ijk, s, F32(2.0))
    assert got[4] > 0


def _all_sign_patterns():
    pats = []
    for bits in range(1, 255):
        pats.append([-1.0 if bits >> c & 1 else 1.0 for c in range(8)])
    return np.array(pats)


def test_every_mixed_cell(shim):
    rng = np.random.default_rng(2)
    sign = _all_sign_patterns()
    assert len(sign) == 254
    mags = [rng.uniform(1e-3, 2.0, sign.shape), np.full(sign.shape, 1e-300), np.full(sign.shape, 1e300),
            rng.choice([0.0, 5e-324, 1e-200, 1.0, 1e200], sign.shape)]
    g = rng.integers(-1000, 1000, (len(sign), 3))
    s = F32(0.37)
    for mag in mags:
        f = sign * mag
        f = np.where(f == 0, np.where(sign < 0, -5e-324, 0.0), f)     # keep the sides: +0 is outside
        for zero in (0.0, -0.0):                                         # a signed zero is outside either way
            f2 = f.copy()
            f2[:, 7] = np.where(sign[:, 7] > 0, zero, f2[:, 7])
            mixed = np.zeros(len(f2), np.uint8)
            v, nv = np.zeros((len(f2), 3), F32), np.zeros((len(f2), 3), F32)
            shim.s3s_host_cells(_p(g), _p(f2), len(f2), s, _p(mixed), _p(v), _p(nv))
            assert mixed.all() and mixed_ref(f2).all()
            assert np.array_equal(v.view(np.uint32), vertex_ref(g, f2, F64(s)).view(np.uint32))
            assert np.array_equal(nv.view(np.uint32), normal_ref(f2).view(np.uint32))
    # one-sided cells are not mixed; a zero and a cancelling gradient give a zero normal
    f = np.array([[1.0] * 8, [-1.0] * 8, [0.0] * 8, [-0.0] * 8, [1, -1, -1, 1, 1, -1, -1, 1.0],
                  [1e300, -1e300, 1e300, -1e300, 1e300, -1e300, 1e300, -1e300]])
    mixed = np.zeros(len(f), np.uint8)
    v, nv = np.zeros((len(f), 3), F32), np.zeros((len(f), 3), F32)
    shim.s3s_host_cells(_p(np.zeros((len(f), 3), np.int64)), _p(f), len(f), s, _p(mixed), _p(v), _p(nv))
    assert list(mixed) == [0, 0, 0, 0, 1, 1]
    assert np.array_equal(nv.view(np.uint32), normal_ref(f).view(np.uint32))
    assert not nv[:5].any()                            # zero gradient (cells 0-4) ...
    assert not nv[5].any()                             # ... and an infinite length


def test_colour_offsets_and_winding(shim):
    sums = np.arange(0, 8 * 255 + 1, dtype=np.uint32)
    out = np.zeros(len(sums), np.uint8)
    shim.s3s_host_colour(_p(sums), len(sums), _p(out))
    assert np.array_equal(out, ((sums.astype(np.int64) + 4) // 8).astype(np.uint8))
    k_of, d_of = np.zeros(27, np.int32), np.zeros((27, 3), np.int32)
    shim.s3s_host_offsets(_p(k_of), _p(d_of))
    assert list(k_of) == list(range(27))
    assert [tuple(d) for d in d_of] == [(dx, dy, dz) for dz in (-1, 0, 1) for dy in (-1, 0, 1) for dx in (-1, 0, 1)]
    for a in range(3):
        for lower in (0, 1):
            off, tri = np.zeros((4, 3), np.int32), np.zeros(6, np.int32)
            shim.s3s_host_quad(a, lower, _p(off), _p(tri))
            assert np.array_equal(off, quad_ref(a))
            assert [tuple(t) for t in tri.reshape(2, 3)] == triangles_ref([0, 1, 2, 3], lower)
            # the right-hand normal of both triangles, with each vertex at its cell's centre, points along +e_a when
            # the lower end is inside, else along -e_a
            c = quad_ref(a) + 0.5
            for t in tri.reshape(2, 3):
                nrm = np.cross(c[t[1]] - c[t[0]], c[t[2]] - c[t[0]])
                want = np.eye(3)[a] * (1 if lower else -1)
                assert np.dot(nrm, want) > 0 and np.allclose(np.cross(nrm, want), 0)


# ---- whole extractions --------------------------------------------------------------------------------------------
@pytest.mark.parametrize("seed", [0, 1, 2, 3])
def test_random_small_models(shim, seed):
    rng = np.random.default_rng(10 + seed)
    s = F32(rng.uniform(0.1, 2.0))
    xyz, nrm, rgb, ijk = random_model(rng, int(rng.integers(20, 200)), s)
    for md in (F32(1.0) * s, F32(2.0) * s, F32(3.5) * s):
        a = host_extract(shim, xyz, nrm, rgb, ijk, s, md)
        b = extract_ref(xyz, nrm, rgb, ijk, s, md)
        assert_same_surface(a, b)
        assert len(a[0]) > 0 and (len(a[3]) > 0 or md < 2 * s)


def test_closed_sphere(shim):
    s = F32(0.25)
    xyz, nrm, rgb, ijk = sphere_model(s, 2.0)
    a = host_extract(shim, xyz, nrm, rgb, ijk, s, 2 * s)
    b = extract_ref(xyz, nrm, rgb, ijk, s, 2 * s)
    assert_same_surface(a, b)
    vx, _, _, faces, _, undefined = a
    assert len(faces) > 100
    e = np.sort(np.concatenate([faces[:, [0, 1]], faces[:, [1, 2]], faces[:, [2, 0]]]), axis=1)
    _, cnt = np.unique(e, axis=0, return_counts=True)
    assert (cnt == 2).all()
    assert len(vx) - len(cnt) + len(faces) == 2


def test_single_voxel(shim):
    s = F32(0.5)
    xyz = np.array([[0.2, 0.3, 0.26]], F32)
    nrm = np.array([[0.0, 0.0, 1.0]], F32)
    rgb = np.array([[9, 99, 199]], np.uint8)
    ijk = voxel_ijk(xyz, s)
    for md in (s, 2 * s, 3 * s):
        a = host_extract(shim, xyz, nrm, rgb, ijk, s, F32(md))
        assert_same_surface(a, extract_ref(xyz, nrm, rgb, ijk, s, F32(md)))
        assert len(a[0]) > 0 and (a[2] == [[9, 99, 199]]).all()
        assert (np.abs(a[0][:, 2] - F32(0.26)) < 1e-6).all()          # the plane z = 0.26, within R of the point
