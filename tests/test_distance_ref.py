"""The numpy reference of the sample-to-surface distances (scan3d_voxel_surface_distance, scan3d_voxel_surface_distance_dev,
scan3d_mesh_distance_dev; include/scan3d.h and 3dscan_b200/common/scan3d_distance_math.h have the rules):
distance_ref(samples, xyz, faces, R) gives the per-sample outputs and the result dict the GPU must match byte for
byte.  It is checked here against a brute-force plain-Python loop over all faces, and against exact values on an
axis-aligned cube and an icosphere."""
import math

import numpy as np
import pytest

F32 = np.float32
I_MIN, I_MAX = -(1 << 20), 1 << 20
BLOCK = 256


def _dot(u, v):
    return (u[..., 0] * v[..., 0] + u[..., 1] * v[..., 1]) + u[..., 2] * v[..., 2]


def _along(s, t, u):
    return s + t[:, None] * u


def _segment(p, s, e):
    u = e - s
    t = _dot(p - s, u)
    m = _dot(u, u)
    q = e.copy()
    lo = t <= 0
    q[lo] = s[lo]
    mid = ~lo & (t < m)
    q[mid] = _along(s[mid], t[mid] / m[mid], u[mid])
    return q


def _edges(p, a, b, c):
    best_q = _segment(p, a, b)
    best = _dot(p - best_q, p - best_q)
    for s, e in ((b, c), (c, a)):
        q = _segment(p, s, e)
        d = _dot(p - q, p - q)
        w = d < best
        best_q[w], best[w] = q[w], d[w]
    return best_q


def normal_ref(a, b, c):
    ab, ac = b - a, c - a
    N = np.stack([ab[:, 1] * ac[:, 2] - ab[:, 2] * ac[:, 1], ab[:, 2] * ac[:, 0] - ab[:, 0] * ac[:, 2],
                  ab[:, 0] * ac[:, 1] - ab[:, 1] * ac[:, 0]], 1)
    return N, _dot(N, N)


def closest_ref(p, a, b, c):
    """Ericson's ClosestPtPointTriangle with the header's fallback, vectorised over rows of float64 [m][3]"""
    m = len(p)
    N, l2 = normal_ref(a, b, c)
    q = np.zeros((m, 3))
    fb = l2 == 0
    done = fb.copy()
    ab, ac = b - a, c - a
    ap, bp, cp = p - a, p - b, p - c
    d1, d2 = _dot(ab, ap), _dot(ac, ap)
    d3, d4 = _dot(ab, bp), _dot(ac, bp)
    d5, d6 = _dot(ab, cp), _dot(ac, cp)
    vc = d1 * d4 - d3 * d2
    vb = d5 * d2 - d1 * d6
    va = d3 * d6 - d5 * d4
    e, g = d4 - d3, d5 - d6
    with np.errstate(divide="ignore", invalid="ignore"):
        r = ~done & (d1 <= 0) & (d2 <= 0)
        q[r], done = a[r], done | r
        r = ~done & (d3 >= 0) & (d4 <= d3)
        q[r], done = b[r], done | r
        r = ~done & (vc <= 0) & (d1 >= 0) & (d3 <= 0)
        den = d1 - d3
        ok = r & (den > 0)
        q[ok] = _along(a[ok], d1[ok] / den[ok], ab[ok])
        fb, done = fb | (r & ~ok), done | r
        r = ~done & (d6 >= 0) & (d5 <= d6)
        q[r], done = c[r], done | r
        r = ~done & (vb <= 0) & (d2 >= 0) & (d6 <= 0)
        den = d2 - d6
        ok = r & (den > 0)
        q[ok] = _along(a[ok], d2[ok] / den[ok], ac[ok])
        fb, done = fb | (r & ~ok), done | r
        r = ~done & (va <= 0) & (e >= 0) & (g >= 0)
        den = e + g
        ok = r & (den > 0)
        q[ok] = _along(b[ok], e[ok] / den[ok], (c - b)[ok])
        fb, done = fb | (r & ~ok), done | r
        r = ~done
        den = (va + vb) + vc
        ok = r & (den > 0)
        inv = 1.0 / den[ok]
        q[ok] = _along(_along(a[ok], vb[ok] * inv, ab[ok]), vc[ok] * inv, ac[ok])
        fb = fb | (r & ~ok)
    if fb.any():
        q[fb] = _edges(p[fb], a[fb], b[fb], c[fb])
    d = p - q
    return _dot(d, d), _dot(d, N)


def cell_edge(R):
    return float(F32(R)) * (1.0 + 2.0 ** -20)


def cells_ref(v, S):
    """per value: its cell, and whether it is finite and in the key range"""
    with np.errstate(invalid="ignore", over="ignore"):
        f = np.floor(np.asarray(v, np.float64) / S)
        ok = np.isfinite(f) & (f >= I_MIN) & (f < I_MAX)
    return np.where(ok, f, 0).astype(np.int64), ok


def face_boxes(xyz, faces, S):
    """cell boxes lo, hi [f][3], whether every corner's cell is in range, the entries (clamped at 2^32)"""
    c = xyz[faces].astype(F32)                                  # [f][3 corners][3]
    lo, lok = cells_ref(c.min(1), S)
    hi, hok = cells_ref(c.max(1), S)
    ok = lok.all(1) & hok.all(1)
    n = np.prod(np.where(ok[:, None], hi - lo + 1, 0).astype(object), axis=1) if len(faces) else np.zeros(0)
    ent = np.array([min(int(x), 1 << 32) for x in n], np.uint64)
    return lo, hi, ok, ent


def _key(c):
    return ((c[..., 0] - I_MIN) << 42) | ((c[..., 1] - I_MIN) << 21) | (c[..., 2] - I_MIN)


def candidates(samples, xyz, faces, S):
    """the (sample, face) pairs of the index rule, each once, and the samples' invalid and in-range flags"""
    p = samples.astype(np.float64)
    invalid = ~np.isfinite(p).all(1)
    cs, ok = cells_ref(p, S)
    inr = ok.all(1) & ~invalid
    live = (faces[:, 0] != faces[:, 1]) & (faces[:, 1] != faces[:, 2]) & (faces[:, 0] != faces[:, 2])
    lo, hi, fok, _ = face_boxes(xyz, faces, S)
    sel = np.flatnonzero(live & fok)
    span = (hi[sel] - lo[sel] + 1)
    cnt = span.prod(1) if len(sel) else np.zeros(0, np.int64)
    fid = np.repeat(sel, cnt)
    k = np.arange(len(fid)) - np.repeat(np.cumsum(cnt) - cnt, cnt)
    sp = np.repeat(span, cnt, axis=0)
    off = np.stack([k % sp[:, 0], (k // sp[:, 0]) % sp[:, 1], k // (sp[:, 0] * sp[:, 1])], 1) if len(fid) else \
        np.zeros((0, 3), np.int64)
    ekey = _key(np.repeat(lo[sel], cnt, axis=0) + off) if len(fid) else np.zeros(0, np.int64)
    order = np.argsort(ekey, kind="stable")
    ekey, fid = ekey[order], fid[order]
    si = np.flatnonzero(inr)
    nb = np.array([(dx, dy, dz) for dz in (-1, 0, 1) for dy in (-1, 0, 1) for dx in (-1, 0, 1)], np.int64)
    cc = cs[si][:, None, :] + nb[None]                            # [s][27][3]
    inkey = ((cc >= I_MIN) & (cc < I_MAX)).all(2)
    keys = _key(np.where(inkey[..., None], cc, 0))
    a = np.searchsorted(ekey, keys, "left")
    b = np.searchsorted(ekey, keys, "right")
    n = np.where(inkey, b - a, 0).reshape(-1)
    ps = np.repeat(np.repeat(si, 27), n)
    start = np.repeat(a.reshape(-1), n) + (np.arange(n.sum()) - np.repeat(np.cumsum(n) - n, n))
    pf = fid[start] if len(start) else np.zeros(0, np.int64)
    pair = np.unique(np.stack([ps, pf], 1), axis=0) if len(ps) else np.zeros((0, 2), np.int64)
    return pair, invalid


def _block_sum(v):
    """the header's order: a halving tree per warp, the 8 warps in order, then the block partials by 256 threads"""
    nb = max(1, -(-len(v) // BLOCK))
    x = np.zeros(nb * BLOCK)
    x[:len(v)] = v
    x = x.reshape(nb, BLOCK // 32, 32)
    for h in (16, 8, 4, 2, 1):
        x = x[..., :h] + x[..., h:2 * h]
    w = x[..., 0]
    part = w[:, 0].copy()
    for k in range(1, BLOCK // 32):
        part = part + w[:, k]
    tb = -(-nb // BLOCK) * BLOCK
    y = np.zeros(tb)
    y[:nb] = part
    y = y.reshape(-1, BLOCK)
    acc = np.zeros(BLOCK)
    for r in y:
        acc = acc + r
    for h in (128, 64, 32, 16, 8, 4, 2, 1):
        acc = acc[:h] + acc[h:2 * h]
    return float(acc[0])


def distance_ref(samples, xyz, faces, R, is_sample=None):
    """(dist float32 [n], face int32 [n], result dict) of the header's rules; is_sample: the surface route's model
    mask (None: every row is a sample)"""
    samples = np.ascontiguousarray(samples, F32).reshape(-1, 3)
    xyz = np.ascontiguousarray(xyz, F32).reshape(-1, 3)
    faces = np.ascontiguousarray(faces, np.int32).reshape(-1, 3).astype(np.int64)
    n = len(samples)
    mask = np.ones(n, bool) if is_sample is None else np.asarray(is_sample, bool)
    S = cell_edge(R)
    r2 = float(F32(R)) * float(F32(R))
    idx = np.flatnonzero(mask)
    pair, invalid_s = candidates(samples[idx], xyz, faces, S)
    ps, pf = idx[pair[:, 0]] if len(pair) else np.zeros(0, np.int64), pair[:, 1]
    X = xyz.astype(np.float64)
    d2, s = closest_ref(samples[ps].astype(np.float64), X[faces[pf, 0]], X[faces[pf, 1]], X[faces[pf, 2]])
    q = d2 <= r2
    ps, pf, d2, s = ps[q], pf[q], d2[q], s[q]
    order = np.lexsort((pf, d2, ps))
    ps, pf, d2, s = ps[order], pf[order], d2[order], s[order]
    first = np.ones(len(ps), bool)
    first[1:] = ps[1:] != ps[:-1]
    ps, pf, d2, s = ps[first], pf[first], d2[first], s[first]
    root = np.sqrt(d2)
    dist = np.full(n, np.nan, F32)
    face = np.full(n, -1, np.int32)
    sd = np.where(s < 0, -root, root).astype(F32)
    dist[ps], face[ps] = sd, pf
    dv, d2v = np.zeros(n), np.zeros(n)
    dv[ps], d2v[ps] = root, d2
    m = len(ps)
    sum_d, sum_d2 = _block_sum(dv), _block_sum(d2v)
    if m:
        mx = root.max()
        max_sample = int(ps[root == mx].min())
    else:
        mx, max_sample = 0.0, -1
    _, _, fok, ent = face_boxes(xyz, faces, S)
    live = (faces[:, 0] != faces[:, 1]) & (faces[:, 1] != faces[:, 2]) & (faces[:, 0] != faces[:, 2])
    res = dict(samples=int(mask.sum()), matched=m, invalid=int(invalid_s.sum()), inside=int((s < 0).sum()),
               max_sample=max_sample, max=float(mx), mean=sum_d / m if m else 0.0,
               rms=math.sqrt(sum_d2 / m) if m else 0.0,
               min_signed=float(sd.min()) if m else 0.0, max_signed=float(sd.max()) if m else 0.0,
               entries=int(ent[live].astype(object).sum()) if live.any() else 0)
    return dist, face, res


# ---- an independent plain-Python restatement over all faces ----
def _pdot(u, v):
    return (u[0] * v[0] + u[1] * v[1]) + u[2] * v[2]


def _psub(u, v):
    return [u[0] - v[0], u[1] - v[1], u[2] - v[2]]


def _pseg(p, s, e):
    u = _psub(e, s)
    t = _pdot(_psub(p, s), u)
    if t <= 0:
        return list(s)
    m = _pdot(u, u)
    if t >= m:
        return list(e)
    t = t / m
    return [s[k] + t * u[k] for k in range(3)]


def _pclosest(p, a, b, c):
    ab, ac = _psub(b, a), _psub(c, a)
    N = [ab[1] * ac[2] - ab[2] * ac[1], ab[2] * ac[0] - ab[0] * ac[2], ab[0] * ac[1] - ab[1] * ac[0]]

    def edges():
        best, bq = None, None
        for s, e in ((a, b), (b, c), (c, a)):
            q = _pseg(p, s, e)
            d = _pdot(_psub(p, q), _psub(p, q))
            if best is None or d < best:
                best, bq = d, q
        return bq

    def solve():
        if _pdot(N, N) == 0:
            return edges()
        ap = _psub(p, a)
        d1, d2 = _pdot(ab, ap), _pdot(ac, ap)
        if d1 <= 0 and d2 <= 0:
            return list(a)
        bp = _psub(p, b)
        d3, d4 = _pdot(ab, bp), _pdot(ac, bp)
        if d3 >= 0 and d4 <= d3:
            return list(b)
        vc = d1 * d4 - d3 * d2
        if vc <= 0 and d1 >= 0 and d3 <= 0:
            den = d1 - d3
            return [a[k] + (d1 / den) * ab[k] for k in range(3)] if den > 0 else edges()
        cp = _psub(p, c)
        d5, d6 = _pdot(ab, cp), _pdot(ac, cp)
        if d6 >= 0 and d5 <= d6:
            return list(c)
        vb = d5 * d2 - d1 * d6
        if vb <= 0 and d2 >= 0 and d6 <= 0:
            den = d2 - d6
            return [a[k] + (d2 / den) * ac[k] for k in range(3)] if den > 0 else edges()
        va = d3 * d6 - d5 * d4
        e, g = d4 - d3, d5 - d6
        if va <= 0 and e >= 0 and g >= 0:
            den = e + g
            bc = _psub(c, b)
            return [b[k] + (e / den) * bc[k] for k in range(3)] if den > 0 else edges()
        den = (va + vb) + vc
        if not den > 0:
            return edges()
        inv = 1.0 / den
        v, w = vb * inv, vc * inv
        t = [a[k] + v * ab[k] for k in range(3)]
        return [t[k] + w * ac[k] for k in range(3)]

    q = solve()
    d = _psub(p, q)
    return _pdot(d, d), _pdot(d, N)


def brute_ref(samples, xyz, faces, R):
    r2 = float(F32(R)) * float(F32(R))
    out_d, out_f = [], []
    for p in samples.astype(np.float64).tolist():
        best = None
        if all(math.isfinite(x) for x in p):
            for fi, (i, j, k) in enumerate(faces.tolist()):
                if i == j or j == k or i == k:
                    continue
                d2, s = _pclosest(p, *(xyz[v].astype(np.float64).tolist() for v in (i, j, k)))
                if d2 <= r2 and (best is None or (d2, fi) < best[:2]):
                    best = (d2, fi, s)
        if best is None:
            out_d.append(np.nan)
            out_f.append(-1)
        else:
            r = math.sqrt(best[0])
            out_d.append(-r if best[2] < 0 else r)
            out_f.append(best[1])
    return np.array(out_d, F32), np.array(out_f, np.int32)


# ---- test meshes ----
def cube(size=1.0, origin=(0.0, 0.0, 0.0)):
    """an axis-aligned cube with outward faces (two per side)"""
    o = np.array(origin, np.float64)
    v = np.array([[x, y, z] for z in (0, 1) for y in (0, 1) for x in (0, 1)], np.float64) * size + o
    quads = [(0, 2, 3, 1), (4, 5, 7, 6), (0, 1, 5, 4), (2, 6, 7, 3), (0, 4, 6, 2), (1, 3, 7, 5)]
    f = []
    for a, b, c, d in quads:
        f += [(a, b, c), (a, c, d)]
    return v.astype(F32), np.array(f, np.int32)


def icosphere(level=2, r=1.0):
    t = (1 + 5 ** 0.5) / 2
    v = [(-1, t, 0), (1, t, 0), (-1, -t, 0), (1, -t, 0), (0, -1, t), (0, 1, t), (0, -1, -t), (0, 1, -t), (t, 0, -1),
         (t, 0, 1), (-t, 0, -1), (-t, 0, 1)]
    v = [np.array(x, np.float64) / np.linalg.norm(x) for x in v]
    f = [(0, 11, 5), (0, 5, 1), (0, 1, 7), (0, 7, 10), (0, 10, 11), (1, 5, 9), (5, 11, 4), (11, 10, 2), (10, 7, 6),
         (7, 1, 8), (3, 9, 4), (3, 4, 2), (3, 2, 6), (3, 6, 8), (3, 8, 9), (4, 9, 5), (2, 4, 11), (6, 2, 10),
         (8, 6, 7), (9, 8, 1)]
    for _ in range(level):
        mid, nf = {}, []

        def m(a, b):
            k = (min(a, b), max(a, b))
            if k not in mid:
                x = v[a] + v[b]
                v.append(x / np.linalg.norm(x))
                mid[k] = len(v) - 1
            return mid[k]
        for a, b, c in f:
            ab, bc, ca = m(a, b), m(b, c), m(c, a)
            nf += [(a, ab, ca), (b, bc, ab), (c, ca, bc), (ab, bc, ca)]
        f = nf
    return (np.array(v) * r).astype(F32), np.array(f, np.int32)


def random_mesh(seed, nv=120, nf=300, scale=4.0):
    rng = np.random.default_rng(seed)
    xyz = (rng.normal(size=(nv, 3)) * scale).astype(F32)
    faces = rng.integers(0, nv, (nf, 3)).astype(np.int32)
    faces[::17, 2] = faces[::17, 0]                                     # degenerate
    faces[1::23] = [0, 1, 2]                                            # duplicates
    xyz[5] = xyz[6]                                                     # a zero-length side
    xyz[9] = (xyz[7] + xyz[8]) / 2                                      # collinear corners
    return xyz, faces


def random_samples(seed, n, scale=5.0):
    rng = np.random.default_rng(seed)
    s = (rng.normal(size=(n, 3)) * scale).astype(F32)
    s[::31, 1] = np.nan
    s[1::37, 0] = np.inf
    return s


# ---- tests ----
@pytest.mark.parametrize("seed", range(4))
def test_reference_against_brute_force(seed):
    xyz, faces = random_mesh(seed)
    samples = random_samples(seed + 10, 300)
    samples[:40] = xyz[faces[:40, 0]]                                   # on vertices
    samples[40:80] = (xyz[faces[40:80, 0]] + xyz[faces[40:80, 1]]) / 2  # on edges
    samples[80:120] = xyz[faces[80:120]].mean(1)                        # inside faces
    for R in (1.0, 3.0, 40.0):
        dist, face, res = distance_ref(samples, xyz, faces, R)
        bd, bf = brute_ref(samples, xyz, faces, R)
        assert np.array_equal(face, bf)
        assert np.array_equal(dist.view(np.uint32), bd.view(np.uint32))
        assert res["matched"] == int((face >= 0).sum())
        assert res["invalid"] == int((~np.isfinite(samples).all(1)).sum()) > 0
        assert res["samples"] == 300


def test_cube_exact_values():
    xyz, faces = cube(2.0)
    R = 1.0
    s = np.array([[1.0, 1.0, -0.25],       # 0.25 below the bottom centre: outside
                  [1.0, 1.0, 0.25],        # inside, nearest the bottom
                  [-0.25, 1.0, -0.5],      # nearest the edge x = 0, z = 0
                  [-0.25, -0.5, -0.75],    # nearest the corner 0
                  [2.5, 0.5, 0.75],        # outside the side x = 2
                  [np.nan, 0, 0],          # invalid
                  [10.0, 10.0, 10.0],      # unmatched
                  [1e30, 0.0, 0.0]], F32)  # cell out of the key range
    dist, face, res = distance_ref(s, xyz, faces, R)
    bd, bf = brute_ref(s[:5], xyz, faces, R)
    assert np.array_equal(face[:5], bf) and np.array_equal(dist[:5].view(np.uint32), bd.view(np.uint32))
    assert dist[0] == F32(0.25) and dist[1] == F32(-0.25)
    assert dist[2] == F32(math.sqrt(0.25 ** 2 + 0.5 ** 2))
    assert dist[3] == F32(math.sqrt(0.25 ** 2 + 0.5 ** 2 + 0.75 ** 2))
    assert dist[4] == F32(0.5)
    assert np.isnan(dist[5:]).all() and (face[5:] == -1).all()
    # the bottom centre lies on the diagonal of its two triangles: the tie goes to the smaller face
    assert face[0] == 0 and face[1] == 0
    # the edge sample is equidistant from the bottom and the x = 0 side: the smaller index wins
    d_all = [brute_ref(s[2:3], xyz, faces[f:f + 1], R)[0][0] for f in range(12)]
    tied = [f for f in range(12) if d_all[f] == d_all[face[2]]]
    assert len(tied) >= 2 and face[2] == min(tied)
    assert res["invalid"] == 1 and res["matched"] == 5 and res["inside"] == 1
    assert res["max"] == math.sqrt(0.25 ** 2 + 0.5 ** 2 + 0.75 ** 2) and res["max_sample"] == 3
    assert res["min_signed"] == F32(-0.25) and res["max_signed"] == dist[3]


def test_icosphere_samples_on_the_circumsphere():
    xyz, faces = icosphere(2, 1.0)
    rng = np.random.default_rng(3)
    d = rng.normal(size=(2000, 3))
    s = (d / np.linalg.norm(d, axis=1, keepdims=True)).astype(F32)
    X = xyz.astype(np.float64)
    N = np.cross(X[faces[:, 1]] - X[faces[:, 0]], X[faces[:, 2]] - X[faces[:, 0]])
    inr = np.min(np.abs((N * X[faces[:, 0]]).sum(1)) / np.linalg.norm(N, axis=1))
    assert (N * X[faces[:, 0]]).sum(1).min() > 0                       # outward faces
    dist, face, res = distance_ref(s, xyz, faces, 0.25)
    assert res["matched"] == 2000 and (face >= 0).all()
    assert (dist >= 0).all() and dist.max() <= (1.0 - inr) * (1 + 1e-5) + 1e-6


def test_zero_area_faces_give_no_nan():
    xyz = np.array([[0, 0, 0], [1, 0, 0], [2, 0, 0], [1, 0, 0], [1e20, -1e20, 1], [1, 1, 0], [0, 0, 1]], F32)
    faces = np.array([[0, 1, 2], [1, 3, 0], [0, 2, 1]], np.int32)       # collinear, a repeated point, reversed
    rng = np.random.default_rng(0)
    s = (rng.normal(size=(200, 3)) * 2).astype(F32)
    dist, face, res = distance_ref(s, xyz, faces, 10.0)
    assert res["matched"] == 200 and not np.isnan(dist).any()
    bd, bf = brute_ref(s, xyz, faces, 10.0)
    assert np.array_equal(face, bf) and np.array_equal(dist.view(np.uint32), bd.view(np.uint32))
    # the rounding case of the header: an edge divisor that rounds to 0 on a face of non-zero area
    p = np.array([[1e20, -1e20, 1.0]])
    a, b, c = np.zeros((1, 3)), np.array([[1.0, 1.0, 0.0]]), np.array([[0.0, 0.0, 1.0]])
    d2, s2 = closest_ref(p, a, b, c)
    assert np.isfinite(d2).all() and np.isfinite(s2).all()
    assert (d2[0], s2[0]) == _pclosest(p[0].tolist(), a[0].tolist(), b[0].tolist(), c[0].tolist())


def test_entries_and_boxes_at_cell_boundaries():
    R = 1.0
    S = cell_edge(R)
    below = float(np.nextafter(F32(S), F32(0)))
    xyz = np.array([[0, 0, 0], [S, 0, 0], [0, S, 0], [below, 0, 0], [-1e-30, 0, 0], [3 * S, 2 * S, 0]], F32)
    faces = np.array([[0, 1, 2], [0, 3, 2], [4, 3, 2], [0, 5, 2], [0, 0, 1]], np.int32)
    lo, hi, ok, ent = face_boxes(xyz, faces, S)
    assert ok.all()

    def cell(v):
        return math.floor(float(F32(v)) / S)
    want = []
    for f in faces:
        c = xyz[f].astype(np.float64)
        n = 1
        for k in range(3):
            n *= cell(c[:, k].max()) - cell(c[:, k].min()) + 1
        want.append(n)
    assert list(ent) == want
    # F32(S) may round below S: its cell is then 0; a tiny negative coordinate is in cell -1
    assert want[1] == 2 * 1 * 1 and want[2] == 2 * 2 * 1
    # the total leaves the degenerate face out
    _, _, res = distance_ref(np.zeros((0, 3), F32), xyz, faces, R)
    assert res["entries"] == sum(want[:4])
    # the clamp at 2^32 and the key range
    big = np.array([[-1e5, -1e5, -1e5], [1e5, 1e5, 1e5], [0, 1e5, 0]], F32)
    _, _, ok, ent = face_boxes(big, np.array([[0, 1, 2]], np.int32), cell_edge(0.15))
    assert ok.all() and int(ent[0]) == 1 << 32
    _, _, ok, _ = face_boxes(big, np.array([[0, 1, 2]], np.int32), cell_edge(1e-3))
    assert not ok.any()


def test_block_sum_order():
    rng = np.random.default_rng(1)
    v = rng.random(70000) * 1e3
    got = _block_sum(v)
    assert abs(got - math.fsum(v)) <= 1e-9 * abs(got)
    assert _block_sum(np.zeros(0)) == 0.0
