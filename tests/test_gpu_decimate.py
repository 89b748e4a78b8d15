"""GPU checks of the surface simplification (scan3d_voxel_surface_decimate): bit parity with decimate_ref of
tests/test_decimate_ref.py on random clouds, a dense sphere, the ctx route and a surface after components, at every
cell ratio from 1 to 256; the geometry of a simplified sphere; the state rules, errors and launch count; and the
largest piece of the noise-free multi-view scene."""
import ctypes as C
import math

import numpy as np
import pytest

from gpu_common import s3
from test_decimate_ref import decimate_ref
from test_gpu_align import CENTRE, SMALL, _ctx, _scene, _spacing, _torch
from test_gpu_components import CEN, RADIUS, S, _sphere, _sphere_and_islands
from test_gpu_surface import _cloud, _edges, _merge, _same, _surface
from test_gpu_voxel import C1, _read_ply, _voxel_size
from test_gpu_voxel import _scene as _voxel_scene
from test_surface_math_host import sphere_model

pytestmark = pytest.mark.gpu

F32 = np.float32
LAUNCHES = 12
RATIOS = (1, 2, 4, 8, 256)


def _decimate(ctx, cell):
    before = ctx.launch_count()
    res = ctx.surface_decimate(cell)
    assert ctx.launch_count() == before + LAUNCHES
    return res, ctx.voxel_surface_mesh()


def _check(ctx, s, raw, extract, ratios=RATIOS):
    """for each ratio: extract again, simplify, compare with the reference; the second ratio twice"""
    out = {}
    for r in ratios + ratios[1:2]:
        _same(extract(), raw)
        cell = F32(r * s)
        res, mesh = _decimate(ctx, cell)
        want = decimate_ref(raw, s, cell)
        _same(mesh, want[:4])
        assert res == dict(vertices=len(want[0]), faces=len(want[3]), collapsed_faces=want[4],
                           duplicate_faces=want[5], mean_fallbacks=want[6]), r
        if r in out:
            _same(mesh, out[r][1])
        out[r] = (res, mesh, want)
        print(f"H/s {r}: {len(raw[0])} -> {res['vertices']} vertices, {len(raw[3])} -> {res['faces']} faces, "
              f"{res['collapsed_faces']} collapsed, {res['duplicate_faces']} duplicates, "
              f"{res['mean_fallbacks']} fallbacks")
    return out


@pytest.mark.parametrize("seed", [0, 1])
def test_parity_random_clouds(seed):
    rng = np.random.default_rng(seed)
    ctx = _ctx()
    s = F32(0.2)
    p, n, c = _cloud(rng, 40000)
    _merge(ctx, s, [(p, n, c)])
    raw = _surface(ctx, max_distance=F32(2 * s))[1]
    assert len(raw[3]) > 1000
    _check(ctx, s, raw, lambda: _surface(ctx, max_distance=F32(2 * s))[1])
    ctx.close()


def test_parity_dense_sphere():
    ctx = _ctx()
    s = F32(0.1)
    p, n, c, _ = sphere_model(s, 2.5)
    _merge(ctx, s, [(p, n, c)])
    raw = _surface(ctx)[1]
    _check(ctx, s, raw, lambda: _surface(ctx)[1])
    ctx.close()


def test_parity_ctx_route_640x480():
    cfg, cal, stack, roi = _scene(SMALL)
    ctx = s3.Scan3D(cfg, 0, cal)
    ctx.set_texture(np.random.default_rng(5).integers(0, 256, (cfg.H, cfg.W, 3), dtype=np.uint8))
    for k, theta in enumerate((0.0, 20.0, 40.0)):
        ctx.set_registration(True, theta, *CENTRE)
        n = ctx.reconstruct(stack, roi)
        ctx.build_mesh(math.inf)
        if k == 0:
            s = F32(2.0 * _spacing(ctx))
            ctx.voxel_begin(s, 3 * n)
        ctx.voxel_add()
    ctx.voxel_finish()
    raw = _surface(ctx)[1]
    assert len(raw[3]) > 1000
    _check(ctx, s, raw, lambda: _surface(ctx)[1])
    ctx.close()


def test_parity_after_components():
    ctx = _ctx()
    _sphere_and_islands(ctx)

    def largest():
        _surface(ctx)
        ctx.surface_components(0, 1)
        return ctx.voxel_surface_mesh()
    raw = largest()
    _check(ctx, S, raw, largest)
    ctx.close()


def _edge_counts(faces):
    """(boundary edges, non-manifold edges) of a mesh: undirected edges in one face, in more than two"""
    und, cnt = np.unique(np.sort(_edges(faces), axis=1), axis=0, return_counts=True)
    return int((cnt == 1).sum()), int((cnt > 2).sum())


def test_geometry_of_a_simplified_sphere():
    ctx = _ctx()
    raw = _sphere_and_islands(ctx, islands=False)
    nf = len(raw[3])

    def radial_rms(x):
        return float(np.sqrt(np.mean((np.linalg.norm(x.astype(np.float64) - CEN, axis=1) - RADIUS) ** 2)))
    for r in (2, 4, 8):
        _surface(ctx)
        res, (xyz, nrm, rgb, faces) = _decimate(ctx, F32(r * S))
        want = decimate_ref(raw, S, F32(r * S))
        _same((xyz, nrm, rgb, faces), want[:4])
        assert nf / len(faces) >= r * r / 4
        e_quadric, e_mean = radial_rms(xyz), radial_rms(want[7]["mean"])
        assert e_quadric < e_mean
        x = xyz.astype(np.float64)
        fn = np.cross(x[faces[:, 1]] - x[faces[:, 0]], x[faces[:, 2]] - x[faces[:, 0]])
        outward = float(((fn * (x[faces].mean(1) - CEN)).sum(1) > 0).mean())
        assert outward >= 0.99
        comp = ctx.surface_components(1, 0)
        assert comp["kept"] == 1
        boundary, nonmanifold = _edge_counts(faces)
        print(f"sphere r {RADIUS} s {S} H/s {r}: {nf} -> {len(faces)} faces ({nf / len(faces):.1f}x), "
              f"{res['vertices']} vertices, {res['mean_fallbacks']} fallbacks; radial RMS {e_quadric:.3g} (quadric) vs "
              f"{e_mean:.3g} (mean); outward {outward:.5f}; {boundary} boundary, {nonmanifold} non-manifold edges; "
              f"components {comp['components']}")
    ctx.close()


def test_rules_state_errors_and_launch_count(tmp_path):
    ctx = _ctx()
    L, h = ctx.L, ctx.h
    out = s3.DecimateResultC()
    vbuf = np.zeros(8, np.int64)

    def run(cell):
        return L.scan3d_voxel_surface_decimate(h, F32(cell), C.byref(out))

    def table():
        return L.scan3d_get_surface_components(h, vbuf.ctypes.data_as(C.c_void_p), None, None, 8)

    before = ctx.launch_count()
    assert run(4 * S) == -3                                        # before any surface
    assert ctx.launch_count() == before
    raw = _sphere_and_islands(ctx)
    acc = b"".join(a.tobytes() for a in ctx.voxels())
    src = _torch((_sphere(S, RADIUS, CEN)[0][::5] + F32(0.01)).astype(F32))
    kw = dict(max_iterations=3, apply=False, stop_rotation=0.0, stop_translation=0.0)
    r1 = ctx.align_dev(src, 0.2, **kw)
    # argument errors: nothing launched, the surface stays byte-identical
    before = ctx.launch_count()
    assert L.scan3d_voxel_surface_decimate(None, F32(4 * S), C.byref(out)) == -4
    assert L.scan3d_voxel_surface_decimate(h, F32(4 * S), None) == -4
    for bad in (math.nan, math.inf, -math.inf, 0.0, -1.0, S * F32(0.999), 257 * S, 1e30):
        assert run(bad) == -4, bad
    assert ctx.launch_count() == before
    _same(ctx.voxel_surface_mesh(), raw)
    # a component table made before is stale afterwards; components after work
    ctx.surface_components(0, 0)
    assert table() == 0
    res, mesh = _decimate(ctx, F32(4 * S))
    assert table() == -3
    _same(mesh, decimate_ref(raw, S, F32(4 * S))[:4])
    # a second simplification is refused until a new extraction
    before = ctx.launch_count()
    assert run(4 * S) == -3 and b"already" in L.scan3d_last_error(h)
    assert ctx.launch_count() == before
    _same(ctx.voxel_surface_mesh(), mesh)
    comp = ctx.surface_components(1, 0)
    assert table() == 0 and comp["faces"] == res["faces"] and comp["vertices"] <= res["vertices"]
    assert run(4 * S) == -3                                        # components do not clear the refusal
    _same(_surface(ctx)[1], raw)
    res, mesh = _decimate(ctx, F32(4 * S))
    # the PLY writer writes the simplified surface
    path = str(tmp_path / "simple.ply")
    ctx.write_voxel_surface_ply(path, binary=True)
    head, body = _read_ply(path)
    nv, nf = len(mesh[0]), len(mesh[3])
    assert f"element vertex {nv}" in head and f"element face {nf}" in head
    vt = np.dtype([("xyz", "<f4", 3), ("n", "<f4", 3), ("rgb", "u1", 3)])
    ft = np.dtype([("k", "u1"), ("v", "<i4", 3)])
    v = np.frombuffer(body, vt, nv)
    f = np.frombuffer(body, ft, nf, offset=nv * vt.itemsize)
    _same((v["xyz"].copy(), v["n"].copy(), v["rgb"].copy(), f["v"].copy()), mesh)
    # the accumulator is unchanged, an align gives what it gave before and leaves the surface
    assert b"".join(x.tobytes() for x in ctx.voxels()) == acc
    r2 = ctx.align_dev(src, 0.2, **kw)
    assert r1.T.tobytes() == r2.T.tobytes() and (r1.pairs_first, r1.rms_last) == (r2.pairs_first, r2.rms_last)
    _same(ctx.voxel_surface_mesh(), mesh)
    # an empty surface: every launch, 0 / 0
    ctx.voxel_begin(S, 16)
    far = _torch(np.array([[1.0, 1.0, 1.0]], F32))
    ctx.voxel_add_dev(far, None, None)                            # a model without normals gives an empty surface
    ctx.voxel_finish()
    assert _surface(ctx)[0]["faces"] == 0
    res, mesh = _decimate(ctx, F32(2 * S))
    assert res == dict(vertices=0, faces=0, collapsed_faces=0, duplicate_faces=0, mean_fallbacks=0)
    assert [len(a) for a in mesh] == [0, 0, 0, 0]
    # begin, add and finish make the simplified surface stale
    p, nn, c = _sphere(S, RADIUS, CEN)
    tp, tn, tc = _torch(p), _torch(nn), _torch(c)
    for step in ("begin", "add", "finish"):
        ctx.voxel_begin(S, len(p))
        ctx.voxel_add_dev(tp, tn, tc)
        ctx.voxel_finish()
        _surface(ctx)
        assert run(4 * S) == 0
        if step == "begin":
            ctx.voxel_begin(S, len(p))
        elif step == "add":
            ctx.voxel_add_dev(tp, tn, tc)
        else:
            ctx.voxel_finish()
        assert L.scan3d_get_voxel_surface(h, None, None, None, None, 0, 0) == -3, step
        assert run(4 * S) == -3, step
    del src, far, tp, tn, tc
    ctx.close()


def test_largest_piece_of_the_noise_free_scene():
    """The largest component of eight merged views of the sphere alone (test_gpu_components' scene), simplified at
    H = 4 s: against the reference, and what it does to the face count and the distance from the sphere."""
    params = s3.default_synth_params(noise_sigma=0.0)
    cfg, cal, _, stack, roi, truth = _voxel_scene(C1, params=params, want_truth=True)
    centre = np.array(CENTRE)
    on_sphere = np.abs(np.linalg.norm(truth.astype(np.float64) - centre, axis=2) - 25.0) < 1e-3
    roi = (roi * on_sphere).astype(np.uint8)
    ctx = s3.Scan3D(cfg, 0, cal)
    s = None
    for k in range(8):
        ctx.set_registration(True, 45.0 * k, *CENTRE)
        n = ctx.reconstruct(stack, roi)
        ctx.build_mesh(math.inf)
        if s is None:
            s = _voxel_size(ctx.points())
            ctx.voxel_begin(s, 8 * n)
        ctx.voxel_add()
    ctx.voxel_finish()
    _surface(ctx)
    ctx.surface_components(0, 1)
    big = ctx.voxel_surface_mesh()
    res, mesh = _decimate(ctx, F32(4 * s))
    want = decimate_ref(big, F32(s), F32(4 * s))
    _same(mesh, want[:4])

    def off(m):
        return float(np.abs(np.linalg.norm(m[0].astype(np.float64) - centre, axis=1) - 25.0).max())
    used = np.unique(mesh[3])
    before, after = off(big), off((mesh[0][used],))
    boundary, nonmanifold = _edge_counts(mesh[3])
    print(f"voxel {s:.4f}: largest component {len(big[0])} vertices, {len(big[3])} faces, max |r - 25| {before:.4f}; "
          f"H = 4 s: {res['vertices']} vertices ({len(used)} in faces), {res['faces']} faces, "
          f"{res['mean_fallbacks']} fallbacks, max |r - 25| {after:.4f}; {boundary} boundary, {nonmanifold} "
          f"non-manifold edges")
    # measured on a B200 (1000 W power limit): voxel 0.1318, largest component 557 592 vertices, 1 109 222 faces, max
    # |r - 25| 0.4808; at H = 4 s 34 404 vertices (34 274 in faces), 68 972 faces (16.1x fewer), 1179 fallbacks, max
    # |r - 25| 0.4330; 975 boundary and 2259 non-manifold edges.  Margins: 5 % on the reduction, 0.02 mm on the distance.
    assert len(big[3]) / res["faces"] >= 15.3
    assert after <= 0.453 and after < before
    ctx.close()
