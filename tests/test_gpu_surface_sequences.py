"""GPU checks of the held voxel surface through long mixed call sequences: every call runs on a context and on the
numpy model of tests/surface_sequence_model.py, which chains the stage references on its own previous output.  After
every step the return code, the result dict, the launch count, the held surface byte for byte, whether the surface and
the component table getters succeed, and the table itself when it is current must all equal the model's.

The scripted sequences each aim at one hazard of the state the stages share: a long chain against the chained
references; smoothing and filling, which swap only part of the surface with the spare set; the _dev routes, which share
each stage's grow-only workspace with the surface route, on meshes much larger and much smaller than the held surface;
a small surface followed by a much larger one; argument and state errors in the middle of a chain; and the context's
pixel route around the surface.  Seeded random sequences mix all of them; a failure prints the steps so far."""
import ctypes as C
import importlib
import math

import numpy as np
import pytest

import surface_sequence_model as sm
from surface_sequence_model import OK, STATE, SurfaceModel
from test_fill_math_host import build_host_lib, host_polygon
from test_fill_ref import polygon_faces_ref
from test_gpu_align import CENTRE, SMALL, _ctx, _spacing, _torch
from test_gpu_align import _scene as _pixel_scene
from test_gpu_surface import _cloud
from test_smooth_ref import odd_mesh
from test_surface_math_host import model_ijk

s3 = importlib.import_module("3dscan_b200")
pytestmark = pytest.mark.gpu

F32 = np.float32
S = F32(0.2)
POINT_BLOCK = 1024
NUMPY_EDGES = 64
_HOST = []


@pytest.fixture(scope="module", autouse=True)
def _host_lib(tmp_path_factory):
    _HOST.append(build_host_lib(tmp_path_factory.mktemp("fillhost")))
    yield
    _HOST.clear()


def _polygon(p, rims, exists):
    """the numpy DP for small holes, the header compiled for the host for large ones (tests/test_gpu_fill.py)"""
    if len(p) <= NUMPY_EDGES:
        return polygon_faces_ref(p, rims, exists)
    return host_polygon(_HOST[0], p, rims, exists)[0]


def _byref(x, null):
    return None if null else C.byref(x)


class Run:
    """one context and its model, stepped together"""

    def __init__(self, ctx):
        self.ctx, self.L, self.h = ctx, ctx.L, ctx.h
        self.model = SurfaceModel(polygon=_polygon)
        self.added = []
        self.log = []
        self._keep = []

    # ---- the merge ---------------------------------------------------------------------------------------------------
    def merge(self, s, parts, max_voxels=None):
        """begin, add each part from device memory, finish; the model takes the finish outputs"""
        self.begin(s, max_voxels or 2 * sum(len(p[0]) for p in parts))
        for p in parts:
            self.add_dev(p)
        self.finish()

    def begin(self, s, max_voxels):
        self.ctx.voxel_begin(s, max_voxels)
        self.model.begin(s)
        self.added = []
        self._record("begin", dict(voxel_size=float(s), max_voxels=max_voxels))

    def add_dev(self, part):
        t = [_torch(a) for a in part]
        self._keep.append(t)
        self.ctx.voxel_add_dev(*t)
        self.added.append(part[0])
        self.model.add()
        self._record("add_dev", dict(points=len(part[0])))

    def add_ctx(self):
        self.added.append(self.ctx.points())
        self.ctx.voxel_add()
        self.model.add()
        self._record("voxel_add", {})

    def finish(self):
        self.ctx.voxel_finish()
        self.ctx.sync()
        xyz, nrm, rgb, _ = self.ctx.voxels()
        ijk = model_ijk(np.concatenate(self.added), self.model.voxel_size)
        assert len(ijk) == len(xyz)
        self.model.finish((xyz, nrm, rgb, ijk))
        self._record("finish", dict(voxels=len(xyz)))

    # ---- one step of the surface route ---------------------------------------------------------------------------------
    def step(self, entry, args=None):
        before = self.ctx.launch_count()
        kw, want = sm.run(self.model, entry, args or {})
        self._record(entry, kw)
        rc, got = getattr(self, "_" + entry)(**kw)
        self._expect(rc == want.rc, f"return code {rc}, the model says {want.rc}")
        if rc == OK:
            self._expect(got == want.result, f"result\n  {got}\nthe model says\n  {want.result}")
        self._expect(self.ctx.launch_count() - before == want.launches,
                     f"{self.ctx.launch_count() - before} launches, the model says {want.launches}")
        self.check()
        return rc, got

    def _extract(self, max_distance, max_points, null=False):
        r = s3.SurfaceResultC()
        rc = self.L.scan3d_voxel_surface(self.h, _byref(s3.SurfaceParams(max_distance, max_points), null), C.byref(r))
        return rc, dict(vertices=r.vertices, faces=r.faces, lattice_points=r.lattice_points,
                        undefined_points=r.undefined_points)

    def _components(self, min_faces, max_components, null=False):
        r = s3.ComponentsResultC()
        rc = self.L.scan3d_voxel_surface_components(self.h, _byref(s3.ComponentsParams(min_faces, max_components), null),
                                                    C.byref(r))
        return rc, {name: getattr(r, name) for name, _ in s3.ComponentsResultC._fields_}

    def _decimate(self, cell_size, null=False):
        r = s3.DecimateResultC()
        rc = self.L.scan3d_voxel_surface_decimate(self.h, cell_size, _byref(r, null))
        return rc, {name: getattr(r, name) for name, _ in s3.DecimateResultC._fields_}

    def _smooth(self, iterations, lam, mu, null=False):
        r = s3.SmoothResultC()
        rc = self.L.scan3d_voxel_surface_smooth(self.h, C.byref(s3.SmoothParams(iterations, lam, mu)), _byref(r, null))
        return rc, s3.Scan3D._smooth_result(r)

    def _fill(self, max_edges, null=False):
        r = s3.FillResultC()
        rc = self.L.scan3d_voxel_surface_fill_holes(self.h, max_edges, _byref(r, null))
        return rc, s3.Scan3D._fill_result(r)

    def _repair(self, flags, null=False):
        r = s3.RepairResultC()
        rc = self.L.scan3d_voxel_surface_repair(self.h, flags, _byref(r, null))
        return rc, s3.Scan3D._repair_result(r)

    def _orient(self, null=False):
        r = s3.OrientResultC()
        rc = self.L.scan3d_voxel_surface_orient(self.h, _byref(r, null))
        return rc, s3.Scan3D._orient_result(r)

    def _measure(self, null=False):
        r = s3.MeasureResultC()
        rc = self.L.scan3d_voxel_surface_measure(self.h, _byref(r, null))
        return rc, s3.Scan3D._measure_result(r)

    # ---- one call of a _dev route, on a mesh (xyz, normals, rgb, faces) in device memory -------------------------------
    def dev(self, entry, mesh, **kw):
        xyz, nrm, _, faces = mesh
        self._record(entry + "_dev", dict(kw, vertices=len(xyz), faces=len(faces)))
        tx, tn, tf = _torch(xyz), _torch(nrm), _torch(faces)
        m, ctx = self.model, self.ctx
        before = ctx.launch_count()
        if entry == "components":
            want = m.components_dev(faces, len(xyz))
            labels, c = ctx.mesh_components_dev(tf, len(xyz))
            got, out = dict(components=c), (labels.cpu().numpy(),)
        elif entry == "smooth":
            want = m.smooth_dev(xyz, nrm, faces, **kw)
            got = ctx.mesh_smooth_dev(tx, tf, tn, kw["iterations"], kw["lam"], kw["mu"])
            out = (tx.cpu().numpy(), tn.cpu().numpy())
        elif entry == "fill":
            want = m.fill_dev(xyz, faces, **kw)
            add, got = ctx.mesh_fill_holes_dev(tx, tf, kw["max_edges"])
            out = (add.cpu().numpy(),)
        elif entry == "repair":
            want = m.repair_dev(xyz, faces, **kw)
            f, src, got = ctx.mesh_repair_dev(tx, tf, bool(kw["flags"] & 1), bool(kw["flags"] & 2))
            out = (f.cpu().numpy(), src.cpu().numpy())
        elif entry == "orient":
            want = m.orient_dev(xyz, nrm, faces)
            got = ctx.mesh_orient_dev(tx, tf, tn)
            out = (tf.cpu().numpy(), tn.cpu().numpy())
        else:
            want = m.measure_dev(xyz, faces)
            got, out = ctx.mesh_measure_dev(tx, tf), None
        self._expect(got == want.result, f"result\n  {got}\nthe model says\n  {want.result}")
        self._expect(ctx.launch_count() - before == want.launches, "launches")
        if out is not None:
            self._expect(_same(out, want.out), "the _dev route's output differs from its reference")
        self.check()
        return got

    # ---- the state after every step -------------------------------------------------------------------------------
    def check(self):
        m, L, h = self.model, self.L, self.h
        rc = L.scan3d_get_voxel_surface(h, None, None, None, None, 0, 0)
        self._expect(rc == m.get_surface().rc, f"scan3d_get_voxel_surface returns {rc}")
        if rc == OK:
            want = m.mesh
            nv, nf = len(want[0]), len(want[3])
            # one row more than the model holds, filled with a marker: the context must not hold more
            got = (np.full((nv + 1, 3), -7, F32), np.full((nv + 1, 3), -7, F32), np.full((nv + 1, 3), 7, np.uint8),
                   np.full((nf + 1, 3), -7, np.int32))
            assert L.scan3d_get_voxel_surface(h, *[a.ctypes.data_as(C.c_void_p) for a in got], nv + 1, nf + 1) == OK
            self._expect((got[0][-1] == -7).all() and (got[3][-1] == -7).all(), "the context holds more than the model")
            self._expect(_same(tuple(a[:-1] for a in got), want), "the held surface differs from the model's")
        rc = L.scan3d_get_surface_components(h, None, None, None, 0)
        self._expect(rc == m.get_components().rc, f"scan3d_get_surface_components returns {rc}")
        if rc == OK:
            v, f, kept = m.table
            c = len(v)
            gv, gf, gk = np.full(c + 1, -7, np.int64), np.full(c + 1, -7, np.int64), np.full(c + 1, 7, np.uint8)
            assert L.scan3d_get_surface_components(h, gv.ctypes.data_as(C.c_void_p), gf.ctypes.data_as(C.c_void_p),
                                                   gk.ctypes.data_as(C.c_void_p), c + 1) == OK
            self._expect(gv[-1] == -7 and gf[-1] == -7 and gk[-1] == 7, "the context's table has more components")
            self._expect(np.array_equal(gv[:c], v) and np.array_equal(gf[:c], f) and
                         np.array_equal(gk[:c], kept.astype(np.uint8)), "the component table differs from the model's")

    def _record(self, entry, kw):
        self.log.append(f"{len(self.log):3d} {entry}({', '.join(f'{k}={v}' for k, v in kw.items())})")

    def _expect(self, ok, what):
        if not ok:
            raise AssertionError(f"{what}\nsteps so far:\n" + "\n".join(self.log))

    def close(self):
        import torch
        torch.cuda.synchronize()
        self._keep.clear()
        self.ctx.close()


def _same(got, want):
    return all(x.shape == y.shape and x.dtype == y.dtype and np.array_equal(x.view(np.uint8), y.view(np.uint8))
               for x, y in zip(got, want))


def _parts(rng, n, r=3.0, cap=0.8, touch=0.4, islands=3):
    """a noisy sphere of radius r open above z = cap r, a smaller sphere that touches it, and single far voxels"""
    p, nrm, c = _cloud(rng, n, r)
    keep = p[:, 2] - F32(0.2) < cap * r
    parts = [(p[keep], nrm[keep], c[keep])]
    q, m, d = _cloud(rng, int(n * touch * touch), touch * r)
    parts.append(((q + np.array([(1 + touch) * r, 0, 0], F32)).astype(F32), m, d))
    far = (np.array([[0.0, 0.0, 3.0]]) * r + np.arange(islands)[:, None] * [2.0 * r, 0.0, 0.0]).astype(F32)
    parts.append((far, np.tile(np.array([[0.0, 0.6, 0.8]], F32), (islands, 1)), np.full((islands, 3), 9, np.uint8)))
    return parts


def _surface_scene(run, seed, n=20000, **kw):
    run.merge(S, _parts(np.random.default_rng(seed), n, **kw))
    rc, res = run.step("extract")
    assert rc == OK
    return res


def _tiled(mesh, copies=8):
    """copies of a mesh side by side: as many times the vertices and faces"""
    xyz, nrm, rgb, faces = mesh
    shift = float(np.abs(xyz).max(initial=1.0)) * 3
    return (np.concatenate([xyz + F32(k * shift) for k in range(copies)]).astype(F32), np.tile(nrm, (copies, 1)),
            np.tile(rgb, (copies, 1)), np.concatenate([faces + k * len(xyz) for k in range(copies)]).astype(np.int32))


def _small(seed):
    xyz, nrm, faces = odd_mesh(np.random.default_rng(seed), 300, 500)
    return xyz, nrm, np.zeros(xyz.shape, np.uint8), faces


def test_long_chain_against_the_chained_references():
    run = Run(_ctx())
    res = _surface_scene(run, 0)
    print(f"raw surface: {res}")
    codes = [run.step(entry, args)[0] for entry, args in sm.LONG_CHAIN]
    # the smoothed surface's decimation is refused, the new extraction's accepted
    assert codes == [OK] * 6 + [STATE] + [OK] * 3
    # a repair that changes the raw surface and a fill that adds faces after it: refused until the next extraction
    run.step("extract")
    run.step("repair", dict(flags=sm.BOTH))
    run.step("fill", dict(max_edges=22))
    assert run.model.filled_after_repair
    assert run.step("decimate", dict(ratio=4))[0] == STATE
    run.step("extract")
    assert run.step("decimate", dict(ratio=4))[0] == OK
    run.close()


def test_partial_swaps():
    """smooth swaps positions and normals only, fill the faces only: every byte of the held surface, the vertices no
    stage moved included, must stay the model's"""
    run = Run(_ctx())
    _surface_scene(run, 1)
    for entry, args in sm.PARTIAL_SWAPS:
        run.step(entry, args)
    # a decimation of a fresh surface after the partial swaps, then the same mix again
    run.step("extract")
    run.step("decimate", dict(ratio=2))
    for entry, args in sm.PARTIAL_SWAPS:
        run.step(entry, args)
    run.close()


DEV_STAGES = {
    "components": ("components", dict(min_faces=0, max_components=0), {}),
    "smooth": ("smooth", sm.SMOOTH, sm.SMOOTH),
    "fill": ("fill", dict(max_edges=22), dict(max_edges=1024)),
    "repair": ("repair", dict(flags=sm.BOTH), dict(flags=sm.BOTH)),
    "orient": ("orient", {}, {}),
    "measure": ("measure", {}, {}),
}


@pytest.mark.parametrize("size", ["larger", "smaller"])
def test_dev_calls_between_surface_calls(size):
    """each stage's surface route, then its _dev route on a mesh about 8 times larger (or much smaller) than the held
    surface with the component table current, then the surface route again"""
    run = Run(_ctx())
    _surface_scene(run, 2)
    for k, (stage, (entry, args, dev_args)) in enumerate(DEV_STAGES.items()):
        run.step(entry, args)
        run.step("components", dict(min_faces=0, max_components=0))
        mesh = _tiled(run.model.mesh) if size == "larger" else _small(k)
        if size == "larger":
            assert len(mesh[3]) >= 8 * len(run.model.mesh[3]) > 0
        run.dev(stage, mesh, **dev_args)
        run.step(entry, args)
    run.close()


def test_shrink_then_grow():
    """one kept component leaves a small surface; a model with several times more voxels then runs the full chain, so
    the compaction offsets and the spare set cross POINT_BLOCK boundaries in both directions"""
    run = Run(_ctx())
    _surface_scene(run, 3, n=8000, islands=5)
    rc, res = run.step("components", dict(min_faces=0, max_components=1))
    small = (res["vertices"], res["faces"])
    for entry, args in sm.FULL_CHAIN:
        run.step(entry, args)
    run.merge(S, _parts(np.random.default_rng(4), 100000, r=8.0))
    rc, big = run.step("extract")
    print(f"small surface {small}, large surface {big['vertices'], big['faces']}")
    assert big["faces"] > 3 * small[1] and big["vertices"] > 3 * small[0] and min(small) > POINT_BLOCK
    for entry, args in sm.FULL_CHAIN:
        run.step(entry, args)
    # and back to a small one
    run.merge(S, _parts(np.random.default_rng(5), 8000))
    run.step("extract")
    for entry, args in sm.FULL_CHAIN:
        run.step(entry, args)
    run.close()


def test_errors_in_the_middle_of_a_chain():
    run = Run(_ctx())
    _surface_scene(run, 6)
    for entry, args in sm.ERRORS_MID_CHAIN:
        run.step(entry, args)
    # state errors: after an add every surface entry and both getters refuse, and a finish does not bring the surface
    # back; the next extraction matches the model
    run.add_dev(_parts(np.random.default_rng(7), 2000)[0])
    for entry, args in [("extract", {}), ("components", dict(min_faces=0, max_components=0)), ("decimate", dict(ratio=2)),
                        ("smooth", sm.SMOOTH), ("fill", dict(max_edges=8)), ("repair", dict(flags=sm.BOTH)),
                        ("orient", {}), ("measure", {})]:
        assert run.step(entry, args)[0] == STATE
    run.finish()
    assert run.step("measure")[0] == STATE
    for entry, args in [("extract", {}), ("components", dict(min_faces=1, max_components=1)), ("decimate", dict(ratio=3)),
                        ("measure", {})]:
        assert run.step(entry, args)[0] == OK
    run.begin(S, 10)
    run.check()
    run.close()


def test_the_context_route_around_the_surface():
    """reconstruct, build_mesh and an align that moves the points leave the surface and the table current; an add, a
    finish or a begin make them stale"""
    cfg, cal, stack, roi = _pixel_scene(SMALL)
    ctx = s3.Scan3D(cfg, 0, cal)
    ctx.set_texture(np.random.default_rng(5).integers(0, 256, (cfg.H, cfg.W, 3), dtype=np.uint8))
    run = Run(ctx)
    ctx.set_registration(True, 0.0, *CENTRE)
    n = ctx.reconstruct(stack, roi)
    ctx.build_mesh(math.inf)
    s = F32(5 * _spacing(ctx))
    run.begin(s, 3 * n)
    run.add_ctx()
    run.finish()
    assert run.step("extract")[1]["faces"] > 1000
    run.step("components", dict(min_faces=1, max_components=0))
    ctx.set_registration(True, 20.0, *CENTRE)
    ctx.reconstruct(stack, roi)
    run.check()
    ctx.build_mesh(math.inf)
    run.check()
    ctx.align(F32(4 * s), max_iterations=3, apply=True)
    run.check()
    run.step("smooth", sm.SMOOTH)
    ctx.build_mesh(math.inf)
    run.add_ctx()
    assert run.step("measure")[0] == STATE
    run.finish()
    assert run.step("smooth", sm.SMOOTH)[0] == STATE
    run.step("extract")
    run.step("repair", dict(flags=sm.BOTH))
    run.step("decimate", dict(ratio=2))
    ctx.reconstruct(stack, roi)
    ctx.align(F32(4 * s), max_iterations=2, apply=True)
    run.step("orient")
    run.begin(s, 3 * n)
    run.check()
    run.close()


def _random_step(rng, run):
    """one step of a random sequence: a surface entry or a _dev call with valid or invalid arguments, or an add"""
    pick = lambda xs: xs[rng.integers(len(xs))]
    entry = pick(["extract", "components", "components", "decimate", "smooth", "fill", "fill", "repair", "orient",
                  "measure", "dev", "dev", "dev", "add"])
    null = rng.random() < 0.05
    if entry == "extract":
        if "VOXELS" not in run.model.current:
            run.finish()
        args = dict(null=null)
    elif entry == "components":
        args = dict(min_faces=pick([0, 0, 1, 5, 50, -1]), max_components=pick([0, 0, 1, 2, 4, -2]), null=null)
    elif entry == "decimate":
        args = dict(ratio=pick([1.0, 2.0, 3.5, 4.0, 0.9, 300.0]), null=null)
    elif entry == "smooth":
        args = dict(iterations=pick([0, 1, 3, 10, -1]), lam=pick([0.5, 0.33, 1.0, 0.0]),
                    mu=pick([-0.53, 0.0, -1.0, 0.2]), null=null)
    elif entry == "fill":
        args = dict(max_edges=pick([3, 8, 22, 22, 23, 64, 1024, 2]), null=null)
    elif entry == "repair":
        args = dict(flags=pick([1, 2, 3, 3, 0, 4]), null=null)
    elif entry in ("orient", "measure"):
        args = dict(null=null)
    elif entry == "add":
        run.add_dev(_parts(rng, 2000, islands=1)[0])
        return
    else:
        stage = pick(list(DEV_STAGES))
        held = run.model.mesh
        mesh = _tiled(held, int(rng.integers(2, 9))) if held is not None and rng.random() < 0.5 else \
            _small(int(rng.integers(1000)))
        run.dev(stage, mesh, **DEV_STAGES[stage][2])
        return
    run.step(entry, args)


@pytest.mark.parametrize("seed", [11, 12, 13])
def test_random_sequences(seed):
    rng = np.random.default_rng(seed)
    run = Run(_ctx())
    _surface_scene(run, seed, n=int(rng.integers(8000, 25000)))
    for _ in range(36):
        _random_step(rng, run)
    print("\n".join(run.log))
    run.close()
