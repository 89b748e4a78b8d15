"""CPU checks of the surface-sequence model (tests/surface_sequence_model.py) that tests/test_gpu_surface_sequences.py
holds a context to: the staleness each entry causes agrees with the dependency table that tests/test_results_host.py
pins against csrc/scan3d_results.h, chains of references keep producing valid meshes whose counts match the result
dicts, and every scripted sequence runs to completion with the return codes the header's rules give."""
import itertools

import numpy as np
import pytest

import surface_sequence_model as sm
from surface_sequence_model import ARG, OK, STATE, SurfaceModel
from test_results_host import DOWNSTREAM, ENTRY
from test_surface_math_host import random_model, sphere_model

F32 = np.float32
S = F32(0.2)


def scene(s=S, r=2.0, cap=0.8):
    """a sphere open above z = cap r, a smaller sphere that touches it, and a rough slab far from both"""
    a = sphere_model(s, r)
    keep = a[0][:, 2] - F32(-0.2) < cap * r
    a = tuple(x[keep] for x in a)
    b = sphere_model(s, 0.45 * r, centre=(0.3 + 1.4 * r, -0.2, 0.1))
    x, n, c, ijk = random_model(np.random.default_rng(1), 120, s)
    slab = ((x + F32(9 * r)).astype(F32), n, c, ijk + np.floor(F32(9 * r) / s).astype(np.int64))
    return sm.voxel_model([a, b, slab])


def _model(voxels=None):
    m = SurfaceModel()
    m.begin(S)
    m.finish(scene() if voxels is None else voxels)
    return m


def _closure(start, ops):
    """the results current after ops on start, by the closure rule of test_results_host"""
    cur = set(start)
    for op, r in ops:
        cur -= DOWNSTREAM[r] | ({r} if op == "drop" else set())
        if op == "produce":
            cur.add(r)
    return cur


def _valid(mesh, res=None):
    xyz, nrm, rgb, faces = mesh
    assert xyz.dtype == nrm.dtype == np.float32 and rgb.dtype == np.uint8 and faces.dtype == np.int32
    assert xyz.shape == nrm.shape == rgb.shape == (len(xyz), 3) and faces.shape == (len(faces), 3)
    assert ((faces >= 0) & (faces < len(xyz))).all()
    if res is not None and "vertices" in res:
        assert (res["vertices"], res["faces"]) == (len(xyz), len(faces))


# the model's entries on the surface, with the ops of test_results_host's ENTRY they must agree with; fill and repair
# drop the component table (the header: they make it stale), orient and measure change nothing
SURFACE_ENTRIES = {
    "extract": ({}, ENTRY["voxel_surface"]),
    "components": (dict(min_faces=0, max_components=0), ENTRY["components"]),
    "decimate": (dict(ratio=2), ENTRY["decimate"]),
    "smooth": (sm.SMOOTH, ENTRY["smooth"]),
    "fill": (dict(max_edges=8), [("drop", "COMPONENTS")]),
    "repair": (dict(flags=sm.BOTH), [("drop", "COMPONENTS")]),
    "orient": ({}, []),
    "measure": ({}, []),
}


def test_staleness_agrees_with_the_dependency_table():
    base = _model()
    base.extract(**sm.resolve(base, "extract", {}))
    held = base.mesh
    optional = ("COMPONENTS", "SIMPLIFIED", "SMOOTHED")
    seen = set()
    for entry, (kw, ops) in SURFACE_ENTRIES.items():
        for k in range(len(optional) + 1):
            for extra in itertools.combinations(optional, k):
                start = {"ACCUMULATOR", "VOXELS", "SURFACE", *extra}
                m = _model(base.voxels)
                m.mesh, m.current = held, set(start)
                _, step = sm.run(m, entry, kw)
                if step.rc == OK:
                    assert m.current == _closure(start, ops), (entry, extra)
                    seen.add(entry)
                else:
                    assert (entry, step.rc) == ("decimate", STATE) and set(extra) & {"SIMPLIFIED", "SMOOTHED"}
                    assert m.current == start and m.mesh is held
    assert seen == set(SURFACE_ENTRIES)
    # the merge's entries, from every state with a surface
    for k in range(len(optional) + 1):
        for extra in itertools.combinations(optional, k):
            start = {"ACCUMULATOR", "VOXELS", "SURFACE", *extra}
            for entry, name, args in (("begin", "voxel_begin", (S,)), ("add", "voxel add", ()),
                                      ("finish", "voxel_finish", (base.voxels,))):
                m = _model(base.voxels)
                m.current = set(start)
                getattr(m, entry)(*args)
                assert m.current == _closure(start, ENTRY[name]), (entry, extra)


def test_every_surface_entry_needs_a_surface():
    m = SurfaceModel()
    assert m.extract(0.4, 100).rc == STATE                             # before begin
    m.begin(S)
    assert m.extract(0.4, 100).rc == STATE                             # before the first finish
    for entry, (kw, _) in SURFACE_ENTRIES.items():
        if entry != "extract":
            assert getattr(m, entry)(**sm.resolve(m, entry, kw)).rc == STATE, entry
    m.finish(scene())
    m.add()
    assert m.extract(0.4, 100).rc == STATE and m.get_surface().rc == STATE


@pytest.mark.parametrize("name", ["LONG_CHAIN", "PARTIAL_SWAPS", "FULL_CHAIN", "ERRORS_MID_CHAIN"])
def test_scripted_sequences_run_on_the_model(name):
    m = _model()
    kw, step = sm.run(m, "extract", {})
    assert step.rc == OK and step.result["faces"] > 1000
    _valid(m.mesh, step.result)
    codes = []
    for entry, args in getattr(sm, name):
        before = (m.mesh, set(m.current), m.table, m.repaired, m.filled_after_repair)
        kw, step = sm.run(m, entry, args)
        codes.append(step.rc)
        assert step.rc in (OK, ARG, STATE), (entry, kw)
        if step.rc != OK:
            assert step.launches == 0 and (m.mesh, m.current, m.table, m.repaired, m.filled_after_repair) == before
            continue
        assert step.launches > 0
        _valid(m.mesh, step.result)
        if entry == "components":
            v, f, kept = m.table                         # the table covers the surface as it was
            assert (v.sum(), f.sum()) == (len(before[0][0]), len(before[0][3])) and len(v) == len(kept)
    if name == "LONG_CHAIN":
        # the smoothed surface is refused, the new extraction simplified
        assert codes == [OK] * 6 + [STATE, OK, OK, OK]
        assert m.current >= {"SURFACE", "SIMPLIFIED"} and "SMOOTHED" not in m.current
    if name == "ERRORS_MID_CHAIN":
        assert codes[-3:] == [ARG, STATE, OK]                      # smoothed: refused after the argument check
        assert codes.count(OK) == 7
    if name == "FULL_CHAIN":
        assert OK in codes and all(c == OK for c in codes)


def test_extraction_resets_the_flags_and_the_decimation_rules():
    m = _model()
    sm.run(m, "extract", {})
    raw = m.mesh
    # a repair that changed the surface, then a fill that added faces: refused until the next extraction
    rep = m.repair(sm.BOTH)
    fil = m.fill(22)
    assert rep.result["faces"] < len(raw[3]) or rep.result["vertices_added"] > 0
    assert fil.result["faces_added"] > 0 and m.repaired and m.filled_after_repair
    assert sm.run(m, "decimate", dict(ratio=4))[1].rc == STATE
    assert m.fill_cap() == 22
    sm.run(m, "extract", {})
    assert not m.repaired and not m.filled_after_repair and m.current == {"ACCUMULATOR", "VOXELS", "SURFACE"}
    assert sm.run(m, "decimate", dict(ratio=4))[1].rc == OK and m.fill_cap() == 1024
    # a fill before the repair leaves it decimatable
    sm.run(m, "extract", {})
    m.fill(22)
    m.repair(sm.BOTH)
    assert sm.run(m, "decimate", dict(ratio=4))[1].rc == OK
    # an extraction that needs more lattice points than max_points leaves no surface
    kw, step = sm.run(m, "extract", {})
    assert m.extract(kw["max_distance"], step.result["lattice_points"] - 1).rc == sm.CONFIG
    assert m.get_surface().rc == STATE and m.get_components().rc == STATE


def test_dev_entries_change_no_state():
    m = _model()
    sm.run(m, "extract", {})
    m.components(0, 0)
    state = (m.mesh, set(m.current), m.table)
    xyz, nrm, _, faces = m.mesh
    assert m.components_dev(faces, len(xyz)).result["components"] == len(m.table[0])
    assert m.smooth_dev(xyz, nrm, faces, **sm.SMOOTH).rc == OK
    assert m.fill_dev(xyz, faces, 1024).rc == OK and m.fill_dev(xyz, faces, 1025).rc == ARG
    assert m.repair_dev(xyz, faces, sm.BOTH).rc == OK and m.repair_dev(xyz, faces, 0).rc == ARG
    assert m.orient_dev(xyz, nrm, faces).rc == OK and m.measure_dev(xyz, faces).rc == OK
    assert (m.mesh, m.current, m.table) == state
