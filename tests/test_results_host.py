"""Which of a context's results are current, s3d::Results (csrc/scan3d_results.h), checked on the CPU:
tests/results_host.cpp is compiled against the header alone.  Each C entry is replayed as the drops and produces it
makes on success, and the whole readiness is checked after every entry of the sequences include/scan3d.h documents."""
import os
import subprocess

import pytest

HERE = os.path.dirname(os.path.abspath(__file__))

PIXEL = ["WRAPPED_V", "WRAPPED_H", "UNWRAPPED_V", "UNWRAPPED_H", "CPMAP", "VALID", "XYZ", "POINTS", "POINT_COLOURS",
         "MESH"]
MODEL = ["ACCUMULATOR", "VOXELS", "SURFACE", "COMPONENTS", "SIMPLIFIED", "SMOOTHED"]
ALL = PIXEL + MODEL

# everything computed from each result, directly or not, written out by hand
DOWNSTREAM = {
    "WRAPPED_V": {"UNWRAPPED_V", "CPMAP", "VALID", "XYZ", "POINTS", "POINT_COLOURS", "MESH"},
    "WRAPPED_H": {"UNWRAPPED_H", "CPMAP", "VALID", "XYZ", "POINTS", "POINT_COLOURS", "MESH"},
    "UNWRAPPED_V": {"CPMAP", "VALID", "XYZ", "POINTS", "POINT_COLOURS", "MESH"},
    "UNWRAPPED_H": {"CPMAP", "VALID", "XYZ", "POINTS", "POINT_COLOURS", "MESH"},
    "CPMAP": {"XYZ", "POINTS", "POINT_COLOURS", "MESH"},
    "VALID": {"XYZ", "POINTS", "POINT_COLOURS", "MESH"},
    "XYZ": {"POINTS", "POINT_COLOURS", "MESH"},
    "POINTS": {"POINT_COLOURS", "MESH"},
    "POINT_COLOURS": set(),
    "MESH": set(),
    "ACCUMULATOR": {"VOXELS", "SURFACE", "COMPONENTS", "SIMPLIFIED", "SMOOTHED"},
    "VOXELS": {"SURFACE", "COMPONENTS", "SIMPLIFIED", "SMOOTHED"},
    "SURFACE": {"COMPONENTS", "SIMPLIFIED", "SMOOTHED"},
    "COMPONENTS": set(),
    "SIMPLIFIED": set(),
    "SMOOTHED": set(),
}


def _d(*names):
    return [("drop", n) for n in names]


def _p(*names):
    return [("produce", n) for n in names]


# The operations of each entry on success, in the order the entry makes them.
ENTRY = {
    "wrapped(0)": _d("WRAPPED_V") + _p("WRAPPED_V"),
    "wrapped(1)": _d("WRAPPED_H") + _p("WRAPPED_H"),
    "unwrap(0)": _d("UNWRAPPED_V") + _p("UNWRAPPED_V"),
    "unwrap(1)": _d("UNWRAPPED_H") + _p("UNWRAPPED_H"),
    "c_p_map": _d("CPMAP", "VALID") + _p("CPMAP", "VALID"),
    "triangulate": _d("XYZ") + _p("XYZ"),
    "compact": _d("POINTS") + _p("POINTS"),
    "compact, texture set": _d("POINTS") + _p("POINTS", "POINT_COLOURS"),
    "reconstruct dirs=2": _d("WRAPPED_V", "WRAPPED_H") + _p("UNWRAPPED_V", "UNWRAPPED_H", "VALID", "CPMAP", "POINTS"),
    "reconstruct dirs=2, texture set": _d("WRAPPED_V", "WRAPPED_H")
    + _p("UNWRAPPED_V", "UNWRAPPED_H", "VALID", "CPMAP", "POINTS", "POINT_COLOURS"),
    "reconstruct dirs=1": _d("WRAPPED_V", "WRAPPED_H") + _p("UNWRAPPED_V", "VALID"),
    "set_points_buffer": _d("POINTS"),
    "align with apply": _d("MESH"),
    "build_mesh": _d("MESH") + _p("MESH"),
    "set_texture(NULL)": _d("POINT_COLOURS"),
    "voxel_begin": _d("ACCUMULATOR") + _p("ACCUMULATOR"),
    "voxel add": _d("VOXELS"),
    "voxel_finish": _d("VOXELS") + _p("VOXELS"),
    "voxel_surface": _d("SURFACE") + _p("SURFACE"),
    "components": _d("COMPONENTS") + _p("COMPONENTS"),
    "decimate": _d("COMPONENTS") + _p("SIMPLIFIED"),
    "smooth": _p("SMOOTHED"),
}
# the stage route of a reconstruct: every pixel result dropped, then the stage entries chained
ENTRY["reconstruct stage route dirs=2"] = _d("WRAPPED_V", "WRAPPED_H") + sum(
    (ENTRY[e] for e in ("wrapped(0)", "unwrap(0)", "wrapped(1)", "unwrap(1)", "c_p_map", "triangulate", "compact")), [])
ENTRY["reconstruct stage route dirs=1"] = (_d("WRAPPED_V", "WRAPPED_H") + ENTRY["wrapped(0)"] + ENTRY["unwrap(0)"]
                                           + _p("VALID"))


@pytest.fixture(scope="module")
def replay(tmp_path_factory):
    exe = str(tmp_path_factory.mktemp("results") / "results_host")
    subprocess.check_call(["/usr/bin/g++", "-O1", "-std=c++17", "-Wall", "-Werror", "-o", exe,
                           os.path.join(HERE, "results_host.cpp")])

    def run(ops):
        args = [f"{op}:{name}" for op, name in ops]
        lines = subprocess.run([exe] + args, capture_output=True, text=True, check=True).stdout.splitlines()
        assert len(lines) == len(ops)
        return [set() if l == "-" else set(l.split()) for l in lines]

    def entries(steps):
        """the readiness after each entry of steps, a list of (entry, readiness expected after it)"""
        ops = sum((ENTRY[e] for e, _ in steps), [])
        states = run(ops)
        k = 0
        for e, want in steps:
            k += len(ENTRY[e])
            assert states[k - 1] == set(want), f"after {e}"

    run.entries = entries
    return run


def test_drop_and_produce_follow_the_closure(replay):
    for r in ALL:
        everything = [("produce", n) for n in ALL]
        # drop: r and everything computed from it
        assert replay(everything + [("drop", r)])[-1] == set(ALL) - {r} - DOWNSTREAM[r], r
        # produce: everything computed from the old r, r itself current
        assert replay(everything + [("produce", r)])[-1] == set(ALL) - DOWNSTREAM[r], r
        assert replay([("produce", r)])[-1] == {r}
        assert replay([("drop", r)])[-1] == set()


def test_stage_entries_in_the_reference_order(replay):
    replay.entries([
        ("wrapped(0)", {"WRAPPED_V"}),
        ("unwrap(0)", {"WRAPPED_V", "UNWRAPPED_V"}),
        ("wrapped(1)", {"WRAPPED_V", "UNWRAPPED_V", "WRAPPED_H"}),
        ("unwrap(1)", {"WRAPPED_V", "UNWRAPPED_V", "WRAPPED_H", "UNWRAPPED_H"}),
        ("c_p_map", {"WRAPPED_V", "UNWRAPPED_V", "WRAPPED_H", "UNWRAPPED_H", "CPMAP", "VALID"}),
        ("triangulate", {"WRAPPED_V", "UNWRAPPED_V", "WRAPPED_H", "UNWRAPPED_H", "CPMAP", "VALID", "XYZ"}),
        ("compact, texture set", set(PIXEL) - {"MESH"}),
        ("build_mesh", set(PIXEL)),
        # new inputs of one direction: the other direction's phases stay, everything merged from both goes
        ("unwrap(1)", {"WRAPPED_V", "UNWRAPPED_V", "WRAPPED_H", "UNWRAPPED_H"}),
        ("c_p_map", {"WRAPPED_V", "UNWRAPPED_V", "WRAPPED_H", "UNWRAPPED_H", "CPMAP", "VALID"}),
        ("wrapped(0)", {"WRAPPED_V", "WRAPPED_H", "UNWRAPPED_H"}),
    ])


def test_single_pass_reconstruct(replay):
    after = {"UNWRAPPED_V", "UNWRAPPED_H", "CPMAP", "VALID", "POINTS"}
    replay.entries([
        ("wrapped(0)", {"WRAPPED_V"}),
        ("reconstruct dirs=2", after),                 # the wrapped phases and masks stay in registers
        ("build_mesh", after | {"MESH"}),
        ("reconstruct dirs=2, texture set", after | {"POINT_COLOURS"}),
        # a stage entry after it: VALID goes, the other direction's unwrapped phase stays
        ("wrapped(0)", {"WRAPPED_V", "UNWRAPPED_H"}),
        ("unwrap(0)", {"WRAPPED_V", "UNWRAPPED_V", "UNWRAPPED_H"}),
        ("c_p_map", {"WRAPPED_V", "UNWRAPPED_V", "UNWRAPPED_H", "CPMAP", "VALID"}),
    ])
    replay.entries([("reconstruct dirs=1", {"UNWRAPPED_V", "VALID"})])


def test_stage_route_of_a_reconstruct(replay):
    replay.entries([
        ("reconstruct dirs=2", {"UNWRAPPED_V", "UNWRAPPED_H", "CPMAP", "VALID", "POINTS"}),
        ("build_mesh", {"UNWRAPPED_V", "UNWRAPPED_H", "CPMAP", "VALID", "POINTS", "MESH"}),
        ("reconstruct stage route dirs=2", set(PIXEL) - {"POINT_COLOURS", "MESH"}),
    ])
    replay.entries([("reconstruct stage route dirs=1", {"WRAPPED_V", "UNWRAPPED_V", "VALID"})])


def test_points_colours_and_mesh(replay):
    points = {"UNWRAPPED_V", "UNWRAPPED_H", "CPMAP", "VALID", "POINTS"}
    replay.entries([
        # set_texture(A), reconstruct: the points carry A's colours
        ("reconstruct dirs=2, texture set", points | {"POINT_COLOURS"}),
        ("build_mesh", points | {"POINT_COLOURS", "MESH"}),
        # the points move, their colours stay theirs
        ("align with apply", points | {"POINT_COLOURS"}),
        ("build_mesh", points | {"POINT_COLOURS", "MESH"}),
        ("set_texture(NULL)", points | {"MESH"}),
        # reconstruct without a texture, then set_texture(B): B colours no point computed before it
        ("reconstruct dirs=2", points),
        ("build_mesh", points | {"MESH"}),
        ("set_points_buffer", points - {"POINTS"}),
    ])
    replay.entries([
        ("wrapped(0)", {"WRAPPED_V"}), ("unwrap(0)", {"WRAPPED_V", "UNWRAPPED_V"}),
        ("wrapped(1)", {"WRAPPED_V", "UNWRAPPED_V", "WRAPPED_H"}),
        ("unwrap(1)", {"WRAPPED_V", "UNWRAPPED_V", "WRAPPED_H", "UNWRAPPED_H"}),
        ("c_p_map", {"WRAPPED_V", "UNWRAPPED_V", "WRAPPED_H", "UNWRAPPED_H", "CPMAP", "VALID"}),
        ("triangulate", set(PIXEL) - {"POINTS", "POINT_COLOURS", "MESH"}),
        ("compact", set(PIXEL) - {"POINT_COLOURS", "MESH"}),
        ("build_mesh", set(PIXEL) - {"POINT_COLOURS"}),
        ("compact, texture set", set(PIXEL) - {"MESH"}),
        ("triangulate", set(PIXEL) - {"POINTS", "POINT_COLOURS", "MESH"}),
    ])


def test_model_stages(replay):
    acc, vox = {"ACCUMULATOR"}, {"ACCUMULATOR", "VOXELS"}
    srf = vox | {"SURFACE"}
    replay.entries([
        ("voxel_begin", acc),
        ("voxel add", acc),
        ("voxel add", acc),
        ("voxel_finish", vox),
        ("voxel_surface", srf),
        ("components", srf | {"COMPONENTS"}),
        ("smooth", srf | {"COMPONENTS", "SMOOTHED"}),
        ("components", srf | {"COMPONENTS", "SMOOTHED"}),     # components keep the smoothing
        ("voxel_surface", srf),                                # a new extraction: neither simplified nor smoothed
        ("components", srf | {"COMPONENTS"}),
        ("decimate", srf | {"SIMPLIFIED"}),                    # the component table is stale
        ("components", srf | {"SIMPLIFIED", "COMPONENTS"}),
        ("smooth", srf | {"SIMPLIFIED", "COMPONENTS", "SMOOTHED"}),
        ("components", srf | {"SIMPLIFIED", "COMPONENTS", "SMOOTHED"}),
        # the pixel path does not touch the model, and the model does not touch the points
        ("reconstruct dirs=2", srf | {"SIMPLIFIED", "COMPONENTS", "SMOOTHED", "UNWRAPPED_V", "UNWRAPPED_H", "CPMAP",
                                      "VALID", "POINTS"}),
        ("voxel add", acc | {"UNWRAPPED_V", "UNWRAPPED_H", "CPMAP", "VALID", "POINTS"}),
    ])
    full = ["voxel_begin", "voxel_finish", "voxel_surface", "decimate", "components", "smooth"]
    for last, want in (("voxel add", acc), ("voxel_finish", vox), ("voxel_begin", acc)):
        states = replay(sum((ENTRY[e] for e in full + [last]), []))
        assert states[-len(ENTRY[last]) - 1] == srf | {"SIMPLIFIED", "COMPONENTS", "SMOOTHED"}
        assert states[-1] == want, last
