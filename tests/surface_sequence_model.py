"""A numpy model of one context's voxel-model state, for sequences of surface calls.

SurfaceModel mirrors what include/scan3d.h says a context holds between calls: the held voxel surface, the component
table, which of the model results are current (VOXELS, SURFACE, COMPONENTS, SIMPLIFIED, SMOOTHED, and ACCUMULATOR, which
begin makes current), and the two facts since the last extraction that the decimation's rules read: a repair or an
orientation changed the surface, and a fill added faces after that.  Every entry returns a Step: the return code the
header promises, the result dict, and the launches it makes; the state changes only when the header says so.  The
surface is always computed by the references (extract_ref, labels_ref / keep_ref / compact_ref, decimate_ref, smooth_ref,
fill_ref, repair_ref, orient_ref, measure_ref) from the model's own previous surface, never from a GPU's.  The voxel
outputs a finish produces are an input here: the merge has its own tests.

The rules are written from the header's text, one entry at a time; tests/test_surface_sequence_model.py checks the
staleness they imply against the dependency table of tests/test_results_host.py."""
import math
from dataclasses import dataclass, field

import numpy as np

from test_components_ref import compact_ref, keep_ref, labels_ref
from test_decimate_ref import decimate_ref
from test_fill_ref import fill_ref, polygon_faces_ref
from test_orient_ref import measure_ref, orient_ref
from test_repair_ref import FACES, VERTICES, apply_source, repair_ref
from test_smooth_ref import passes_of, smooth_ref
from test_surface_math_host import extract_ref

F32, F64 = np.float32, np.float64
OK, CONFIG, STATE, ARG = 0, -1, -3, -4
FILL_NETS_MAX_EDGES, FILL_MAX_EDGES = 22, 1024
SMOOTH_MAX_ITERATIONS = 4096
RATIO_MAX = 256

# launches of each entry when it succeeds (include/scan3d.h); an argument or state error launches nothing
EXTRACT_LAUNCHES = 3 + 8 + 1
COMPONENTS_LAUNCHES, COMPONENTS_DEV_LAUNCHES = 16, 7
DECIMATE_LAUNCHES = 12
FILL_LAUNCHES = 10
REPAIR_LAUNCHES = 12
ORIENT_LAUNCHES, MEASURE_LAUNCHES = 8, 7


def smooth_launches(iterations, mu):
    return 7 + passes_of(iterations, mu) + 2



@dataclass
class Step:
    rc: int
    result: dict = None
    launches: int = 0
    out: tuple = None          # what a _dev entry writes to caller memory


def _finite(x):
    return math.isfinite(float(x))


@dataclass
class SurfaceModel:
    polygon: object = polygon_faces_ref        # one hole's triangulation for fill_ref
    current: set = field(default_factory=set)
    voxel_size: float = None                   # of the last begin, as a float32
    voxels: tuple = None                       # (xyz, normals, rgb, merge indices) of the last finish
    mesh: tuple = None                         # (xyz, normals, rgb, faces) of the held surface
    table: tuple = None                        # (vertices, faces, kept) per component of the last components call
    repaired: bool = False                     # since the extraction: a repair or an orientation changed the surface
    filled_after_repair: bool = False          # ... and a fill added faces after that

    # ---- the merge: begin, add and finish -------------------------------------------------------------------------
    def begin(self, voxel_size):
        """a begin resets the accumulator: the voxel outputs, the surface and all computed from it are stale"""
        self.current = {"ACCUMULATOR"}
        self.voxel_size = F32(voxel_size)
        return Step(OK)

    def add(self):
        """an add makes the voxel outputs of the last finish stale, and with them the surface"""
        self.current &= {"ACCUMULATOR"}
        return Step(OK)

    def finish(self, voxels):
        """new voxel outputs: the surface of the old ones is stale"""
        self.current = {"ACCUMULATOR", "VOXELS"}
        self.voxels = voxels
        return Step(OK)

    # ---- the getters ------------------------------------------------------------------------------------------------
    def get_surface(self):
        return Step(OK if "SURFACE" in self.current else STATE)

    def get_components(self):
        return Step(OK if "COMPONENTS" in self.current else STATE)

    # ---- the surface route ------------------------------------------------------------------------------------------
    def extract(self, max_distance, max_points, null=False):
        if null or not (_finite(max_distance) and max_distance > 0) or not 1 <= max_points < 2 ** 31:
            return Step(ARG)
        if "VOXELS" not in self.current:
            return Step(STATE)
        # a new extraction: neither simplified nor smoothed, no component table, nothing repaired or filled
        self.current -= {"SURFACE", "COMPONENTS", "SIMPLIFIED", "SMOOTHED"}
        self.repaired = self.filled_after_repair = False
        xyz, nrm, rgb, ijk = self.voxels
        vx, vn, vr, faces, lattice, undefined = extract_ref(xyz, nrm, rgb, ijk, self.voxel_size, F32(max_distance))
        if lattice > max_points:                 # found on the device: the counting launches ran, no surface
            return Step(CONFIG, launches=EXTRACT_LAUNCHES - 1)
        self.mesh = (vx, vn, vr, faces)
        self.current.add("SURFACE")
        return Step(OK, dict(vertices=len(vx), faces=len(faces), lattice_points=lattice, undefined_points=undefined),
                    EXTRACT_LAUNCHES)

    def components(self, min_faces, max_components, null=False):
        if null or min_faces < 0 or max_components < 0:
            return Step(ARG)
        if "SURFACE" not in self.current:
            return Step(STATE)
        xyz, _, _, faces = self.mesh
        labels, c = labels_ref(faces, len(xyz))
        vcount, fcount, kept = keep_ref(labels, faces, c, min_faces, max_components)
        self.mesh = compact_ref(self.mesh, labels, kept)
        self.table = (vcount, fcount, kept)
        # the table is of the surface as it is now; whether it was simplified or smoothed stays
        self.current.add("COMPONENTS")
        return Step(OK, dict(components=c, kept=int(kept.sum()), vertices=len(self.mesh[0]), faces=len(self.mesh[3]),
                             largest_faces=int(fcount.max(initial=0))), COMPONENTS_LAUNCHES)

    def decimate(self, cell_size, null=False):
        if null or not _finite(cell_size):
            return Step(ARG)
        if "SURFACE" not in self.current:
            return Step(STATE)
        H, s = F64(F32(cell_size)), F64(self.voxel_size)
        if not (s <= H <= RATIO_MAX * s):
            return Step(ARG)
        # simplified once; never a smoothed surface; never one filled after a repair changed it
        if self.current & {"SIMPLIFIED", "SMOOTHED"} or self.filled_after_repair:
            return Step(STATE)
        out = decimate_ref(self.mesh, self.voxel_size, F32(cell_size))
        self.mesh = out[:4]
        self.current.discard("COMPONENTS")
        self.current.add("SIMPLIFIED")
        return Step(OK, dict(vertices=len(out[0]), faces=len(out[3]), collapsed_faces=out[4], duplicate_faces=out[5],
                             mean_fallbacks=out[6]), DECIMATE_LAUNCHES)

    @staticmethod
    def _smooth_args(iterations, lam, mu):
        lam, mu = F32(lam), F32(mu)
        return 0 <= iterations <= SMOOTH_MAX_ITERATIONS and 0 < lam <= 1 and -1 <= mu <= 0

    def smooth(self, iterations, lam, mu, null=False):
        if null or not self._smooth_args(iterations, lam, mu):
            return Step(ARG)
        if "SURFACE" not in self.current:
            return Step(STATE)
        xyz, nrm, rgb, faces = self.mesh
        out, onrm, info = smooth_ref(xyz, nrm, faces, iterations, lam, mu)
        # faces, colours and the vertex order stay: the component table stays current
        self.mesh = (out, onrm, rgb, faces)
        self.current.add("SMOOTHED")
        return Step(OK, info, smooth_launches(iterations, mu))

    def fill_cap(self):
        """the largest max_edges: a surface neither simplified nor smoothed stays decimatable only with small holes"""
        return FILL_MAX_EDGES if self.current & {"SIMPLIFIED", "SMOOTHED"} else FILL_NETS_MAX_EDGES

    def fill(self, max_edges, null=False):
        if null:
            return Step(ARG)
        if "SURFACE" not in self.current:
            return Step(STATE)
        if not 3 <= max_edges <= self.fill_cap():
            return Step(ARG)
        xyz, nrm, rgb, faces = self.mesh
        add, info = fill_ref(xyz, faces, max_edges, self.polygon)
        self.mesh = (xyz, nrm, rgb, np.concatenate([faces, add]).astype(np.int32))
        self.current.discard("COMPONENTS")
        if len(add) and self.repaired:
            self.filled_after_repair = True
        return Step(OK, info, FILL_LAUNCHES)

    def repair(self, flags, null=False):
        if null or flags <= 0 or flags & ~(FACES | VERTICES):
            return Step(ARG)
        if "SURFACE" not in self.current:
            return Step(STATE)
        xyz, nrm, rgb, faces = self.mesh
        out, src, info = repair_ref(xyz, faces, flags)
        self.mesh = (apply_source(xyz, src), apply_source(nrm, src), np.concatenate([rgb, rgb[src]]), out)
        # the vertex count can change: the table is stale; simplified and smoothed stay as they were
        self.current.discard("COMPONENTS")
        if info["faces"] < len(faces) or len(src):
            self.repaired = True
        return Step(OK, info, REPAIR_LAUNCHES)

    def orient(self, null=False):
        if null:
            return Step(ARG)
        if "SURFACE" not in self.current:
            return Step(STATE)
        xyz, nrm, rgb, faces = self.mesh
        out, onrm, info = orient_ref(xyz, faces, nrm)
        self.mesh = (xyz, onrm, rgb, out)
        # the component table stays current; flips count as a repair that changed the surface
        if info["flipped_faces"]:
            self.repaired = True
        return Step(OK, info, ORIENT_LAUNCHES)

    def measure(self, null=False):
        if null:
            return Step(ARG)
        if "SURFACE" not in self.current:
            return Step(STATE)
        return Step(OK, measure_ref(self.mesh[0], self.mesh[3]), MEASURE_LAUNCHES)

    # ---- the _dev routes: any mesh in caller memory; they change no state -------------------------------------------
    @staticmethod
    def _mesh_args(n_vertices, n_faces):
        return 0 <= n_vertices < 2 ** 31 and 0 <= n_faces < 2 ** 31

    def components_dev(self, faces, n_vertices):
        if not self._mesh_args(n_vertices, len(faces)):
            return Step(ARG)
        labels, c = labels_ref(faces, n_vertices)
        return Step(OK, dict(components=c), COMPONENTS_DEV_LAUNCHES, (labels,))

    def smooth_dev(self, xyz, normals, faces, iterations, lam, mu):
        if not self._smooth_args(iterations, lam, mu) or not self._mesh_args(len(xyz), len(faces)):
            return Step(ARG)
        out, onrm, info = smooth_ref(xyz, normals, faces, iterations, lam, mu)
        return Step(OK, info, smooth_launches(iterations, mu), (out, onrm))

    def fill_dev(self, xyz, faces, max_edges):
        if not 3 <= max_edges <= FILL_MAX_EDGES or not self._mesh_args(len(xyz), len(faces)):
            return Step(ARG)
        add, info = fill_ref(xyz, faces, max_edges, self.polygon)
        return Step(OK, info, FILL_LAUNCHES, (add,))

    def repair_dev(self, xyz, faces, flags):
        if flags <= 0 or flags & ~(FACES | VERTICES) or not self._mesh_args(len(xyz), len(faces)):
            return Step(ARG)
        out, src, info = repair_ref(xyz, faces, flags)
        return Step(OK, info, REPAIR_LAUNCHES, (out, src))

    def orient_dev(self, xyz, normals, faces):
        if not self._mesh_args(len(xyz), len(faces)):
            return Step(ARG)
        out, onrm, info = orient_ref(xyz, faces, normals)
        return Step(OK, info, ORIENT_LAUNCHES, (out, onrm))

    def measure_dev(self, xyz, faces):
        if not self._mesh_args(len(xyz), len(faces)):
            return Step(ARG)
        return Step(OK, measure_ref(xyz, faces), MEASURE_LAUNCHES)


# ---- scripted sequences of surface entries -------------------------------------------------------------------------
# (entry, arguments); decimate takes cell_size as a multiple of the voxel size (ratio), extract defaults to
# max_distance = 2 voxel_size and 64 lattice points per voxel (always enough: a voxel's 27 cells have 64 corners)
SMOOTH = dict(iterations=10, lam=0.5, mu=-0.53)
BOTH = FACES | VERTICES

# every stage in the recommended order, then a decimation the rules refuse, a new extraction and one they accept
LONG_CHAIN = [("smooth", SMOOTH), ("components", dict(min_faces=0, max_components=1)), ("fill", dict(max_edges=1024)),
              ("repair", dict(flags=BOTH)), ("orient", {}), ("measure", {}), ("decimate", dict(ratio=4)),
              ("extract", {}), ("decimate", dict(ratio=4)), ("measure", {})]

# smoothing swaps only the positions and normals with the spare set, filling only the faces: alternate them so the
# held and spare sets hold buffers of different generations, then swap whole sets
PARTIAL_SWAPS = [("fill", dict(max_edges=8)), ("smooth", SMOOTH), ("fill", dict(max_edges=22)),
                 ("smooth", dict(iterations=3, lam=0.7, mu=-0.72)), ("fill", dict(max_edges=1024)),
                 ("smooth", dict(iterations=5, lam=0.3, mu=0.0)), ("components", dict(min_faces=1, max_components=0)),
                 ("repair", dict(flags=BOTH)), ("smooth", dict(iterations=1, lam=1.0, mu=-1.0))]

# the full chain after a new extraction
FULL_CHAIN = [("components", dict(min_faces=1, max_components=0)), ("repair", dict(flags=BOTH)), ("orient", {}),
              ("decimate", dict(ratio=2)), ("repair", dict(flags=BOTH)), ("fill", dict(max_edges=1024)),
              ("smooth", SMOOTH), ("components", dict(min_faces=0, max_components=2)), ("measure", {})]

NAN = float("nan")
# argument and state errors between valid calls: each must leave the state as it was and launch nothing
ERRORS_MID_CHAIN = [
    ("components", dict(min_faces=0, max_components=0)),
    ("components", dict(min_faces=-1, max_components=0)), ("components", dict(min_faces=0, max_components=-1)),
    ("components", dict(min_faces=0, max_components=0, null=True)),
    ("decimate", dict(ratio=0.5)), ("decimate", dict(ratio=257)), ("decimate", dict(cell_size=NAN)),
    ("decimate", dict(cell_size=float("inf"))), ("decimate", dict(ratio=4, null=True)),
    ("fill", dict(max_edges=2)), ("fill", dict(max_edges=23)), ("fill", dict(max_edges=-5)),
    ("fill", dict(max_edges=22, null=True)),
    ("smooth", dict(SMOOTH, iterations=-1)), ("smooth", dict(SMOOTH, iterations=4097)), ("smooth", dict(SMOOTH, lam=0.0)),
    ("smooth", dict(SMOOTH, lam=1.5)), ("smooth", dict(SMOOTH, lam=NAN)), ("smooth", dict(SMOOTH, mu=0.1)),
    ("smooth", dict(SMOOTH, mu=-1.5)), ("smooth", dict(SMOOTH, mu=NAN)), ("smooth", dict(SMOOTH, null=True)),
    ("repair", dict(flags=0)), ("repair", dict(flags=4)), ("repair", dict(flags=-1)), ("repair", dict(flags=BOTH, null=True)),
    ("orient", dict(null=True)), ("measure", dict(null=True)),
    ("extract", dict(max_distance=0.0)), ("extract", dict(max_distance=NAN)), ("extract", dict(max_points=0)),
    ("extract", dict(max_points=2 ** 31)), ("extract", dict(null=True)),
    ("fill", dict(max_edges=22)),                          # valid: the cap of an unrefined surface
    ("repair", dict(flags=BOTH)),
    ("smooth", SMOOTH),
    ("decimate", dict(ratio=4)),                           # refused: smoothed
    ("fill", dict(max_edges=1025)), ("fill", dict(max_edges=1024)),
    ("components", dict(min_faces=-3, max_components=1)),
    ("components", dict(min_faces=1, max_components=1)),
    ("decimate", dict(ratio=0.5)),                         # the argument error comes first
    ("decimate", dict(ratio=4)),
    ("measure", {}),
]


def resolve(model, entry, kw):
    """the concrete arguments of a scripted step for the model's state (the voxel size of the last begin)"""
    kw = dict(kw)
    s = model.voxel_size
    if entry == "decimate" and "ratio" in kw:
        kw["cell_size"] = float(F32(kw.pop("ratio") * s))
    if entry == "extract":
        kw.setdefault("max_distance", float(F32(2 * s)))
        kw.setdefault("max_points", min(max(64 * len(model.voxels[0]), 1), 2 ** 31 - 1))
    return kw


def run(model, entry, kw):
    """one scripted step on the model: (concrete arguments, Step)"""
    kw = resolve(model, entry, kw)
    return kw, getattr(model, entry)(**kw)


def voxel_model(parts):
    """the voxel outputs (xyz, normals, rgb, merge indices) of pieces already merged, each (xyz, normals, rgb, ijk):
    concatenated, a voxel that a later piece repeats kept at its first place"""
    xyz, nrm, rgb, ijk = (np.concatenate(a) for a in zip(*parts))
    _, first = np.unique(ijk, axis=0, return_index=True)
    first = np.sort(first)
    return xyz[first], nrm[first], rgb[first], ijk[first]
