"""scan3d-b200: B200-native reconstruction hot path of pranavkantgaur/3dscan.

Thin ctypes binding over the two in-tree native libraries:

  lib/libscan3d.so       CUDA kernels + the C ABI of include/scan3d.h (the product)
  lib/libscan3d_host.so  C++ host side: file formats, synthetic captures (include/scan3d_host.h)

There is no Python or CPU compute path: if libscan3d.so is missing or no CUDA device is usable,
every compute call raises.  (The package directory name starts with a digit; import it with
importlib.import_module("3dscan_b200").)
"""
import ctypes as C
import math
import os

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
_LIBDIR = os.environ.get("SCAN3D_LIBDIR") or os.path.join(_HERE, "lib")   # override: a trace-enabled build (tools/trace_fused.py)

# ---- scan3d_plane ----
PLANE_WRAPPED_V, PLANE_WRAPPED_H, PLANE_UNWRAPPED_V, PLANE_UNWRAPPED_H = 0, 1, 2, 3
PLANE_CODE_V, PLANE_CODE_H, PLANE_MASK, PLANE_VALID, PLANE_CPMAP, PLANE_XYZ = 4, 5, 6, 7, 8, 9
PLANE_MASK_H = 10
FLAG_POINT_PIXELS = 1
FLAG_FAST_TRIANGULATION = 2
FLAG_MODULATION_MASK = 4
FLAG_STRICT_REFERENCE = 8

_PLANE_DTYPE = {
    PLANE_WRAPPED_V: (np.float32, ()), PLANE_WRAPPED_H: (np.float32, ()),
    PLANE_UNWRAPPED_V: (np.float32, ()), PLANE_UNWRAPPED_H: (np.float32, ()),
    PLANE_CODE_V: (np.int16, ()), PLANE_CODE_H: (np.int16, ()),
    PLANE_MASK: (np.uint8, ()), PLANE_MASK_H: (np.uint8, ()), PLANE_VALID: (np.uint8, ()),
    PLANE_CPMAP: (np.int32, (2,)), PLANE_XYZ: (np.float64, (3,)),
}


class Config(C.Structure):
    _fields_ = [(n, C.c_int32) for n in
                ("W", "H", "PW", "PH", "N", "M_v", "M_h", "fw_v", "fw_h", "dirs", "row0", "H_total")]
    _fields_ += [("flags", C.c_uint32)]


class Calib(C.Structure):
    _fields_ = [("Kc", C.c_double * 9), ("dc", C.c_double * 5), ("Kp", C.c_double * 9),
                ("dp", C.c_double * 5), ("rc", C.c_double * 3), ("tc", C.c_double * 3),
                ("rp", C.c_double * 3), ("tp", C.c_double * 3)]


class SynthParams(C.Structure):
    _fields_ = [("sphere_c", C.c_double * 3), ("sphere_r", C.c_double), ("plane_z", C.c_double),
                ("albedo_lo", C.c_double), ("albedo_hi", C.c_double), ("ambient_max", C.c_double),
                ("noise_sigma", C.c_double), ("roi_fraction", C.c_double), ("true_pi", C.c_int32),
                ("projector_pixelated", C.c_int32), ("seed", C.c_uint64)]


class AlignParams(C.Structure):
    _fields_ = [("T_init", C.c_double * 16), ("max_distance", C.c_float), ("max_iterations", C.c_int32),
                ("stride", C.c_int32), ("stop_rotation", C.c_double), ("stop_translation", C.c_double),
                ("apply", C.c_int32)]


class AlignResultC(C.Structure):
    _fields_ = [("T", C.c_double * 16), ("iterations", C.c_int32), ("status", C.c_int32),
                ("pairs_first", C.c_int64), ("pairs_last", C.c_int64), ("rms_first", C.c_double),
                ("rms_last", C.c_double)]


class AlignResult:
    """scan3d_align_result: T (4x4 float64, p_model = T p_source), iterations, status (0 converged, 1 iteration
    limit, 2 too few pairs / singular system), pairs_first / pairs_last, rms_first / rms_last."""

    def __init__(self, r):
        self.T = np.array(list(r.T), np.float64).reshape(4, 4)
        self.iterations, self.status = r.iterations, r.status
        self.pairs_first, self.pairs_last = r.pairs_first, r.pairs_last
        self.rms_first, self.rms_last = r.rms_first, r.rms_last

    def __repr__(self):
        return (f"AlignResult(status={self.status}, iterations={self.iterations}, pairs={self.pairs_first}->"
                f"{self.pairs_last}, rms={self.rms_first:.6g}->{self.rms_last:.6g})")


class SurfaceParams(C.Structure):
    _fields_ = [("max_distance", C.c_float), ("max_points", C.c_int64)]


class SurfaceResultC(C.Structure):
    _fields_ = [("vertices", C.c_int64), ("faces", C.c_int64), ("lattice_points", C.c_int64),
                ("undefined_points", C.c_int64)]


class ComponentsParams(C.Structure):
    _fields_ = [("min_faces", C.c_int64), ("max_components", C.c_int64)]


class ComponentsResultC(C.Structure):
    _fields_ = [("components", C.c_int64), ("kept", C.c_int64), ("vertices", C.c_int64), ("faces", C.c_int64),
                ("largest_faces", C.c_int64)]


class DecimateResultC(C.Structure):
    _fields_ = [("vertices", C.c_int64), ("faces", C.c_int64), ("collapsed_faces", C.c_int64),
                ("duplicate_faces", C.c_int64), ("mean_fallbacks", C.c_int64)]


class SmoothParams(C.Structure):
    _fields_ = [("iterations", C.c_int32), ("lam", C.c_float), ("mu", C.c_float)]


class SmoothResultC(C.Structure):
    _fields_ = [("vertices", C.c_int64), ("faces", C.c_int64), ("held_vertices", C.c_int64),
                ("isolated_vertices", C.c_int64), ("passes", C.c_int64), ("max_displacement", C.c_double)]


class FillResultC(C.Structure):
    _fields_ = [("vertices", C.c_int64), ("faces", C.c_int64), ("boundary_edges", C.c_int64), ("holes", C.c_int64),
                ("filled", C.c_int64), ("faces_added", C.c_int64), ("open_edges", C.c_int64)]


# the largest hole scan3d_voxel_surface_fill_holes accepts on a surface that is neither simplified nor smoothed (which
# stays decimatable after the fill), and on any other mesh (include/scan3d.h)
FILL_NETS_MAX_EDGES = 22
FILL_MAX_EDGES = 1024


class RepairResultC(C.Structure):
    _fields_ = [(name, C.c_int64) for name in (
        "vertices", "faces", "degenerate_faces", "duplicate_faces", "nonmanifold_edges", "nonmanifold_faces",
        "split_vertices", "vertices_added", "boundary_edges", "inconsistent_edges")]


class OrientResultC(C.Structure):
    _fields_ = [(name, C.c_int64) for name in (
        "vertices", "faces", "degenerate_faces", "patches", "closed_patches", "nonorientable_patches", "flipped_faces",
        "flipped_normals", "inconsistent_edges_before", "inconsistent_edges")]


class MeasureResultC(C.Structure):
    _fields_ = [(name, C.c_int64) for name in (
        "vertices", "faces", "degenerate_faces", "patches", "closed_patches", "nonorientable_patches",
        "unreferenced_vertices", "edges", "boundary_edges", "nonmanifold_edges", "inconsistent_edges",
        "euler_characteristic", "watertight")] + [
        ("area", C.c_double), ("volume", C.c_double), ("bbox_min", C.c_float * 3), ("bbox_max", C.c_float * 3)]


class DistanceParams(C.Structure):
    _fields_ = [("max_distance", C.c_float)]


class DistanceResultC(C.Structure):
    _fields_ = [(name, C.c_int64) for name in ("samples", "matched", "invalid", "inside", "max_sample")] + [
        ("max", C.c_double), ("mean", C.c_double), ("rms", C.c_double), ("min_signed", C.c_float),
        ("max_signed", C.c_float), ("entries", C.c_int64)]


# the steps of scan3d_voxel_surface_repair and scan3d_mesh_repair_dev (include/scan3d.h)
REPAIR_FACES = 1
REPAIR_VERTICES = 2


# voxel_surface's default max_points per merged voxel: the smallest power of two >= 1.5x the largest lattice points
# per voxel measured on tools/bench_surface.py's workloads (29.2 on workload A, profiles/r3_bench_surface.json).  64 is
# also the most a voxel can add (the 4 x 4 x 4 corners of its 27 cells), so the default never overflows; pass
# max_points from a previous result's lattice_points to hold less memory.
SURFACE_POINTS_PER_VOXEL = 64


class Scan3DError(RuntimeError):
    pass


def make_config(W, H, PW=0, PH=0, N=3, M_v=1, M_h=1, fw_v=1, fw_h=1, dirs=2, row0=0, H_total=0,
                flags=0):
    return Config(W, H, PW, PH, N, M_v, M_h, fw_v, fw_h, dirs, row0, H_total or H, flags)


def make_calib(Kc, dc, Kp, dp, rc, tc, rp, tp):
    cal = Calib()
    for name, val, n in (("Kc", Kc, 9), ("dc", dc, 5), ("Kp", Kp, 9), ("dp", dp, 5),
                         ("rc", rc, 3), ("tc", tc, 3), ("rp", rp, 3), ("tp", tp, 3)):
        a = np.ascontiguousarray(val, np.float64).reshape(-1)
        assert a.size == n, (name, a.size)
        getattr(cal, name)[:] = a.tolist()
    return cal


def calib_to_dict(cal):
    return {k: np.array(list(getattr(cal, k))) for k in ("Kc", "dc", "Kp", "dp", "rc", "tc", "rp", "tp")}


# ------------------------------------------------------------------------------------------
_cuda = None
_host = None


def _load(name):
    path = os.path.join(_LIBDIR, name)
    if not os.path.exists(path):
        raise Scan3DError(
            f"{path} is missing: build it with `python 3dscan_b200/build.py` "
            "(there is no CPU fallback for the CUDA path)")
    return C.CDLL(path)


def cuda_lib():
    """libscan3d.so with argtypes set.  Loading works without a GPU; compute calls do not."""
    global _cuda
    if _cuda is not None:
        return _cuda
    L = _load("libscan3d.so")
    vp, i32, i64 = C.c_void_p, C.c_int, C.c_int64
    L.scan3d_version.restype = i32
    L.scan3d_create.argtypes = [C.POINTER(Config), i32, C.POINTER(vp)]
    L.scan3d_destroy.argtypes = [vp]
    L.scan3d_destroy.restype = None
    L.scan3d_last_error.argtypes = [vp]
    L.scan3d_last_error.restype = C.c_char_p
    L.scan3d_set_stream.argtypes = [vp, vp]
    L.scan3d_sync.argtypes = [vp]
    L.scan3d_set_calibration.argtypes = [vp, C.POINTER(Calib)]
    L.scan3d_get_projection_matrices.argtypes = [vp, vp, vp]
    L.scan3d_set_texture.argtypes = [vp, vp]
    for fn in ("scan3d_compute_wrapped_phase", "scan3d_compute_wrapped_phase_dev",
               "scan3d_unwrap_phase", "scan3d_unwrap_phase_dev"):
        getattr(L, fn).argtypes = [vp, i32, vp, vp]
    L.scan3d_compute_c_p_map.argtypes = [vp]
    L.scan3d_triangulate.argtypes = [vp]
    L.scan3d_compact_points.argtypes = [vp, C.POINTER(i64)]
    L.scan3d_stack_bytes.argtypes = [C.POINTER(Config)]
    L.scan3d_stack_bytes.restype = i64
    L.scan3d_reconstruct.argtypes = [vp, vp, vp, C.POINTER(i64)]
    L.scan3d_reconstruct_dev.argtypes = [vp, vp, vp]
    L.scan3d_plane_bytes.argtypes = [vp, i32]
    L.scan3d_plane_bytes.restype = i64
    L.scan3d_get_plane.argtypes = [vp, i32, vp]
    L.scan3d_device_plane.argtypes = [vp, i32]
    L.scan3d_device_plane.restype = vp
    L.scan3d_get_code_i32.argtypes = [vp, i32, vp]
    L.scan3d_get_cpmap_i64.argtypes = [vp, vp]
    L.scan3d_point_count.argtypes = [vp, C.POINTER(i64)]
    L.scan3d_get_points.argtypes = [vp, vp, vp, vp, i64]
    for fn in ("scan3d_device_points", "scan3d_device_point_pixels", "scan3d_device_point_count"):
        getattr(L, fn).argtypes = [vp]
        getattr(L, fn).restype = vp
    L.scan3d_write_ply.argtypes = [vp, C.c_char_p, i32]
    L.scan3d_write_pcd.argtypes = [vp, C.c_char_p]
    L.scan3d_launch_count.argtypes = [vp]
    L.scan3d_set_points_buffer.argtypes = [vp, vp, i64]
    L.scan3d_pattern_bytes.argtypes = [C.POINTER(Config), i32]
    L.scan3d_pattern_bytes.restype = i64
    L.scan3d_generate_patterns.argtypes = [vp, i32, vp]
    L.scan3d_generate_patterns_dev.argtypes = [vp, i32, vp]
    f32 = C.c_float
    L.scan3d_undistort_frames.argtypes = [vp, i32, vp, i32, vp]
    L.scan3d_undistort_frames_dev.argtypes = [vp, i32, vp, i32, vp]
    L.scan3d_get_undistort_map.argtypes = [vp, i32, vp, vp]
    L.scan3d_roi_fill.argtypes = [vp, vp, vp, vp]
    L.scan3d_roi_fill_dev.argtypes = [vp, vp, vp, vp]
    L.scan3d_register_points.argtypes = [vp, vp, vp, i64, f32, f32, f32, f32]
    L.scan3d_set_registration.argtypes = [vp, i32, f32, f32, f32, f32]
    L.scan3d_set_cta_limit.argtypes = [vp, i32]
    L.scan3d_reconstruct_raw.argtypes = [vp, vp, vp, C.POINTER(i64)]
    L.scan3d_reconstruct_raw_dev.argtypes = [vp, vp, vp]
    L.scan3d_register_points_dev.argtypes = [vp, vp, vp, i64, f32, f32, f32, f32]
    L.scan3d_register_rotation.argtypes = [f32, vp]
    L.scan3d_peer_alloc.argtypes = [i32, i64, C.POINTER(vp), C.c_char_p]
    L.scan3d_peer_free.argtypes = [i32, vp]
    L.scan3d_peer_open.argtypes = [i32, C.c_char_p, C.POINTER(vp)]
    L.scan3d_peer_close.argtypes = [i32, vp]
    L.scan3d_launch_count.restype = i64
    L.scan3d_build_mesh.argtypes = [vp, C.c_float]
    L.scan3d_mesh_face_count.argtypes = [vp, C.POINTER(i64)]
    L.scan3d_get_mesh.argtypes = [vp, vp, vp, i64]
    for fn in ("scan3d_device_mesh_faces", "scan3d_device_point_normals"):
        getattr(L, fn).argtypes = [vp]
        getattr(L, fn).restype = vp
    L.scan3d_write_mesh_ply.argtypes = [vp, C.c_char_p, i32]
    L.scan3d_voxel_begin.argtypes = [vp, C.c_float, i64]
    L.scan3d_voxel_add_points.argtypes = [vp]
    L.scan3d_voxel_add_points_dev.argtypes = [vp, vp, vp, vp, i64]
    L.scan3d_voxel_finish.argtypes = [vp]
    L.scan3d_voxel_count.argtypes = [vp, C.POINTER(i64), C.POINTER(i64)]
    L.scan3d_get_voxels.argtypes = [vp, vp, vp, vp, vp, i64]
    L.scan3d_write_voxel_ply.argtypes = [vp, C.c_char_p, i32]
    L.scan3d_align_to_voxels.argtypes = [vp, C.POINTER(AlignParams), C.POINTER(AlignResultC)]
    L.scan3d_align_to_voxels_dev.argtypes = [vp, vp, i64, C.POINTER(AlignParams), C.POINTER(AlignResultC)]
    L.scan3d_voxel_surface.argtypes = [vp, C.POINTER(SurfaceParams), C.POINTER(SurfaceResultC)]
    L.scan3d_get_voxel_surface.argtypes = [vp, vp, vp, vp, vp, i64, i64]
    L.scan3d_write_voxel_surface_ply.argtypes = [vp, C.c_char_p, i32]
    L.scan3d_voxel_surface_components.argtypes = [vp, C.POINTER(ComponentsParams), C.POINTER(ComponentsResultC)]
    L.scan3d_get_surface_components.argtypes = [vp, vp, vp, vp, i64]
    L.scan3d_mesh_components_dev.argtypes = [vp, vp, i64, i64, vp, C.POINTER(i64)]
    L.scan3d_voxel_surface_decimate.argtypes = [vp, C.c_float, C.POINTER(DecimateResultC)]
    L.scan3d_voxel_surface_smooth.argtypes = [vp, C.POINTER(SmoothParams), C.POINTER(SmoothResultC)]
    L.scan3d_mesh_smooth_dev.argtypes = [vp, vp, vp, i64, vp, i64, C.POINTER(SmoothParams), C.POINTER(SmoothResultC)]
    L.scan3d_voxel_surface_fill_holes.argtypes = [vp, i32, C.POINTER(FillResultC)]
    L.scan3d_mesh_fill_holes_dev.argtypes = [vp, vp, i64, vp, i64, i32, vp, i64, C.POINTER(FillResultC)]
    L.scan3d_voxel_surface_repair.argtypes = [vp, i32, C.POINTER(RepairResultC)]
    L.scan3d_mesh_repair_dev.argtypes = [vp, vp, i64, vp, i64, i32, vp, vp, i64, C.POINTER(RepairResultC)]
    L.scan3d_voxel_surface_orient.argtypes = [vp, C.POINTER(OrientResultC)]
    L.scan3d_mesh_orient_dev.argtypes = [vp, vp, vp, i64, vp, i64, C.POINTER(OrientResultC)]
    L.scan3d_voxel_surface_measure.argtypes = [vp, C.POINTER(MeasureResultC)]
    L.scan3d_mesh_measure_dev.argtypes = [vp, vp, i64, vp, i64, C.POINTER(MeasureResultC)]
    L.scan3d_voxel_surface_distance.argtypes = [vp, C.POINTER(DistanceParams), vp, vp, C.POINTER(DistanceResultC)]
    L.scan3d_voxel_surface_distance_dev.argtypes = [vp, vp, i64, C.POINTER(DistanceParams), vp, vp,
                                                    C.POINTER(DistanceResultC)]
    L.scan3d_mesh_distance_dev.argtypes = [vp, vp, i64, vp, i64, vp, i64, C.POINTER(DistanceParams), vp, vp,
                                           C.POINTER(DistanceResultC)]
    L.scan3d_debug_atan2.argtypes = [vp, vp, vp, vp, i32, i32]
    L.scan3d_debug_divcheck.argtypes = [vp, C.POINTER(C.c_uint64)]
    _cuda = L
    return L


def host_lib():
    global _host
    if _host is not None:
        return _host
    L = _load("libscan3d_host.so")
    vp, i32, i64 = C.c_void_p, C.c_int, C.c_int64
    L.scan3d_read_bmp8.argtypes = [C.c_char_p, C.POINTER(i32), C.POINTER(i32), vp, i64]
    L.scan3d_read_bmp_bgr.argtypes = [C.c_char_p, C.POINTER(i32), C.POINTER(i32), vp, i64]
    L.scan3d_write_bmp8.argtypes = [C.c_char_p, i32, i32, vp]
    L.scan3d_read_cv_matrix.argtypes = [C.c_char_p, C.c_char_p, i32, i32, vp]
    L.scan3d_load_calibration.argtypes = [C.c_char_p, C.POINTER(Calib)]
    L.scan3d_load_captured_set.argtypes = [C.c_char_p, C.POINTER(Config), vp]
    L.scan3d_write_ply_points.argtypes = [C.c_char_p, vp, vp, i64, i32]
    L.scan3d_write_pcd_points.argtypes = [C.c_char_p, vp, vp, i64]
    L.scan3d_host_last_error.restype = C.c_char_p
    L.scan3d_synth_default_params.argtypes = [C.POINTER(SynthParams)]
    L.scan3d_synth_default_params.restype = None
    L.scan3d_synth_stack.argtypes = [C.POINTER(Config), C.POINTER(Calib), C.POINTER(SynthParams), vp, vp, vp, i32]
    L.scan3d_synth_pattern_row.argtypes = [i32, i32, i32, i32, i32, vp]
    L.scan3d_scale_calibration.argtypes = [C.POINTER(Calib), C.c_double, C.c_double, C.POINTER(Calib)]
    L.scan3d_scale_calibration.restype = None
    _host = L
    return L


def _ptr(a):
    if a is None:
        return None
    if isinstance(a, int):
        return C.c_void_p(a)
    return a.ctypes.data_as(C.c_void_p)


# ------------------------------------------------------------------------------------------
# host side helpers
# ------------------------------------------------------------------------------------------
def stack_planes(cfg):
    n = cfg.N + 2 * cfg.M_v
    if cfg.dirs == 2:
        n += cfg.N + 2 * cfg.M_h
    return n


def split_stack(cfg, stack):
    """stack [NF][H][W] -> dict of views fringe_v, gray_v, inv_v (, fringe_h, gray_h, inv_h)."""
    out, o = {}, 0
    for d, key in enumerate(("v", "h")[:cfg.dirs]):
        M = cfg.M_v if d == 0 else cfg.M_h
        out["fringe_" + key] = stack[o:o + cfg.N]; o += cfg.N
        out["gray_" + key] = stack[o:o + M]; o += M
        out["inv_" + key] = stack[o:o + M]; o += M
    return out


def default_synth_params(**kw):
    p = SynthParams()
    host_lib().scan3d_synth_default_params(C.byref(p))
    for k, v in kw.items():
        if k == "sphere_c":
            p.sphere_c[:] = list(v)
        else:
            setattr(p, k, v)
    return p


def synth_stack(cfg, cal, params=None, want_truth=False, threads=0, out=None, roi_out=None):
    """Synthetic captured stack [NF][H][W] u8 + full-frame ROI [H_total][W] u8 (+ truth XYZ)."""
    params = params or default_synth_params()
    nf = stack_planes(cfg)
    stack = out if out is not None else np.empty((nf, cfg.H, cfg.W), np.uint8)
    roi = roi_out if roi_out is not None else np.empty((cfg.H_total or cfg.H, cfg.W), np.uint8)
    truth = np.empty((cfg.H, cfg.W, 3), np.float32) if want_truth else None
    rc = host_lib().scan3d_synth_stack(C.byref(cfg), C.byref(cal), C.byref(params), _ptr(stack),
                                       _ptr(roi), _ptr(truth), threads)
    if rc:
        raise Scan3DError(f"scan3d_synth_stack failed: {rc}")
    return (stack, roi, truth) if want_truth else (stack, roi)


def synth_pattern_row(kind, n_or_m, fw, k, length):
    out = np.empty(length, np.uint8)
    rc = host_lib().scan3d_synth_pattern_row(kind, n_or_m, fw, k, length, _ptr(out))
    if rc:
        raise Scan3DError("scan3d_synth_pattern_row failed")
    return out


def scale_calibration(cal, cam_scale, proj_scale):
    out = Calib()
    host_lib().scan3d_scale_calibration(C.byref(cal), cam_scale, proj_scale, C.byref(out))
    return out


def load_calibration(root):
    cal = Calib()
    rc = host_lib().scan3d_load_calibration(root.encode(), C.byref(cal))
    if rc:
        raise Scan3DError(host_lib().scan3d_host_last_error().decode())
    return cal


def load_captured_set(root, cfg):
    stack = np.empty((stack_planes(cfg), cfg.H, cfg.W), np.uint8)
    rc = host_lib().scan3d_load_captured_set(root.encode(), C.byref(cfg), _ptr(stack))
    if rc:
        raise Scan3DError(host_lib().scan3d_host_last_error().decode())
    return stack


def read_bmp8(path):
    w, h = C.c_int(), C.c_int()
    L = host_lib()
    if L.scan3d_read_bmp8(path.encode(), C.byref(w), C.byref(h), None, 0):
        raise Scan3DError(L.scan3d_host_last_error().decode())
    buf = np.empty((h.value, w.value), np.uint8)
    if L.scan3d_read_bmp8(path.encode(), C.byref(w), C.byref(h), _ptr(buf), buf.size):
        raise Scan3DError(L.scan3d_host_last_error().decode())
    return buf


def read_bmp_bgr(path):
    """cvLoadImage(path) in colour: [H][W][3] B,G,R (8/save_point_cloud.cpp:59 loads the texture this way)."""
    w, h = C.c_int(), C.c_int()
    L = host_lib()
    if L.scan3d_read_bmp_bgr(path.encode(), C.byref(w), C.byref(h), None, 0):
        raise Scan3DError(L.scan3d_host_last_error().decode())
    buf = np.empty((h.value, w.value, 3), np.uint8)
    if L.scan3d_read_bmp_bgr(path.encode(), C.byref(w), C.byref(h), _ptr(buf), buf.size):
        raise Scan3DError(L.scan3d_host_last_error().decode())
    return buf


# ------------------------------------------------------------------------------------------
# the context (device side)
# ------------------------------------------------------------------------------------------
class Scan3D:
    """One reconstruction context = one GPU, one stream, one frame shape (include/scan3d.h)."""

    def __init__(self, cfg, device=0, calib=None, stream=None):
        self.L = cuda_lib()
        self.cfg = cfg
        self.h = C.c_void_p()
        rc = self.L.scan3d_create(C.byref(cfg), device, C.byref(self.h))
        if rc:
            msg = self.L.scan3d_last_error(None).decode()
            raise Scan3DError(f"scan3d_create failed ({rc}): {msg}")
        if stream is not None:
            self._ck(self.L.scan3d_set_stream(self.h, C.c_void_p(stream)))
        if calib is not None:
            self.set_calibration(calib)

    def _ck(self, rc):
        if rc:
            raise Scan3DError(f"scan3d error {rc}: {self.L.scan3d_last_error(self.h).decode()}")

    def close(self):
        if self.h:
            self.L.scan3d_destroy(self.h)
            self.h = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    # -- setup
    def set_stream(self, stream):
        self._ck(self.L.scan3d_set_stream(self.h, C.c_void_p(stream) if stream else None))

    def set_calibration(self, cal):
        self._ck(self.L.scan3d_set_calibration(self.h, C.byref(cal)))

    def projection_matrices(self):
        a, b = np.empty(12), np.empty(12)
        self._ck(self.L.scan3d_get_projection_matrices(self.h, _ptr(a), _ptr(b)))
        return a.reshape(3, 4), b.reshape(3, 4)

    def set_texture(self, bgr):
        self._ck(self.L.scan3d_set_texture(self.h, _ptr(None if bgr is None else np.ascontiguousarray(bgr, np.uint8))))

    def sync(self):
        self._ck(self.L.scan3d_sync(self.h))

    # -- stage entries (host numpy arrays, or ints = device pointers with dev=True)
    def compute_wrapped_phase(self, direction, fringe, roi, dev=False):
        f = self.L.scan3d_compute_wrapped_phase_dev if dev else self.L.scan3d_compute_wrapped_phase
        self._ck(f(self.h, direction, _ptr(fringe), _ptr(roi)))

    def unwrap_phase(self, direction, gray, inv, dev=False):
        f = self.L.scan3d_unwrap_phase_dev if dev else self.L.scan3d_unwrap_phase
        self._ck(f(self.h, direction, _ptr(gray), _ptr(inv)))

    def compute_c_p_map(self):
        self._ck(self.L.scan3d_compute_c_p_map(self.h))

    def triangulate(self):
        self._ck(self.L.scan3d_triangulate(self.h))

    def compact_points(self):
        n = C.c_int64()
        self._ck(self.L.scan3d_compact_points(self.h, C.byref(n)))
        return n.value

    # -- fused entry
    def reconstruct(self, stack, roi):
        n = C.c_int64()
        self._ck(self.L.scan3d_reconstruct(self.h, _ptr(stack), _ptr(roi), C.byref(n)))
        return n.value

    def set_cta_limit(self, ctas_per_sm):
        """several contexts on several streams of one GPU: this context's kernel takes at most that many CTA slots per SM"""
        self._ck(self.L.scan3d_set_cta_limit(self.h, int(ctas_per_sm)))

    def set_registration(self, enable, theta_deg=0.0, tx=0.0, ty=0.0, tz=0.0):
        """register_point_clouds' transform folded into the point store of the following reconstructions."""
        self._ck(self.L.scan3d_set_registration(self.h, int(bool(enable)), theta_deg, tx, ty, tz))

    def reconstruct_raw(self, raw_stack, roi):
        """raw captures (before the capture loop's cvUndistort2) -> (registered) points in one call."""
        raw_stack = np.ascontiguousarray(raw_stack, np.uint8)
        roi = np.ascontiguousarray(roi, np.uint8)
        n = C.c_int64()
        self._ck(self.L.scan3d_reconstruct_raw(self.h, _ptr(raw_stack), _ptr(roi), C.byref(n)))
        return n.value

    def reconstruct_raw_dev(self, stack_ptr, roi_ptr):
        self._ck(self.L.scan3d_reconstruct_raw_dev(self.h, C.c_void_p(stack_ptr), C.c_void_p(roi_ptr)))

    def reconstruct_dev(self, stack_ptr, roi_ptr):
        self._ck(self.L.scan3d_reconstruct_dev(self.h, C.c_void_p(stack_ptr), C.c_void_p(roi_ptr)))

    # -- results
    def plane(self, which):
        dt, tail = _PLANE_DTYPE[which]
        out = np.empty((self.cfg.H, self.cfg.W) + tail, dt)
        self._ck(self.L.scan3d_get_plane(self.h, which, _ptr(out)))
        return out

    def device_plane(self, which):
        return self.L.scan3d_device_plane(self.h, which)

    def code_i32(self, direction):
        out = np.empty((self.cfg.H, self.cfg.W), np.int32)
        self._ck(self.L.scan3d_get_code_i32(self.h, direction, _ptr(out)))
        return out

    def cpmap_i64(self):
        out = np.empty((self.cfg.H * self.cfg.W, 2), np.int64)
        self._ck(self.L.scan3d_get_cpmap_i64(self.h, _ptr(out)))
        return out

    def point_count(self):
        n = C.c_int64()
        self._ck(self.L.scan3d_point_count(self.h, C.byref(n)))
        return n.value

    def points(self, want_pix=False, want_rgb=False):
        n = self.point_count()
        xyz = np.empty((n, 3), np.float32)
        pix = np.empty(n, np.uint32) if want_pix else None
        rgb = np.empty((n, 3), np.uint8) if want_rgb else None
        self._ck(self.L.scan3d_get_points(self.h, _ptr(xyz), _ptr(pix), _ptr(rgb), n))
        out = (xyz,)
        if want_pix:
            out += (pix,)
        if want_rgb:
            out += (rgb,)
        return out if len(out) > 1 else xyz

    def device_points(self):
        return self.L.scan3d_device_points(self.h)

    def device_point_count(self):
        return self.L.scan3d_device_point_count(self.h)

    def generate_patterns(self, direction):
        """generate_pattern() on the GPU: u8 [N + 2M][PH][PW] (fringe, Gray, inverse Gray) of one direction."""
        M = self.cfg.M_v if direction == 0 else self.cfg.M_h
        out = np.empty((self.cfg.N + 2 * M, self.cfg.PH, self.cfg.PW), np.uint8)
        self._ck(self.L.scan3d_generate_patterns(self.h, int(direction), _ptr(out)))
        return out

    def generate_patterns_dev(self, direction, dev_ptr):
        self._ck(self.L.scan3d_generate_patterns_dev(self.h, int(direction), C.c_void_p(dev_ptr)))

    # -- either side of the path (SURVEY.md 8 f2 / f4)
    def _kind_shape(self, device_kind):
        return (self.cfg.H, self.cfg.W) if device_kind == 0 else (self.cfg.PH, self.cfg.PW)

    def undistort_frames(self, frames, device_kind=0):
        """cvUndistort2 of u8 frames [n][H][W] (camera, device_kind 0) or [n][PH][PW] (projector, 1)."""
        frames = np.ascontiguousarray(frames, np.uint8)
        H, W = self._kind_shape(device_kind)
        if frames.ndim != 3 or frames.shape[1:] != (H, W):
            raise Scan3DError(f"frames must be [n][{H}][{W}] u8, got {frames.shape}")
        out = np.empty_like(frames)
        if frames.shape[0] == 0:
            return out
        self._ck(self.L.scan3d_undistort_frames(self.h, int(device_kind), _ptr(frames), frames.shape[0], _ptr(out)))
        return out

    def undistort_frames_dev(self, src_ptr, n_frames, dst_ptr, device_kind=0):
        self._ck(self.L.scan3d_undistort_frames_dev(self.h, int(device_kind), C.c_void_p(src_ptr), int(n_frames),
                                                    C.c_void_p(dst_ptr)))

    def undistort_map(self, device_kind=0):
        """cv::undistort's fixed-point map: (xy int16 [H][W][2], frac uint16 [H][W])."""
        H, W = self._kind_shape(device_kind)
        xy = np.empty((H, W, 2), np.int16)
        fr = np.empty((H, W), np.uint16)
        self._ck(self.L.scan3d_get_undistort_map(self.h, int(device_kind), _ptr(xy), _ptr(fr)))
        return xy, fr

    def roi_fill(self, outline):
        """image_scissor's fill: (selected_region u8 [H_total][W], outline image after the in-place fill)."""
        outline = np.ascontiguousarray(outline, np.uint8)
        if outline.shape != (self.cfg.H_total, self.cfg.W):
            raise Scan3DError(f"outline must be [{self.cfg.H_total}][{self.cfg.W}] u8, got {outline.shape}")
        roi = np.empty_like(outline)
        filled = np.empty_like(outline)
        self._ck(self.L.scan3d_roi_fill(self.h, _ptr(outline), _ptr(roi), _ptr(filled)))
        return roi, filled

    def register_points(self, xyz, theta_deg, tx, ty, tz):
        """register_point_clouds' transform of one cloud (f32 [n][3]) captured at turntable angle theta_deg."""
        xyz = np.ascontiguousarray(xyz, np.float32).reshape(-1, 3)
        out = np.empty_like(xyz)
        if xyz.shape[0] == 0:
            return out
        self._ck(self.L.scan3d_register_points(self.h, _ptr(xyz), _ptr(out), xyz.shape[0], theta_deg, tx, ty, tz))
        return out

    def register_points_dev(self, src_ptr, dst_ptr, n, theta_deg, tx, ty, tz):
        self._ck(self.L.scan3d_register_points_dev(self.h, C.c_void_p(src_ptr), C.c_void_p(dst_ptr), int(n),
                                                   theta_deg, tx, ty, tz))

    def write_ply(self, path, binary=False):
        self._ck(self.L.scan3d_write_ply(self.h, path.encode(), 1 if binary else 0))

    def write_pcd(self, path):
        self._ck(self.L.scan3d_write_pcd(self.h, path.encode()))

    # -- camera-grid mesh of the points (include/scan3d.h has the exact rules)
    def build_mesh(self, max_edge=math.inf):
        """Triangles between neighbouring valid pixels whose edges are at most max_edge long, and per-point normals
        (asynchronous; after reconstruct / compact_points)."""
        self._ck(self.L.scan3d_build_mesh(self.h, max_edge))

    def mesh(self):
        """(faces int32 [n][3] point indices, normals float32 [point_count][3]) of the last build_mesh."""
        nf = C.c_int64()
        self._ck(self.L.scan3d_mesh_face_count(self.h, C.byref(nf)))
        faces = np.empty((nf.value, 3), np.int32)
        normals = np.empty((self.point_count(), 3), np.float32)
        self._ck(self.L.scan3d_get_mesh(self.h, _ptr(faces), _ptr(normals), nf.value))
        return faces, normals

    def write_mesh_ply(self, path, binary=False):
        self._ck(self.L.scan3d_write_mesh_ply(self.h, path.encode(), 1 if binary else 0))

    # -- voxel-grid merge of registered views (include/scan3d.h has the exact rules)
    def voxel_begin(self, voxel_size, max_voxels):
        """Reset the ctx's merge accumulator: voxels of edge voxel_size, up to max_voxels of them."""
        self._ck(self.L.scan3d_voxel_begin(self.h, voxel_size, int(max_voxels)))
        self._voxel_size = float(C.c_float(voxel_size).value)

    def voxel_add(self):
        """Add the ctx's current points (with the fresh mesh's normals and the texture's colours); asynchronous."""
        self._ck(self.L.scan3d_voxel_add_points(self.h))

    def voxel_add_dev(self, xyz, normals=None, rgb=None, n=None):
        """Add n points from device memory on the ctx's GPU: torch tensors or raw pointers (then n is required);
        normals / rgb None mean zeros.  Asynchronous on the ctx stream."""
        def dptr(a):
            return None if a is None else C.c_void_p(a if isinstance(a, int) else a.data_ptr())
        if n is None:
            n = xyz.shape[0]
        self._ck(self.L.scan3d_voxel_add_points_dev(self.h, dptr(xyz), dptr(normals), dptr(rgb), int(n)))

    def voxel_finish(self):
        self._ck(self.L.scan3d_voxel_finish(self.h))

    def voxel_count(self):
        """(voxels, dropped points) of the last voxel_finish (synchronises)."""
        v, d = C.c_int64(), C.c_int64()
        self._ck(self.L.scan3d_voxel_count(self.h, C.byref(v), C.byref(d)))
        return v.value, d.value

    def voxels(self):
        """(xyz float32 [v][3], normals float32 [v][3], rgb uint8 [v][3], counts uint32 [v]) in first-point order."""
        v, _ = self.voxel_count()
        out = (np.empty((v, 3), np.float32), np.empty((v, 3), np.float32), np.empty((v, 3), np.uint8),
               np.empty(v, np.uint32))
        self._ck(self.L.scan3d_get_voxels(self.h, *[_ptr(a) for a in out], v))
        return out

    def write_voxel_ply(self, path, binary=False):
        self._ck(self.L.scan3d_write_voxel_ply(self.h, path.encode(), 1 if binary else 0))

    # -- triangle surface of the voxel outputs (include/scan3d.h has the exact rules)
    def voxel_surface(self, max_distance=None, max_points=None):
        """Extract the surface of the outputs of the last voxel_finish; synchronises once and returns a dict with
        vertices, faces, lattice_points and undefined_points.  max_distance None = 2 voxel_size; max_points None =
        SURFACE_POINTS_PER_VOXEL * the voxel count (within [1, 2^31 - 1])."""
        if max_distance is None:
            max_distance = 2.0 * self._voxel_size
        if max_points is None:
            max_points = min(max(SURFACE_POINTS_PER_VOXEL * self.voxel_count()[0], 1), 2 ** 31 - 1)
        p = SurfaceParams(max_distance, int(max_points))
        r = SurfaceResultC()
        self._ck(self.L.scan3d_voxel_surface(self.h, C.byref(p), C.byref(r)))
        self._surface_counts = (r.vertices, r.faces)
        self._surface_refined = False
        return dict(vertices=r.vertices, faces=r.faces, lattice_points=r.lattice_points,
                    undefined_points=r.undefined_points)

    def voxel_surface_mesh(self):
        """(xyz float32 [v][3], normals float32 [v][3], rgb uint8 [v][3], faces int32 [f][3]) of the last
        voxel_surface."""
        v, f = getattr(self, "_surface_counts", (0, 0))
        out = (np.empty((v, 3), np.float32), np.empty((v, 3), np.float32), np.empty((v, 3), np.uint8),
               np.empty((f, 3), np.int32))
        self._ck(self.L.scan3d_get_voxel_surface(self.h, *[_ptr(a) for a in out], v, f))
        return out

    def write_voxel_surface_ply(self, path, binary=False):
        self._ck(self.L.scan3d_write_voxel_surface_ply(self.h, path.encode(), 1 if binary else 0))

    # -- connected components (include/scan3d.h has the exact rules)
    def surface_components(self, min_faces=0, max_components=0):
        """Label the held voxel surface and keep, in place, its components with at least min_faces faces, at most
        max_components of them (0 = no limit) by faces descending; synchronises once and returns a dict with
        components, kept, vertices, faces and largest_faces.  voxel_surface_mesh() then returns the kept surface."""
        p = ComponentsParams(int(min_faces), int(max_components))
        r = ComponentsResultC()
        self._ck(self.L.scan3d_voxel_surface_components(self.h, C.byref(p), C.byref(r)))
        self._surface_counts = (r.vertices, r.faces)
        self._components = r.components
        return dict(components=r.components, kept=r.kept, vertices=r.vertices, faces=r.faces,
                    largest_faces=r.largest_faces)

    def surface_component_table(self):
        """(vertices int64 [c], faces int64 [c], kept bool [c]) per component of the last surface_components, in id
        order."""
        c = getattr(self, "_components", 0)
        v, f, k = np.empty(c, np.int64), np.empty(c, np.int64), np.empty(c, np.uint8)
        self._ck(self.L.scan3d_get_surface_components(self.h, _ptr(v), _ptr(f), _ptr(k), c))
        return v, f, k.astype(bool)

    def mesh_components_dev(self, faces, n_vertices):
        """Connected components of a triangle mesh on the ctx's GPU: faces is a CUDA int32 tensor [f][3].  torch's
        current stream is synchronised first, so faces written there are ready and the new labels tensor is not in
        use by earlier work.  Returns (labels int32 tensor [n_vertices], component count)."""
        import torch
        if not (isinstance(faces, torch.Tensor) and faces.is_cuda and faces.dtype == torch.int32 and faces.dim() == 2
                and faces.shape[1] == 3):
            raise Scan3DError("faces must be a CUDA int32 tensor of shape [f][3]")
        faces = faces.contiguous()
        labels = torch.empty(int(n_vertices), dtype=torch.int32, device=faces.device)
        torch.cuda.current_stream(faces.device).synchronize()
        n = C.c_int64()
        self._ck(self.L.scan3d_mesh_components_dev(self.h, C.c_void_p(faces.data_ptr()), faces.shape[0],
                                                   int(n_vertices), C.c_void_p(labels.data_ptr()), C.byref(n)))
        return labels, n.value

    # -- simplification of the voxel surface (include/scan3d.h has the exact rules)
    def surface_decimate(self, cell_size):
        """Replace the held voxel surface, in place, by its vertex clustering on a grid of edge cell_size (voxel_size
        to 256 voxel_size) with quadric placement; synchronises once and returns a dict with vertices, faces,
        collapsed_faces, duplicate_faces and mean_fallbacks.  voxel_surface_mesh() then returns the simplified
        surface; the component table goes stale."""
        r = DecimateResultC()
        self._ck(self.L.scan3d_voxel_surface_decimate(self.h, float(cell_size), C.byref(r)))
        self._surface_counts = (r.vertices, r.faces)
        self._components = 0
        self._surface_refined = True
        return dict(vertices=r.vertices, faces=r.faces, collapsed_faces=r.collapsed_faces,
                    duplicate_faces=r.duplicate_faces, mean_fallbacks=r.mean_fallbacks)

    # -- smoothing of the voxel surface and of device meshes (include/scan3d.h has the exact rules)
    @staticmethod
    def _smooth_result(r):
        return dict(vertices=r.vertices, faces=r.faces, held_vertices=r.held_vertices,
                    isolated_vertices=r.isolated_vertices, passes=r.passes, max_displacement=r.max_displacement)

    def surface_smooth(self, iterations=10, lam=0.5, mu=-0.53):
        """Taubin lambda|mu smoothing of the held voxel surface, in place (MeshLab's defaults); boundary and
        non-manifold vertices are held.  Synchronises once and returns a dict with vertices, faces, held_vertices,
        isolated_vertices, passes and max_displacement.  voxel_surface_mesh() then returns the smoothed surface; the
        component table stays valid."""
        r = SmoothResultC()
        self._ck(self.L.scan3d_voxel_surface_smooth(self.h, C.byref(SmoothParams(int(iterations), lam, mu)),
                                                    C.byref(r)))
        self._surface_counts = (r.vertices, r.faces)
        self._surface_refined = True
        return self._smooth_result(r)

    def mesh_smooth_dev(self, xyz, faces, normals=None, iterations=10, lam=0.5, mu=-0.53):
        """surface_smooth() for a triangle mesh on the ctx's GPU, in place: xyz a CUDA float32 tensor [v][3], faces a
        CUDA int32 tensor [f][3], normals None or a CUDA float32 tensor [v][3] (then recomputed).  torch's current
        stream is synchronised first, so data written there is ready.  Returns the dict of surface_smooth()."""
        import torch

        def ok(t, dtype, rows):
            return (isinstance(t, torch.Tensor) and t.is_cuda and t.dtype == dtype and t.dim() == 2 and
                    t.shape[1] == 3 and t.is_contiguous() and (rows is None or t.shape[0] == rows))
        if not ok(xyz, torch.float32, None):
            raise Scan3DError("xyz must be a contiguous CUDA float32 tensor of shape [v][3]")
        if not ok(faces, torch.int32, None):
            raise Scan3DError("faces must be a contiguous CUDA int32 tensor of shape [f][3]")
        if normals is not None and not ok(normals, torch.float32, xyz.shape[0]):
            raise Scan3DError("normals must be None or a contiguous CUDA float32 tensor of the shape of xyz")
        torch.cuda.current_stream(xyz.device).synchronize()
        r = SmoothResultC()
        self._ck(self.L.scan3d_mesh_smooth_dev(self.h, C.c_void_p(xyz.data_ptr()),
                                               None if normals is None else C.c_void_p(normals.data_ptr()),
                                               xyz.shape[0], C.c_void_p(faces.data_ptr()), faces.shape[0],
                                               C.byref(SmoothParams(int(iterations), lam, mu)), C.byref(r)))
        return self._smooth_result(r)

    # -- hole filling of the voxel surface and of device meshes (include/scan3d.h has the exact rules)
    @staticmethod
    def _fill_result(r):
        return dict(vertices=r.vertices, faces=r.faces, boundary_edges=r.boundary_edges, holes=r.holes,
                    filled=r.filled, faces_added=r.faces_added, open_edges=r.open_edges)

    def surface_fill_holes(self, max_edges=None):
        """Close, in place, the holes of the held voxel surface whose boundary loops have at most max_edges edges by
        minimum-weight triangulation (Liepa's weight).  max_edges None = the largest allowed: FILL_NETS_MAX_EDGES on a
        surface that is neither simplified nor smoothed (it stays decimatable), else FILL_MAX_EDGES.  Synchronises
        twice and returns a dict with vertices, faces, boundary_edges, holes, filled, faces_added and open_edges.
        voxel_surface_mesh() then returns the filled surface; the component table goes stale."""
        if max_edges is None:
            max_edges = FILL_MAX_EDGES if getattr(self, "_surface_refined", False) else FILL_NETS_MAX_EDGES
        r = FillResultC()
        self._ck(self.L.scan3d_voxel_surface_fill_holes(self.h, int(max_edges), C.byref(r)))
        self._surface_counts = (r.vertices, r.faces)
        self._components = 0
        return self._fill_result(r)

    def mesh_fill_holes_dev(self, xyz, faces, max_edges=FILL_MAX_EDGES):
        """surface_fill_holes() for a triangle mesh on the ctx's GPU: xyz a CUDA float32 tensor [v][3], faces a CUDA
        int32 tensor [f][3]; neither is changed.  torch's current stream is synchronised first, so data written there
        is ready.  Returns (the added faces, a new CUDA int32 tensor [faces_added][3], the dict of
        surface_fill_holes())."""
        import torch

        def ok(t, dtype):
            return (isinstance(t, torch.Tensor) and t.is_cuda and t.dtype == dtype and t.dim() == 2 and
                    t.shape[1] == 3 and t.is_contiguous())
        if not ok(xyz, torch.float32):
            raise Scan3DError("xyz must be a contiguous CUDA float32 tensor of shape [v][3]")
        if not ok(faces, torch.int32):
            raise Scan3DError("faces must be a contiguous CUDA int32 tensor of shape [f][3]")
        torch.cuda.current_stream(xyz.device).synchronize()
        rows = faces.shape[0]
        for attempt in range(2):
            out = torch.empty((max(rows, 1), 3), dtype=torch.int32, device=xyz.device)
            r = FillResultC()
            rc = self.L.scan3d_mesh_fill_holes_dev(self.h, C.c_void_p(xyz.data_ptr()), xyz.shape[0],
                                                   C.c_void_p(faces.data_ptr()), faces.shape[0], int(max_edges),
                                                   C.c_void_p(out.data_ptr()), rows, C.byref(r))
            if rc == -1 and attempt == 0 and r.faces_added > rows:   # SCAN3D_ERR_CONFIG
                rows = r.faces_added                        # too small: once more with the reported size
                continue
            self._ck(rc)
            return out[:r.faces_added], self._fill_result(r)

    # -- repair of non-manifold edges and vertices of the voxel surface and of device meshes (include/scan3d.h has the
    # exact rules)
    @staticmethod
    def _repair_result(r):
        return {name: getattr(r, name) for name, _ in RepairResultC._fields_}

    @staticmethod
    def _repair_flags(faces, vertices):
        return (REPAIR_FACES if faces else 0) | (REPAIR_VERTICES if vertices else 0)

    def surface_repair(self, faces=True, vertices=True):
        """Repair, in place, the non-manifold edges (faces=True: duplicate faces and the extra faces of edges in more
        than two, by area) and the non-manifold vertices (vertices=True: one new vertex per extra fan) of the held
        voxel surface; degenerate faces always go.  Synchronises twice and returns a dict with the fields of
        scan3d_repair_result.  voxel_surface_mesh() then returns the repaired surface; the component table goes
        stale."""
        r = RepairResultC()
        self._ck(self.L.scan3d_voxel_surface_repair(self.h, self._repair_flags(faces, vertices), C.byref(r)))
        self._surface_counts = (r.vertices, r.faces)
        self._components = 0
        return self._repair_result(r)

    def mesh_repair_dev(self, xyz, faces, repair_faces=True, vertices=True):
        """surface_repair() for a triangle mesh on the ctx's GPU (repair_faces is surface_repair's faces): xyz a CUDA
        float32 tensor [v][3], faces a CUDA int32 tensor [f][3]; neither is changed.  torch's current stream is
        synchronised first, so data written there is ready.  Returns (the repaired faces, a new CUDA int32 tensor
        [faces][3]; the source vertex of each added vertex, a new CUDA int32 tensor [vertices_added], for extending
        attribute arrays with a gather; the dict of surface_repair())."""
        import torch

        def ok(t, dtype):
            return (isinstance(t, torch.Tensor) and t.is_cuda and t.dtype == dtype and t.dim() == 2 and
                    t.shape[1] == 3 and t.is_contiguous())
        if not ok(xyz, torch.float32):
            raise Scan3DError("xyz must be a contiguous CUDA float32 tensor of shape [v][3]")
        if not ok(faces, torch.int32):
            raise Scan3DError("faces must be a contiguous CUDA int32 tensor of shape [f][3]")
        torch.cuda.current_stream(xyz.device).synchronize()
        nf = faces.shape[0]
        out = torch.empty((max(nf, 1), 3), dtype=torch.int32, device=xyz.device)
        src = torch.empty(max(3 * nf, 1), dtype=torch.int32, device=xyz.device)   # a new vertex per corner at most
        r = RepairResultC()
        self._ck(self.L.scan3d_mesh_repair_dev(self.h, C.c_void_p(xyz.data_ptr()), xyz.shape[0],
                                               C.c_void_p(faces.data_ptr()), nf,
                                               self._repair_flags(repair_faces, vertices), C.c_void_p(out.data_ptr()),
                                               C.c_void_p(src.data_ptr()), 3 * nf, C.byref(r)))
        return out[:r.faces], src[:r.vertices_added], self._repair_result(r)

    # -- coherent orientation and measures of the voxel surface and of device meshes (include/scan3d.h has the exact
    # rules)
    @staticmethod
    def _orient_result(r):
        return {name: getattr(r, name) for name, _ in OrientResultC._fields_}

    @staticmethod
    def _measure_result(r):
        out = {name: getattr(r, name) for name, _ in MeasureResultC._fields_}
        out["watertight"] = bool(r.watertight)
        out["bbox_min"], out["bbox_max"] = tuple(r.bbox_min), tuple(r.bbox_max)
        return out

    @staticmethod
    def _mesh_tensors(xyz, faces, normals=None):
        import torch

        def ok(t, dtype, rows):
            return (isinstance(t, torch.Tensor) and t.is_cuda and t.dtype == dtype and t.dim() == 2 and
                    t.shape[1] == 3 and t.is_contiguous() and (rows is None or t.shape[0] == rows))
        if not ok(xyz, torch.float32, None):
            raise Scan3DError("xyz must be a contiguous CUDA float32 tensor of shape [v][3]")
        if not ok(faces, torch.int32, None):
            raise Scan3DError("faces must be a contiguous CUDA int32 tensor of shape [f][3]")
        if normals is not None and not ok(normals, torch.float32, xyz.shape[0]):
            raise Scan3DError("normals must be None or a contiguous CUDA float32 tensor of the shape of xyz")
        torch.cuda.current_stream(xyz.device).synchronize()

    def surface_orient(self):
        """Orient the faces of the held voxel surface coherently, in place: per patch of faces joined across edges of
        two faces, the fewest flips that make it consistent, closed patches with their normals outward; a vertex all of
        whose faces flipped has its normal negated.  Synchronises once and returns a dict with the fields of
        scan3d_orient_result.  The component table stays current."""
        r = OrientResultC()
        self._ck(self.L.scan3d_voxel_surface_orient(self.h, C.byref(r)))
        return self._orient_result(r)

    def mesh_orient_dev(self, xyz, faces, normals=None):
        """surface_orient() for a triangle mesh on the ctx's GPU, in place: xyz a CUDA float32 tensor [v][3] (read),
        faces a CUDA int32 tensor [f][3] (the flips are written into it), normals None or a CUDA float32 tensor [v][3].
        torch's current stream is synchronised first, so data written there is ready.  Returns the dict of
        surface_orient()."""
        self._mesh_tensors(xyz, faces, normals)
        r = OrientResultC()
        self._ck(self.L.scan3d_mesh_orient_dev(self.h, C.c_void_p(xyz.data_ptr()),
                                               None if normals is None else C.c_void_p(normals.data_ptr()),
                                               xyz.shape[0], C.c_void_p(faces.data_ptr()), faces.shape[0],
                                               C.byref(r)))
        return self._orient_result(r)

    def surface_measure(self):
        """The area, signed volume, bounding box and topology (edges by kind, patches, Euler characteristic, watertight)
        of the held voxel surface: a dict with the fields of scan3d_measure_result (watertight a bool, the boxes
        tuples).  Changes nothing; synchronises once."""
        r = MeasureResultC()
        self._ck(self.L.scan3d_voxel_surface_measure(self.h, C.byref(r)))
        return self._measure_result(r)

    def mesh_measure_dev(self, xyz, faces):
        """surface_measure() for a triangle mesh on the ctx's GPU: xyz a CUDA float32 tensor [v][3], faces a CUDA int32
        tensor [f][3]; neither is changed.  torch's current stream is synchronised first."""
        self._mesh_tensors(xyz, faces)
        r = MeasureResultC()
        self._ck(self.L.scan3d_mesh_measure_dev(self.h, C.c_void_p(xyz.data_ptr()), xyz.shape[0],
                                                C.c_void_p(faces.data_ptr()), faces.shape[0], C.byref(r)))
        return self._measure_result(r)

    # -- distances of samples from a triangle surface within a radius (include/scan3d.h has the exact rules)
    @staticmethod
    def _distance_result(r):
        return {name: getattr(r, name) for name, _ in DistanceResultC._fields_}

    @staticmethod
    def _distance_outputs(samples, n):
        import torch
        dev = samples.device
        return (torch.empty(n, dtype=torch.float32, device=dev), torch.empty(n, dtype=torch.int32, device=dev))

    @staticmethod
    def _samples_tensor(samples):
        import torch
        if not (isinstance(samples, torch.Tensor) and samples.is_cuda and samples.dtype == torch.float32 and
                samples.dim() == 2 and samples.shape[1] == 3 and samples.is_contiguous()):
            raise Scan3DError("samples must be a contiguous CUDA float32 tensor of shape [n][3]")
        torch.cuda.current_stream(samples.device).synchronize()

    def surface_distance(self, max_distance, per_sample=False):
        """The distances of the merge's model (the voxel outputs with a non-zero normal) from the held voxel surface,
        each to its nearest face within max_distance, signed by that face's normal (negative inside an outward
        surface).  Returns a dict with the fields of scan3d_distance_result (max is the one-sided Hausdorff distance
        within max_distance); with per_sample=True, (dist, face, dict): CUDA tensors indexed by voxel ordinal, NaN and
        -1 for a voxel that is not matched or not in the model.  Changes nothing; synchronises twice."""
        import torch
        p = DistanceParams(max_distance)
        r = DistanceResultC()
        if not per_sample:
            self._ck(self.L.scan3d_voxel_surface_distance(self.h, C.byref(p), None, None, C.byref(r)))
            return self._distance_result(r)
        n = self.voxel_count()[0]                       # the outputs of the last finish: no SURFACE without them
        dev = torch.device("cuda", torch.cuda.current_device())
        dist = torch.empty(n, dtype=torch.float32, device=dev)
        face = torch.empty(n, dtype=torch.int32, device=dev)
        torch.cuda.current_stream(dev).synchronize()
        self._ck(self.L.scan3d_voxel_surface_distance(self.h, C.byref(p), C.c_void_p(dist.data_ptr()) if n else None,
                                                      C.c_void_p(face.data_ptr()) if n else None, C.byref(r)))
        return dist, face, self._distance_result(r)

    def surface_distance_dev(self, samples, max_distance):
        """surface_distance() for samples of the caller: a CUDA float32 tensor [n][3] on the ctx's GPU (a view's
        device_points(), for instance) against the held voxel surface.  torch's current stream is synchronised first.
        Returns (dist, face, dict): dist float32 [n] signed, NaN when invalid or unmatched; face int32 [n], -1 then."""
        self._samples_tensor(samples)
        n = samples.shape[0]
        dist, face = self._distance_outputs(samples, n)
        p = DistanceParams(max_distance)
        r = DistanceResultC()
        self._ck(self.L.scan3d_voxel_surface_distance_dev(self.h, C.c_void_p(samples.data_ptr()), n, C.byref(p),
                                                          C.c_void_p(dist.data_ptr()), C.c_void_p(face.data_ptr()),
                                                          C.byref(r)))
        return dist, face, self._distance_result(r)

    def mesh_distance_dev(self, samples, xyz, faces, max_distance):
        """surface_distance_dev() against any triangle mesh on the ctx's GPU: xyz a CUDA float32 tensor [v][3], faces
        a CUDA int32 tensor [f][3] (the camera-grid mesh included); nothing is changed."""
        self._samples_tensor(samples)
        self._mesh_tensors(xyz, faces)
        n = samples.shape[0]
        dist, face = self._distance_outputs(samples, n)
        p = DistanceParams(max_distance)
        r = DistanceResultC()
        self._ck(self.L.scan3d_mesh_distance_dev(self.h, C.c_void_p(samples.data_ptr()), n,
                                                 C.c_void_p(xyz.data_ptr()), xyz.shape[0],
                                                 C.c_void_p(faces.data_ptr()), faces.shape[0], C.byref(p),
                                                 C.c_void_p(dist.data_ptr()), C.c_void_p(face.data_ptr()),
                                                 C.byref(r)))
        return dist, face, self._distance_result(r)

    # -- scan-to-model alignment against the voxel outputs (include/scan3d.h has the exact rules)
    @staticmethod
    def _align_params(max_distance, max_iterations, stride, T_init, apply, stop_rotation, stop_translation):
        p = AlignParams()
        T = np.eye(4) if T_init is None else np.asarray(T_init, np.float64).reshape(4, 4)
        p.T_init[:] = T.reshape(-1).tolist()
        p.max_distance = max_distance
        p.max_iterations = int(max_iterations)
        p.stride = int(stride)
        p.stop_rotation = stop_rotation
        p.stop_translation = 1e-4 * float(C.c_float(max_distance).value) if stop_translation is None else stop_translation
        p.apply = int(bool(apply))
        return p

    def align(self, max_distance, max_iterations=30, stride=1, T_init=None, apply=True, stop_rotation=1e-6,
              stop_translation=None):
        """Point-to-plane ICP of the ctx's current points against the outputs of the last voxel_finish; with apply the
        points are transformed in place (the mesh goes stale).  stop_translation None = 1e-4 * max_distance.
        Synchronises once; returns an AlignResult."""
        p = self._align_params(max_distance, max_iterations, stride, T_init, apply, stop_rotation, stop_translation)
        r = AlignResultC()
        self._ck(self.L.scan3d_align_to_voxels(self.h, C.byref(p), C.byref(r)))
        return AlignResult(r)

    def align_dev(self, xyz, max_distance, max_iterations=30, stride=1, T_init=None, apply=True, stop_rotation=1e-6,
                  stop_translation=None, n=None):
        """align() for n points in device memory on the ctx's GPU: a torch tensor [n][3] float32, or a raw pointer
        (then n is required); with apply they are transformed in place."""
        if n is None:
            n = xyz.shape[0]
        ptr = C.c_void_p(xyz if isinstance(xyz, int) else xyz.data_ptr())
        p = self._align_params(max_distance, max_iterations, stride, T_init, apply, stop_rotation, stop_translation)
        r = AlignResultC()
        self._ck(self.L.scan3d_align_to_voxels_dev(self.h, ptr, int(n), C.byref(p), C.byref(r)))
        return AlignResult(r)

    def set_points_buffer(self, dev_ptr, capacity_points):
        """Compacted points go to this device pointer (may be another GPU's memory mapped here); 0/None restores."""
        self._ck(self.L.scan3d_set_points_buffer(self.h, C.c_void_p(dev_ptr) if dev_ptr else None, int(capacity_points)))

    def launch_count(self):
        return int(self.L.scan3d_launch_count(self.h))

    def debug_divcheck(self):
        n = C.c_uint64()
        self._ck(self.L.scan3d_debug_divcheck(self.h, C.byref(n)))
        return n.value

    def debug_atan2(self, y, x, mode):
        y = np.ascontiguousarray(y, np.float64)
        x = np.ascontiguousarray(x, np.float64)
        out = np.empty(y.shape, np.float32)
        self._ck(self.L.scan3d_debug_atan2(self.h, _ptr(y), _ptr(x), _ptr(out), y.size, mode))
        return out


def register_rotation(theta_deg):
    """The 4x4 float matrix register_point_clouds builds for turntable angle theta_deg (its Pi = 22/7)."""
    R = np.empty(16, np.float32)
    cuda_lib().scan3d_register_rotation(theta_deg, _ptr(R))
    return R.reshape(4, 4)


# ---------------------------------------------------------------------------------------------
# peer memory helpers (row-sharded mode, 3dscan_b200/sharding.py)
# ---------------------------------------------------------------------------------------------
def peer_alloc(device, nbytes):
    """(device pointer, 64-byte CUDA IPC handle) of a new block on `device`."""
    p, h = C.c_void_p(), C.create_string_buffer(64)
    rc = cuda_lib().scan3d_peer_alloc(int(device), int(nbytes), C.byref(p), h)
    if rc:
        raise Scan3DError(f"scan3d_peer_alloc failed ({rc})")
    return int(p.value), bytes(h.raw)


def peer_free(device, ptr):
    cuda_lib().scan3d_peer_free(int(device), C.c_void_p(ptr))


def peer_open(device, handle):
    """Maps another process's block for kernels running on `device`; returns the local pointer."""
    p = C.c_void_p()
    rc = cuda_lib().scan3d_peer_open(int(device), C.create_string_buffer(bytes(handle), 64), C.byref(p))
    if rc:
        raise Scan3DError(f"scan3d_peer_open failed ({rc})")
    return int(p.value)


def peer_close(device, ptr):
    cuda_lib().scan3d_peer_close(int(device), C.c_void_p(ptr))


def wrap_device(ptr, shape, typestr):
    """torch view of a raw device buffer (no copy, no ownership)."""
    import torch

    class _Holder:
        pass
    h = _Holder()
    h.__cuda_array_interface__ = {"shape": tuple(shape), "typestr": typestr, "data": (int(ptr), False), "version": 2}
    return torch.as_tensor(h, device="cuda")
