"""CPU-side checks: the C-ABI libraries load without a GPU and export every symbol that
include/*.h declares; host-side logic (file formats, pattern conventions, synthetic scenes)."""
import ctypes as C
import importlib
import os
import re

import numpy as np
import pytest

import oracle_ffi as o
from helpers import GOLDEN, load_c1_full, load_calib_c1

s3 = importlib.import_module("3dscan_b200")
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _declared(header):
    text = open(os.path.join(ROOT, "include", header)).read()
    text = re.sub(r"/\*.*?\*/", "", text, flags=re.S)
    return sorted(set(re.findall(r"\b(scan3d_[a-z0-9_]+)\s*\(", text)))


def test_cuda_library_exports_every_declared_symbol():
    L = s3.cuda_lib()
    names = _declared("scan3d.h")
    assert len(names) >= 30
    for n in names:
        assert hasattr(L, n), n
    assert L.scan3d_version() == 100


def test_host_library_exports_every_declared_symbol():
    L = s3.host_lib()
    for n in _declared("scan3d_host.h"):
        assert hasattr(L, n), n


def test_config_validation_without_gpu():
    L = s3.cuda_lib()
    h = C.c_void_p()
    bad = s3.make_config(0, 10)
    assert L.scan3d_create(C.byref(bad), 0, C.byref(h)) == -1
    assert b"W/H" in L.scan3d_last_error(None)
    bad = s3.make_config(64, 64, 64, 64, N=2, M_v=4, M_h=4)
    assert L.scan3d_create(C.byref(bad), 0, C.byref(h)) == -1
    cfg = s3.make_config(4096, 3000, 4096, 3000, 8, 10, 10, 4, 4, 2)
    assert L.scan3d_stack_bytes(C.byref(cfg)) == 56 * 4096 * 3000


def test_no_cpu_fallback_without_gpu():
    try:
        import torch
        if torch.cuda.is_available():
            pytest.skip("GPU present")
    except ImportError:
        pass
    with pytest.raises(s3.Scan3DError):
        s3.Scan3D(s3.make_config(64, 64, 64, 64, 3, 4, 4, 4, 4, 2), 0)


def test_pattern_rows_match_reference_generated_patterns():
    k = np.load(os.path.join(GOLDEN, "pattern_kat.npz"))
    for i in range(3):
        assert np.array_equal(s3.synth_pattern_row(0, 3, 32, i, 1280), k["fringe_v_row0"][i])
        assert np.array_equal(s3.synth_pattern_row(0, 3, 32, i, 720), k["fringe_h_col0"][i])
    for i in range(6):
        assert np.array_equal(s3.synth_pattern_row(1, 6, 32, i, 1280), k["gray_v_row0"][i])
        assert np.array_equal(s3.synth_pattern_row(2, 6, 32, i, 1280), k["inv_v_row0"][i])
    for i in range(5):
        assert np.array_equal(s3.synth_pattern_row(1, 5, 32, i, 720), k["gray_h_col0"][i])
        assert np.array_equal(s3.synth_pattern_row(2, 5, 32, i, 720), k["inv_h_col0"][i])
    # stale images of earlier 4-step (fw 16) and 5-step (fw 32) runs pin those expressions too
    assert np.array_equal(s3.synth_pattern_row(0, 4, 16, 3, 1024), k["fringe4_k3_v_row0"])
    assert np.array_equal(s3.synth_pattern_row(0, 4, 16, 3, 768), k["fringe4_k3_h_col0"])
    assert np.array_equal(s3.synth_pattern_row(0, 5, 32, 4, 1024), k["fringe5_k4_v_row0"])
    assert np.array_equal(s3.synth_pattern_row(0, 5, 32, 4, 768), k["fringe5_k4_h_col0"])


def _cal():
    c = load_calib_c1()
    args = [c[k] for k in ("Kc", "dc", "Kp", "dp", "rc", "tc", "rp", "tp")]
    return s3.make_calib(*args), o.make_calib(*args)


def test_synthetic_scene_reconstructs_through_the_oracle():
    """noise-free stack -> oracle -> the scene comes back (the generator and the decode agree)."""
    cal, ocal = _cal()
    cfg = s3.make_config(400, 300, 320, 180, 4, 6, 5, 8, 8, 2)
    cal2 = s3.scale_calibration(cal, 0.25, 0.25)
    c2 = s3.calib_to_dict(cal2)
    ocal2 = o.make_calib(*[c2[k] for k in ("Kc", "dc", "Kp", "dp", "rc", "tc", "rp", "tp")])
    p = s3.default_synth_params(noise_sigma=0.0, ambient_max=0.0, albedo_lo=1.0)
    stack, roi, truth = s3.synth_stack(cfg, cal2, p, want_truth=True)
    d = s3.split_stack(cfg, stack)
    r = o.reconstruct({k: getattr(cfg, k) for k in ("W", "H", "PW", "PH", "N", "M_v", "M_h", "fw_v", "fw_h", "dirs")},
                      ocal2, d["fringe_v"], d["gray_v"], d["inv_v"], d["fringe_h"], d["gray_h"], d["inv_h"], roi)
    assert r.count > 20000
    err = np.linalg.norm(r.pts - truth.reshape(-1, 3)[r.pix], axis=1)
    assert np.median(err) < 0.5          # mm; the scene is ~100 mm from the camera
    assert (err < 2.0).mean() > 0.97


def test_synth_is_deterministic_and_row_shardable():
    cal, _ = _cal()
    full = s3.make_config(160, 48, 128, 96, 3, 5, 5, 4, 4, 2)
    a, roi = s3.synth_stack(full, cal)
    b, _ = s3.synth_stack(full, cal)
    assert np.array_equal(a, b)
    part = s3.make_config(160, 20, 128, 96, 3, 5, 5, 4, 4, 2, row0=10, H_total=48)
    c, roi2 = s3.synth_stack(part, cal)
    assert np.array_equal(c, a[:, 10:30]) and np.array_equal(roi, roi2)
    assert 0.6 < roi.mean() < 0.8


def _cv_xml(path, name, arr):
    """A matrix file as OpenCV's cvSave writes it (opencv_storage, doubles as %.16e)."""
    arr = np.asarray(arr, np.float64)
    rows, cols = (arr.shape[0], 1) if arr.ndim == 1 else arr.shape
    os.makedirs(os.path.dirname(path), exist_ok=True)
    data = " ".join("%.16e" % v for v in arr.ravel())
    with open(path, "w") as f:
        f.write(f'<?xml version="1.0"?>\n<opencv_storage>\n<{name} type_id="opencv-matrix">\n  <rows>{rows}</rows>\n'
                f"  <cols>{cols}</cols>\n  <dt>d</dt>\n  <data>\n    {data}</data></{name}>\n</opencv_storage>\n")


def _cv_bmp8(path, img):
    """An 8-bit grey BMP as cvSaveImage writes it: 256-entry grey palette, bottom-up rows padded to 4 bytes."""
    H, W = img.shape
    stride = (W + 3) & ~3
    rows = np.zeros((H, stride), np.uint8)
    rows[:, :W] = img[::-1]
    pal = np.repeat(np.arange(256, dtype=np.uint8), 4).reshape(256, 4)
    pal[:, 3] = 0
    off = 14 + 40 + 1024
    hdr = b"BM" + (off + rows.size).to_bytes(4, "little") + bytes(4) + off.to_bytes(4, "little")
    info = b"".join(v.to_bytes(n, "little") for v, n in ((40, 4), (W, 4), (H, 4), (1, 2), (8, 2), (0, 4), (rows.size, 4),
                                                          (0, 4), (0, 4), (0, 4), (0, 4)))
    os.makedirs(os.path.dirname(path), exist_ok=True)
    with open(path, "wb") as f:
        f.write(hdr + info + pal.tobytes() + rows.tobytes())


def test_reference_tree_loaders(tmp_path):
    """load_calibration / load_captured_set on a tree laid out like the reference's: its calibration matrices
    (tests/golden/calib_c1.json) and its whole captured scan (tests/golden/c1_full.npz) in the files and formats the
    reference stores them in."""
    root =str(tmp_path / "M_tech_project_console")
    c = load_calib_c1()
    for path, name, key in (("/Camera_calibration/Matrices/cam_intrinsic_mat.xml", "cam_intrinsic_mat", "Kc"),
                            ("/Camera_calibration/Matrices/cam_distortion_vect.xml", "cam_distortion_vect", "dc"),
                            ("/Projector_calibration/Matrices/proj_intrinsic_mat.xml", "proj_intrinsic_mat", "Kp"),
                            ("/Projector_calibration/Matrices/proj_distortion_vect.xml", "proj_distortion_vect", "dp"),
                            ("/Triangulation/Camera_extrinsic_parametrs/world_to_cam_rot_vect.xml", "world_to_cam_rot_vect", "rc"),
                            ("/Triangulation/Camera_extrinsic_parametrs/world_to_cam_trans_vect.xml", "world_to_cam_trans_vect", "tc"),
                            ("/Triangulation/Projector_extrinsic_parametrs/world_to_proj_rot_vect.xml", "world_to_proj_rot_vect", "rp"),
                            ("/Triangulation/Projector_extrinsic_parametrs/world_to_proj_trans_vect.xml", "world_to_proj_trans_vect", "tp")):
        _cv_xml(root + path, name, c[key].reshape(3, 3) if key in ("Kc", "Kp") else c[key])
    d = load_c1_full()
    want = []
    for name, key in (("Vertical", "v"), ("Horizontal", "h")):
        fr = f"{root}/Captured_patterns/Fringe_patterns/{name}/Undistorted/"
        gc = f"{root}/Captured_patterns/Coded_patterns/Gray_coded/{name}/Undistorted/"
        for prefix, folder, frames in (("", fr, d[f"fringe_{key}"]), ("", gc, d[f"gray_{key}"]), ("inverse_", gc, d[f"inv_{key}"])):
            for i, img in enumerate(frames):
                _cv_bmp8(f"{folder}{prefix}Gray_captured_image_{i}.bmp", img)
            want.append(frames)

    cal = s3.load_calibration(root)
    for k in ("Kc", "dc", "Kp", "dp", "rc", "tc", "rp", "tp"):
        assert np.array_equal(np.array(list(getattr(cal, k))), c[k])
    cfg = s3.make_config(1600, 1200, 1280, 720, 3, 6, 5, 32, 32, 2)
    stack = s3.load_captured_set(root, cfg)
    assert stack.shape == (28, 1200, 1600)
    assert np.array_equal(stack, np.concatenate(want))


def test_bmp_and_ply_roundtrip(tmp_path):
    img = np.random.default_rng(1).integers(0, 256, (37, 53), dtype=np.uint8)
    p = str(tmp_path / "a.bmp")
    assert s3.host_lib().scan3d_write_bmp8(p.encode(), 53, 37, img.ctypes.data_as(C.c_void_p)) == 0
    assert np.array_equal(s3.read_bmp8(p), img)
    xyz = np.random.default_rng(2).normal(size=(11, 3)).astype(np.float32)
    q = str(tmp_path / "a.ply")
    assert s3.host_lib().scan3d_write_ply_points(q.encode(), xyz.ctypes.data_as(C.c_void_p), None, 11, 0) == 0
    body = open(q).read().split("end_header\n")[1]
    got = np.loadtxt(body.splitlines())[:, :3].astype(np.float32)
    assert np.array_equal(got, xyz)
    # PCD (pcl::io::savePCDFileASCII layout): 8 significant digits, rgb packed into a float
    rgb = np.random.default_rng(3).integers(0, 256, (11, 3), dtype=np.uint8)
    r = str(tmp_path / "a.pcd")
    assert s3.host_lib().scan3d_write_pcd_points(r.encode(), xyz.ctypes.data_as(C.c_void_p), rgb.ctypes.data_as(C.c_void_p), 11) == 0
    lines = open(r).read().splitlines()
    assert lines[1] == "VERSION 0.7" and lines[2] == "FIELDS x y z rgb" and lines[9] == "POINTS 11" and lines[10] == "DATA ascii"
    rows = np.array([[float(v) for v in ln.split()] for ln in lines[11:]])
    assert rows.shape == (11, 4)
    assert np.allclose(rows[:, :3], xyz, rtol=5e-8, atol=0)
    packed = (rgb[:, 0].astype(np.uint32) << 16) | (rgb[:, 1].astype(np.uint32) << 8) | rgb[:, 2]
    assert np.allclose(rows[:, 3], packed.view(np.float32).astype(np.float64), rtol=5e-8, atol=0)


def test_new_entry_points_reject_bad_arguments_without_a_gpu():
    """Argument checks that run before any CUDA call."""
    L = s3.cuda_lib()
    cfg = s3.make_config(64, 16, 1280, 720, 3, 6, 5, 32, 32, 2)
    assert L.scan3d_pattern_bytes(C.byref(cfg), 0) == (3 + 12) * 1280 * 720
    assert L.scan3d_pattern_bytes(C.byref(cfg), 1) == (3 + 10) * 1280 * 720
    assert L.scan3d_pattern_bytes(C.byref(cfg), 2) == 0
    assert L.scan3d_generate_patterns(None, 0, None) != 0
    assert L.scan3d_set_points_buffer(None, None, 0) != 0
    p = C.c_void_p()
    assert L.scan3d_peer_alloc(0, 0, C.byref(p), C.create_string_buffer(64)) != 0     # zero bytes
    assert L.scan3d_peer_open(0, None, C.byref(p)) != 0


def test_ply_reader_round_trip(tmp_path):
    """scan3d_read_ply_points (pcl::io::loadPLYFile's job in 9/register_point_clouds.cpp:66,87) reads back what
    scan3d_write_ply_points wrote, ascii and binary, bit for bit (%.9g round-trips a float)."""
    H = s3.host_lib()
    H.scan3d_write_ply_points.argtypes = [C.c_char_p, C.c_void_p, C.c_void_p, C.c_int64, C.c_int]
    H.scan3d_read_ply_points.argtypes = [C.c_char_p, C.c_void_p, C.c_void_p, C.c_int64, C.POINTER(C.c_int64)]
    rng = np.random.default_rng(12)
    xyz = (rng.normal(size=(777, 3)) * [1e-3, 50, 4e5]).astype(np.float32)
    rgb = rng.integers(0, 256, (777, 3), dtype=np.uint8)
    for binary in (0, 1):
        path = str(tmp_path / f"c{binary}.ply").encode()
        assert H.scan3d_write_ply_points(path, xyz.ctypes.data_as(C.c_void_p), rgb.ctypes.data_as(C.c_void_p), 777, binary) == 0
        n = C.c_int64()
        assert H.scan3d_read_ply_points(path, None, None, 0, C.byref(n)) == 0 and n.value == 777
        x2 = np.empty_like(xyz)
        c2 = np.empty_like(rgb)
        assert H.scan3d_read_ply_points(path, x2.ctypes.data_as(C.c_void_p), c2.ctypes.data_as(C.c_void_p), 777, C.byref(n)) == 0
        assert np.array_equal(x2.view(np.uint32), xyz.view(np.uint32)) and np.array_equal(c2, rgb)
        assert H.scan3d_read_ply_points(path, x2.ctypes.data_as(C.c_void_p), None, 10, C.byref(n)) == -4   # buffer too small
    # a PCL-style header: doubles, an extra property, no colours
    p = tmp_path / "pcl.ply"
    p.write_text("ply\nformat ascii 1.0\nelement vertex 2\nproperty double x\nproperty double y\nproperty double z\n"
                 "property float curvature\nend_header\n1.5 2.5 -3 0.1\n4 5 6 0.2\n")
    x3 = np.empty((2, 3), np.float32)
    c3 = np.empty((2, 3), np.uint8)
    n = C.c_int64()
    assert H.scan3d_read_ply_points(str(p).encode(), x3.ctypes.data_as(C.c_void_p), c3.ctypes.data_as(C.c_void_p), 2, C.byref(n)) == 0
    assert np.array_equal(x3, np.array([[1.5, 2.5, -3], [4, 5, 6]], np.float32)) and not c3.any()
    assert H.scan3d_read_ply_points(str(tmp_path / "missing.ply").encode(), None, None, 0, C.byref(n)) == -5


def test_aux_entries_reject_bad_arguments_without_gpu():
    L = s3.cuda_lib()
    assert L.scan3d_undistort_frames(None, 0, None, 1, None) == -4
    assert L.scan3d_roi_fill(None, None, None, None) == -4
    assert L.scan3d_register_points(None, None, None, 0, 0.0, 0.0, 0.0, 0.0) == -4
    R = np.empty(16, np.float32)
    assert L.scan3d_register_rotation(36.0, R.ctypes.data_as(C.c_void_p)) == 0      # host arithmetic (libm), no GPU needed
    assert np.array_equal(R.reshape(4, 4), o.register_rotation(36.0))


def test_compat_library_exports_the_reference_named_functions():
    """libscan3d_compat.so carries the reference's own stage functions with C++ linkage
    (PROJECT_GLOBAL/intermodule_dependencies.h:10-25 + the capture / scissor / registration entries)."""
    s3.cuda_lib(); s3.host_lib()            # its dependencies, resolved through $ORIGIN
    L = C.CDLL(os.path.join(ROOT, "3dscan_b200", "lib", "libscan3d_compat.so"))
    for sym in ("_Z16generate_patternv", "_Z13load_matricesv", "_Z21compute_wrapped_phasei", "_Z12unwrap_phasei",
                "_Z15compute_c_p_mapv", "_Z11triangulatev", "_Z16save_point_cloudj", "_Z16reconstruct_scanj",
                "_Z21register_point_cloudsjffff", "_Z18image_scissor_fillPKh", "_Z17undistort_capturePKhPhi",
                "_Z18scan3d_compat_initPKciiiii", "_Z22scan3d_compat_shutdownv", "_Z17scan3d_compat_ctxv"):
        assert hasattr(L, sym), sym
    for glob in ("selected_region", "valid_map", "code_vertical", "unwrapped_phi_horizontal", "c_p_map", "intersection_points",
                 "number_of_patterns_fringe", "fringe_width_pixels_vertical", "Camera_imagewidth"):
        C.c_void_p.in_dll(L, glob)


def test_reference_main_example_builds_and_fails_loudly_without_a_gpu(tmp_path):
    """examples/m_tech_console.cpp links against the three libraries; without a CUDA device it must stop with the
    library's error instead of computing anything on the CPU."""
    import subprocess
    libdir = os.path.join(ROOT, "3dscan_b200", "lib")
    exe = str(tmp_path / "m_tech_console")
    subprocess.check_call(["/usr/bin/g++", "-O2", "-std=c++17", "-Wall", "-I", os.path.join(ROOT, "include"),
                           os.path.join(ROOT, "examples", "m_tech_console.cpp"), "-L", libdir, "-lscan3d_compat",
                           "-lscan3d_host", "-lscan3d", "-Wl,-rpath," + libdir, "-o", exe])
    assert subprocess.run([exe], capture_output=True).returncode == 2          # usage
    try:
        import torch
        if torch.cuda.is_available():
            return
    except ImportError:
        pass
    r = subprocess.run([exe, str(tmp_path)], capture_output=True, text=True)
    assert r.returncode != 0 and "scan3d_create" in r.stderr


def test_colour_bmp_loads_as_the_grey_image_opencv_returns(tmp_path):
    """cvLoadImage(file, CV_LOAD_IMAGE_GRAYSCALE) on a 24-bit BMP (3/wrapped_phase.cpp:44, 4/phase_unwrap.cpp:78-90):
    scan3d_read_bmp8 gives the same bytes as cv2.imread(..., IMREAD_GRAYSCALE) (fixed-point BGR weights, padded rows)."""
    g = np.load(os.path.join(GOLDEN, "f4_kat.npz"))
    p = tmp_path / "colour.bmp"
    p.write_bytes(g["bmp24_bytes"].tobytes())
    assert np.array_equal(s3.read_bmp8(str(p)), g["bmp24_grey"])


def test_colour_bmp_reader_and_malformed_files(tmp_path):
    """scan3d_read_bmp_bgr = cvLoadImage in colour (8/save_point_cloud.cpp:59-66: texture.bmp, split into B, G, R);
    truncated or inconsistent headers are refused instead of read past (palette and pixel-data bounds)."""
    import cv2
    g = np.load(os.path.join(GOLDEN, "f4_kat.npz"))
    p = tmp_path / "colour.bmp"
    raw = g["bmp24_bytes"].tobytes()
    p.write_bytes(raw)
    assert np.array_equal(s3.read_bmp_bgr(str(p)), cv2.imread(str(p), cv2.IMREAD_COLOR))
    # an 8-bit palettised file through both readers
    grey = (np.arange(12 * 20, dtype=np.uint32).reshape(12, 20) * 7 % 256).astype(np.uint8)
    q = tmp_path / "grey.bmp"
    s3.write_bmp8(str(q), grey) if hasattr(s3, "write_bmp8") else cv2.imwrite(str(q), grey)
    assert np.array_equal(s3.read_bmp8(str(q)), grey)
    assert np.array_equal(s3.read_bmp_bgr(str(q)), np.repeat(grey[:, :, None], 3, axis=2))
    ok = q.read_bytes()
    bad = []
    bad.append(ok[:60])                                                     # cut inside the palette
    bad.append(ok[:len(ok) - 5])                                            # cut inside the pixel data
    bad.append(ok[:10] + (2 ** 31 - 1).to_bytes(4, "little") + ok[14:])     # pixel-data offset far outside the file
    bad.append(ok[:14] + (5000).to_bytes(4, "little") + ok[18:])            # info-header size larger than the file
    bad.append(ok[:10] + (20).to_bytes(4, "little") + ok[14:])              # pixel data overlapping the header
    for i, b in enumerate(bad):
        f = tmp_path / ("bad%d.bmp" % i)
        f.write_bytes(b)
        for reader in (s3.read_bmp8, s3.read_bmp_bgr):
            with pytest.raises(s3.Scan3DError):
                reader(str(f))
