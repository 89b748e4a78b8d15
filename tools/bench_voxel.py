#!/usr/bin/env python
"""Throughput of the voxel-grid merge (scan3d_voxel_begin / add_points_dev / finish) on the 12 MP configuration
(bench.py's c3 workload, fast triangulation mode, seed 0x3D5CA9, a texture set and a mesh built for every view):
    python tools/bench_voxel.py [REPS] > profiles/r3_bench_voxel.json

Two workloads, reconstructed with scan3d_set_registration about the sphere centre into device buffers before any
timing (points, mesh normals, colours copied out of the context):
  A  throughput:     8 whole views at 45 degree steps (~8.7 M points each)
  B  heavy overlap: 36 views of the sphere alone (ROI = pixels whose truth point lies on it) at 10 degree steps
The voxel is 2x the median distance between horizontally adjacent points of view 0; max_voxels is 1.25x the voxel
count of an untimed first pass.  Each repetition times begin + every add + finish with CUDA events on the ctx stream
(after a warm-up repetition); the adds and the finish are also timed on their own.  Bytes are algorithmic: 27 B per
input point (xyz, normal, rgb read once) and 31 B per output voxel (xyz, normal, rgb, count written once).
A separate, untimed torch.profiler pass over one repetition gives the per-kernel split."""
import importlib
import json
import os
import subprocess
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
for p in (ROOT, os.path.join(ROOT, "tests")):
    sys.path.insert(0, p)
sys.dont_write_bytecode = True
s3 = importlib.import_module("3dscan_b200")
from helpers import load_calib_c1, scaled_calib   # noqa: E402  (calibration fixture only)

import torch  # noqa: E402

W, H, PW, PH = 4096, 3000, 4096, 3000
REPS = int(sys.argv[1]) if len(sys.argv) > 1 else 10
CENTRE = (60.0, 40.0, -30.0)
peak = 6456.0
try:
    peak = float(json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))["hbm_gbs"])
except Exception:
    pass


def gpu_info():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i", "0"],
                             capture_output=True, text=True, timeout=30).stdout.strip()
        name, plim = [x.strip() for x in out.split(",")]
        return name, plim
    except Exception:
        return torch.cuda.get_device_name(0), None


def capture_views(ctx, stack, roi, angles):
    """(xyz, normals, rgb) device tensors of each registered view, and the point counts"""
    views = []
    for theta in angles:
        ctx.set_registration(True, theta, *CENTRE)
        n = ctx.reconstruct(stack, roi)
        ctx.build_mesh(float("inf"))
        ctx.sync()
        L, h = ctx.L, ctx.h
        xyz = s3.wrap_device(ctx.device_points(), (n, 3), "<f4").clone()
        nrm = s3.wrap_device(L.scan3d_device_point_normals(h), (n, 3), "<f4").clone()
        _, rgb = ctx.points(want_rgb=True)
        views.append((xyz, nrm, torch.from_numpy(rgb).cuda()))
    torch.cuda.synchronize()
    return views


def median_spacing(ctx, xyz0):
    """median distance between horizontally adjacent valid pixels' points of the last reconstruct (view 0 here)"""
    pix = np.flatnonzero(ctx.plane(s3.PLANE_VALID).reshape(-1))
    p = xyz0.cpu().numpy().astype(np.float64)
    adj = (pix[1:] == pix[:-1] + 1) & (pix[1:] % W != 0)
    d = np.linalg.norm(p[1:][adj] - p[:-1][adj], axis=1)
    return float(np.median(d[d > 0]))


def merge(ctx, views, voxel, max_voxels, ev=None):
    if ev:
        ev[0].record(stream)
    ctx.voxel_begin(voxel, max_voxels)
    if ev:
        ev[1].record(stream)
    for xyz, nrm, rgb in views:
        ctx.voxel_add_dev(xyz, nrm, rgb)
    if ev:
        ev[2].record(stream)
    ctx.voxel_finish()
    if ev:
        ev[3].record(stream)


def run(name, ctx, views, voxel):
    points = sum(v[0].shape[0] for v in views)
    merge(ctx, views, voxel, points)                      # untimed first pass: the voxel count
    voxels, dropped = ctx.voxel_count()
    max_voxels = int(1.25 * voxels)
    merge(ctx, views, voxel, max_voxels)                  # warm-up at the timed capacity
    ctx.sync()
    t_all, t_begin, t_adds, t_fin = [], [], [], []
    for _ in range(REPS):
        ev = [torch.cuda.Event(enable_timing=True) for _ in range(4)]
        merge(ctx, views, voxel, max_voxels, ev)
        ev[3].synchronize()
        t_all.append(ev[0].elapsed_time(ev[3]) * 1e3)
        t_begin.append(ev[0].elapsed_time(ev[1]) * 1e3)
        t_adds.append(ev[1].elapsed_time(ev[2]) * 1e3)
        t_fin.append(ev[2].elapsed_time(ev[3]) * 1e3)
    assert ctx.voxel_count() == (voxels, dropped)
    us = float(np.median(t_all))
    add_us = float(np.median(t_adds)) / len(views)
    nbytes = 27 * points + 31 * voxels
    add_bytes = 27 * points / len(views)
    res = dict(workload=name, views=len(views), points=points, voxel_size=round(voxel, 6), max_voxels=max_voxels,
               voxels=voxels, dropped=dropped, reps=REPS,
               us_begin_adds_finish=round(us, 1), us_begin=round(float(np.median(t_begin)), 1),
               us_per_add=round(add_us, 1), us_finish=round(float(np.median(t_fin)), 1),
               spread_us=[round(min(t_all), 1), round(max(t_all), 1)],
               algorithmic_bytes=nbytes, achieved_gbs=round(nbytes / us / 1e3, 1),
               frac=round(nbytes / us / 1e3 / peak, 3),
               add_gbs=round(add_bytes / add_us / 1e3, 1), add_frac=round(add_bytes / add_us / 1e3 / peak, 3),
               peak_gbs=peak)
    # per-kernel split of one repetition, in a separate profiled pass
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        merge(ctx, views, voxel, max_voxels)
        ctx.sync()
    split = {}
    for e in prof.key_averages():
        t = getattr(e, "self_device_time_total", 0)
        if t > 0:
            split[e.key[:60]] = dict(us=round(t, 1), calls=e.count)
    res["kernel_split_us"] = split
    return res


c = scaled_calib(load_calib_c1(), W / 1600.0, PW / 1280.0)
cal = s3.make_calib(*[c[k] for k in ("Kc", "dc", "Kp", "dp", "rc", "tc", "rp", "tp")])
cfg = s3.make_config(W, H, PW, PH, 8, 10, 10, 4, 4, 2, flags=s3.FLAG_FAST_TRIANGULATION)
params = s3.default_synth_params(seed=0x3D5CA9)
stack, roi, truth = s3.synth_stack(cfg, cal, params, want_truth=True)
stream = torch.cuda.Stream()
ctx = s3.Scan3D(cfg, 0, cal, stream=stream.cuda_stream)
ctx.set_texture(np.random.default_rng(0x3D5CA9).integers(0, 256, (H, W, 3), dtype=np.uint8))

views_a = capture_views(ctx, stack, roi, [45.0 * k for k in range(8)])
ctx.set_registration(True, 0.0, *CENTRE)
ctx.reconstruct(stack, roi)
voxel = 2.0 * median_spacing(ctx, views_a[0][0])
on_sphere = np.abs(np.linalg.norm(truth.astype(np.float64) - np.array(CENTRE), axis=2) - params.sphere_r) < 1e-3
roi_b = (roi * on_sphere).astype(np.uint8)
views_b = capture_views(ctx, stack, roi_b, [10.0 * k for k in range(36)])
del stack, truth

name, plim = gpu_info()
out = dict(kernel="scan3d_voxel_begin + scan3d_voxel_add_points_dev per view + scan3d_voxel_finish",
           scan="4096x3000 c3 synthetic scan, 8-step, 10+10 bits, fast triangulation, seed 0x3D5CA9, texture, mesh",
           gpu=name, power_limit=plim, median_spacing_x2=round(voxel, 6),
           A=run("A: 8 whole views at 45 deg", ctx, views_a, voxel),
           B=run("B: 36 sphere-only views at 10 deg", ctx, views_b, voxel))
print(json.dumps(out, indent=1), flush=True)
ctx.close()
