#!/usr/bin/env python
"""Cost of the scan-to-model alignment (scan3d_align_to_voxels_dev) on the 12 MP configuration (bench.py's c3 workload,
fast triangulation mode, seed 0x3D5CA9, a texture set and a mesh built for every view):
    python tools/bench_align.py [REPS] > profiles/r3_bench_align.json

Model: tools/bench_voxel.py's workload A, 8 whole views registered at 45 degree steps about the sphere centre, merged
at 2x the median horizontal spacing.  Source: the 45 degree view once more, registered with a perturbed angle (45.3)
and pivot (+0.2 mm in x, -0.1 mm in z), ~8.7 M points in device memory; T_true maps it onto the model's copy of that
view.  Timed with CUDA events on the ctx stream after a warm-up (each timed call ends in the entry's synchronisation):
  index + 1 and index + 9 iterations at stride 1 and at stride 16, with the stop test off (every iteration runs), so
  one iteration = (t9 - t1) / 8 and the index build = t1 - one iteration;
  the whole coarse-to-fine alignment: max_distance 1.0 mm at stride 16, then 0.15 mm at stride 1 with T_init = I
  after the applied coarse call (default iteration limit and stop test), the source restored before each repetition.
A separate, untimed torch.profiler pass over one coarse-to-fine alignment gives the per-kernel split."""
import importlib
import json
import math
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
THETA, THETA_P, PIVOT_P = 45.0, 45.3, (CENTRE[0] + 0.2, CENTRE[1], CENTRE[2] - 0.1)
COARSE, FINE = dict(max_distance=1.0, stride=16), dict(max_distance=0.15, stride=1)


def gpu_info():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i", "0"],
                             capture_output=True, text=True, timeout=30).stdout.strip()
        name, plim = [x.strip() for x in out.split(",")]
        return name, plim
    except Exception:
        return torch.cuda.get_device_name(0), None


def registration(theta, pivot):
    """register_point_clouds' transform as a 4x4: p -> R (p - pivot) + pivot"""
    R = s3.register_rotation(theta).astype(np.float64)[:3, :3]
    T = np.eye(4)
    T[:3, :3] = R
    T[:3, 3] = np.asarray(pivot) - R @ np.asarray(pivot)
    return T


c = scaled_calib(load_calib_c1(), W / 1600.0, PW / 1280.0)
cal = s3.make_calib(*[c[k] for k in ("Kc", "dc", "Kp", "dp", "rc", "tc", "rp", "tp")])
cfg = s3.make_config(W, H, PW, PH, 8, 10, 10, 4, 4, 2, flags=s3.FLAG_FAST_TRIANGULATION)
params = s3.default_synth_params(seed=0x3D5CA9)
stack, roi = s3.synth_stack(cfg, cal, params)
stream = torch.cuda.Stream()
ctx = s3.Scan3D(cfg, 0, cal, stream=stream.cuda_stream)
ctx.set_texture(np.random.default_rng(0x3D5CA9).integers(0, 256, (H, W, 3), dtype=np.uint8))

# the model: workload A of tools/bench_voxel.py
views = []
for k in range(8):
    ctx.set_registration(True, 45.0 * k, *CENTRE)
    n = ctx.reconstruct(stack, roi)
    ctx.build_mesh(math.inf)
    ctx.sync()
    views.append((s3.wrap_device(ctx.device_points(), (n, 3), "<f4").clone(),
                  s3.wrap_device(ctx.L.scan3d_device_point_normals(ctx.h), (n, 3), "<f4").clone()))
    if k == 0:
        pix = np.flatnonzero(ctx.plane(s3.PLANE_VALID).reshape(-1))
        p0 = ctx.points().astype(np.float64)
        adj = (pix[1:] == pix[:-1] + 1) & (pix[1:] % W != 0)
        d = np.linalg.norm(p0[1:][adj] - p0[:-1][adj], axis=1)
        voxel = 2.0 * float(np.median(d[d > 0]))
torch.cuda.synchronize()
points = sum(v[0].shape[0] for v in views)
ctx.voxel_begin(voxel, points)
for xyz, nrm in views:
    ctx.voxel_add_dev(xyz, nrm)
ctx.voxel_finish()
voxels, _ = ctx.voxel_count()
ctx.voxel_begin(voxel, int(1.25 * voxels))
for xyz, nrm in views:
    ctx.voxel_add_dev(xyz, nrm)
ctx.voxel_finish()
assert ctx.voxel_count()[0] == voxels
del views

# the source
ctx.set_registration(True, THETA_P, *PIVOT_P)
n_src = ctx.reconstruct(stack, roi)
ctx.sync()
source = s3.wrap_device(ctx.device_points(), (n_src, 3), "<f4").clone()
work = source.clone()
del stack
T_true = registration(THETA, CENTRE) @ np.linalg.inv(registration(THETA_P, PIVOT_P))
torch.cuda.synchronize()


def timed(fn, reps=REPS):
    fn()                                                   # warm-up
    ts = []
    for _ in range(reps):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(stream)
        fn()
        e1.record(stream)
        e1.synchronize()
        ts.append(e0.elapsed_time(e1) * 1e3)
    return float(np.median(ts)), [round(min(ts), 1), round(max(ts), 1)]


def fixed(iters, stride):
    return lambda: ctx.align_dev(source, FINE["max_distance"], max_iterations=iters, stride=stride, apply=False,
                                 stop_rotation=0.0, stop_translation=0.0)


def coarse_to_fine():
    with torch.cuda.stream(stream):
        work.copy_(source)
    a = ctx.align_dev(work, **COARSE)
    b = ctx.align_dev(work, **FINE, T_init=np.eye(4))
    return a, b


res = dict(kernel="scan3d_align_to_voxels_dev", gpu=None, power_limit=None,
           scan="4096x3000 c3 synthetic scan, 8-step, 10+10 bits, fast triangulation, seed 0x3D5CA9, texture, mesh",
           model=f"tools/bench_voxel.py workload A: 8 views at 45 deg, {points} points -> {voxels} voxels",
           voxel_size=round(voxel, 6), source_points=n_src,
           source=f"the {THETA} deg view registered at {THETA_P} deg about pivot {PIVOT_P}",
           coarse=COARSE, fine=FINE, reps=REPS)
for stride in (1, 16):
    t1, s1 = timed(fixed(1, stride))
    t9, s9 = timed(fixed(9, stride))
    it = (t9 - t1) / 8
    res[f"stride{stride}"] = dict(samples=math.ceil(n_src / stride), us_index_plus_1_iteration=round(t1, 1),
                                  us_index_plus_9_iterations=round(t9, 1), us_per_iteration=round(it, 1),
                                  us_index=round(t1 - it, 1), spread_1=s1, spread_9=s9)
t_all, s_all = timed(coarse_to_fine)
a, b = coarse_to_fine()
T = b.T @ a.T
E = T @ np.linalg.inv(T_true)
res["coarse_to_fine"] = dict(
    us=round(t_all, 1), spread_us=s_all,
    coarse=dict(iterations=a.iterations, status=a.status, pairs_first=a.pairs_first, pairs_last=a.pairs_last,
                rms_first=a.rms_first, rms_last=a.rms_last),
    fine=dict(iterations=b.iterations, status=b.status, pairs_first=b.pairs_first, pairs_last=b.pairs_last,
              rms_first=b.rms_first, rms_last=b.rms_last),
    error_vs_T_true=dict(rotation_deg=float(np.degrees(np.arccos(np.clip((np.trace(E[:3, :3]) - 1) / 2, -1, 1)))),
                         translation_mm=float(np.linalg.norm(E[:3, 3]))))
# per-kernel split of one coarse-to-fine alignment, in a separate profiled pass
from torch.profiler import ProfilerActivity, profile  # noqa: E402
with profile(activities=[ProfilerActivity.CUDA]) as prof:
    coarse_to_fine()
    ctx.sync()
split = {}
for e in prof.key_averages():
    t = getattr(e, "self_device_time_total", 0)
    if t > 0:
        split[e.key[:60]] = dict(us=round(t, 1), calls=e.count)
res["kernel_split_us"] = split
res["gpu"], res["power_limit"] = gpu_info()
print(json.dumps(res, indent=1), flush=True)
ctx.close()
