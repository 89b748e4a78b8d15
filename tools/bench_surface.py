#!/usr/bin/env python
"""Cost of the surface extraction (scan3d_voxel_surface) on workloads A and B of tools/bench_voxel.py (the 12 MP c3
scan, fast triangulation, seed 0x3D5CA9, a texture and a mesh per view):
    python tools/bench_surface.py [REPS] > profiles/r3_bench_surface.json

  A  8 whole views at 45 degree steps (~24 M voxels)
  B  36 views of the sphere alone at 10 degree steps
The voxel is 2x the median distance between horizontally adjacent points of view 0 and R = 2 voxels.  Each workload is
merged once; an untimed first extraction at a generous max_points (16, 32 or 48 per voxel) gives the lattice point count, and the timed ones run
at max_points = 1.25x that count.  Each repetition times one scan3d_voxel_surface call (which synchronises once and
queues the emission) plus a stream synchronise with CUDA events on the ctx stream, after a warm-up.  A separate
torch.profiler pass over one extraction gives the per-kernel split.  Device memory is what torch.cuda.mem_get_info
reports in use beyond the merge before and after the first extraction (the ctx's surface buffers and the index)."""
import importlib
import json
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
for p in (ROOT, os.path.join(ROOT, "tests"), os.path.join(ROOT, "tools")):
    sys.path.insert(0, p)
sys.dont_write_bytecode = True
s3 = importlib.import_module("3dscan_b200")
from helpers import load_calib_c1, scaled_calib   # noqa: E402  (calibration fixture only)

import torch  # noqa: E402

W, H, PW, PH = 4096, 3000, 4096, 3000
REPS = int(sys.argv[1]) if len(sys.argv) > 1 else 10
CENTRE = (60.0, 40.0, -30.0)


def gpu_info():
    import subprocess
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i", "0"],
                             capture_output=True, text=True, timeout=30).stdout.strip()
        name, plim = [x.strip() for x in out.split(",")]
        return name, plim
    except Exception:
        return torch.cuda.get_device_name(0), None


def capture_views(ctx, stack, roi, angles):
    views = []
    for theta in angles:
        ctx.set_registration(True, theta, *CENTRE)
        n = ctx.reconstruct(stack, roi)
        ctx.build_mesh(float("inf"))
        ctx.sync()
        xyz = s3.wrap_device(ctx.device_points(), (n, 3), "<f4").clone()
        nrm = s3.wrap_device(ctx.L.scan3d_device_point_normals(ctx.h), (n, 3), "<f4").clone()
        _, rgb = ctx.points(want_rgb=True)
        views.append((xyz, nrm, torch.from_numpy(rgb).cuda()))
    torch.cuda.synchronize()
    return views


def median_spacing(ctx, xyz0):
    pix = np.flatnonzero(ctx.plane(s3.PLANE_VALID).reshape(-1))
    p = xyz0.cpu().numpy().astype(np.float64)
    adj = (pix[1:] == pix[:-1] + 1) & (pix[1:] % W != 0)
    d = np.linalg.norm(p[1:][adj] - p[:-1][adj], axis=1)
    return float(np.median(d[d > 0]))


def run(name, ctx, views, voxel):
    ctx.voxel_begin(voxel, sum(v[0].shape[0] for v in views))
    for v in views:
        ctx.voxel_add_dev(*v)
    ctx.voxel_finish()
    voxels, _ = ctx.voxel_count()
    R = 2.0 * voxel
    torch.cuda.synchronize()
    free0, _ = torch.cuda.mem_get_info()
    for per_voxel in (16, 32, 48):                     # at most 64 lattice points per voxel
        try:
            first = ctx.voxel_surface(R, min(per_voxel * voxels, 2 ** 31 - 1))
            break
        except s3.Scan3DError:
            pass
    ctx.sync()
    free1, _ = torch.cuda.mem_get_info()
    max_points = int(1.25 * first["lattice_points"])
    ctx.voxel_surface(R, max_points)                    # warm-up at the timed capacity
    ctx.sync()
    times = []
    for _ in range(REPS):
        ev = [torch.cuda.Event(enable_timing=True) for _ in range(2)]
        ev[0].record(stream)
        res = ctx.voxel_surface(R, max_points)
        ev[1].record(stream)
        ev[1].synchronize()
        times.append(ev[0].elapsed_time(ev[1]))
    assert res == first, (res, first)
    out = dict(workload=name, views=len(views), voxels=voxels, voxel_size=round(voxel, 6), max_distance=round(R, 6),
               max_points=max_points, reps=REPS, ms_per_extraction=round(float(np.median(times)), 2),
               spread_ms=[round(min(times), 2), round(max(times), 2)],
               lattice_points=first["lattice_points"], undefined_points=first["undefined_points"],
               lattice_points_per_voxel=round(first["lattice_points"] / voxels, 3),
               vertices=first["vertices"], faces=first["faces"],
               device_bytes_first_extraction=int(free0 - free1))
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        ctx.voxel_surface(R, max_points)
        ctx.sync()
    split = {}
    for e in prof.key_averages():
        t = getattr(e, "self_device_time_total", 0)
        if t > 0:
            split[e.key[:60]] = dict(us=round(t, 1), calls=e.count)
    out["kernel_split_us"] = split
    return out


def setup():
    """the ctx on its own stream and the c3 scan (stack, roi, truth, synth params) both workloads are captured from"""
    global stream
    c = scaled_calib(load_calib_c1(), W / 1600.0, PW / 1280.0)
    cal = s3.make_calib(*[c[k] for k in ("Kc", "dc", "Kp", "dp", "rc", "tc", "rp", "tp")])
    cfg = s3.make_config(W, H, PW, PH, 8, 10, 10, 4, 4, 2, flags=s3.FLAG_FAST_TRIANGULATION)
    params = s3.default_synth_params(seed=0x3D5CA9)
    stack, roi, truth = s3.synth_stack(cfg, cal, params, want_truth=True)
    stream = torch.cuda.Stream()
    ctx = s3.Scan3D(cfg, 0, cal, stream=stream.cuda_stream)
    ctx.set_texture(np.random.default_rng(0x3D5CA9).integers(0, 256, (H, W, 3), dtype=np.uint8))
    return ctx, stack, roi, truth, params


def workload_a(ctx, stack, roi):
    """(views, voxel size) of workload A"""
    views = capture_views(ctx, stack, roi, [45.0 * k for k in range(8)])
    ctx.set_registration(True, 0.0, *CENTRE)
    ctx.reconstruct(stack, roi)
    return views, 2.0 * median_spacing(ctx, views[0][0])


def workload_b(ctx, stack, roi, truth, params):
    """views of workload B (the voxel size is A's)"""
    on_sphere = np.abs(np.linalg.norm(truth.astype(np.float64) - np.array(CENTRE), axis=2) - params.sphere_r) < 1e-3
    roi_b = (roi * on_sphere).astype(np.uint8)
    return capture_views(ctx, stack, roi_b, [10.0 * k for k in range(36)])


def main():
    ctx, stack, roi, truth, params = setup()
    name, plim = gpu_info()
    result = dict(kernel="scan3d_voxel_surface (R = 2 voxels) + stream synchronise",
                  scan="4096x3000 c3 synthetic scan, 8-step, 10+10 bits, fast triangulation, seed 0x3D5CA9, texture, mesh",
                  gpu=name, power_limit=plim)
    views, voxel = workload_a(ctx, stack, roi)
    result["A"] = run("A: 8 whole views at 45 deg", ctx, views, voxel)
    del views
    torch.cuda.synchronize()
    views = workload_b(ctx, stack, roi, truth, params)
    del stack, truth
    result["B"] = run("B: 36 sphere-only views at 10 deg", ctx, views, voxel)
    print(json.dumps(result, indent=1), flush=True)
    ctx.close()


if __name__ == "__main__":
    main()
