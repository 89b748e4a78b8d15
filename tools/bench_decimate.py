#!/usr/bin/env python
"""Cost of simplifying the voxel surface (scan3d_voxel_surface_decimate) on workloads A and B of tools/bench_surface.py
(same scan, views, voxel size, R = 2 voxels and max_points = 1.25x the lattice points):
    python tools/bench_decimate.py [REPS] > profiles/r3_bench_decimate.json

The input is A's largest component (scan3d_voxel_surface_components with max_components = 1, what a user keeps of
whole views) and B's whole surface.  The call replaces the held surface in place and a surface is simplified once,
so every timed repetition first extracts (and for A cleans) the surface again, untimed, and then times one
scan3d_voxel_surface_decimate call plus a stream synchronise with the host clock, after a warm-up.  Cell sizes are
2, 4 and 8 voxels.  One extraction is timed the same way, for the ratio.  The device bytes are the drop of the
device's free memory over the first simplification, which allocates every buffer the entry owns.  A separate
torch.profiler pass over one call at 4 voxels gives the per-kernel split."""
import json
import os
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "tools"))
sys.dont_write_bytecode = True
import bench_surface as bs  # noqa: E402

import numpy as np  # noqa: E402
import torch  # noqa: E402

REPS = int(sys.argv[1]) if len(sys.argv) > 1 else 10
RATIOS = (2, 4, 8)


def host_ms(fn):
    t0 = time.perf_counter()
    out = fn()
    return out, 1e3 * (time.perf_counter() - t0)


def run(name, ctx, views, voxel, largest):
    ctx.voxel_begin(voxel, sum(v[0].shape[0] for v in views))
    for v in views:
        ctx.voxel_add_dev(*v)
    ctx.voxel_finish()
    voxels, _ = ctx.voxel_count()
    R = 2.0 * voxel
    for per_voxel in (16, 32, 48):                     # at most 64 lattice points per voxel
        try:
            first = ctx.voxel_surface(R, min(per_voxel * voxels, 2 ** 31 - 1))
            break
        except bs.s3.Scan3DError:
            pass
    max_points = int(1.25 * first["lattice_points"])

    def extract():
        r = ctx.voxel_surface(R, max_points)
        ctx.sync()
        return r

    def prepare():
        r = extract()
        if largest:
            r = ctx.surface_components(0, 1)
        ctx.sync()
        return r

    def decimate(cell):
        r = ctx.surface_decimate(cell)
        ctx.sync()
        return r

    src = prepare()
    free0 = torch.cuda.mem_get_info()[0]
    decimate(4 * voxel)                                  # warm-up; allocates every buffer
    device_bytes = free0 - torch.cuda.mem_get_info()[0]
    out = dict(workload=name, input="largest component" if largest else "whole surface", views=len(views),
               voxels=voxels, voxel_size=round(voxel, 6), max_distance=round(R, 6), max_points=max_points,
               vertices_in=src["vertices"], faces_in=src["faces"], reps=REPS, device_bytes=int(device_bytes),
               device_bytes_per_input_vertex=round(device_bytes / max(src["vertices"], 1), 1))
    ext = [host_ms(extract)[1] for _ in range(3)]
    out["ms_per_extraction"] = round(float(np.median(ext)), 2)
    for r in RATIOS:
        times = []
        for _ in range(REPS):
            prepare()
            res, t = host_ms(lambda: decimate(r * voxel))
            times.append(t)
        out[f"H = {r} s"] = dict(ms_per_call=round(float(np.median(times)), 2),
                                 spread_ms=[round(min(times), 2), round(max(times), 2)], result=res,
                                 face_reduction=round(src["faces"] / max(res["faces"], 1), 2))
    out["ms_ratio_to_extraction_at_4s"] = round(out["H = 4 s"]["ms_per_call"] / out["ms_per_extraction"], 4)
    from torch.profiler import ProfilerActivity, profile
    prepare()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        decimate(4 * voxel)
    split = {}
    for e in prof.key_averages():
        t = getattr(e, "self_device_time_total", 0)
        if t > 0:
            split[e.key[:60]] = dict(us=round(t, 1), calls=e.count)
    out["kernel_split_us_at_4s"] = split
    return out


def main():
    ctx, stack, roi, truth, params = bs.setup()
    name, plim = bs.gpu_info()
    result = dict(kernel="scan3d_voxel_surface_decimate + stream synchronise (host clock)",
                  scan="4096x3000 c3 synthetic scan, 8-step, 10+10 bits, fast triangulation, seed 0x3D5CA9, texture, mesh",
                  gpu=name, power_limit=plim)
    views, voxel = bs.workload_a(ctx, stack, roi)
    result["A"] = run("A: 8 whole views at 45 deg", ctx, views, voxel, largest=True)
    print(json.dumps(result["A"]), file=sys.stderr, flush=True)
    del views
    torch.cuda.synchronize()
    views = bs.workload_b(ctx, stack, roi, truth, params)
    del stack, truth
    result["B"] = run("B: 36 sphere-only views at 10 deg", ctx, views, voxel, largest=False)
    print(json.dumps(result, indent=1), flush=True)
    ctx.close()


if __name__ == "__main__":
    main()
