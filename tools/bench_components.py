#!/usr/bin/env python
"""Cost of removing the isolated pieces of the voxel surface (scan3d_voxel_surface_components) on workloads A and B of
tools/bench_surface.py (same scan, views, voxel size, R = 2 voxels and max_points = 1.25x the lattice points):
    python tools/bench_components.py [REPS] > profiles/r3_bench_components.json

The call replaces the held surface in place, so every timed repetition first extracts the raw surface again (untimed)
and then times one scan3d_voxel_surface_components call plus a stream synchronise with the host clock, after a
warm-up.  The rules timed are (0, 0) (labels and counts, every vertex and face copied), min_faces = 1 and
max_components = 1.  One extraction is timed the same way, for the ratio.  A separate torch.profiler pass over one
max_components = 1 call on a raw surface gives the per-kernel split."""
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

REPS = int(sys.argv[1]) if len(sys.argv) > 1 else 5
RULES = {"all (0, 0)": (0, 0), "min_faces 1": (1, 0), "max_components 1": (0, 1)}


def host_ms(fn):
    t0 = time.perf_counter()
    out = fn()
    return out, 1e3 * (time.perf_counter() - t0)


def run(name, ctx, views, voxel):
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

    def clean(rule):
        r = ctx.surface_components(*rule)
        ctx.sync()
        return r

    extract()
    clean((0, 1))                                        # warm-up
    out = dict(workload=name, views=len(views), voxels=voxels, voxel_size=round(voxel, 6), max_distance=round(R, 6),
               max_points=max_points, vertices=first["vertices"], faces=first["faces"], reps=REPS)
    ext = [host_ms(extract)[1] for _ in range(3)]
    out["ms_per_extraction"] = round(float(np.median(ext)), 2)
    for label, rule in RULES.items():
        times = []
        for _ in range(REPS):
            extract()
            res, t = host_ms(lambda: clean(rule))
            times.append(t)
        out[label] = dict(ms_per_call=round(float(np.median(times)), 2),
                          spread_ms=[round(min(times), 2), round(max(times), 2)], result=res)
    res = out["max_components 1"]["result"]
    out["components"] = res["components"]
    out["largest_share_of_faces"] = round(res["largest_faces"] / max(first["faces"], 1), 6)
    out["ms_ratio_to_extraction"] = round(out["max_components 1"]["ms_per_call"] / out["ms_per_extraction"], 4)
    from torch.profiler import ProfilerActivity, profile
    extract()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        clean((0, 1))
    split = {}
    for e in prof.key_averages():
        t = getattr(e, "self_device_time_total", 0)
        if t > 0:
            split[e.key[:60]] = dict(us=round(t, 1), calls=e.count)
    out["kernel_split_us"] = split
    return out


def main():
    ctx, stack, roi, truth, params = bs.setup()
    name, plim = bs.gpu_info()
    result = dict(kernel="scan3d_voxel_surface_components + stream synchronise (host clock)",
                  scan="4096x3000 c3 synthetic scan, 8-step, 10+10 bits, fast triangulation, seed 0x3D5CA9, texture, mesh",
                  gpu=name, power_limit=plim)
    views, voxel = bs.workload_a(ctx, stack, roi)
    result["A"] = run("A: 8 whole views at 45 deg", ctx, views, voxel)
    print(json.dumps(result["A"]), file=sys.stderr, flush=True)
    del views
    torch.cuda.synchronize()
    views = bs.workload_b(ctx, stack, roi, truth, params)
    del stack, truth
    result["B"] = run("B: 36 sphere-only views at 10 deg", ctx, views, voxel)
    print(json.dumps(result, indent=1), flush=True)
    ctx.close()


if __name__ == "__main__":
    main()
