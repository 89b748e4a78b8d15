#!/usr/bin/env python
"""Cost of hole filling (scan3d_voxel_surface_fill_holes, scan3d_mesh_fill_holes_dev) on the workloads of
tools/bench_surface.py (same scan, views, voxel size, R = 2 voxels and max_points = 1.25x the lattice points):
    python tools/bench_fill.py [REPS] > profiles/r3_bench_fill.json

  A raw       A's largest component (scan3d_voxel_surface_components with max_components = 1) at the unrefined
              surface's cap, max_edges = 22
  A smoothed  the same after 10 Taubin iterations (MeshLab's defaults), max_edges = 1024
  B           B's whole surface, max_edges = 22
  C3          the camera-grid mesh of view 0 of the c3 scan (scan3d_build_mesh, no edge limit) through
              scan3d_mesh_fill_holes_dev, max_edges = 1024, into a preallocated output of n_faces rows
Every timed repetition first rebuilds its input, untimed, then times one call (which synchronises twice) with the host
clock, after a warm-up; the median of REPS (default 5) and the spread are reported.  A separate torch.profiler pass
over one call gives the per-kernel split.  One extraction of A is timed the same way for the aim: a fill of A in at
most 10 % of it."""
import ctypes as C
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

s3 = bs.s3
REPS = int(sys.argv[1]) if len(sys.argv) > 1 else 5


def host_ms(fn):
    t0 = time.perf_counter()
    out = fn()
    return out, 1e3 * (time.perf_counter() - t0)


def measure(out, prepare, fill):
    """fills out with the median time, spread, result and kernel split of fill() on inputs rebuilt by prepare()"""
    prepare()
    fill()                                               # warm-up; allocates every buffer
    times = []
    for _ in range(REPS):
        prepare()
        res, t = host_ms(fill)
        times.append(t)
    out.update(reps=REPS, ms_per_call=round(float(np.median(times)), 3),
               spread_ms=[round(min(times), 3), round(max(times), 3)], result=res)
    from torch.profiler import ProfilerActivity, profile
    prepare()
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        fill()
    split = {}
    for e in prof.key_averages():
        t = getattr(e, "self_device_time_total", 0)
        if t > 0:
            split[e.key[:60]] = dict(us=round(t, 1), calls=e.count)
    out["kernel_split_us"] = split


def surface_workloads(ctx, views, voxel, largest, cases):
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
        except s3.Scan3DError:
            pass
    max_points = int(1.25 * first["lattice_points"])

    def extract():
        r = ctx.voxel_surface(R, max_points)
        ctx.sync()
        return r
    extract()
    ms_extraction = round(float(np.median([host_ms(extract)[1] for _ in range(3)])), 2)
    outs = {}
    for name, smoothed, max_edges in cases:
        def prepare():
            r = extract()
            if largest:
                r = ctx.surface_components(0, 1)
            if smoothed:
                ctx.surface_smooth(10)
            ctx.sync()
            return r
        src = prepare()
        out = dict(input=("largest component" if largest else "whole surface") + (", smoothed" if smoothed else ""),
                   views=len(views), voxels=voxels, voxel_size=round(voxel, 6), vertices=src["vertices"],
                   faces=src["faces"], max_edges=max_edges, ms_per_extraction=ms_extraction)
        measure(out, prepare, lambda: ctx.surface_fill_holes(max_edges))
        out["ms_over_extraction"] = round(out["ms_per_call"] / ms_extraction, 4)
        outs[name] = out
        print(json.dumps(out), file=sys.stderr, flush=True)
    return outs


def camera_workload(ctx, stack, roi):
    L, h = ctx.L, ctx.h
    state = {}

    def prepare():
        ctx.set_registration(True, 0.0, *bs.CENTRE)
        state["n"] = ctx.reconstruct(stack, roi)
        ctx.build_mesh(float("inf"))
        nf = C.c_int64()
        L.scan3d_mesh_face_count(h, C.byref(nf))
        state["nf"] = nf.value
        if state.get("out") is None or state["out"].shape[0] < max(nf.value, 1):
            state["out"] = torch.empty((max(nf.value, 1), 3), dtype=torch.int32, device="cuda")
        torch.cuda.synchronize()

    def fill():
        r = s3.FillResultC()
        ctx._ck(L.scan3d_mesh_fill_holes_dev(h, L.scan3d_device_points(h), state["n"], L.scan3d_device_mesh_faces(h),
                                             state["nf"], 1024, C.c_void_p(state["out"].data_ptr()), state["nf"],
                                             C.byref(r)))
        return s3.Scan3D._fill_result(r)

    prepare()
    out = dict(input="camera-grid mesh of view 0 (scan3d_mesh_fill_holes_dev)", vertices=state["n"], faces=state["nf"],
               max_edges=1024)
    measure(out, prepare, fill)
    return out


def main():
    ctx, stack, roi, truth, params = bs.setup()
    name, plim = bs.gpu_info()
    result = dict(kernel="scan3d_voxel_surface_fill_holes / scan3d_mesh_fill_holes_dev (host clock, two synchronises)",
                  scan="4096x3000 c3 synthetic scan, 8-step, 10+10 bits, fast triangulation, seed 0x3D5CA9, texture, mesh",
                  gpu=name, power_limit=plim)
    result["C3"] = camera_workload(ctx, stack, roi)
    print(json.dumps(result["C3"]), file=sys.stderr, flush=True)
    views, voxel = bs.workload_a(ctx, stack, roi)
    result.update(surface_workloads(ctx, views, voxel, True, [("A raw", False, 22), ("A smoothed", True, 1024)]))
    del views
    torch.cuda.synchronize()
    views = bs.workload_b(ctx, stack, roi, truth, params)
    del stack, truth
    result.update(surface_workloads(ctx, views, voxel, False, [("B", False, 22)]))
    a, b = result["A raw"], result["A smoothed"]
    result["aim"] = dict(rule="a fill of A's largest component in at most 10 % of A's extraction",
                         raw_ratio=a["ms_over_extraction"], smoothed_ratio=b["ms_over_extraction"],
                         met=max(a["ms_over_extraction"], b["ms_over_extraction"]) <= 0.10)
    print(json.dumps(result, indent=1), flush=True)
    ctx.close()


if __name__ == "__main__":
    main()
