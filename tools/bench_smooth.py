#!/usr/bin/env python
"""Cost of smoothing (scan3d_voxel_surface_smooth, scan3d_mesh_smooth_dev) on the workloads of tools/bench_surface.py
(same scan, views, voxel size, R = 2 voxels and max_points = 1.25x the lattice points):
    python tools/bench_smooth.py [REPS] > profiles/r3_bench_smooth.json

  A   A's largest component (scan3d_voxel_surface_components with max_components = 1, what a user keeps of whole views)
  B   B's whole surface
  C3  the camera-grid mesh of view 0 of the c3 scan (scan3d_build_mesh, no edge limit), smoothed in place on the ctx's
      own buffers through scan3d_mesh_smooth_dev
Every timed repetition first rebuilds its input, untimed (a new extraction, or a new reconstruct and mesh), then times
one call plus a stream synchronise with the host clock, after a warm-up; the median and the spread are reported, at
iterations 1, 10 and 50 with MeshLab's lambda = 0.5, mu = -0.53.  ms per pass is the slope between 10 and 50
iterations (80 passes).  The context's smoothing buffers are grow-only and shared by the three workloads (run in the
order C3, A, B), so device_bytes_growth is only what a workload's first call added (the drop of the device's free
memory); device_bytes_owned is what the context holds for the workload by include/scan3d.h's sizes (81 B per vertex,
96 B per face, and for a surface 24 B per vertex of the spare surface set).  A separate torch.profiler pass
over one call at 10 iterations gives the per-kernel split, and the gather's bytes per pass (neighbour rows at 4 B and neighbour positions at 24 B per row entry,
then degree, row end, held flag, own position and the write at 57 B per vertex) over its mean kernel time give its rate.
Those are the bytes the algorithm reads, not DRAM traffic: neighbours are mostly close in index order, so many of the
position loads hit L2 and the rate can exceed HBM's.
One extraction of A is timed the same way for the aim: 10 iterations in at most 10 % of it."""
import json
import os
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "tools"))
sys.dont_write_bytecode = True
import bench_surface as bs  # noqa: E402

import ctypes as C  # noqa: E402

import numpy as np  # noqa: E402
import torch  # noqa: E402

s3 = bs.s3
REPS = int(sys.argv[1]) if len(sys.argv) > 1 else 10
ITERATIONS = (1, 10, 50)


def host_ms(fn):
    t0 = time.perf_counter()
    out = fn()
    return out, 1e3 * (time.perf_counter() - t0)


def row_entries(faces):
    """twice the distinct undirected edges of faces [f][3] (numpy int32), counted on the GPU"""
    f = torch.from_numpy(np.ascontiguousarray(faces)).cuda().long()
    a = torch.cat([f[:, 0], f[:, 1], f[:, 2]])
    b = torch.cat([f[:, 1], f[:, 2], f[:, 0]])
    keep = a != b
    a, b = a[keep], b[keep]
    key = torch.minimum(a, b) * (1 << 32) + torch.maximum(a, b)
    return 2 * int(torch.unique(key).numel())


def measure(out, n_vertices, n_faces, entries, prepare, smooth, surface):
    """fills out with the timings, bytes and split of smooth(iterations) on inputs rebuilt by prepare()"""
    prepare()
    torch.cuda.synchronize()
    free0 = torch.cuda.mem_get_info()[0]
    smooth(10)                                           # warm-up; allocates every buffer
    out["device_bytes_growth"] = int(free0 - torch.cuda.mem_get_info()[0])
    out["device_bytes_owned"] = (81 + (24 if surface else 0)) * max(n_vertices, 1) + 16 * max(6 * n_faces, 64)
    out.update(vertices=n_vertices, faces=n_faces, row_entries=entries, reps=REPS)
    for it in ITERATIONS:
        times = []
        for _ in range(REPS):
            prepare()
            res, t = host_ms(lambda: smooth(it))
            times.append(t)
        out[f"iterations {it}"] = dict(ms_per_call=round(float(np.median(times)), 3),
                                       spread_ms=[round(min(times), 3), round(max(times), 3)], result=res)
    t10, t50 = out["iterations 10"]["ms_per_call"], out["iterations 50"]["ms_per_call"]
    out["ms_per_pass"] = round((t50 - t10) / 80, 4)
    from torch.profiler import ProfilerActivity, profile
    prepare()
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        smooth(10)
    split = {}
    for e in prof.key_averages():
        t = getattr(e, "self_device_time_total", 0)
        if t > 0:
            split[e.key[:60]] = dict(us=round(t, 1), calls=e.count)
    out["kernel_split_us_at_10"] = split
    gather = [v for k, v in split.items() if "k_sm_pass" in k]
    if gather:
        us = gather[0]["us"] / gather[0]["calls"]
        nbytes = 28 * entries + 57 * n_vertices
        out["gather"] = dict(us_per_pass=round(us, 2), bytes_per_pass=nbytes,
                             gb_per_s=round(nbytes / (us * 1e-6) / 1e9, 1))


def surface_workload(name, ctx, views, voxel, largest):
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

    def prepare():
        r = extract()
        if largest:
            r = ctx.surface_components(0, 1)
        ctx.sync()
        return r

    def smooth(it):
        r = ctx.surface_smooth(it)
        ctx.sync()
        return r

    src = prepare()
    entries = row_entries(ctx.voxel_surface_mesh()[3])
    out = dict(workload=name, input="largest component" if largest else "whole surface", views=len(views),
               voxels=voxels, voxel_size=round(voxel, 6), max_distance=round(R, 6), max_points=max_points)
    extract()
    out["ms_per_extraction"] = round(float(np.median([host_ms(extract)[1] for _ in range(max(REPS // 2, 3))])), 2)
    measure(out, src["vertices"], src["faces"], entries, prepare, smooth, surface=True)
    out["ms_10_iterations_over_extraction"] = round(out["iterations 10"]["ms_per_call"] / out["ms_per_extraction"], 4)
    return out


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

    def smooth(it):
        p, r = s3.SmoothParams(it, 0.5, -0.53), s3.SmoothResultC()
        ctx._ck(L.scan3d_mesh_smooth_dev(h, L.scan3d_device_points(h), L.scan3d_device_point_normals(h), state["n"],
                                         L.scan3d_device_mesh_faces(h), state["nf"], C.byref(p), C.byref(r)))
        return s3.Scan3D._smooth_result(r)

    prepare()
    entries = row_entries(ctx.mesh()[0])
    out = dict(workload="C3: camera-grid mesh of view 0 (scan3d_mesh_smooth_dev, in place)")
    measure(out, state["n"], state["nf"], entries, prepare, smooth, surface=False)
    return out


def main():
    ctx, stack, roi, truth, params = bs.setup()
    name, plim = bs.gpu_info()
    result = dict(kernel="scan3d_voxel_surface_smooth / scan3d_mesh_smooth_dev + stream synchronise (host clock)",
                  scan="4096x3000 c3 synthetic scan, 8-step, 10+10 bits, fast triangulation, seed 0x3D5CA9, texture, mesh",
                  gpu=name, power_limit=plim)
    result["C3"] = camera_workload(ctx, stack, roi)
    print(json.dumps(result["C3"]), file=sys.stderr, flush=True)
    views, voxel = bs.workload_a(ctx, stack, roi)
    result["A"] = surface_workload("A: 8 whole views at 45 deg", ctx, views, voxel, largest=True)
    print(json.dumps(result["A"]), file=sys.stderr, flush=True)
    del views
    torch.cuda.synchronize()
    views = bs.workload_b(ctx, stack, roi, truth, params)
    del stack, truth
    result["B"] = surface_workload("B: 36 sphere-only views at 10 deg", ctx, views, voxel, largest=False)
    a = result["A"]
    result["aim"] = dict(rule="10 lambda|mu iterations on A's largest component in at most 10 % of A's extraction",
                         ratio=a["ms_10_iterations_over_extraction"], met=a["ms_10_iterations_over_extraction"] <= 0.10)
    print(json.dumps(result, indent=1), flush=True)
    ctx.close()


if __name__ == "__main__":
    main()
