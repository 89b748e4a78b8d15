#!/usr/bin/env python
"""Cost of the coherent orientation and of the measures (scan3d_voxel_surface_orient / _measure,
scan3d_mesh_orient_dev / scan3d_mesh_measure_dev) on the workloads of tools/bench_repair.py (same scan, views, voxel
size, R = 2 voxels and max_points = 1.25x the lattice points):
    python tools/bench_orient.py > profiles/r3_bench_orient.json

  A raw                  A's largest component (scan3d_voxel_surface_components with max_components = 1)
  A decimated repaired   the same after scan3d_voxel_surface_decimate at 4 voxels and a repair with both steps
  B                      B's whole surface, then filled (max_edges 22) for its area and volume
  C3                     the camera-grid mesh of view 0 of the c3 scan (scan3d_build_mesh, no edge limit) through the
                         dev routes, in place
Orientation and measure are timed separately: every timed repetition first rebuilds its input, untimed, then times one
call (which synchronises once) with the host clock, after a warm-up; the median of 5 and the spread are reported, and
a separate torch.profiler pass over one call gives the per-kernel split.  Each surface workload also reports the
open_edges of a hole fill without and with the orientation first.  B is the sphere of the default scene of
host/scan3d_synth.cpp, so its filled volume is compared with 4/3 pi r^3.  One extraction of A is timed the same way
for the aim: an orientation and a measure of A in at most 10 % of it each."""
import ctypes as C
import json
import math
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "tools"))
sys.dont_write_bytecode = True
import bench_fill as bf  # noqa: E402
import bench_surface as bs  # noqa: E402

import numpy as np  # noqa: E402
import torch  # noqa: E402

s3 = bs.s3


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
    ms_extraction = round(float(np.median([bf.host_ms(extract)[1] for _ in range(3)])), 2)
    outs = {}
    for name, decimated in cases:
        def prepare():
            r = extract()
            if largest:
                r = ctx.surface_components(0, 1)
            if decimated:
                r = ctx.surface_decimate(4 * voxel)
                r = ctx.surface_repair()
            ctx.sync()
            return r
        src = prepare()
        max_edges = 1024 if decimated else 22
        out = dict(input=("largest component" if largest else "whole surface") +
                   (", decimated at 4 voxels and repaired" if decimated else ""),
                   views=len(views), voxels=voxels, voxel_size=round(voxel, 6), vertices=src["vertices"],
                   faces=src["faces"], ms_per_extraction=ms_extraction)
        out["orient"], out["measure"] = {}, {}
        bf.measure(out["orient"], prepare, ctx.surface_orient)
        bf.measure(out["measure"], prepare, ctx.surface_measure)
        for k in ("orient", "measure"):
            out[k]["ms_over_extraction"] = round(out[k]["ms_per_call"] / ms_extraction, 4)
        prepare()
        without = ctx.surface_fill_holes(max_edges)
        measured = ctx.surface_measure()
        prepare()
        ctx.surface_orient()
        with_orient = ctx.surface_fill_holes(max_edges)
        out["fill"] = dict(max_edges=max_edges, without_orient=without, after_orient=with_orient,
                           measure_after_fill_without_orient=measured, measure_after_orient_and_fill=ctx.surface_measure())
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
        torch.cuda.synchronize()

    def orient():
        r = s3.OrientResultC()
        ctx._ck(L.scan3d_mesh_orient_dev(h, L.scan3d_device_points(h), None, state["n"], L.scan3d_device_mesh_faces(h),
                                         state["nf"], C.byref(r)))
        return s3.Scan3D._orient_result(r)

    def measure():
        r = s3.MeasureResultC()
        ctx._ck(L.scan3d_mesh_measure_dev(h, L.scan3d_device_points(h), state["n"], L.scan3d_device_mesh_faces(h),
                                          state["nf"], C.byref(r)))
        return s3.Scan3D._measure_result(r)

    prepare()
    out = dict(input="camera-grid mesh of view 0 (scan3d_mesh_orient_dev, scan3d_mesh_measure_dev)",
               vertices=state["n"], faces=state["nf"], orient={}, measure={})
    bf.measure(out["orient"], prepare, orient)
    bf.measure(out["measure"], prepare, measure)
    return out


def main():
    ctx, stack, roi, truth, params = bs.setup()
    name, plim = bs.gpu_info()
    result = dict(kernel="scan3d_voxel_surface_orient / _measure, scan3d_mesh_orient_dev / _measure_dev (host clock, "
                         "one synchronise)",
                  scan="4096x3000 c3 synthetic scan, 8-step, 10+10 bits, fast triangulation, seed 0x3D5CA9, texture, mesh",
                  gpu=name, power_limit=plim)
    result["C3"] = camera_workload(ctx, stack, roi)
    print(json.dumps(result["C3"]), file=sys.stderr, flush=True)
    views, voxel = bs.workload_a(ctx, stack, roi)
    result.update(surface_workloads(ctx, views, voxel, True, [("A raw", False), ("A decimated repaired", True)]))
    del views
    torch.cuda.synchronize()
    views = bs.workload_b(ctx, stack, roi, truth, params)
    del stack, truth
    result.update(surface_workloads(ctx, views, voxel, False, [("B", False)]))
    r = float(params.sphere_r)
    filled = result["B"]["fill"]["measure_after_orient_and_fill"]
    sphere = 4.0 / 3.0 * math.pi * r ** 3
    result["B sphere"] = dict(scene_sphere_radius=r, volume_4_3_pi_r3=sphere, filled_volume=filled["volume"],
                              filled_area=filled["area"], area_4_pi_r2=4.0 * math.pi * r * r,
                              volume_ratio=filled["volume"] / sphere, watertight=filled["watertight"])
    a = result["A raw"]
    result["aim"] = dict(rule="an orientation and a measure of A's largest component each in at most 10 % of A's "
                              "extraction",
                         orient_ratio=a["orient"]["ms_over_extraction"], measure_ratio=a["measure"]["ms_over_extraction"],
                         met=a["orient"]["ms_over_extraction"] <= 0.10 and a["measure"]["ms_over_extraction"] <= 0.10)
    print(json.dumps(result, indent=1), flush=True)
    ctx.close()


if __name__ == "__main__":
    main()
