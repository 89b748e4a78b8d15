#!/usr/bin/env python
"""Cost of the non-manifold repair (scan3d_voxel_surface_repair, scan3d_mesh_repair_dev) with both steps on the
workloads of tools/bench_fill.py (same scan, views, voxel size, R = 2 voxels and max_points = 1.25x the lattice
points):
    python tools/bench_repair.py [REPS] > profiles/r3_bench_repair.json

  A raw        A's largest component (scan3d_voxel_surface_components with max_components = 1)
  A decimated  the same after scan3d_voxel_surface_decimate at 4 voxels, where clusters join sheets
  B            B's whole surface
  C3           the camera-grid mesh of view 0 of the c3 scan (scan3d_build_mesh, no edge limit) through
               scan3d_mesh_repair_dev, into preallocated outputs of n_faces face rows and 3 n_faces source rows
Every timed repetition first rebuilds its input, untimed, then times one call (which synchronises twice) with the host
clock, after a warm-up; the median of REPS (default 5) and the spread are reported.  A separate torch.profiler pass
over one call gives the per-kernel split.  Each workload also reports the open_edges of a hole fill (max_edges 22 on
an unrefined surface, else 1024) without and with the repair first.  One extraction of A is timed the same way for
the aim: a repair of A in at most 10 % of it."""
import ctypes as C
import json
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
            ctx.sync()
            return r
        src = prepare()
        max_edges = 1024 if decimated else 22
        out = dict(input=("largest component" if largest else "whole surface") + (", decimated at 4 voxels" if
                                                                                  decimated else ""),
                   views=len(views), voxels=voxels, voxel_size=round(voxel, 6), vertices=src["vertices"],
                   faces=src["faces"], ms_per_extraction=ms_extraction)
        bf.measure(out, prepare, lambda: ctx.surface_repair())
        out["ms_over_extraction"] = round(out["ms_per_call"] / ms_extraction, 4)
        prepare()
        without = ctx.surface_fill_holes(max_edges)
        prepare()
        ctx.surface_repair()
        with_repair = ctx.surface_fill_holes(max_edges)
        out["fill"] = dict(max_edges=max_edges, without_repair=without, after_repair=with_repair)
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
            state["src"] = torch.empty(max(3 * nf.value, 1), dtype=torch.int32, device="cuda")
        torch.cuda.synchronize()

    def repair():
        r = s3.RepairResultC()
        ctx._ck(L.scan3d_mesh_repair_dev(h, L.scan3d_device_points(h), state["n"], L.scan3d_device_mesh_faces(h),
                                         state["nf"], s3.REPAIR_FACES | s3.REPAIR_VERTICES,
                                         C.c_void_p(state["out"].data_ptr()), C.c_void_p(state["src"].data_ptr()),
                                         3 * state["nf"], C.byref(r)))
        return s3.Scan3D._repair_result(r)

    prepare()
    out = dict(input="camera-grid mesh of view 0 (scan3d_mesh_repair_dev)", vertices=state["n"], faces=state["nf"])
    bf.measure(out, prepare, repair)
    # the fill of the mesh as it is, and of the repaired mesh with the copies appended to the points
    prepare()
    res = repair()
    pts_view = torch.from_numpy(ctx.points()).cuda()
    faces_view = torch.from_numpy(ctx.mesh()[0]).cuda()
    without = ctx.mesh_fill_holes_dev(pts_view, faces_view, 1024)[1]
    rep_pts = torch.cat([pts_view, pts_view[state["src"][:res["vertices_added"]].long()]]).contiguous()
    with_repair = ctx.mesh_fill_holes_dev(rep_pts, state["out"][:res["faces"]].contiguous(), 1024)[1]
    out["fill"] = dict(max_edges=1024, without_repair=without, after_repair=with_repair)
    return out


def main():
    ctx, stack, roi, truth, params = bs.setup()
    name, plim = bs.gpu_info()
    result = dict(kernel="scan3d_voxel_surface_repair / scan3d_mesh_repair_dev, both steps (host clock, two "
                         "synchronises)",
                  scan="4096x3000 c3 synthetic scan, 8-step, 10+10 bits, fast triangulation, seed 0x3D5CA9, texture, mesh",
                  gpu=name, power_limit=plim)
    result["C3"] = camera_workload(ctx, stack, roi)
    print(json.dumps(result["C3"]), file=sys.stderr, flush=True)
    views, voxel = bs.workload_a(ctx, stack, roi)
    result.update(surface_workloads(ctx, views, voxel, True, [("A raw", False), ("A decimated", True)]))
    del views
    torch.cuda.synchronize()
    views = bs.workload_b(ctx, stack, roi, truth, params)
    del stack, truth
    result.update(surface_workloads(ctx, views, voxel, False, [("B", False)]))
    a = result["A raw"]
    result["aim"] = dict(rule="a repair of A's largest component in at most 10 % of A's extraction",
                         raw_ratio=a["ms_over_extraction"], met=a["ms_over_extraction"] <= 0.10)
    print(json.dumps(result, indent=1), flush=True)
    ctx.close()


if __name__ == "__main__":
    main()
