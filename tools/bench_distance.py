#!/usr/bin/env python
"""Cost and result of the sample-to-surface distances (scan3d_voxel_surface_distance, scan3d_voxel_surface_distance_dev,
scan3d_mesh_distance_dev) on the workloads of tools/bench_orient.py (same scan, views, voxel size; the extraction's
R = 2 voxels and max_points = 1.25x the lattice points; the distances' max_distance R = 2 voxels too):
    python tools/bench_distance.py > profiles/r3_bench_distance.json

  model -> A raw         the merged model (voxels with a normal) against A's largest component
  model -> A decimated   ... after scan3d_voxel_surface_decimate at 4 voxels
  model -> A smoothed    ... after scan3d_voxel_surface_smooth, 10 iterations
  model -> A filled      ... after scan3d_voxel_surface_fill_holes (max_edges 22)
  model -> B             B's model against B's whole surface
  C3 view -> A           a registered view's points (device_points of view 0) against A's raw component, dev route
  A raw <-> A decimated  the vertices of each against the other's faces, mesh route, both ways
Every timed repetition first rebuilds its input, untimed, then times one call (which synchronises twice) with the host
clock, after a warm-up; the median of 5 and the spread are reported, and a separate torch.profiler pass over one call
gives the per-kernel split.  The deviation figures (max = the one-sided Hausdorff distance within R, mean, RMS, the
signed extremes, the share inside) are the point: how far decimation, smoothing and filling move A from its data.  One
extraction of A is timed the same way for the aim: model -> A raw in at most 10 % of it."""
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


def _figures(res, voxel):
    out = dict(res)
    for k in ("max", "mean", "rms", "min_signed", "max_signed"):
        out[k + "_voxels"] = round(res[k] / voxel, 4)
    out["inside_share"] = round(res["inside"] / res["matched"], 4) if res["matched"] else 0.0
    return out


def _mesh(ctx):
    xyz, _, _, faces = ctx.voxel_surface_mesh()
    return torch.from_numpy(np.ascontiguousarray(xyz)).cuda(), torch.from_numpy(np.ascontiguousarray(faces)).cuda()


def surface_workloads(ctx, views, voxel, largest, stages, view_points=None):
    ctx.voxel_begin(voxel, sum(v[0].shape[0] for v in views))
    for v in views:
        ctx.voxel_add_dev(*v)
    ctx.voxel_finish()
    voxels, _ = ctx.voxel_count()
    R = 2.0 * voxel
    for per_voxel in (16, 32, 48):
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
    outs, meshes = {}, {}
    for name, stage in stages:
        def prepare():
            r = extract()
            if largest:
                r = ctx.surface_components(0, 1)
            if stage == "decimated":
                r = ctx.surface_decimate(4 * voxel)
            elif stage == "smoothed":
                r = ctx.surface_smooth(10)
            elif stage == "filled":
                r = ctx.surface_fill_holes(22)
            ctx.sync()
            return r
        src = prepare()
        meshes[stage] = _mesh(ctx)
        out = dict(input=("largest component" if largest else "whole surface") + ("" if stage == "raw" else ", " + stage),
                   views=len(views), voxels=voxels, voxel_size=round(voxel, 6), vertices=src["vertices"],
                   faces=src["faces"], max_distance=round(R, 6), ms_per_extraction=ms_extraction)
        out["distance"] = {}
        bf.measure(out["distance"], prepare, lambda: ctx.surface_distance(R))
        out["distance"]["ms_over_extraction"] = round(out["distance"]["ms_per_call"] / ms_extraction, 4)
        out["deviation"] = _figures(out["distance"]["result"], voxel)
        outs[name] = out
        print(json.dumps(out), file=sys.stderr, flush=True)
    if view_points is not None:
        def prepare_raw():
            extract()
            if largest:
                ctx.surface_components(0, 1)
            ctx.sync()
        out = dict(input="view 0's registered points against A's largest component (scan3d_voxel_surface_distance_dev)",
                   samples=int(view_points.shape[0]), max_distance=round(R, 6), distance={})
        bf.measure(out["distance"], prepare_raw, lambda: ctx.surface_distance_dev(view_points, R)[2])
        out["deviation"] = _figures(out["distance"]["result"], voxel)
        outs["C3 view -> A"] = out
        print(json.dumps(out), file=sys.stderr, flush=True)
    if "raw" in meshes and "decimated" in meshes:
        for a, b in (("raw", "decimated"), ("decimated", "raw")):
            (sx, _), (tx, tf) = meshes[a], meshes[b]
            out = dict(input=f"A {a} vertices against A {b} faces (scan3d_mesh_distance_dev)", samples=int(sx.shape[0]),
                       faces=int(tf.shape[0]), max_distance=round(R, 6), distance={})
            bf.measure(out["distance"], torch.cuda.synchronize, lambda: ctx.mesh_distance_dev(sx, tx, tf, R)[2])
            out["deviation"] = _figures(out["distance"]["result"], voxel)
            outs[f"A {a} -> A {b}"] = out
            print(json.dumps(out), file=sys.stderr, flush=True)
    return outs


def main():
    ctx, stack, roi, truth, params = bs.setup()
    name, plim = bs.gpu_info()
    result = dict(kernel="scan3d_voxel_surface_distance, scan3d_voxel_surface_distance_dev, scan3d_mesh_distance_dev "
                         "(host clock, two synchronisations)",
                  scan="4096x3000 c3 synthetic scan, 8-step, 10+10 bits, fast triangulation, seed 0x3D5CA9, texture, mesh",
                  gpu=name, power_limit=plim)
    views, voxel = bs.workload_a(ctx, stack, roi)
    result.update(surface_workloads(ctx, views, voxel, True,
                                    [("model -> A raw", "raw"), ("model -> A decimated", "decimated"),
                                     ("model -> A smoothed", "smoothed"), ("model -> A filled", "filled")],
                                    view_points=views[0][0]))
    del views
    torch.cuda.synchronize()
    views = bs.workload_b(ctx, stack, roi, truth, params)
    del stack, truth
    result.update(surface_workloads(ctx, views, voxel, False, [("model -> B", "raw")]))
    a = result["model -> A raw"]
    result["aim"] = dict(rule="model -> A's largest component in at most 10 % of A's extraction",
                         ratio=a["distance"]["ms_over_extraction"], met=a["distance"]["ms_over_extraction"] <= 0.10)
    print(json.dumps(result, indent=1), flush=True)
    ctx.close()


if __name__ == "__main__":
    main()
