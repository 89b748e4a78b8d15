#!/usr/bin/env python
"""bench.py -- throughput of the reconstruction hot path (BASELINE.json metric) on N B200s.

  python bench.py --gpus N --steps K --warmup W          (N > 1: launched under torchrun)
  python bench.py --impl reference ...                    (CPU oracle port, rank 0 only)
  python bench.py ... --dump-outputs DIR                  (also write what the last timed step computed)

Workload: BASELINE.json configs[2] = synthetic 4096x3000 (12 MP) scans, vertical + horizontal,
8-step phase shift + 10-bit Gray code (56 u8 frames per scan).  A "step" is one pass of the hot
path over one batch of `--batch` scans per GPU, cycled over a ring of `--ring` distinct stacks
resident in HBM (ring bytes >> L2).  With N > 1 this is configs[3]: scans are sharded
frame-parallel, no collective on the data path (weak scaling: per-GPU work is fixed).

Printed JSON (one line, rank 0): value = whole-job Mpix/s with inputs resident in HBM; e2e = the
same metric through the host-buffer C-ABI entry (pinned host stack -> H2D -> kernel -> D2H of the
point cloud); roofline for the fused kernel; cpu_baseline = the oracle port on the host cores.
"""
import argparse
import importlib
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
for p in (ROOT, os.path.join(ROOT, "oracle"), os.path.join(ROOT, "tests")):
    if p not in sys.path:
        sys.path.insert(0, p)
sys.dont_write_bytecode = True      # the benchmark leaves the source tree as it found it (no __pycache__ in it)

import numpy as np

METRIC = "decoded+triangulated Mpix/s"
WORKLOADS = {
    # name: W, H, PW, PH, N, M_v, M_h, fw_v, fw_h, dirs
    "c3_12mp_8step_10bit_vh": (4096, 3000, 4096, 3000, 8, 10, 10, 4, 4, 2),
    "c2_1080p_3step_8bit_v": (1920, 1080, 1920, 1080, 3, 8, 8, 8, 8, 1),
    "c1_1600x1200_3step_6bit_vh": (1600, 1200, 1280, 720, 3, 6, 5, 32, 32, 2),
    # configs[4]: ONE 50 MP frame, row-sharded over the ranks, NCCL gather of the compacted points
    "c5_50mp_rowshard_8step_10bit_vh": (8192, 6144, 8192, 6144, 8, 10, 10, 8, 8, 2),
}


def algorithmic_bytes_per_pixel(N, M_v, M_h, dirs):
    """SURVEY.md 8(d): every input frame read once + 1 B ROI; per direction 4 B phase + 2 B fringe
    order; 1 B valid; both directions: 8 B c_p_map + 12 B point (f = 1 upper bound)."""
    reads = N + 2 * M_v + (N + 2 * M_h if dirs == 2 else 0) + 1
    writes = dirs * 6 + 1 + (20 if dirs == 2 else 0)
    return reads + writes


def measured_peak_gbs():
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            return float(json.load(f)["hbm_gbs"]), "measured"
    except Exception:
        return 6650.0, "fallback"


def ncu_traffic(workload):
    """dram bytes per launch of the fused kernel from the committed ncu capture, if any."""
    try:
        with open(os.path.join(ROOT, "profiles", "fused_kernel_ncu.json")) as f:
            d = json.load(f)
        return d.get(workload, {}).get("dram_bytes_per_launch")
    except Exception:
        return None


def host_threads():
    """All the host cores this process may run on (torchrun exports OMP_NUM_THREADS=1; the oracle
    takes an explicit thread count, so that setting does not throttle the CPU arm)."""
    try:
        return max(1, len(os.sched_getaffinity(0)))
    except AttributeError:
        return max(1, os.cpu_count() or 1)


class ClockSampler:
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.rows, self.proc, self.index = [], None, index

    def start(self):
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", "-i", str(self.index), "--query-gpu=" + self.Q,
                 "--format=csv,noheader,nounits", "-lms", "25"],
                stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._pump, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def wait_first_row(self, timeout=5.0):
        """nvidia-smi takes a few hundred ms to come up on a fresh box: do not start a short timed
        region before it delivers samples."""
        t_end = time.time() + timeout
        while self.proc and not self.rows and time.time() < t_end:
            time.sleep(0.02)

    def _pump(self):
        for line in self.proc.stdout:
            self.rows.append((time.time(), [x.strip() for x in line.split(",")]))

    def stop(self, t0, t1):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        return self.window(t0, t1)

    def window(self, t0, t1):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        rows = [r for t, r in self.rows if t0 <= t <= t1 + 0.05]
        window = "timed region"
        if not rows:     # region shorter than the sampling period: nearest samples either side
            rows = [r for t, r in self.rows if t0 - 0.1 <= t <= t1 + 0.1] or [r for _, r in self.rows[-3:]]
            window = "nearest samples (region shorter than the 25 ms sampling period)"
        sm, reasons, mx, pw = [], set(), None, []
        for r in rows:
            try:
                sm.append(float(r[0])); mx = float(r[1])
                pw.append(float(r[2]))
                for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), r[3:7]):
                    if v.lower().startswith("active"):
                        reasons.add(name)
            except Exception:
                pass
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": mx,
                "reasons": sorted(reasons), "samples": len(sm), "window": window,
                "power_w": float(np.median(pw)) if pw else None}


DUMP_SEED = 0x3D5CA9
DUMP_SAMPLES = 1 << 18      # pixels of every plane and rows of the point cloud written per scan
DUMP_SCANS = 4              # scans written at most: 4 x 2^18 x 40 B = 42 MB


def scan_outputs(s3, ctx, dirs):
    """What a caller of the timed path reads back after a context's last scan (include/scan3d.h results)."""
    out = {"unwrapped_v": ctx.plane(s3.PLANE_UNWRAPPED_V), "code_v": ctx.code_i32(0), "valid": ctx.plane(s3.PLANE_VALID)}
    if dirs == 2:
        out.update(unwrapped_h=ctx.plane(s3.PLANE_UNWRAPPED_H), code_h=ctx.code_i32(1),
                   cpmap=ctx.plane(s3.PLANE_CPMAP), points=ctx.points())
    return out


def oracle_outputs(r, dirs):
    """The same arrays from one oracle reconstruction (--impl reference)."""
    out = {"unwrapped_v": r.unwrapped_v, "code_v": r.code_v, "valid": r.valid_v if dirs == 1 else r.valid}
    if dirs == 2:
        out.update(unwrapped_h=r.unwrapped_h, code_h=r.code_h, cpmap=r.cpmap, points=r.pts)
    return out


def dump_outputs(out_dir, scans, H, W):
    """--dump-outputs: scans = {ring member k: () -> {name: array}} -> out_dir/ring<k>_<name>.npy, float32 (the point
    count float64).  Every per-pixel plane is sampled at one seeded set of DUMP_SAMPLES pixels and the point cloud at
    a seeded set of DUMP_SAMPLES rows (the same for every scan and both arms), so that the files stay below 64 MB."""
    assert len(scans) <= DUMP_SCANS
    os.makedirs(out_dir, exist_ok=True)
    n = DUMP_SAMPLES
    npix = H * W
    pix = np.arange(npix) if npix <= n else np.sort(np.random.default_rng(DUMP_SEED).choice(npix, n, replace=False))
    for k, fetch in sorted(scans.items()):
        for name, a in fetch().items():
            if name == "points":
                np.save(os.path.join(out_dir, "ring%d_point_count.npy" % k), np.array([len(a)], np.float64))
                if len(a) > n:
                    a = a[np.sort(np.random.default_rng(DUMP_SEED + 1).choice(len(a), n, replace=False))]
            else:
                a = np.asarray(a).reshape(npix, -1)[pix]
                a = a[:, 0] if a.shape[1] == 1 else a
            np.save(os.path.join(out_dir, "ring%d_%s.npy" % (k, name)), np.ascontiguousarray(a, np.float32))


def oracle_scan_seconds(cfg, ocal, stack, roi, threads, min_seconds, max_runs):
    from gpu_common import run_oracle
    run_oracle(cfg, ocal, stack, roi, threads=threads)          # warm (page faults, thread pool)
    times = []
    t_all = time.time()
    while len(times) < max_runs and (not times or time.time() - t_all < min_seconds):
        t = time.time()
        run_oracle(cfg, ocal, stack, roi, threads=threads)
        times.append(time.time() - t)
    return float(np.median(times)), len(times)


def bench_rowshard(args, s3, cal, cfg_full, config, rank, world, local_rank, stream, barrier, bpp, steps=None, tag="c5"):
    """configs[4]: one very large frame; rank r decodes + triangulates its block of rows, then the compacted point
    lists are gathered (rank order == raster order) on rank 0.  Returns the result line (rank 0) or None."""
    import importlib
    import torch
    import torch.distributed as dist
    sh = importlib.import_module("3dscan_b200.sharding")
    steps = steps or args.steps
    W, Ht = cfg_full.W, cfg_full.H
    row0, rows = sh.row_block(Ht, rank, world)
    cfg = s3.make_config(W, rows, cfg_full.PW, cfg_full.PH, cfg_full.N, cfg_full.M_v, cfg_full.M_h,
                         cfg_full.fw_v, cfg_full.fw_h, 2, row0=row0, H_total=Ht, flags=cfg_full.flags)
    nf = s3.stack_planes(cfg)
    # two contexts on two streams: the exchange of scan k overlaps the decode of scan k+1
    streams = [stream, torch.cuda.Stream()]
    ctxs = [s3.Scan3D(cfg, local_rank, cal, stream=st.cuda_stream) for st in streams]
    stack_h = torch.empty((nf, rows, W), dtype=torch.uint8, pin_memory=True)
    roi_h = torch.empty((Ht, W), dtype=torch.uint8, pin_memory=True)
    s3.synth_stack(cfg, cal, s3.default_synth_params(seed=0x3D5CA9), out=stack_h.numpy(), roi_out=roi_h.numpy(),
                   threads=max(1, (os.cpu_count() or 8) // max(1, world)))
    stack_d, roi_d = stack_h.to("cuda"), roi_h.to("cuda")
    del stack_h
    total = [0]
    seq = [0]

    def decode(k):
        ctxs[k & 1].reconstruct_dev(stack_d.data_ptr(), roi_d.data_ptr())      # runs on streams[k & 1]

    # --exchange peer (default): the C++ row-shard group (include/scan3d_shard.h): counts over a shared-memory board,
    # one copy-engine push per rank over NVLink to the final raster offset in rank 0's block.
    # --exchange nccl: all-gather of the counts + NCCL send/recv of the points after the kernel.
    group, outs = None, None
    if args.exchange == "peer" or world == 1:
        name = "b%s_%s_%d" % (os.environ.get("MASTER_PORT", "0"), tag, os.getppid() if world > 1 else os.getpid())
        group = sh.RowShardGroup(name, rank, world, local_rank, Ht * W, slots=2)
        for i in range(2):
            group.bind(i, ctxs[i])
    else:
        outs = [torch.empty((Ht * W, 3), dtype=torch.float32, device="cuda") if rank == 0 else None for _ in ctxs]
        srcs = [_wrap_device(torch, c.device_points(), (rows * W, 3), "<f4") for c in ctxs]
        cnts = [_wrap_device(torch, c.device_point_count(), (1,), "<i4") for c in ctxs]

    def step():
        # one scan per step: enqueue the decode of scan k+1, then gather scan k (the host only waits for scan k)
        k = seq[0]
        decode(k + 1)
        if group is not None:
            total[0], _ = group.gather(k & 1, ctxs[k & 1])
            group.release(k & 1)               # (rank 0: nobody consumes the cloud here)
        else:
            with torch.cuda.stream(streams[k & 1]):
                _, counts = sh.gather_points(srcs[k & 1], cnts[k & 1], dst=0, out=outs[k & 1], slot=k & 1)
            total[0] = sum(counts)
        seq[0] = k + 1

    sampler = ClockSampler(local_rank)
    sampler.start()
    decode(0)
    for _ in range(args.warmup):
        step()
    sampler.wait_first_row()
    torch.cuda.synchronize()
    barrier()
    l0 = sum(c.launch_count() for c in ctxs)
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    barrier()
    t0 = time.time()
    ev0.record(stream)
    streams[1].wait_stream(stream)     # both streams start behind ev0
    for _ in range(steps):
        step()
    stream.wait_stream(streams[1])
    ev1.record(stream)
    barrier()
    t1 = time.time()
    ms = ev0.elapsed_time(ev1)
    clocks = sampler.stop(t0, t1)
    tms = torch.tensor([ms], device="cuda", dtype=torch.float64)
    if world > 1:
        dist.all_reduce(tms, op=dist.ReduceOp.MAX)
    ms_max = float(tms.item())
    npix = W * Ht
    value = steps * npix / (ms_max * 1e-3) / 1e6
    peak, peak_kind = measured_peak_gbs()
    ms_scan = ms_max / steps
    achieved = bpp * npix / (ms_scan * 1e-3) / 1e9
    # what bounds the mode: every rank's HBM share of the decode, or rank 0's NVLink ingest of the other ranks' points
    nvlink_gbs = 770.0                                   # measured peer-copy rate per direction (B200_PROFILING.md)
    ingest_bytes = 12.0 * total[0] * (world - 1) / max(1, world)
    floor_hbm_ms = bpp * npix / world / (peak * 1e9) * 1e3
    floor_link_ms = ingest_bytes / (nvlink_gbs * 1e9) * 1e3
    line = None
    if rank == 0:
        cfgd = dict(config)
        cfgd.update({"workload": "c5_50mp_rowshard_8step_10bit_vh", "frame": [W, Ht],
                     "sharding": ("one frame row-sharded over %d rank(s); " % world) +
                     ("counts over a shared-memory board, one copy-engine push per rank over NVLink to the final raster offset in rank 0's block (include/scan3d_shard.h)"
                      if group is not None else "all-gather of counts + NCCL send/recv of compacted points to rank 0") + "; 2 contexts on 2 streams",
                     "rows_per_rank": rows, "scans_per_gpu_per_step": 1, "resident_ring": 1,
                     "l2_policy": "inputs larger than L2 (%.2f GB per GPU)" % (nf * rows * W / 1e9)})
        line = {"metric": METRIC, "value": value, "unit": "Mpix/s", "n_gpus": world, "steps": steps,
                "warmup": args.warmup, "ms_per_step": ms_scan, "higher_is_better": True,
                "scaling": "strong", "vs_baseline": None, "dtype": "f64", "data": "synthetic", "config": cfgd,
                "scans_per_s": steps / (ms_max * 1e-3), "points_last_scan": total[0],
                "gpu_launches": sum(c.launch_count() for c in ctxs) - l0, "clocks": clocks,
                "roofline": {"bound": "hbm" if floor_hbm_ms >= floor_link_ms else "nvlink ingest of rank 0",
                             "achieved": achieved, "peak": peak * world, "unit": "GB/s",
                             "frac": achieved / (peak * world), "traffic": None,
                             "floor_ms_hbm": floor_hbm_ms, "floor_ms_nvlink_ingest": floor_link_ms,
                             "frac_of_binding_floor": max(floor_hbm_ms, floor_link_ms) / ms_scan,
                             "nvlink_ingest_gbs": ingest_bytes / (ms_scan * 1e-3) / 1e9,
                             "peak_kind": "%d x MEASURED_PEAKS.json hbm_gbs; time includes the point gather; NVLink floor = (world-1)/world of the points at the measured 770 GB/s peer-copy rate into rank 0" % world},
                "e2e": None, "cpu_baseline": None}
    torch.cuda.synchronize()
    if group is not None:
        group.close()
    for c in ctxs:
        c.close()
    del stack_d, roi_d
    torch.cuda.empty_cache()
    return line


def _wrap_device(torch, ptr, shape, typestr):
    """torch view of a ctx-owned device buffer (no copy)."""
    class _Holder:
        pass
    h = _Holder()
    h.__cuda_array_interface__ = {"shape": tuple(shape), "typestr": typestr, "data": (int(ptr), False), "version": 2}
    return torch.as_tensor(h, device="cuda")


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--workload", default="c3_12mp_8step_10bit_vh", choices=sorted(WORKLOADS))
    ap.add_argument("--batch", type=int, default=256, help="scans per GPU per step (configs[3]: a batch of 256 scans)")
    ap.add_argument("--ring", type=int, default=4, help="distinct resident stacks per GPU")
    ap.add_argument("--e2e-scans", type=int, default=3, help="scans per e2e step (one lane = one context + host thread per scan)")
    ap.add_argument("--exact-triangulation", action="store_true",
                    help="reference operation order in the normal-equation solve (bit-identical points)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-rowshard", action="store_true", help="N > 1: skip the row-sharded 50 MP frame that rides along")
    ap.add_argument("--contexts", type=int, default=4, help="contexts (each on its own stream) the batch alternates over")
    ap.add_argument("--cta-limit", type=int, default=1, help="CTA slots per SM each context's kernel may take (0 = all)")
    ap.add_argument("--exchange", default="peer", choices=["peer", "nccl"], help="row-shard workload, N>1: how the points reach rank 0")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write what the last step computed as DIR/ring<k>_<name>.npy (rank 0: "
                         "the last scans of up to 4 ring members; seeded samples of planes and points, < 64 MB in all)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.workload.startswith("c5_"):
        ap.error("--dump-outputs covers the frame-parallel workloads, not the row-sharded one")
    if args.warmup < 3:
        args.warmup = 3

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    W, H, PW, PH, N, Mv, Mh, fwv, fwh, dirs = WORKLOADS[args.workload]
    npix = W * H
    bpp = algorithmic_bytes_per_pixel(N, Mv, Mh, dirs)

    # workload definition: the reference's calibration (tests/golden/calib_c1.json) scaled to the frame;
    # nothing under oracle/ is imported on the B200 arm -- only the two CPU legs below load it
    from helpers import load_calib_c1, scaled_calib
    s3 = importlib.import_module("3dscan_b200")
    cal_dict = scaled_calib(load_calib_c1(), W / 1600.0, PW / 1280.0)
    cal_args = [cal_dict[k] for k in ("Kc", "dc", "Kp", "dp", "rc", "tc", "rp", "tp")]
    cal = s3.make_calib(*cal_args)
    flags = 0 if args.exact_triangulation else s3.FLAG_FAST_TRIANGULATION
    cfg = s3.make_config(W, H, PW, PH, N, Mv, Mh, fwv, fwh, dirs, flags=flags)
    config = {"workload": args.workload, "frame": [W, H], "projector": [PW, PH], "phase_steps": N,
              "gray_bits": [Mv, Mh][:dirs], "directions": dirs, "frames_per_scan": s3.stack_planes(cfg),
              "scans_per_gpu_per_step": args.batch, "resident_ring": args.ring, "contexts_per_gpu": args.contexts, "cta_slots_per_sm_per_context": args.cta_limit or "all",
              "sharding": "frame-parallel scans, no collective" if world > 1 else "single GPU",
              "l2_policy": "inputs larger than L2 (ring of distinct stacks, %.2f GB per GPU)"
                           % (args.ring * s3.stack_planes(cfg) * npix / 1e9),
              "algorithmic_bytes_per_pixel": bpp, "fused_cfg": os.environ.get("SCAN3D_FUSED_CFG", "default"),
              "triangulation": "reference operation order (bit-identical points)" if args.exact_triangulation
              else "fused-FMA normal equations (points within 1e-6 relative; decode/c_p_map bit-exact)"}

    # ------------------------------------------------------------------ reference arm (CPU)
    if args.impl == "reference":
        if rank != 0:
            return
        import oracle_ffi as o
        ocal = o.make_calib(*cal_args)
        threads = host_threads()
        stack, roi = s3.synth_stack(cfg, cal, s3.default_synth_params(seed=0x3D5CA9))
        from gpu_common import run_oracle
        for _ in range(args.warmup):
            run_oracle(cfg, ocal, stack, roi, threads=threads)
        t0 = time.time()
        for _ in range(args.steps):
            r = run_oracle(cfg, ocal, stack, roi, threads=threads)
        dt = time.time() - t0
        if args.dump_outputs:
            dump_outputs(args.dump_outputs, {0: lambda: oracle_outputs(r, dirs)}, H, W)     # ring member 0 = this stack
        val = args.steps * npix / dt / 1e6
        config["scans_per_gpu_per_step"] = 1
        line = {"impl": "reference", "metric": METRIC, "value": val, "unit": "Mpix/s", "n_gpus": args.gpus,
                "steps": args.steps, "warmup": args.warmup, "ms_per_step": dt / args.steps * 1e3,
                "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f64",
                "data": "synthetic", "config": config, "scans_per_s": args.steps / dt,
                "cpu_baseline": {"value": val, "unit": "Mpix/s", "cores": threads, "kind": "port",
                                 "sample": "1 full %dx%d scan per step, stages 3-8 incl. full-frame undistort tables, inputs in RAM, no file I/O" % (W, H)},
                "e2e": {"value": val, "unit": "Mpix/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
        print(json.dumps(line))
        return

    # ------------------------------------------------------------------ B200 arm
    import torch
    import torch.distributed as dist
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device -- the product path has no CPU fallback")
    torch.cuda.set_device(local_rank)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    # a dedicated non-default stream: kernels, copies and the timing events all live on it
    stream = torch.cuda.Stream()
    torch.cuda.set_stream(stream)
    if args.workload.startswith("c5_"):
        line = bench_rowshard(args, s3, cal, cfg, config, rank, world, local_rank, stream, barrier, bpp)
        if rank == 0:
            print(json.dumps(line))
        if world > 1:
            dist.destroy_process_group()
        return
    ctx = s3.Scan3D(cfg, local_rank, cal, stream=stream.cuda_stream)
    nf = s3.stack_planes(cfg)
    # Resident ring of distinct scans.  One synthetic capture is rendered on the host (rank 0, all
    # host threads) and broadcast over NCCL; ring member k of rank r is that capture shifted by a
    # rank- and k-specific number of columns (stack and ROI alike): every member is a valid capture
    # of the shifted scene in its own memory, so the ring (>> L2) is never served from cache.
    host_stack = torch.empty((nf, H, W), dtype=torch.uint8, pin_memory=True)
    host_roi = torch.empty((H, W), dtype=torch.uint8, pin_memory=True)
    if rank == 0:
        s3.synth_stack(cfg, cal, s3.default_synth_params(seed=0x3D5CA9), out=host_stack.numpy(), roi_out=host_roi.numpy())
    base_stack = host_stack.to("cuda")
    base_roi = host_roi.to("cuda")
    if world > 1:
        dist.broadcast(base_stack, 0)
        dist.broadcast(base_roi, 0)
        host_stack.copy_(base_stack)      # every rank's e2e leg reads its own pinned copy
        host_roi.copy_(base_roi)
    ring, rois = [], []
    for i in range(args.ring):
        shift = 16 * ((rank * args.ring + i) * 7 % (W // 16))
        ring.append(torch.roll(base_stack, shifts=shift, dims=2) if shift else base_stack)
        rois.append(torch.roll(base_roi, shifts=shift, dims=1) if shift else base_roi)
    torch.cuda.synchronize()

    # --contexts C --cta-limit L: the scans of a batch alternate over C contexts on C streams (still one GPU, still
    # frame-parallel), each context's persistent kernel taking L of the SM's 3 CTA slots: the kernels of 3 scans are
    # resident side by side and the fourth waits in the queue, so one scan's pipeline fill and drain (and its two
    # work-list launches) overlap the steady state of the others
    side_streams = [torch.cuda.Stream() for _ in range(args.contexts - 1)]
    ctxs = [ctx] + [s3.Scan3D(cfg, local_rank, cal, stream=st.cuda_stream) for st in side_streams]

    if args.cta_limit:
        for c in ctxs:
            c.set_cta_limit(args.cta_limit)

    def step():
        for b in range(args.batch):
            k = b % args.ring
            ctxs[b % len(ctxs)].reconstruct_dev(ring[k].data_ptr(), rois[k].data_ptr())

    # ---- burst figure first (GPU still cool, clocks at their maximum): the same schedule over 8 x 16 scans after
    #      3 x 16 warm-up scans, ~35 ms -- what the kernel does before the power cap of a 1.4 s region pulls the SM
    #      clock down (the kernel is SM-bound, so the long-region figure follows that clock)
    def small_step(n=16):
        for b in range(n):
            k = b % args.ring
            ctxs[b % len(ctxs)].reconstruct_dev(ring[k].data_ptr(), rois[k].data_ptr())

    sampler = ClockSampler(local_rank)
    sampler.start()
    for _ in range(3):
        small_step()
    torch.cuda.synchronize()
    sampler.wait_first_row()
    b0, b1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    tb0 = time.time()
    b0.record(stream)
    for st in side_streams:
        st.wait_stream(stream)
    for _ in range(8):
        small_step()
    for st in side_streams:
        stream.wait_stream(st)
    b1.record(stream)
    torch.cuda.synchronize()
    tb1 = time.time()
    burst_us = b0.elapsed_time(b1) * 1e3 / 128
    burst_clocks = sampler.window(tb0, tb1)

    for _ in range(args.warmup):
        step()
    sampler.wait_first_row()
    barrier()
    l0 = sum(c.launch_count() for c in ctxs)
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    barrier()
    t_wall0 = time.time()
    ev0.record(stream)
    for st in side_streams:
        st.wait_stream(stream)         # every stream starts behind ev0 ...
    for _ in range(args.steps):
        step()
    for st in side_streams:
        stream.wait_stream(st)         # ... and ev1 is behind every stream
    ev1.record(stream)
    barrier()
    t_wall1 = time.time()
    ms = ev0.elapsed_time(ev1)
    launches = sum(c.launch_count() for c in ctxs) - l0
    clocks = sampler.stop(t_wall0, t_wall1)
    count = ctx.point_count() if dirs == 2 else 0
    if args.dump_outputs and rank == 0:
        # each context still holds the results of its last scan of the last step (the e2e leg below reuses ctx):
        # the last DUMP_SCANS of them, named by the ring member they read
        last = {}
        for b in range(args.batch):
            last[b % len(ctxs)] = b
        scans = {b % args.ring: ctxs[c] for c, b in sorted(last.items(), key=lambda cb: cb[1])[-DUMP_SCANS:]}
        dump_outputs(args.dump_outputs, {k: (lambda c=c: scan_outputs(s3, c, dirs)) for k, c in scans.items()}, H, W)
    tms = torch.tensor([ms], device="cuda", dtype=torch.float64)
    if world > 1:
        dist.all_reduce(tms, op=dist.ReduceOp.MAX)
    ms_max = float(tms.item())
    total_pix = world * args.steps * args.batch * npix
    value = total_pix / (ms_max * 1e-3) / 1e6

    # ---- roofline of the dominant (only) kernel: algorithmic bytes per launch / avg launch time
    # per scan: 2 tiny work-list kernels + the persistent fused kernel; the whole scan time is
    # charged to the fused kernel (conservative: its own duration is slightly shorter)
    per_launch_s = ms * 1e-3 / (args.steps * args.batch)
    peak, peak_kind = measured_peak_gbs()
    achieved = bpp * npix / per_launch_s / 1e9
    roofline = {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                "traffic": ncu_traffic(args.workload), "peak_kind": peak_kind + " (MEASURED_PEAKS.json hbm_gbs)" if peak_kind == "measured" else "fallback 6.65 TB/s",
                "kernel": ("s3d::k_fused<%d,%d>" if os.environ.get("SCAN3D_FUSED_IMPL") == "6" else "s3d::k_fused7<%d,%d,...>") % (N, dirs), "algorithmic_bytes_per_launch": bpp * npix,
                "avg_launch_us": per_launch_s * 1e6, "launches_per_scan": launches / (args.steps * args.batch), "frac_of_8TBs_nominal": achieved / 8000.0,
                "burst": {"avg_launch_us": burst_us, "frac": bpp * npix / (burst_us * 1e-6) / 1e9 / peak, "scans": 128, "clocks": burst_clocks,
                          "note": "same schedule, 128 scans (~35 ms) before the long region: what the kernel does before a sustained load's power cap pulls the SM clock down"}}

    # ---- e2e: host-buffer entry, pinned input, H2D + kernel + D2H of the point cloud per scan
    e2e = None
    if not args.no_e2e:
        # Two contexts on two host threads (contexts are independent, include/scan3d.h): the D2H of
        # one scan's points and its kernel overlap the H2D of the other scan's stack (PCIe is full
        # duplex); the H2D stream itself is the bound (57 B/pixel in).
        h2d = (nf + 1) * npix
        lanes = args.e2e_scans if args.e2e_scans <= 4 else 2
        e_ctxs = [ctx] + [s3.Scan3D(cfg, local_rank, cal, stream=torch.cuda.Stream().cuda_stream) for _ in range(lanes - 1)]
        for c in e_ctxs:
            c.set_cta_limit(args.cta_limit)
        pts_hosts = [torch.empty((npix, 3), dtype=torch.float32, pin_memory=True) if dirs == 2 else None for _ in e_ctxs]
        out_hosts = [torch.empty((H, W), dtype=torch.float32, pin_memory=True) for _ in e_ctxs]

        def e2e_scan(i):
            c = e_ctxs[i]
            n = c.reconstruct(host_stack.numpy(), host_roi.numpy())
            if dirs == 2:
                c._ck(c.L.scan3d_get_points(c.h, pts_hosts[i].data_ptr(), None, None, n))
                return n * 12 + 8
            c._ck(c.L.scan3d_get_plane(c.h, s3.PLANE_UNWRAPPED_V, out_hosts[i].data_ptr()))
            return npix * 4

        def e2e_lane(i, scans, res):
            for _ in range(scans):
                res[i] = e2e_scan(i)

        def e2e_run(scans_per_lane):
            res = [0] * lanes
            ths = [threading.Thread(target=e2e_lane, args=(i, scans_per_lane, res)) for i in range(lanes)]
            for t in ths:
                t.start()
            for t in ths:
                t.join()
            return res[0]

        d2h = e2e_run(1)
        barrier()
        t0 = time.time()
        e_steps = max(1, min(args.steps, 5))
        d2h = e2e_run(e_steps * args.e2e_scans // lanes)
        barrier()
        dt = time.time() - t0
        for c in e_ctxs[1:]:
            c.close()
        te = torch.tensor([dt], device="cuda", dtype=torch.float64)
        if world > 1:
            dist.all_reduce(te, op=dist.ReduceOp.MAX)
        # what the host->device path of this box can do at best: one large pinned copy, best of 3 (this rank alone)
        probe = torch.empty(256 << 20, dtype=torch.uint8, device="cuda")
        h2d_peak = 0.0
        for _ in range(3):
            torch.cuda.synchronize()
            tp = time.time()
            probe.copy_(host_stack.view(-1)[:probe.numel()], non_blocking=True)
            torch.cuda.synchronize()
            h2d_peak = max(h2d_peak, probe.numel() / (time.time() - tp) / 1e9)
        del probe
        e2e = {"value": world * e_steps * args.e2e_scans * npix / float(te.item()) / 1e6, "unit": "Mpix/s",
               "h2d_bytes_per_step": h2d * args.e2e_scans, "d2h_bytes_per_step": d2h * args.e2e_scans,
               "h2d_gbs_achieved_per_gpu": e_steps * args.e2e_scans * h2d / float(te.item()) / 1e9,
               "h2d_gbs_pinned_copy_peak": h2d_peak,
               "bound": "host->device copies (PCIe): the kernel side is %.0fx faster than the input arrives" % (value / world / max(1e-9, e_steps * args.e2e_scans * npix / float(te.item()) / 1e6)),
               "scans_per_step": args.e2e_scans, "steps": e_steps,
               "api": "scan3d_reconstruct(host stack, host roi) + scan3d_get_points, %d context(s) on %d host thread(s)" % (lanes, lanes)}

    # ---- CPU baseline: the oracle port on this box's host cores, bounded sample (rank 0, N=1 semantics)
    cpu = None
    if rank == 0 and not args.no_cpu_baseline:
        import oracle_ffi as o
        ocal = o.make_calib(*cal_args)
        threads = host_threads()
        sec, runs = oracle_scan_seconds(cfg, ocal, host_stack.numpy(), host_roi.numpy(), threads, 8.0, 4)
        cpu = {"value": npix / sec / 1e6, "unit": "Mpix/s", "cores": threads, "kind": "port",
               "sample": "%d full %dx%d scan(s) of the same workload, median; stages 3-8 incl. full-frame undistort tables; inputs in RAM" % (runs, W, H),
               "seconds_per_scan": sec}
        # SURVEY 8d (i): the reference itself is single-threaded -- one scan on one core beside the all-core figure
        if world == 1:
            try:
                sec1, _ = oracle_scan_seconds(cfg, ocal, host_stack.numpy(), host_roi.numpy(), 1, 0.0, 1)
                cpu["single_thread"] = {"value": npix / sec1 / 1e6, "unit": "Mpix/s", "cores": 1, "seconds_per_scan": sec1}
                cpu["single_thread_value"] = npix / sec1 / 1e6      # (flat copies: nested objects get dropped by some parsers)
                cpu["single_thread_seconds_per_scan"] = sec1
                # BASELINE.md section 3 "ref-faithful": one thread AND the reference's own [col][row] plane layout
                # (row-outer loops striding every plane by H elements, 3/wrapped_phase.cpp:164-183)
                from gpu_common import run_oracle
                rr = run_oracle(cfg, ocal, host_stack.numpy(), host_roi.numpy(), colrow=True)
                cpu["reference_layout_single_thread_value"] = npix / rr.seconds / 1e6
                cpu["reference_layout_single_thread_seconds_per_scan"] = rr.seconds
            except Exception as e:   # the all-core figure above is the contract; this one is extra
                cpu["single_thread"] = {"error": str(e)}

    for c in ctxs[1:]:
        c.close()
    # ---- N > 1: configs[4] rides along (one 50 MP frame row-sharded over the ranks), so that the scaling record
    #      carries it at every GPU count
    rowshard = None
    if world > 1 and not args.no_rowshard and args.workload.startswith("c3_"):
        barrier()
        ctx.close()
        del ring, rois, base_stack, base_roi
        torch.cuda.empty_cache()
        W5, H5, PW5, PH5, N5, Mv5, Mh5, fwv5, fwh5, _ = WORKLOADS["c5_50mp_rowshard_8step_10bit_vh"]
        cal5d = scaled_calib(load_calib_c1(), W5 / 1600.0, PW5 / 1280.0)
        cal5 = s3.make_calib(*[cal5d[k] for k in ("Kc", "dc", "Kp", "dp", "rc", "tc", "rp", "tp")])
        cfg5 = s3.make_config(W5, H5, PW5, PH5, N5, Mv5, Mh5, fwv5, fwh5, 2, flags=flags)
        l5 = bench_rowshard(args, s3, cal5, cfg5, {}, rank, world, local_rank, stream, barrier,
                            algorithmic_bytes_per_pixel(N5, Mv5, Mh5, 2), steps=max(8, min(args.steps, 24)), tag="ride")
        if rank == 0:
            rowshard = {"workload": "c5_50mp_rowshard_8step_10bit_vh", "ms_per_scan": l5["ms_per_step"], "mpix_per_s": l5["value"],
                        "points": l5["points_last_scan"], "frac_of_n_x_hbm": l5["roofline"]["frac"],
                        "floor_ms_hbm": l5["roofline"]["floor_ms_hbm"], "floor_ms_nvlink_ingest": l5["roofline"]["floor_ms_nvlink_ingest"],
                        "frac_of_binding_floor": l5["roofline"]["frac_of_binding_floor"], "bound": l5["roofline"]["bound"],
                        "nvlink_ingest_gbs": l5["roofline"]["nvlink_ingest_gbs"], "exchange": l5["config"]["sharding"], "steps": l5["steps"]}
        ctx = None
    if rank == 0:
        line = {"metric": METRIC, "value": value, "unit": "Mpix/s", "n_gpus": world, "steps": args.steps,
                "warmup": args.warmup, "ms_per_step": ms_max / args.steps, "higher_is_better": True,
                "scaling": "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic", "config": config,
                "scans_per_s": world * args.steps * args.batch / (ms_max * 1e-3),
                "points_last_scan": count, "gpu_launches": launches * world, "gpu_launches_per_rank": launches, "clocks": clocks,
                "roofline": roofline, "e2e": e2e, "cpu_baseline": cpu}
        if rowshard is not None:
            line["rowshard"] = rowshard
        print(json.dumps(line))
    if ctx is not None:
        ctx.close()
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
