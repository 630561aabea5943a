#!/usr/bin/env python
"""Benchmark of the tape-evaluation hot path on B200 (see DESIGN.md, "Measurement").

A step = one pass of the hot path over one frame of synthetic input.

  N = 1 : models/prospero.vm, 2D render 4096x4096 (BASELINE.json configs[1], the configuration the metric
          is quoted on): interval levels [128,32,8] with on-device tape simplification, fill, bulk f32 over
          the surviving leaf tiles.  The line also carries `strong_scaling_base`: the N > 1 workload (below)
          rendered whole on this one GPU, so that every strong-scaling figure has its base in the record.
  N > 1 : ONE fixed workload sharded over the N ranks (strong scaling): models/prospero.vm, 3D render of the
          4096^3 voxel volume (BASELINE.json configs[4]).  Rank r renders the root-tile columns (tx, ty) with
          hash(tx, ty) % N == r (shard.tile_owner) at full depth, packs its 1/N of the heightmap+normals image, ONE NCCL all-gather
          runs INSIDE the timed region, and every rank unpacks the complete frame.  value = 4096^3 voxels /
          max-over-ranks device time.  Before timing, every rank also renders the whole volume alone and the
          run ASSERTS that the sharded frame is byte-identical to it; rank 0 times that single-GPU render
          (`strong_scaling_base`).  A 0.3 ms 2D frame cannot shard (its all-gather alone costs more than the
          frame), which is why the N > 1 workload is the 3D volume; see DESIGN.md section 6.

  python bench.py --gpus N --steps K --warmup W           # CUDA arm
  python bench.py --impl reference --gpus N --steps K ...  # CPU arm (oracle port, all host threads)

Prints ONE JSON line (rank 0).  With --dump-outputs DIR, rank 0 also writes what the last timed step computed as
DIR/<name>.npy (finite float32 / float64), a fixed seeded sample of DUMP_PIXELS pixels per image, so that two
builds can be compared output for output:
  frame2d_distance, _kind, _fill_depth, _inside   N = 1: the 2D frame's RawDistancePixel words, unpacked
  volume3d_depth, _normal      the 3D frame's GeometryPixel depth and normal (N = 1 unless --no-volume, and N > 1)
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

SIZE = 4096
MODEL = "prospero.vm"
METRIC = "Mvoxels/s (prospero 4096^2 2D render, interval + bulk f32)"
METRIC_3D = "Mvoxels/s (prospero 4096^3 3D render sharded over N GPUs, interval + bulk f32 + gradients + 1 all-gather)"
ALGO_BYTES_PER_PIXEL = 4       # SURVEY.md 8(d): one RawDistancePixel written per pixel
ALGO_BYTES_PER_PIXEL_3D = 16   # one GeometryPixel written per pixel
T0 = 128
WORKLOAD_2D = f"models/{MODEL} 2D render {SIZE}x{SIZE}, tile sizes [128,32,8], identity camera"
WORKLOAD_3D = f"models/{MODEL} 3D render {SIZE}^3, tile sizes [128,64,32,16,8], identity camera"
# 2^20 of the 2^24 pixels of a frame: the four 2D arrays (16 MiB) and the 3D depth + normals (20 MiB) stay under 64 MB
DUMP_PIXELS = 1 << 20
DUMP_SEED = 0


def model_text():
    with open(os.path.join(ROOT, "models", MODEL)) as f:
        return f.read()


def sample_pixels(img):
    """The same DUMP_PIXELS pixels (seeded, in row-major order) of an [H, W, ...] image, numpy or CUDA tensor."""
    n = img.shape[0] * img.shape[1]
    idx = np.sort(np.random.default_rng(DUMP_SEED).choice(n, min(DUMP_PIXELS, n), replace=False))
    flat = img.reshape((n,) + tuple(img.shape[2:]))
    if isinstance(img, np.ndarray):
        return flat[idx]
    import torch
    return flat[torch.from_numpy(idx).to(img.device)].cpu().numpy()


def frame2d_outputs(img):
    """RawDistancePixel words unpacked into finite arrays (the words themselves NaN-box the fill pixels): kind 0 =
    distance value, 1 = fill, 2 / 3 / 4 = NaN / +inf / -inf distance; the fill's recursion depth; inside as 0 / 1."""
    from fidget_b200.shape import pixel_inside
    px = sample_pixels(img)
    bits = px.view(np.uint32)
    fill = np.isnan(px) & ((bits & np.uint32(0xFF << 9)) == np.uint32(0xF6 << 9))   # RawDistancePixel::KEY
    kind = np.select([fill, np.isnan(px), px == np.inf, px == -np.inf], [1, 2, 3, 4], 0)
    return {"frame2d_distance": np.where(kind == 0, px, 0).astype(np.float32),
            "frame2d_kind": kind.astype(np.float32),
            "frame2d_fill_depth": np.where(fill, (bits >> 1) & 0xFF, 0).astype(np.float32),
            "frame2d_inside": pixel_inside(px).astype(np.float32)}


def volume3d_outputs(img):
    from fidget_b200.shape import GEOMETRY_PIXEL
    px = np.ascontiguousarray(sample_pixels(img)).view(GEOMETRY_PIXEL).reshape(-1)   # [n, 4] float32 -> n pixels
    return {"volume3d_depth": px["depth"].astype(np.float64), "volume3d_normal": px["normal"]}


def dump_outputs(directory, outputs):
    os.makedirs(directory, exist_ok=True)
    for name, a in outputs.items():
        np.save(os.path.join(directory, name + ".npy"), a)


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled while the timed region runs."""
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, index=0):
        self.rows = []
        self.stop = False
        self.index = index
        self.t = None
        # NVML answers in ~0.1 ms, nvidia-smi (the same counters through a subprocess) in ~50 ms; the
        # timed region of a default run lasts ~10 ms, so NVML is what can sample it more than once
        self.nvml, self.handle = None, None
        try:
            import pynvml
            pynvml.nvmlInit()
            self.handle = pynvml.nvmlDeviceGetHandleByIndex(index)
            self.nvml = pynvml
        except Exception:
            self.nvml = None

    def _sample_nvml(self):
        p, h = self.nvml, self.handle
        sm = p.nvmlDeviceGetClockInfo(h, p.NVML_CLOCK_SM)
        mx = p.nvmlDeviceGetMaxClockInfo(h, p.NVML_CLOCK_SM)
        try:
            r = p.nvmlDeviceGetCurrentClocksEventReasons(h)
        except Exception:
            r = p.nvmlDeviceGetCurrentClocksThrottleReasons(h)
        try:
            w = p.nvmlDeviceGetPowerUsage(h) / 1000.0
        except Exception:
            w = 0.0
        bits = (p.nvmlClocksThrottleReasonHwSlowdown, p.nvmlClocksThrottleReasonHwThermalSlowdown,
                p.nvmlClocksThrottleReasonSwThermalSlowdown, p.nvmlClocksThrottleReasonSwPowerCap)
        self.rows.append([str(sm), str(mx), f"{w:.1f}"] + ["Active" if r & b else "Not Active" for b in bits])

    def _sample(self):
        try:
            out = subprocess.run(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                  "-i", str(self.index)], capture_output=True, text=True, timeout=10).stdout
            for line in out.strip().splitlines():
                self.rows.append([c.strip() for c in line.split(",")])
        except Exception:
            pass

    def _run(self):
        while not self.stop:
            if self.nvml is not None:
                try:
                    self._sample_nvml()
                    time.sleep(0.001)
                    continue
                except Exception:
                    self.nvml = None          # fall back to nvidia-smi for the rest of the run
            self._sample()
            time.sleep(0.05)

    def __enter__(self):
        self.t = threading.Thread(target=self._run, daemon=True)
        self.t.start()
        return self

    def __exit__(self, *a):
        self.stop = True
        self.t.join(timeout=15)
        if not self.rows:
            self._sample()

    def summary(self):
        sm = [float(r[0]) for r in self.rows if r and r[0].replace(".", "").isdigit()]
        mx = [float(r[1]) for r in self.rows if len(r) > 1 and r[1].replace(".", "").isdigit()]
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = sorted({names[i] for r in self.rows if len(r) >= 7 for i in range(4)
                          if r[3 + i].lower().startswith("active")})
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": reasons, "samples": len(self.rows),
                "source": "nvml" if self.nvml is not None else "nvidia-smi"}


def measured_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        with open(p) as f:
            return json.load(f).get("hbm_gbs"), "measured (MEASURED_PEAKS.json)"
    return 6650.0, "fallback (B200_PROFILING.md)"


def ncu_table():
    """Per-kernel ncu figures of the committed capture (profiles/dram_traffic.json): DRAM bytes per launch,
    issue-active %, fp32-pipe %."""
    tp = os.path.join(ROOT, "profiles", "dram_traffic.json")
    if os.path.exists(tp):
        with open(tp) as f:
            return json.load(f)
    return {}


# ---------------------------------------------------------------------------------------------------
# CPU arms (the oracle: test infrastructure, timed here as the reference's CPU path; never the product)
def cpu_baseline(sample_frames=1, threads=None):
    from oracle import oracle as orc
    threads = threads or os.cpu_count() or 1
    t = orc.Tape.from_vm(model_text())
    orc.render2d(t, 512, 512, threads=threads)  # warm the library / page in
    t0 = time.perf_counter()
    for _ in range(sample_frames):
        orc.render2d(t, SIZE, SIZE, threads=threads)
    dt = (time.perf_counter() - t0) / sample_frames
    return {"value": SIZE * SIZE / dt / 1e6, "unit": "Mvoxels/s", "cores": threads, "kind": "port",
            "sample": f"{sample_frames} full {SIZE}x{SIZE} frame(s) of {MODEL}, tile sizes [128,32,8], "
                      f"{threads} threads over root tiles (oracle/vm.cc render2d)",
            "seconds_per_frame": dt}


REF_SAMPLE_COLUMNS = list(range(1, SIZE // T0, 4))   # every 4th column of root tiles: 1/4 of the volume


def cpu_volume_sample(orc, tape, threads):
    """One bounded sample of the 3D workload on the CPU: every 4th column of root tiles (x fixed, all y, full
    depth; the oracle enumerates root tiles x-outer like the reference).  Returns the voxels covered."""
    ry = SIZE // T0
    for tx in REF_SAMPLE_COLUMNS:
        orc.render3d(tape, SIZE, SIZE, SIZE, threads=threads, first_root=tx * ry, n_roots=ry)
    return len(REF_SAMPLE_COLUMNS) * T0 * SIZE * SIZE


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    threads = os.cpu_count() or 1
    from oracle import oracle as orc
    t = orc.Tape.from_vm(model_text())
    world = args.gpus
    if world == 1:
        for _ in range(max(args.warmup, 1)):
            orc.render2d(t, SIZE, SIZE, threads=threads)
        t0 = time.perf_counter()
        for _ in range(args.steps):
            img, _ = orc.render2d(t, SIZE, SIZE, threads=threads)
        dt = (time.perf_counter() - t0) / args.steps
        if args.dump_outputs:
            dump_outputs(args.dump_outputs, frame2d_outputs(img))
        v = SIZE * SIZE / dt / 1e6
        metric = METRIC
        workload = WORKLOAD_2D
        sample = (f"each step = one full {SIZE}x{SIZE} frame, {threads} host threads; the Rust reference cannot be "
                  "built here (no rustc), so this is the C++ oracle port of VmShape + fidget-raster::pixel::render")
    else:
        # same workload as the CUDA arm at N > 1; a step is a bounded sample (1/4 of the root-tile columns)
        steps = args.steps
        cpu_volume_sample(orc, t, threads)
        t0 = time.perf_counter()
        vox = 0
        for _ in range(steps):
            vox += cpu_volume_sample(orc, t, threads)
        dt = (time.perf_counter() - t0) / steps
        v = vox / steps / dt / 1e6
        metric = METRIC_3D
        workload = WORKLOAD_3D
        sample = (f"each step = every 4th column of root tiles ({len(REF_SAMPLE_COLUMNS)} of {SIZE // T0}, full depth) of the "
                  f"{SIZE}^3 volume, {threads} host threads, {steps} timed steps; C++ oracle port of VmShape + "
                  "fidget-raster::voxel::render (no rustc here)")
    line = {
        "impl": "reference", "metric": metric, "value": v, "unit": "Mvoxels/s", "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": dt * 1e3, "higher_is_better": True,
        "scaling": "weak" if world == 1 else "strong", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": workload},
        "cpu_baseline": {"value": v, "unit": "Mvoxels/s", "cores": threads, "kind": "port", "sample": sample},
        "e2e": {"value": v, "unit": "Mvoxels/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line))


# ---------------------------------------------------------------------------------------------------
def time_steps(torch, stream, flush, step, n, sync_all):
    starts = [torch.cuda.Event(enable_timing=True) for _ in range(n)]
    stops = [torch.cuda.Event(enable_timing=True) for _ in range(n)]
    sync_all()
    for i in range(n):
        flush.fill_(i & 255)
        starts[i].record(stream)
        step()
        stops[i].record(stream)
    sync_all()
    return sum(s.elapsed_time(e) for s, e in zip(starts, stops)) / n


def volume_on_one_gpu(torch, fb, cuda, shape, stream, flush, steps=3):
    """The N > 1 workload rendered whole on this GPU: returns (image, ms per render, stats)."""
    cfg = fb.RenderConfig3D(SIZE, SIZE, SIZE)
    img = torch.zeros((SIZE, SIZE, 4), dtype=torch.float32, device=flush.device)
    _, st = fb.render3d(shape, cfg, out=img, stats=True)          # warm-up + census
    fb.render3d(shape, cfg, out=img, asynchronous=True)
    ms = time_steps(torch, stream, flush, lambda: fb.render3d(shape, cfg, out=img, asynchronous=True), steps,
                    torch.cuda.synchronize)
    cuda.synchronize()
    return img, ms, st


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=30)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="cuda")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-volume", action="store_true", help="N = 1: skip the 4096^3 strong-scaling base")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write what the last timed step computed to DIR/<name>.npy (see the module docstring)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.impl == "reference":
        if args.dump_outputs and args.gpus > 1:
            ap.error("--dump-outputs: the reference arm at N > 1 times a sample of the volume, not a whole frame")
        return run_reference(args)
    args.warmup = max(args.warmup, 3)

    import torch
    import torch.distributed as dist
    import fidget_b200 as fb
    from fidget_b200 import shard

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    dev = torch.device("cuda", local)

    cuda = fb.CudaContext(local)
    cuda.set_arena_bytes(8 << 30)
    stream = torch.cuda.current_stream()
    cuda.set_stream(stream.cuda_stream)
    ctx, root = fb.Context.from_text(model_text())
    tape = ctx.tape(root)
    shape = fb.CudaShape(cuda, tape)
    flush = torch.empty(512 << 20, dtype=torch.uint8, device=dev)  # > 126 MB L2
    peak, peak_src = measured_peaks()
    bc = tape.bytecode()

    def sync_all():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def maxrank(x):
        t = torch.tensor([x], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    outputs = {}
    if world == 1:
        line = bench_2d(args, torch, fb, cuda, shape, tape, bc, stream, flush, dev, peak, peak_src, sync_all, outputs)
        if not args.no_volume:
            img3, ms3, st3 = volume_on_one_gpu(torch, fb, cuda, shape, stream, flush)
            if args.dump_outputs:
                outputs.update(volume3d_outputs(img3))
            line["strong_scaling_base"] = {
                "workload": f"models/{MODEL} 3D render {SIZE}^3 (the N > 1 workload), whole volume on 1 GPU",
                "value": SIZE ** 3 / (ms3 * 1e-3) / 1e6, "unit": "Mvoxels/s", "ms_per_step": ms3,
                "kernel_launches_per_step": int(st3["kernel_launches"])}
        if not args.no_cpu_baseline:
            line["cpu_baseline"] = cpu_baseline()
        if args.dump_outputs:
            dump_outputs(args.dump_outputs, outputs)
        print(json.dumps(line))
        return

    # ---------------- N > 1: one 4096^3 volume sharded over the ranks, one all-gather per step ----------------
    cfg3 = fb.RenderConfig3D(SIZE, SIZE, SIZE)
    full, base_ms, base_st = volume_on_one_gpu(torch, fb, cuda, shape, stream, flush)   # every rank: the single-GPU image
    image = torch.zeros((SIZE, SIZE, 4), dtype=torch.float32, device=dev)
    chunk, gathered = shard.tile_buffers(world, SIZE, SIZE, 4, dev)

    def step():
        shard.render3d_tiles(shape, cfg3, image, chunk, gathered)

    for _ in range(args.warmup):
        step()
    sync_all()
    cuda.synchronize()
    same = torch.equal(image.view(torch.int32), full.view(torch.int32))
    ok = torch.tensor([int(same)], device=dev)
    dist.all_reduce(ok, op=dist.ReduceOp.MIN)
    assert int(ok.item()) == 1, "sharded frame differs from the single-GPU frame"
    del full

    with ClockSampler(local) as clocks:
        ms_local = time_steps(torch, stream, flush, step, args.steps, sync_all)
    cuda.synchronize()
    if args.dump_outputs and rank == 0:
        outputs.update(volume3d_outputs(image))   # the assembled frame, before the census render below reuses `image`
    ms_per_step = maxrank(ms_local)
    value = SIZE ** 3 / (ms_per_step * 1e-3) / 1e6

    # where this rank's step goes: its render (CUDA events inside the library), then pack + all-gather + unpack
    from dataclasses import replace
    _, st = fb.render3d(shape, replace(cfg3, interleave=(world, rank), timing=True), out=image, stats=True)
    render_ms = maxrank(st["stage_ms"][15])
    stage = st["stage_ms"]

    # ---- end to end: host bytecode in, assembled frame in pinned host memory (rank 0) out ----
    host_img = torch.empty((SIZE, SIZE, 4), dtype=torch.float32).pin_memory() if rank == 0 else None

    def e2e_step():
        s = fb.CudaShape(cuda, tape)          # uploads the bytecode (H2D) and builds the device tape
        shard.render3d_tiles(s, cfg3, image, chunk, gathered)
        if rank == 0:
            host_img.copy_(image, non_blocking=True)
        torch.cuda.synchronize()
        return s

    for _ in range(2):
        e2e_step()
    sync_all()
    n_e2e = max(3, min(args.steps, 10))
    t0 = time.perf_counter()
    for _ in range(n_e2e):
        e2e_step()
    sync_all()
    e2e_dt = maxrank((time.perf_counter() - t0) / n_e2e)
    img_bytes = SIZE * SIZE * 16
    e2e = {"value": SIZE ** 3 / e2e_dt / 1e6, "unit": "Mvoxels/s", "h2d_bytes_per_step": int(bc.words.nbytes) * world,
           "d2h_bytes_per_step": img_bytes, "ms_per_step": e2e_dt * 1e3,
           "note": "per step: fc_tape_create from host bytecode on every rank + sharded fc_render3d + all-gather + copy of "
                   "the assembled frame into pinned host memory on rank 0; wall clock, max over ranks"}
    if rank == 0:
        algo = SIZE * SIZE * ALGO_BYTES_PER_PIXEL_3D
        line = {
            "metric": METRIC_3D, "value": value, "unit": "Mvoxels/s", "n_gpus": world, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": ms_per_step, "higher_is_better": True, "scaling": "strong",
            "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": {"workload": WORKLOAD_3D, "detail": "BASELINE configs[4]; reference VM default tile sizes",
                       "parallelism": f"{world} ranks, root-tile columns interleaved (spatial hash % {world}), full depth per "
                                      f"column; 1 NCCL all-gather of {chunk.numel() * 4} B per rank inside the timed region",
                       "collective": "ncclAllGather (torch.distributed all_gather_into_tensor), 1 per step",
                       "identity_check": "sharded frame == single-GPU frame, byte for byte, asserted on every rank",
                       "l2": "flushed between steps by a 512 MiB fill outside the event-timed regions"},
            "clocks": clocks.summary(), "e2e": e2e,
            "gpu_launches": (int(st["kernel_launches"]) + 2) * args.steps,
            "strong_scaling_base": {"workload": "the same volume rendered whole by rank 0's GPU alone, same run",
                                    "value": SIZE ** 3 / (base_ms * 1e-3) / 1e6, "unit": "Mvoxels/s",
                                    "ms_per_step": base_ms},
            "roofline": {"bound": "hbm", "kernel": "whole step (k_voxels_3d dominates)", "achieved": algo / (ms_per_step * 1e-3) / 1e9,
                         "peak": peak, "unit": "GB/s", "frac": algo / (ms_per_step * 1e-3) / 1e9 / peak, "traffic": None,
                         "peak_source": peak_src, "algorithmic_bytes": algo,
                         "note": "16 B per pixel of the final image (SURVEY 8d); the step is bound by FP32 issue in the "
                                 "voxel interpreter, not by HBM",
                         "slowest_rank_render_ms": render_ms, "gather_pack_unpack_ms": ms_per_step - render_ms,
                         "rank0_stage_ms": {"interval_levels": [float(x) for x in stage[:5]], "k_voxels_3d": float(stage[9]),
                                            "k_normals_3d": float(stage[10])}},
        }
        if args.dump_outputs:
            dump_outputs(args.dump_outputs, outputs)
        print(json.dumps(line))
    dist.barrier()
    dist.destroy_process_group()


def bench_2d(args, torch, fb, cuda, shape, tape, bc, stream, flush, dev, peak, peak_src, sync_all, outputs):
    cfg = fb.RenderConfig2D(SIZE, SIZE)
    image = torch.zeros((SIZE, SIZE), dtype=torch.float32, device=dev)

    def step():
        fb.render2d(shape, cfg, out=image, asynchronous=True)

    for _ in range(args.warmup):
        step()
    sync_all()
    cuda.synchronize()  # surfaces deferred device errors
    with ClockSampler(dev.index or 0) as clocks:
        ms_per_step = time_steps(torch, stream, flush, step, args.steps, sync_all)
    cuda.synchronize()
    if args.dump_outputs:
        outputs.update(frame2d_outputs(image))    # before the per-kernel timing below renders into `image` again
    value = SIZE * SIZE / (ms_per_step * 1e-3) / 1e6

    # ---- per-kernel timing of one step (CUDA events inside the library, on the launching stream) ----
    tcfg = fb.RenderConfig2D(SIZE, SIZE, timing=True)
    stage = np.zeros(16)
    fstage = np.zeros(16)
    reps = 5
    stats = None
    for _ in range(reps):
        flush.fill_(1)
        _, stats = fb.render2d(shape, tcfg, out=image, stats=True)
        stage += np.array(stats["stage_ms"])
    # the experimental fused tail (FC_FLAG_FUSED_TAIL), for the record
    for _ in range(2):
        fb.render2d(shape, fb.RenderConfig2D(SIZE, SIZE, timing=True, fused_tail=True), out=image, stats=True)
    for _ in range(reps):
        flush.fill_(1)
        _, fstats = fb.render2d(shape, fb.RenderConfig2D(SIZE, SIZE, timing=True, fused_tail=True), out=image, stats=True)
        fstage += np.array(fstats["stage_ms"])
    stage /= reps
    fstage /= reps
    launches_per_step = int(stats["kernel_launches"])
    names = {0: "k_interval_root_coop_2d[L0,128px]", 1: "k_interval_level<2>[L1,32px]",
             2: "k_interval_level<2>[L2,8px]", 8: "k_fill_2d (x3)", 9: "k_pixels_2d"}
    ncu = ncu_table()
    n_fill_px = SIZE * SIZE - int(stats["pixels"])
    written = {0: 0, 1: 0, 2: 0, 8: n_fill_px * 4, 9: int(stats["pixels"]) * 4}     # bytes of the frame each kernel writes
    kernels = {}
    for k, nm in names.items():
        e = ncu.get(nm, {}) if isinstance(ncu.get(nm), dict) else {"dram_bytes": ncu.get(nm)}
        kernels[nm] = {"ms": float(stage[k]), "share": float(stage[k] / max(stage[15], 1e-9)),
                       "frame_bytes_written": written[k], "dram_bytes": e.get("dram_bytes"),
                       "issue_active_pct": e.get("issue_active_pct"), "pipe_fp32_pct": e.get("pipe_fp32_pct")}
    dom = max(names, key=lambda k: stage[k])
    algo = SIZE * SIZE * ALGO_BYTES_PER_PIXEL
    achieved = algo / (ms_per_step * 1e-3) / 1e9
    roofline = {"bound": "hbm", "kernel": "whole frame (dominant kernel: " + names[dom] + ")",
                "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                "traffic": sum(v["dram_bytes"] or 0 for v in kernels.values()) or None, "peak_source": peak_src,
                "algorithmic_bytes": algo,
                "definition": "SURVEY 8(d): 4 B per pixel WRITTEN per step / ms_per_step / measured HBM copy bandwidth; "
                              "traffic = sum of the kernels' dram bytes (ncu --set full, profiles/)",
                "stage_total_ms": float(stage[15]),
                "kernels": kernels,
                "experimental_fused_tail_ms": {"k_interval_root_coop_2d[L0,128px]": float(fstage[0]),
                                               "k_tail_2d (levels 1-2 + leaf pixels + fills, one persistent launch)": float(fstage[12])}}

    # ---- end to end through the public API with HOST buffers ----
    host_img = torch.empty((SIZE, SIZE), dtype=torch.float32).pin_memory()
    host_np = host_img.numpy()

    def e2e_step():
        s = fb.CudaShape(cuda, tape)          # uploads the bytecode (H2D) and builds the device tape
        fb.render2d(s, cfg, out=host_np)      # renders + copies the image back (D2H), synchronous
        return s

    for _ in range(3):
        e2e_step()
    sync_all()
    t0 = time.perf_counter()
    n_e2e = max(5, min(args.steps, 20))
    for _ in range(n_e2e):
        e2e_step()
    sync_all()
    e2e_dt = (time.perf_counter() - t0) / n_e2e
    e2e = {"value": SIZE * SIZE / e2e_dt / 1e6, "unit": "Mvoxels/s",
           "h2d_bytes_per_step": int(bc.words.nbytes), "d2h_bytes_per_step": int(SIZE * SIZE * 4),
           "ms_per_step": e2e_dt * 1e3,
           "note": "fc_tape_create from host bytecode + fc_render2d into a pinned host image, wall clock"}
    # the same call with the smaller output formats (derived on the device from the distance image)
    fmt_lines = {}
    for fmt, shape_, nbytes in (("mask_u8", (SIZE, SIZE), SIZE * SIZE), ("bitmap_1bit", (SIZE, SIZE // 8), SIZE * SIZE // 8),
                                ("rgba8", (SIZE, SIZE, 4), SIZE * SIZE * 4)):
        hbuf = torch.empty(shape_, dtype=torch.uint8).pin_memory().numpy()
        fcfg = fb.RenderConfig2D(SIZE, SIZE, out_format=fmt)

        def fstep():
            s = fb.CudaShape(cuda, tape)
            fb.render2d(s, fcfg, out=hbuf)
            return s

        for _ in range(3):
            fstep()
        t0 = time.perf_counter()
        for _ in range(n_e2e):
            fstep()
        dt = (time.perf_counter() - t0) / n_e2e
        fmt_lines[fmt] = {"value": SIZE * SIZE / dt / 1e6, "unit": "Mvoxels/s", "ms_per_step": dt * 1e3,
                          "d2h_bytes_per_step": nbytes}
    e2e["other_output_formats"] = fmt_lines
    return {
        "metric": METRIC, "value": value, "unit": "Mvoxels/s", "n_gpus": 1, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": ms_per_step, "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": WORKLOAD_2D,
                   "detail": "reference VM default tile sizes, pixel_perfect=false",
                   "parallelism": "single GPU",
                   "l2": "flushed between steps by a 512 MiB fill outside the event-timed regions"},
        "clocks": clocks.summary(), "e2e": e2e,
        "gpu_launches": launches_per_step * args.steps,
        "roofline": roofline,
    }


if __name__ == "__main__":
    main()
