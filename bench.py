#!/usr/bin/env python
"""Benchmark of the camera-ISP hot path (BASELINE.json metric: Gpixel/s packed12 -> RGB8/RGB16 ISP at 1/2/4/8 B200,
achieved HBM GB/s vs peak).

    python bench.py --gpus N --steps K --warmup W [--impl reference] [--workload cfg2|cfg1|cfg1_16|cfg3|cfg3_rot90|cfg5|cfg5_32]
                    [--cameras C] [--dump-outputs DIR]

A step = one pass of the hot path over one batch of synthetic packed12 frames already resident in HBM: the fused
packed12 -> demosaic -> tone map -> quantise sweep of batch k (``Camera32/16.process_packed12``) while the joint
metering of batch k+1 (moving-average update of the 9-float metrics) runs on a side stream -- one CUDA-graph replay
(``graphed.GraphedStream``, double-buffered ingest).  Default workload (N = 1) = BASELINE.json configs[1]: 6 x 5472x3648
packed12 frames -> linear tone map -> RGB16.  With N > 1 (torchrun, one rank per GPU) every rank runs the same per-GPU
batch on its own camera streams (weak scaling, no pixel traffic between GPUs) and the ranks exchange the metering
records over NVLink mailboxes so that all cameras share one exposure (``--shared-exposure``, default for N > 1).
``--cameras C`` instead shards C camera streams over the ranks (BASELINE configs[2]: 12 cameras; strong scaling).

Prints ONE JSON line (keys at the bottom of main()).  The default N = 1 run also times the other BASELINE
configurations (>= 0.5 s each) into ``configs``.  ``--dump-outputs DIR`` writes the outputs of the last of the K timed
steps (rank 0) as float32 ``DIR/out<i>.npy`` (see ``dump_outputs``): the inputs are seeded, so two builds run with the
same arguments can be compared output for output.  ``--impl reference`` times the CPU restatement of the reference path
(oracle/c/isp_oracle.c, OpenMP on all host cores): Taichi, and therefore the reference's own CPU backend, is not
installable in this image.
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

METRIC = "Gpixel/s packed12->RGB8/RGB16 ISP"
WORKLOADS = {
    # name: (frames, H, W, isp dtype, tonemap, out dtype, tonemap kwargs, description)
    "cfg2": (6, 3648, 5472, "f32", "linear", "u16", dict(gamma=1.0),
             "BASELINE configs[1]: 6 x 5472x3648 RGGB packed12 -> Malvar -> linear tonemap -> RGB16 (Camera32)"),
    "cfg1": (1, 3000, 4096, "f32", "reinhard", "u8", dict(gamma=1.0, intensity=1.0, light_adapt=1.0, color_adapt=0.0),
             "BASELINE configs[0]: 1 x 4096x3000 RGGB packed12 -> Malvar -> Reinhard -> RGB8 (Camera32)"),
    "cfg1_16": (6, 3000, 4096, "f16", "reinhard", "u8", dict(gamma=0.6),
                "reference bench/camera_isp.py: 6 x 4096x3000 -> Camera16 -> Reinhard gamma 0.6 -> RGB8"),
    "cfg3": (6, 3000, 4096, "f32", "reinhard", "u8", dict(gamma=0.9, intensity=3.0, light_adapt=0.9, color_adapt=0.0),
             "BASELINE configs[2] shard: 6 cameras x 4096x3000 per GPU, script tone-map settings -> RGB8 (Camera32)"),
    # BASELINE configs[4] per-GPU shard: 8 x 4096x3000 -> full ISP (Camera16, Reinhard script settings) -> bilinear resize
    # to width 1920 (aspect-preserving 1920x1406, the reference-pinned path, SURVEY 8d) -> fp16 output.  Resize runs
    # BEFORE metering / tone map like the reference (camera_isp.py:371-373), inside the sweep (csrc/resize_sweep.cuh).
    "cfg5": (8, 3000, 4096, "f16", "reinhard", "f16", dict(gamma=0.9, intensity=3.0, light_adapt=0.9, color_adapt=0.0),
             "BASELINE configs[4] shard: 8 x 4096x3000 -> ISP + bilinear resize_width 1920 (fused into the sweep) -> Reinhard -> fp16"),
}
# the same with the f32 ISP (Camera32): no f16 rounding of the intermediates to reproduce, fp16 only at the output
WORKLOADS["cfg5_32"] = (8, 3000, 4096, "f32", "reinhard", "f16", dict(gamma=0.9, intensity=3.0, light_adapt=0.9, color_adapt=0.0),
                        "BASELINE configs[4] shard with the f32 ISP: 8 x 4096x3000 -> Camera32 + bilinear resize_width 1920 (fused into the sweep) -> Reinhard -> fp16")
# the rig script's default output orientation (scripts/tonemap_scan.py: transform rotate_90): cfg3 with the image turned by the
# normalise pass of the one-sweep Reinhard form (csrc/fused_isp.cuh reinhard_out_transposed_kernel) -- outputs are (W, H, 3)
WORKLOADS["cfg3_rot90"] = WORKLOADS["cfg3"][:7] + ("BASELINE configs[2] shard as the rig script runs it: 6 x 4096x3000 -> Reinhard -> RGB8, rotate_90 "
                                                   "applied inside the call (Camera32)",)
TRANSFORM = {"cfg3_rot90": "rotate_90"}
RESIZE_WIDTH = {"cfg5": 1920, "cfg5_32": 1920}
OUT_BYTES = {"u8": 1, "u16": 2, "f16": 2, "f32": 4}
# dram__bytes_read.sum + dram__bytes_write.sum of the dominant kernel per launch, from the ncu --set full captures
# summarised under profiles/ (None where no capture exists); the source file is named next to the number
TRAFFIC = {"cfg2": (844.2e6, "profiles/r02_cfg2_sweep_fadd2_ncu.txt (181.0 MB read + 663.2 MB written; the last ~56 MB of writes still in L2)"),
           "cfg3": (500.0e6, "profiles/r02_map16_sweep_ncu.txt (111.7 MB read + 388.3 MB written: packed frames in, u16 map out; the tail of the writes still in L2)"),
           "cfg5": (243.2e6, "profiles/r02_resize_sweep_ncu.txt (148.4 MB read + 94.8 MB written)")}


def synth_frames_np(n, h, w, seed=1234):
    """SURVEY 8d generator on the host (numpy): the frames of the CPU arm"""
    frames = []
    yy, xx = np.mgrid[0:h, 0:w].astype(np.float32)
    for i in range(n):
        r = np.random.default_rng(seed + i)
        base = 0.5 + 0.35 * np.sin(xx / w * (5.1 + i) + 0.3 * i) * np.cos(yy / h * 3.7)
        gains = (0.9, 1.0, 0.7)
        cfa = np.empty((h, w), np.float32)
        cfa[0::2, 0::2] = base[0::2, 0::2] * gains[0]
        cfa[0::2, 1::2] = base[0::2, 1::2] * gains[1]
        cfa[1::2, 0::2] = base[1::2, 0::2] * gains[1]
        cfa[1::2, 1::2] = base[1::2, 1::2] * gains[2]
        cfa += 0.05 + 0.02 * (r.random((h, w), dtype=np.float32) - 0.5)
        v = np.clip(np.rint(np.clip(cfa, 0, 1) * 4095), 0, 4095).astype(np.uint32)
        p0, p1 = v[:, 0::2], v[:, 1::2]
        out = np.empty((h, w // 2, 3), np.uint8)
        out[..., 0] = p0 & 0xFF
        out[..., 1] = ((p1 & 0xF) << 4) | (p0 >> 8)
        out[..., 2] = p1 >> 4
        frames.append(out.reshape(h, w * 3 // 2))
    return frames


def synth_frames(n, h, w, seed, device):
    """SURVEY 8d generator on the device: smooth HDR-ish field x channel gains + 2 % noise, mosaiced (RGGB), 12 bit,
    packed with the standard layout (packed.encode12, bit-exact against the golden vectors).  Deterministic in
    (seed, camera index), so that rank 0 can rebuild every rank's frames for the N > 1 parity check."""
    import torch
    from taichi_image_b200 import packed
    yy = torch.arange(h, device=device, dtype=torch.float32)[:, None] / h
    xx = torch.arange(w, device=device, dtype=torch.float32)[None, :] / w
    gains = ((0, 0, 0.9), (0, 1, 1.0), (1, 0, 1.0), (1, 1, 0.7))
    frames = []
    for i in range(n):
        g = torch.Generator(device=device).manual_seed(seed + i)
        base = 0.5 + 0.35 * torch.sin(xx * (5.1 + (seed + i) % 7) + 0.3 * ((seed + i) % 11)) * torch.cos(yy * 3.7)
        cfa = torch.empty((h, w), device=device)
        for dy, dx, gain in gains:
            cfa[dy::2, dx::2] = base[dy::2, dx::2] * gain
        cfa += 0.05 + 0.02 * (torch.rand((h, w), generator=g, device=device) - 0.5)
        frames.append(packed.encode12(torch.round(cfa.clamp(0, 1) * 4095).to(torch.int32).to(torch.uint16)))
    return frames


class ClockSampler:
    """nvidia-smi clocks / throttle reasons during the timed region (B200_PROFILING.md recipe)."""
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.rows, self.proc = [], None
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(index), f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-lms", "20"], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append((time.time(), [x.strip() for x in line.split(",")]))

    def window(self, t0, t1):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        rows = [r for t, r in self.rows if t0 <= t <= t1]
        sm, mx, reasons = [], None, set()
        names = ("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap")
        for r in rows:
            try:
                sm.append(float(r[0])); mx = float(r[1])
            except Exception:
                continue
            for nme, val in zip(names, r[3:7]):
                if val.lower().startswith("active"):
                    reasons.add(nme)
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": mx, "reasons": sorted(reasons), "samples": len(sm)}

    def stop(self):
        if self.proc is not None:
            time.sleep(0.05)
            self.proc.terminate()


def measured_peak():
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            return float(json.load(f)["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    except Exception:
        return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


def host_threads() -> int:
    """all host cores this process may use (torchrun exports OMP_NUM_THREADS=1, which must not cap the CPU arm)"""
    try:
        return max(1, len(os.sched_getaffinity(0)))
    except AttributeError:
        return max(1, os.cpu_count() or 1)


def _oracle_kwargs(workload, threads):
    n, h, w, isp_dt, tonemap, out_dt, tm, _ = WORKLOADS[workload]
    kw = dict(pattern="RGGB", cam16=isp_dt == "f16", out_dtype="u16" if out_dt == "u16" else "u8", tonemap=tonemap,
              stride=8, nthreads=threads, **tm)
    rw = RESIZE_WIDTH.get(workload, 0)
    if rw:
        s = rw / w
        kw["resize"] = ((rw, round(h * s)), (s, s))
    return kw


def cpu_baseline(workload, budget_s=20.0, threads=0):
    """C/OpenMP restatement of the reference path on the host cores, on a bounded sample: whole frames of the workload
    (same size, same tone map, same dtype), one per repetition."""
    from oracle import c_oracle
    n, h, w, isp_dt, tonemap, out_dt, tm, _ = WORKLOADS[workload]
    frame = synth_frames_np(1, h, w)[0]
    threads = threads or host_threads()
    kw = _oracle_kwargs(workload, threads)
    c_oracle.process([frame], **kw)                 # warm-up (page faults, thread pool)
    t0 = time.perf_counter()
    reps = 0
    while True:
        c_oracle.process([frame], **kw)
        reps += 1
        if time.perf_counter() - t0 > budget_s or reps >= 50:
            break
    dt = (time.perf_counter() - t0) / reps
    return {"value": h * w / dt / 1e9, "unit": "Gpixel/s", "cores": threads, "kind": "port",
            "sample": f"{reps} x one {w}x{h} frame of the workload through oracle/c/isp_oracle.c "
                      f"(literal 13-tap demosaic, metering, {tonemap}, {out_dt}); Taichi CPU backend not installable"}


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    n, h, w, isp_dt, tonemap, out_dt, tm, desc = WORKLOADS[args.workload]
    from oracle import c_oracle
    frame = synth_frames_np(1, h, w)[0]
    cores = host_threads()
    kw = _oracle_kwargs(args.workload, cores)
    steps = min(args.steps, 60)                     # bounded: one frame takes ~0.1 s on the host cores
    for _ in range(min(args.warmup, 5)):
        c_oracle.process([frame], **kw)
    t0 = time.perf_counter()
    for _ in range(steps):
        c_oracle.process([frame], **kw)
    dt = time.perf_counter() - t0
    value = steps * h * w / dt / 1e9
    sample = (f"each step = one {w}x{h} frame of the workload through oracle/c/isp_oracle.c "
              f"(OpenMP, {cores} threads); the reference's Taichi CPU backend is not installable here")
    emit({
        "impl": "reference", "metric": METRIC, "value": value, "unit": "Gpixel/s", "n_gpus": args.gpus,
        "steps": steps, "warmup": min(args.warmup, 5), "ms_per_step": dt / steps * 1e3, "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "f32" if isp_dt == "f32" else "f16", "data": "synthetic",
        "config": {"workload": desc, "sample": sample},
        "cpu_baseline": {"value": value, "unit": "Gpixel/s", "cores": cores, "kind": "port", "sample": sample},
        "e2e": {"value": value, "unit": "Gpixel/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    })


_REAL_STDOUT = None


def emit(line: dict):
    """the ONE JSON line on the real stdout (everything else -- NCCL's version banner, library chatter -- was
    redirected to stderr at start-up)"""
    data = (json.dumps(line) + "\n").encode()
    if _REAL_STDOUT is None:
        sys.stdout.write(data.decode()); sys.stdout.flush()
    else:
        os.write(_REAL_STDOUT, data)


class Ctx:
    """per-process state shared by the workloads"""

    def __init__(self, args):
        import torch
        import torch.distributed as dist
        self.torch, self.dist, self.args = torch, dist, args
        self.world = int(os.environ.get("WORLD_SIZE", "1"))
        self.rank = int(os.environ.get("RANK", "0"))
        self.local_rank = int(os.environ.get("LOCAL_RANK", "0"))
        assert torch.cuda.is_available(), "bench.py needs a CUDA device (no CPU fallback)"
        self.device = torch.device("cuda", self.local_rank)
        torch.cuda.set_device(self.device)
        if self.world > 1:
            dist.init_process_group("nccl", device_id=self.device)     # rendezvous, mailbox handles, timing reductions only
        self.peak, self.peak_src = measured_peak()
        self.sampler = ClockSampler(self.local_rank) if self.rank == 0 else None

    def barrier(self):
        if self.world > 1:
            self.dist.barrier()

    def max_over_ranks(self, x: float) -> float:
        if self.world == 1:
            return x
        t = self.torch.tensor([x], device=self.device, dtype=self.torch.float64)
        self.dist.all_reduce(t, op=self.dist.ReduceOp.MAX)
        return float(t.item())


def uses_map16(isp_dt, out_dt, tm):
    """Camera32 Reinhard -> u8 takes the one-sweep u16-map path (taichi_image_b200/camera_isp.py:_fused_params) unless
    B200ISP_REINHARD_EXACT=1 keeps the exact max sweep + write sweep"""
    return (isp_dt == "f32" and out_dt == "u8" and float(tm.get("color_adapt", 0.0)) == 0.0 and 0.3 <= float(tm.get("gamma", 1.0)) <= 1.0
            and os.environ.get("B200ISP_REINHARD_EXACT", "0") != "1")


def launches_per_step(tonemap, isp_dt, resize, shared, lookahead, map16=False):
    """launches of OUR kernels per step, counted from the launch plan (DESIGN.md section 3):
    sweep: linear 1; Reinhard Camera32 -> u8 map sweep + normalise + the two gated fallback sweeps = 4 (exact form: max sweep +
    write sweep = 2); Camera16 store sweep + normalise = 2;
    resizing ISP: sweep + orphan columns (+ normalise for Reinhard) = 2 / 3;
    metering: cooperative 1; as look-ahead on the side stream 2; shared exposure 2 (exchange inside the kernels)"""
    sweep = (3 if tonemap == "reinhard" else 2) if resize else (2 if tonemap == "reinhard" else 1)
    if map16:
        sweep = 4
    return sweep + (2 if (shared or lookahead) else 1)


DUMP_BYTES = 48 << 20      # what --dump-outputs writes at most, sample index included


def dump_outputs(outs, directory):
    """The outputs of one step as float32 ``out<i>.npy`` (exact for u8 / u16 / f16): whole when all of them fit
    DUMP_BYTES, otherwise the same sample of flat element indices from each -- drawn without replacement by
    ``np.random.default_rng(0)`` and sorted, so it depends on the output shape only -- stored as float64
    ``sample_index.npy``."""
    import torch
    os.makedirs(directory, exist_ok=True)
    numel = outs[0].numel()
    k = DUMP_BYTES // (4 * len(outs) + 8)
    idx = None
    if 4 * numel * len(outs) > DUMP_BYTES:
        idx = np.sort(np.random.default_rng(0).choice(numel, k, replace=False))
        np.save(os.path.join(directory, "sample_index.npy"), idx.astype(np.float64))
        idx = torch.from_numpy(idx).to(outs[0].device)
    for i, o in enumerate(outs):
        v = o.float()                                   # before the gather: CUDA has none for uint16
        np.save(os.path.join(directory, f"out{i}.npy"), (v if idx is None else v.reshape(-1)[idx]).cpu().numpy())


def run_workload(ctx: Ctx, name: str, steps: int, warmup: int, min_seconds: float = 0.0, shared=None, cameras: int = 0,
                 isolate: bool = True, dump_dir=None):
    """Times `steps` steps of workload `name` (max over ranks, CUDA events), then -- when min_seconds > 0 -- keeps the same
    steps running for at least that long (timed the same way: the sustained figure with the clocks sampled under it).
    dump_dir: where rank 0 writes the outputs of the last of the `steps` timed steps (dump_outputs).
    Returns a dict of results plus the live objects the caller may reuse (isp, frames)."""
    torch = ctx.torch
    import taichi_image_b200 as tib
    from taichi_image_b200.graphed import GraphedStream
    args = ctx.args
    n, h, w, isp_dt, tonemap, out_dt, tm, desc = WORKLOADS[name]
    world, rank, device = ctx.world, ctx.rank, ctx.device
    cam_ids = list(range(rank * n, rank * n + n))
    if cameras:                       # strong scaling: `cameras` streams sharded over the ranks
        from taichi_image_b200.distributed import shard_cameras
        assert cameras >= world, "every rank needs at least one camera stream (it takes part in the exposure exchange)"
        cam_ids = list(shard_cameras(cameras, world, rank))
        n = len(cam_ids)
    shared = (world > 1) if shared is None else shared
    cam = tib.camera_isp.Camera16 if isp_dt == "f16" else tib.camera_isp.Camera32
    resize_w = RESIZE_WIDTH.get(name, 0)
    base = cam(tib.bayer.BayerPattern.RGGB, moving_alpha=0.1, device=device, resize_width=resize_w, demosaic=args.demosaic,
               transform=tib.interpolate.ImageTransform[TRANSFORM.get(name, "none")])
    isp = base
    if shared:
        from taichi_image_b200.distributed import SharedExposure
        isp = SharedExposure(base)
    # per-camera seeds: camera c of the rig always gets the same frame, whichever rank owns it
    frames = [synth_frames(1, h, w, 1234 + 17 * c, device)[0] for c in cam_ids]
    frames_b = [f.clone() for f in frames]                       # second ingest buffer set (double-buffered stream)
    plan = base._resize_plan(h, w)
    ho, wo = (h, w) if plan is None else (plan[0][1], plan[0][0])
    flip = base._fused_flip(h, tonemap, tib.as_dtype(out_dt), tm.get("gamma", 1.0), tm.get("color_adapt", 0.0))
    assert flip or name not in TRANSFORM, "the transform of this workload must be applied inside the fused call"
    oshape = (wo, ho, 3) if flip & 4 else (ho, wo, 3)
    outs = [torch.empty(oshape, dtype=tib.as_dtype(out_dt).torch, device=device) for _ in range(n)]
    px_per_step = n * h * w
    alg_bytes = px_per_step * 1.5 + n * ho * wo * 3 * OUT_BYTES[out_dt]

    graphed = None
    if args.graph and args.lookahead and n > 0:
        graphed = GraphedStream(isp, frames, outs, tonemap=tonemap, dtype=out_dt, next_frames=frames_b,
                                rows_per_task=args.rows_per_task, **tm)

    def step():
        if n == 0:
            return
        if graphed is not None:
            graphed.step()
        else:
            isp.process_packed12(frames, tonemap=tonemap, dtype=out_dt, out=outs, rows_per_task=args.rows_per_task,
                                 lookahead=frames if args.lookahead else None, **tm)

    def timed(k):
        start, stop = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        torch.cuda.synchronize()
        ctx.barrier()
        t0 = time.time()
        start.record()
        for _ in range(k):
            step()
        stop.record()
        torch.cuda.synchronize()
        t1 = time.time()
        ctx.barrier()
        return ctx.max_over_ranks(start.elapsed_time(stop)), t0, t1

    # The dominant kernel timed ALONE (same process, same resident inputs, CUDA events recorded by the library on the
    # launching stream right before / after the launch): inside the timed region it shares the GPU with the look-ahead
    # metering of the next batch.  Timed once right after the warm-up (the conditions MEASURED_PEAKS.json's burst copy
    # bandwidth was taken under) and once more after the sustained window.
    def kernel_alone():
        iso = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(10)]
        for a, b in iso:
            a.record(); b.record()
        torch.cuda.synchronize()
        for a, b in iso:
            base._run_fused(frames, tonemap, tib.as_dtype(out_dt), outs, tm, update_metering=False,
                            rows_per_task=args.rows_per_task, profile_events=(a, b), flip=flip)
        torch.cuda.synchronize()
        return sum(a.elapsed_time(b) for a, b in iso[2:]) / len(iso[2:])

    def roofline_of(kern_ms):
        if resize_w:
            kern, kern_bytes = "isp::stream2_resize_kernel (sweep + bilinear down-scaling) + orphan columns", \
                px_per_step * 1.5 + n * ho * wo * 3 * (OUT_BYTES[isp_dt] if tonemap == "reinhard" else OUT_BYTES[out_dt])
        elif tonemap == "reinhard" and isp_dt == "f16":
            kern, kern_bytes = "isp::stream2_kernel<EpiReinhardMax2, STORE> (map sweep: packed in, f16 map out)", px_per_step * (1.5 + 6.0)
        elif tonemap == "reinhard" and uses_map16(isp_dt, out_dt, tm):
            kern, kern_bytes = "isp::stream2_kernel<EpiReinhardMax2<Camera32>, STORE> (map sweep: packed in, u16 fixed-point map out)", px_per_step * (1.5 + 6.0)
        elif tonemap == "reinhard":
            kern, kern_bytes = "isp::stream2_kernel<EpiReinhard2> (write sweep of the max + write pair)", alg_bytes
        else:
            kern, kern_bytes = "isp::stream2_kernel<EpiLinear2> (fused packed12 sweep, pair engine)", alg_bytes
        achieved = kern_bytes / (kern_ms * 1e-3) / 1e9
        traffic = TRAFFIC.get(name)
        return {"bound": "hbm", "achieved": achieved, "peak": ctx.peak, "unit": "GB/s", "frac": achieved / ctx.peak,
                "kernel": kern, "kernel_ms": kern_ms, "algorithmic_bytes_per_launch": kern_bytes,
                "peak_source": ctx.peak_src, "bytes_per_pixel": kern_bytes / px_per_step,
                "timing": "kernel timed alone right after the warm-up: 8 launches, CUDA events recorded by the library "
                          "around the launch on the launching stream",
                "traffic": traffic[0] if traffic else None, "traffic_source": traffic[1] if traffic else None}

    for _ in range(max(warmup, 3)):
        step()
    kern_ms_cool = kernel_alone() if (isolate and n > 0) else None
    total_px = world * px_per_step if not cameras else cameras * h * w
    ms, t0, t1 = timed(steps)
    if dump_dir and rank == 0 and n > 0:
        dump_outputs(outs, dump_dir)
    res = {"workload": desc, "value": total_px * steps / (ms * 1e-3) / 1e9, "ms_per_step": ms / steps, "steps": steps,
           "frames_per_gpu": n, "height": h, "width": w, "tonemap": tonemap, "out_dtype": out_dt, "isp_dtype": isp_dt}
    clocks = ctx.sampler.window(t0, t1) if ctx.sampler else None
    if clocks is not None:
        clocks["window"] = "timed region"
    if min_seconds > 0:
        k2 = max(steps, int(min_seconds * 1e3 / max(ms / steps, 1e-3)) + 1)
        k2 = int(ctx.max_over_ranks(float(k2)))
        ms2, t0s, t1s = timed(k2)
        res["sustained"] = {"value": total_px * k2 / (ms2 * 1e-3) / 1e9, "ms_per_step": ms2 / k2, "steps": k2,
                            "seconds": ms2 * 1e-3}
        if ctx.sampler:
            res["sustained"]["clocks"] = ctx.sampler.window(t0s, t1s)
            if clocks is not None and not clocks.get("samples"):
                clocks = dict(res["sustained"]["clocks"], window=f"the {ms2 * 1e-3:.2f} s sustained window right after the (too short) timed region")
    res["clocks"] = clocks

    if isolate and n > 0:
        hot_ms = kernel_alone()
        res["roofline"] = roofline_of(kern_ms_cool)
        res["roofline"]["after_sustained_window"] = {"kernel_ms": hot_ms, "frac": res["roofline"]["algorithmic_bytes_per_launch"] / (hot_ms * 1e-3) / 1e9 / ctx.peak,
                                                     "note": "the same isolated timing repeated right after the sustained window (power-capped clocks)"}
        res["step_gbps"] = alg_bytes / (res["ms_per_step"] * 1e-3) / 1e9
        res["step_frac_of_peak"] = res["step_gbps"] / ctx.peak
    res["gpu_launches_per_step"] = launches_per_step(tonemap, isp_dt, bool(resize_w), shared, bool(args.lookahead),
                                                      map16=tonemap == "reinhard" and not resize_w and uses_map16(isp_dt, out_dt, tm))
    res["_live"] = dict(isp=isp, base=base, frames=frames, outs=outs, n=n, cam_ids=cam_ids, shared=shared, tm=tm)
    return res


def parity_across_ranks(ctx: Ctx, name: str, live, cameras: int):
    """N > 1: every rank's metrics must be bit-identical, and equal to (a) the same split reduction emulated on rank 0
    over ALL ranks' frames (bit-exact) and (b) the single-call joint metering of all frames (reduction order aside)."""
    torch, dist = ctx.torch, ctx.dist
    import taichi_image_b200 as tib
    from taichi_image_b200.distributed import shard_cameras
    n, h, w, isp_dt, tonemap, out_dt, tm, _ = WORKLOADS[name]
    base = live["base"]
    mine = base.metrics.detach().clone().reshape(1, 9)
    allm = torch.empty((ctx.world, 9), dtype=torch.float32, device=ctx.device)
    dist.all_gather_into_tensor(allm, mine)
    out = {"ranks_bit_identical": bool((allm.view(torch.int32) == allm[0:1].view(torch.int32)).all().item())}
    if ctx.rank == 0:
        per_rank = [list(shard_cameras(cameras, ctx.world, r)) for r in range(ctx.world)] if cameras else \
                   [list(range(r * n, r * n + n)) for r in range(ctx.world)]
        cam = tib.camera_isp.Camera16 if isp_dt == "f16" else tib.camera_isp.Camera32
        rw = RESIZE_WIDTH.get(name, 0)
        shards = [[synth_frames(1, h, w, 1234 + 17 * c, ctx.device)[0] for c in ids] for ids in per_rank]
        # (a) the split reduction of every rank, emulated here: phase1 / phase2 per shard, folded in rank order.  With
        # constant frames the moving average is stationary after the first update (lerp of identical values), so one
        # update from zero metrics reproduces the ranks' state.
        emu = [cam(tib.bayer.BayerPattern.RGGB, moving_alpha=0.1, device=ctx.device, resize_width=rw) for _ in shards]
        for e in emu:
            e._metrics_and_alpha()
        live_shards = [(e, s) for e, s in zip(emu, shards) if s]
        g1 = torch.stack([e.meter_phase1(s) for e, s in live_shards]).contiguous()
        g2 = torch.stack([e.meter_phase2(s, g1, 0.0) for e, s in live_shards]).contiguous()
        emu[0].meter_finalize(g1, g2, 0.0)
        # (b) one joint call over all cameras
        joint = cam(tib.bayer.BayerPattern.RGGB, moving_alpha=0.1, device=ctx.device, resize_width=rw)
        flat = [f for s in shards for f in s]
        joint._metrics_and_alpha()
        joint.meter_packed12(flat, 0.0)
        torch.cuda.synchronize()
        m0 = allm[0].cpu().numpy()
        out["equals_emulated_split_bit_exact"] = bool(np.array_equal(m0, emu[0].metrics.cpu().numpy()))
        out["max_rel_diff_vs_joint_single_gpu"] = float(np.max(np.abs(m0 - joint.metrics.cpu().numpy()) / np.maximum(np.abs(m0), 1e-6)))
        out["cameras_total"] = len(flat)
        ok = out["ranks_bit_identical"] and out["max_rel_diff_vs_joint_single_gpu"] < 5e-6
        out["status"] = "ok" if ok else "MISMATCH"
    return out


def host_copy_ceiling(ctx: Ctx, seconds=0.25, mbytes=256):
    """pinned-memory H2D || D2H memcpy rate of this process while every rank does the same: the ceiling of the e2e leg"""
    torch = ctx.torch
    nb = mbytes << 20
    h_in, h_out = torch.empty(nb, dtype=torch.uint8, pin_memory=True), torch.empty(nb, dtype=torch.uint8, pin_memory=True)
    d_in, d_out = torch.empty(nb, dtype=torch.uint8, device=ctx.device), torch.empty(nb, dtype=torch.uint8, device=ctx.device)
    s1, s2 = torch.cuda.Stream(ctx.device), torch.cuda.Stream(ctx.device)
    torch.cuda.synchronize()
    ctx.barrier()
    t0 = time.perf_counter()
    reps = 0
    while time.perf_counter() - t0 < seconds:
        with torch.cuda.stream(s1):
            d_in.copy_(h_in, non_blocking=True)
        with torch.cuda.stream(s2):
            h_out.copy_(d_out, non_blocking=True)
        reps += 1
        if reps % 4 == 0:
            torch.cuda.synchronize()
    torch.cuda.synchronize()
    dt = time.perf_counter() - t0
    ctx.barrier()
    each = reps * nb / dt / 1e9
    tot = each * 2
    if ctx.world > 1:
        t = torch.tensor([tot], device=ctx.device, dtype=torch.float64)
        ctx.dist.all_reduce(t)
        tot = float(t.item())
    return {"h2d_gbs_per_rank": each, "d2h_gbs_per_rank": each, "all_ranks_both_directions_gbs": tot,
            "how": f"{mbytes} MB pinned buffers, H2D and D2H on two streams concurrently, all ranks at once, {seconds} s"}


def run_e2e(ctx: Ctx, name: str, live, ksteps: int, yuv420=False):
    """end to end through the public API with HOST buffers: pinned host -> H2D -> fused ISP -> D2H -> pinned host"""
    torch = ctx.torch
    from taichi_image_b200.pipeline import RigPipeline
    n, h, w, isp_dt, tonemap, out_dt, tm, desc = WORKLOADS[name]
    n = live["n"]
    if n == 0:
        return None
    pipe = RigPipeline(live["isp"], n, h, w, tonemap=tonemap, dtype=out_dt, depth=2, yuv420=yuv420, **live["tm"])
    pinned = [f.cpu().pin_memory() for f in live["frames"]]
    for _ in range(3):
        pipe.process(pinned)
    torch.cuda.synchronize()
    ctx.barrier()
    t_a = time.perf_counter()
    tickets, checksum = [], 0
    for i in range(ksteps):
        tickets.append(pipe.submit(pinned))
        if len(tickets) == 2:
            checksum += int(pipe.result(tickets.pop(0))[0].reshape(-1)[0])
    while tickets:
        checksum += int(pipe.result(tickets.pop(0))[0].reshape(-1)[0])
    torch.cuda.synchronize()
    dt = ctx.max_over_ranks(time.perf_counter() - t_a)
    px = ctx.world * n * h * w
    return {"value": px * ksteps / dt / 1e9, "unit": "Gpixel/s", "h2d_bytes_per_step": pipe.h2d_bytes_per_step,
            "d2h_bytes_per_step": pipe.d2h_bytes_per_step, "steps": ksteps, "workload": desc + (" -> planar YUV 4:2:0" if yuv420 else ""),
            "host_gbs": ctx.world * (pipe.h2d_bytes_per_step + pipe.d2h_bytes_per_step) * ksteps / dt / 1e9,
            "pipeline": "pinned host -> H2D -> fused ISP -> D2H -> pinned host, 2 slots, 3 streams", "checksum": checksum}


def main():
    global _REAL_STDOUT
    sys.stdout.flush()
    _REAL_STDOUT = os.dup(1)
    os.dup2(2, 1)                      # fd 1 -> stderr for native libraries and stray prints
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=200, help="timed steps of the workload: `value` and --dump-outputs come "
                    "from exactly these (the sustained window and the other configurations are timed separately)")
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--workload", default="cfg2", choices=sorted(WORKLOADS))
    ap.add_argument("--cameras", type=int, default=0, help="shard this many camera streams over the ranks (strong scaling; "
                    "BASELINE configs[2]: --workload cfg3 --cameras 12)")
    ap.add_argument("--shared-exposure", type=int, default=-1, help="exchange the metering records across ranks (default: on for N > 1)")
    ap.add_argument("--rows-per-task", type=int, default=0)
    ap.add_argument("--demosaic", default="malvar", choices=["malvar", "bilinear"],
                    help="bilinear: the north_star's alternative demosaic inside the fused sweep (not the BASELINE configuration)")
    ap.add_argument("--e2e-steps", type=int, default=12)
    ap.add_argument("--lookahead", type=int, default=1, help="meter the next batch on a side stream under this batch's sweep "
                    "(camera-stream mode; 0 = strictly serial steps)")
    ap.add_argument("--graph", type=int, default=1, help="replay the step (sweep k || metering k+1) as a CUDA graph; 0 = eager calls")
    ap.add_argument("--configs", type=int, default=-1, help="also time the other BASELINE configurations into `configs` "
                    "(default: on for the plain N = 1 run of the default workload)")
    ap.add_argument("--min-seconds", type=float, default=0.5, help="length of the sustained window after the K timed steps")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the outputs of the last timed step of the workload to DIR/out<i>.npy (float32; a fixed "
                         "sample of at most 48 MiB in all, see dump_outputs)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.impl == "reference":
        if args.dump_outputs:
            ap.error("--dump-outputs writes the outputs of the CUDA path (--impl b200)")
        return run_reference(args)

    ctx = Ctx(args)
    world, rank = ctx.world, ctx.rank
    shared = (world > 1) if args.shared_exposure < 0 else bool(args.shared_exposure)
    name = args.workload
    top = run_workload(ctx, name, args.steps, args.warmup, min_seconds=args.min_seconds, shared=shared, cameras=args.cameras,
                       dump_dir=args.dump_outputs)
    live = top.pop("_live")
    n, h, w, isp_dt, tonemap, out_dt, tm, desc = WORKLOADS[name]

    parity = None
    if world > 1 and shared:
        parity = parity_across_ranks(ctx, name, live, args.cameras)

    e2e = None
    if not args.no_e2e:
        e2e = run_e2e(ctx, name, live, args.e2e_steps)
        if e2e is not None:
            e2e["host_ceiling"] = host_copy_ceiling(ctx)

    # the shared-exposure step at N = 1 (exchange with itself: same kernels, same launch count as N > 1), so that the
    # scaling run compares like with like
    shared_n1 = None
    if world == 1 and not shared and not args.cameras and args.configs != 0:
        r = run_workload(ctx, name, max(args.steps, 50), args.warmup, min_seconds=0.3, shared=True, isolate=False)
        r.pop("_live")
        shared_n1 = {"value": r["value"], "ms_per_step": r["ms_per_step"], "sustained": r.get("sustained"),
                     "note": "the same step with the shared-exposure exchange on (world 1: the rank exchanges with itself)"}

    configs, e2e_variants = None, None
    want_configs = (world == 1 and name == "cfg2" and not args.cameras) if args.configs < 0 else bool(args.configs)
    if want_configs:
        configs = []
        for other in ("cfg1", "cfg3", "cfg3_rot90", "cfg1_16", "cfg5"):
            if other == name:
                continue
            r = run_workload(ctx, other, 50, args.warmup, min_seconds=args.min_seconds)
            lv = r.pop("_live")
            item = {"workload": r["workload"], "value": r["sustained"]["value"], "ms_per_step": r["sustained"]["ms_per_step"],
                    "timed_seconds": r["sustained"]["seconds"], "steps": r["sustained"]["steps"],
                    "roofline": {k: r["roofline"][k] for k in ("frac", "kernel", "kernel_ms", "achieved", "bytes_per_pixel", "traffic", "traffic_source", "after_sustained_window")},
                    "step_frac_of_peak": r["step_frac_of_peak"], "clocks": r["sustained"].get("clocks")}
            if not args.no_e2e and other in ("cfg3", "cfg1_16"):
                # the metric's own dtype (RGB8) and the 1.5 B/px planar YUV 4:2:0 output end to end
                e2e_variants = e2e_variants or []
                e2e_variants.append(run_e2e(ctx, other, lv, args.e2e_steps))
                e2e_variants.append(run_e2e(ctx, other, lv, args.e2e_steps, yuv420=True))
            configs.append(item)
            del lv

    if ctx.sampler:
        ctx.sampler.stop()
    if rank != 0:
        if world > 1:
            ctx.dist.destroy_process_group()
        return

    cpu = None
    if not args.no_cpu_baseline and world == 1:
        cpu = cpu_baseline(name)

    scaling = "strong" if args.cameras else "weak"
    config = {"workload": desc, "frames_per_gpu": top["frames_per_gpu"], "height": h, "width": w, "tonemap": tonemap, "out_dtype": out_dt,
              "shared_exposure": bool(shared), "lookahead_metering": bool(args.lookahead),
              "cuda_graph": bool(args.graph and args.lookahead), "ingest": "double-buffered (two input buffer sets alternate)",
              "l2": "inputs+outputs per step exceed the 126 MB L2 (no flush needed)" if n * h * w * 4.5 > 200e6
                    else "per-step working set near L2 size: stated, not flushed; two input sets alternate"}
    if args.cameras:
        from taichi_image_b200.distributed import max_cameras_per_rank
        config.update({"cameras_total": args.cameras, "cameras_on_busiest_rank": max_cameras_per_rank(args.cameras, world),
                       "ideal_speedup_cap": args.cameras / max_cameras_per_rank(args.cameras, world)})
    line = {
        "metric": METRIC, "value": top["value"], "unit": "Gpixel/s", "n_gpus": world, "steps": args.steps,
        "warmup": max(args.warmup, 3), "ms_per_step": top["ms_per_step"], "higher_is_better": True, "scaling": scaling,
        "vs_baseline": None, "dtype": isp_dt, "data": "synthetic", "config": config, "clocks": top["clocks"],
        "sustained": top.get("sustained"),
        "gpu_launches": top["gpu_launches_per_step"] * args.steps,
        "roofline": top.get("roofline"), "step_gbps": top.get("step_gbps"), "step_frac_of_peak": top.get("step_frac_of_peak"),
        "e2e": e2e, "e2e_variants": e2e_variants, "cpu_baseline": cpu, "configs": configs,
        "shared_exposure_at_n1": shared_n1, "parity_nranks": parity,
    }
    emit(line)
    if world > 1:
        ctx.dist.destroy_process_group()


if __name__ == "__main__":
    main()
