#!/usr/bin/env python
"""bench.py -- frames/s of the per-frame hot path on synthetic 640x512 uint16 IR movies.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--dump-outputs DIR]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N ... bench.py --gpus N ...

`--dump-outputs DIR` writes what the last timed step returned on rank 0 as DIR/<name>.npy (float32, a
fixed sample of frames; float64 for the statistics), so that two builds can be compared output for
output: the inputs depend only on the arguments.

A "step" is one pass of the full per-frame pipeline (bad-pixel correct -> Gaussian u16->f32 ->
sub-pixel translate with per-frame shifts -> delta + byte-plane pre-coder -> min/max/histogram)
over one chunk of synthetic frames that is already resident in HBM.  Work per GPU is fixed
(weak scaling); frames are sharded by contiguous GOP-aligned ranges and the only collective is
the all-reduce of the statistics (outside the per-step path; timed once and reported).

One JSON line on rank 0 (the driver's contract): `value` = whole-job frames/s (device-timed,
max over ranks); `roofline` = the dominant kernel against the measured HBM copy peak; `e2e` =
the same metric through the public API with pinned HOST buffers (H2D + D2H inside the timed
region); `cpu_baseline` = the reference's CPU code on this box's cores (N=1 only).
`--impl reference` times the reference's own CPU implementation instead.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

W, H = 640, 512
GOP = 50
SIGMA = 1.0
METRIC = "frames/s at 640x512 u16 (full per-frame pipeline: bad-pixel correct + gaussian + translate + pre-coder)"
# algorithmic bytes per pixel of each kernel (SURVEY.md 8d): every input byte read once, every
# output byte written once
BYTES_PER_PX = {"bp_correct": 4, "gaussian_u16_f32": 6, "translate_u16": 4, "precode_delta_split": 4, "stats_minmax_hist": 2,
                # the statistics ride along in the pre-coder's pass: the frames are read once, the planes written once
                "precode_delta_split_stats": 4}


def ncu_traffic(kernel, frames):
    """DRAM bytes (read + write) of one launch of `kernel` over `frames` frames, from the committed
    ncu capture (profiles/ncu_traffic.json, one `ncu --set full` launch, scaled per frame)."""
    try:
        with open(os.path.join(ROOT, "profiles", "ncu_traffic.json")) as f:
            t = json.load(f)["kernels"][kernel]
        return t["dram_bytes_per_frame"] * frames
    except Exception:
        return None


def hbm_peak():
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            return float(json.load(f)["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
    except Exception:
        return 6650.0, "fallback (B200_PROFILING.md)"


# ------------------------------------------------------------------------------------------------
# synthetic movie (SURVEY.md 8d): smooth background + drifting hot spot + noise + stuck pixels
# ------------------------------------------------------------------------------------------------
def synth_movie_torch(nframes, first_frame, device, seed=1234):
    import torch

    g = torch.Generator(device=device).manual_seed(seed + first_frame)
    y = torch.arange(H, device=device, dtype=torch.float32).view(1, H, 1)
    x = torch.arange(W, device=device, dtype=torch.float32).view(1, 1, W)
    bg = 8000 + 2000 * torch.exp(-(((x - W / 2) / (0.23 * W)) ** 2) - ((y - H / 2) / (0.23 * H)) ** 2)
    gb = torch.Generator(device="cpu").manual_seed(4321)
    nbad = round(1e-3 * W * H)
    bad = torch.randperm(W * H, generator=gb)[:nbad].to(device)
    out = torch.empty((nframes, H, W), dtype=torch.uint16, device=device)
    step = 256
    for a in range(0, nframes, step):
        b = min(nframes, a + step)
        t = torch.arange(first_frame + a, first_frame + b, device=device, dtype=torch.float32).view(-1, 1, 1)
        cx, cy = W * 0.3 + 0.05 * t, H * 0.6 - 0.05 * t
        spot = 1500 * torch.exp(-(((x - cx) / 12.0) ** 2) - ((y - cy) / 12.0) ** 2)
        f = bg + spot + 3.0 * torch.randn((b - a, H, W), generator=g, device=device)
        f = f.clamp_(0, 16383).to(torch.int32)
        f = f.view(b - a, -1)
        f[:, bad[: nbad // 2]] = 0
        f[:, bad[nbad // 2:]] = 16000
        out.view(torch.int16)[a:b] = f.view(b - a, H, W).to(torch.int16)  # values < 2**15: same bits as uint16
    return out


def synth_movie_numpy(nframes, seed=1234):
    import numpy as np

    rng = np.random.default_rng(seed)
    y, x = np.mgrid[0:H, 0:W].astype(np.float32)
    bg = 8000 + 2000 * np.exp(-(((x - W / 2) / (0.23 * W)) ** 2) - ((y - H / 2) / (0.23 * H)) ** 2)
    nbad = round(1e-3 * W * H)
    bad = np.random.default_rng(4321).choice(W * H, nbad, replace=False)
    mov = np.empty((nframes, H, W), dtype=np.uint16)
    for t in range(nframes):
        cx, cy = W * 0.3 + 0.05 * t, H * 0.6 - 0.05 * t
        spot = 1500 * np.exp(-(((x - cx) / 12.0) ** 2) - ((y - cy) / 12.0) ** 2)
        f = np.clip(bg + spot + rng.normal(0, 3, (H, W)), 0, 16383).astype(np.uint16)
        f.flat[bad[: nbad // 2]] = 0
        f.flat[bad[nbad // 2:]] = 16000
        mov[t] = f
    return mov


# ------------------------------------------------------------------------------------------------
# clocks during the timed region
# ------------------------------------------------------------------------------------------------
class ClockSampler:
    FIELDS = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
              "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        self.rows = []
        self.proc = None
        self.gpu = gpu_index

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--id={self.gpu}", f"--query-gpu={self.FIELDS}",
                                          "--format=csv,noheader,nounits", "-lms", "100"], stdout=subprocess.PIPE,
                                         stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._read, daemon=True)
            self.thread.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in self.rows:
            if len(r) < 6:
                continue
            try:
                sm.append(float(r[0]))
                mx.append(float(r[1]))
            except ValueError:
                continue
            for n, v in zip(names, r[2:6]):
                if v.lower().startswith("active"):
                    reasons.add(n)
        if not sm:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["no samples"]}
        sm.sort()
        return {"sm_mhz": sm[len(sm) // 2], "sm_max_mhz": max(mx), "reasons": sorted(reasons), "samples": len(sm)}


# ------------------------------------------------------------------------------------------------
# CPU arms (the only place bench.py executes oracle/)
# ------------------------------------------------------------------------------------------------
def cpu_pipeline_fn():
    """Returns (fn(frames, dx, dy) -> None, kind): the reference's CPU path for one batch of
    frames -- oracle/_ref (the reference's own sources, stock flags) when it was built, else the
    C port."""
    import numpy as np

    from oracle import oracle as O

    port = O.Port()
    if O.have_ref():
        ref, kind = O.Ref(), "reference"
    else:
        ref, kind = port, "port"

    def make_state(first):
        return ref.bad_pixels_create(first)

    def run(handle, frames, dx, dy):
        for i, f in enumerate(frames):
            c = ref.bad_pixels_correct(handle, f)
            ref.gaussian_filter(c, SIGMA)
            r = ref.translate(c, dx[i], dy[i], "nearest", 0)
            port.split_444(r)  # the writer's byte-plane split (video_io cannot be built here: C restatement)

    return make_state, run, kind


def time_cpu(frames, dx, dy, threads):
    """frames/s of the CPU path over `frames`, frame-parallel over `threads` Python threads
    (ctypes releases the GIL; each call is the reference's stock single-threaded code)."""
    import numpy as np

    make_state, run, kind = cpu_pipeline_fn()
    handle = make_state(frames[0])
    run(handle, frames[:2], dx, dy)  # warm-up
    parts = np.array_split(np.arange(len(frames)), threads)
    t0 = time.perf_counter()
    if threads == 1:
        run(handle, frames, dx, dy)
    else:
        ths = [threading.Thread(target=run, args=(handle, frames[p[0]:p[-1] + 1], dx[p[0]:p[-1] + 1], dy[p[0]:p[-1] + 1]))
               for p in parts if len(p)]
        for t in ths:
            t.start()
        for t in ths:
            t.join()
    el = time.perf_counter() - t0
    return len(frames) / el, kind, el


def run_reference(args, out):
    """--impl reference: the reference's own CPU implementation of the path on this box's host
    cores, every step a bounded sample of the same workload."""
    import numpy as np

    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    cores = os.cpu_count() or 1
    sample = max(64, 8 * cores)
    mov = synth_movie_numpy(sample)
    rng = np.random.default_rng(777)
    dx = rng.uniform(-3, 3, sample).astype(np.float32)
    dy = rng.uniform(-3, 3, sample).astype(np.float32)
    kind = "port"
    for _ in range(args.warmup):
        _, kind, _ = time_cpu(mov, dx, dy, cores)
    total = 0.0
    for _ in range(args.steps):
        fps, kind, el = time_cpu(mov, dx, dy, cores)
        total += el
    value = sample * args.steps / total
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": "frames/s", "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": 1e3 * total / args.steps, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "u16", "data": "synthetic",
        "config": workload_config(sample, args.gpus) | {"note": "CPU arm: every step is a bounded sample of the workload"},
        "cpu_baseline": {"value": value, "unit": "frames/s", "cores": cores, "kind": kind,
                         "sample": f"{sample} frames of 640x512 per step, frame-parallel over {cores} threads, "
                                   f"each call the stock single-threaded reference code"},
        "e2e": {"value": value, "unit": "frames/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    out.emit(line)


# ------------------------------------------------------------------------------------------------
# the other BASELINE.json configs, each kernel alone (device-resident inputs far larger than L2)
# ------------------------------------------------------------------------------------------------
def synth_frames_torch(n, h, w, device, seed):
    """IR-like frames of any size (same recipe as synth_movie_torch, without the drifting spot)."""
    import torch

    g = torch.Generator(device=device).manual_seed(seed)
    y = torch.arange(h, device=device, dtype=torch.float32).view(1, h, 1)
    x = torch.arange(w, device=device, dtype=torch.float32).view(1, 1, w)
    bg = 8000 + 2000 * torch.exp(-(((x - w / 2) / (0.23 * w)) ** 2) - ((y - h / 2) / (0.23 * h)) ** 2)
    out = torch.empty((n, h, w), dtype=torch.uint16, device=device)
    step = max(1, (64 << 20) // (h * w * 4))
    for a in range(0, n, step):
        b = min(n, a + step)
        f = (bg + 3.0 * torch.randn((b - a, h, w), generator=g, device=device)).clamp_(0, 16383).to(torch.int16)
        out.view(torch.int16)[a:b] = f
    npx = h * w
    bad = torch.randperm(npx, generator=torch.Generator(device="cpu").manual_seed(4321))[: max(2, round(1e-3 * npx))].to(device)
    fv = out.view(torch.int16).view(n, -1)
    fv[:, bad[: len(bad) // 2]] = 0
    fv[:, bad[len(bad) // 2:]] = 16000
    return out


def measure_configs(dev, rank, world, dist, peak, reps=3):
    """BASELINE.json configs[0], [1], [3], [4] (C1, C2, C4, C5; C3 is the headline): every kernel of the path alone on
    device-resident movies of ~1.3 GB, CUDA events, one warm-up + median of `reps`, max over ranks.  Returns the `configs`
    object of the JSON line: {config: {case: {ms, gbs, frac, frames, frame}}}."""
    import statistics

    import torch

    from librir_b200 import movie, signal_processing as sp, video_io as vio

    INNER = 4  # launches per timed region: the host's work for launch i + 1 (tensor-map encoding, pointer queries, Python) then
    #            runs under launch i instead of in front of a 0.2 ms kernel; every input is far larger than L2

    def timed(fn):
        fn()
        times = []
        for _ in range(reps):
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            torch.cuda.synchronize()
            e0.record()
            for _i in range(INNER):
                fn()
            e1.record()
            torch.cuda.synchronize()
            times.append(e0.elapsed_time(e1) / INNER)
        t = torch.tensor([statistics.median(times)], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t[0])

    def cell(ms, bytes_per_px, n, h, w, **extra):
        gbs = bytes_per_px * n * h * w / (ms * 1e-3) / 1e9
        d = {"ms": round(ms, 4), "gbs": round(gbs, 1), "frac": round(gbs / peak, 3), "frames": n, "frame": [w, h],
             "frames_per_s_per_gpu": round(n / (ms * 1e-3))}
        d.update(extra)
        return d

    out = {}
    # ---- C1 / C2: 640x512 x 1000 ------------------------------------------------------------------
    n, h, w = 1000, H, W
    frames = synth_frames_torch(n, h, w, dev, 1234 + rank)
    bp = sp.BadPixels(frames[0])
    o16 = torch.empty_like(frames)
    o32 = torch.empty((n, h, w), dtype=torch.float32, device=dev)
    lo = torch.empty((n, h, w), dtype=torch.uint8, device=dev)
    hi = torch.empty_like(lo)
    c1 = {"what": "640x512 x 1000 frames, each kernel alone (bad-pixel correct, Gaussian at the three named sigmas, translate (1.3, -2.7) nearest)"}
    c1["bp_correct"] = cell(timed(lambda: bp.correct_batch(frames, out=o16)), 4, n, h, w)
    for sg in (0.5, 1.0, 2.0):
        c1[f"gaussian_u16_f32_sigma{sg}"] = cell(timed(lambda: sp.gaussian_filter_batch(frames, sg, out=o32)), 6, n, h, w, sigma=sg)
    c1["translate_u16"] = cell(timed(lambda: sp.translate_batch(frames, 1.3, -2.7, "nearest", background=0, out=o16)), 4, n, h, w)
    out["C1"] = c1
    c2 = {"what": "640x512 x 1000 frames through the pre-coder and back (GOP 50)"}
    c2["precode_split"] = cell(timed(lambda: vio.precode_movie(frames, GOP, False, 0, out=(lo, hi))), 4, n, h, w)
    c2["precode_delta_split"] = cell(timed(lambda: vio.precode_movie(frames, GOP, True, 0, out=(lo, hi))), 4, n, h, w)
    c2["decode_delta_merge"] = cell(timed(lambda: vio.decode_movie(lo, hi, GOP, True, 0, out=o16)), 4, n, h, w)
    c2["round_trip_is_identity"] = bool(torch.equal(o16.view(torch.int16), frames.view(torch.int16)))
    out["C2"] = c2
    del frames, o16, o32, lo, hi, bp
    torch.cuda.empty_cache()
    # ---- C4: 1024x1024, per-frame shifts, statistics and their all-reduce INSIDE the step ---------
    n, h, w = 600, 1024, 1024
    frames = synth_frames_torch(n, h, w, dev, 777 + rank)
    o16 = torch.empty_like(frames)
    g = torch.Generator(device=dev).manual_seed(777 + rank)
    dx = torch.rand(n, generator=g, device=dev) * 6 - 3
    dy = torch.rand(n, generator=g, device=dev) * 6 - 3
    stats = movie.MovieStats(dev)

    def c4_step():
        sp.translate_batch(frames, dx, dy, "nearest", background=0, out=o16)
        stats.reset()
        stats.update(o16)
        stats.all_reduce()

    c4_step()  # NCCL set-up of the shapes
    ms = timed(c4_step)
    out["C4"] = {"what": "1024x1024 x 600 frames per GPU per step: translate with per-frame shifts U(-3,3) + min/max/histogram + their "
                         "all-reduce (NCCL) inside the step",
                 "step": cell(ms, 6, n, h, w, frames_per_s_all_gpus=round(n * world / (ms * 1e-3))),
                 "translate_u16": cell(timed(lambda: sp.translate_batch(frames, dx, dy, "nearest", background=0, out=o16)), 4, n, h, w),
                 "stats_minmax_hist": cell(timed(lambda: stats.update(o16)), 2, n, h, w)}
    del frames, o16
    torch.cuda.empty_cache()
    # ---- C5: frame-size sweep ---------------------------------------------------------------------
    c5 = {"what": "each kernel alone per frame size, ~1.3 GB of input per launch; fractions of the measured copy bandwidth"}
    for w, h in [(320, 256), (640, 512), (1024, 1024), (1280, 1024), (2048, 2048)]:
        n = max(50, int(1.3e9 / (w * h * 2)) // 50 * 50)
        frames = synth_frames_torch(n, h, w, dev, 99 + rank)
        bp = sp.BadPixels(frames[0])
        o16 = torch.empty_like(frames)
        o32 = torch.empty((n, h, w), dtype=torch.float32, device=dev)
        lo = torch.empty((n, h, w), dtype=torch.uint8, device=dev)
        hi = torch.empty_like(lo)
        g = torch.Generator(device=dev).manual_seed(5 + rank)
        dx = torch.rand(n, generator=g, device=dev) * 6 - 3
        dy = torch.rand(n, generator=g, device=dev) * 6 - 3
        stats = movie.MovieStats(dev)
        c5[f"{w}x{h}"] = {
            "bp_correct": cell(timed(lambda: bp.correct_batch(frames, out=o16)), 4, n, h, w),
            "gaussian_u16_f32": cell(timed(lambda: sp.gaussian_filter_batch(frames, SIGMA, out=o32)), 6, n, h, w),
            "translate_u16": cell(timed(lambda: sp.translate_batch(frames, dx, dy, "nearest", background=0, out=o16)), 4, n, h, w),
            "precode_delta_split": cell(timed(lambda: vio.precode_movie(frames, GOP, True, 0, out=(lo, hi))), 4, n, h, w),
            "stats_minmax_hist": cell(timed(lambda: stats.update(frames)), 2, n, h, w),
        }
        del frames, o16, o32, lo, hi, bp
        torch.cuda.empty_cache()
    out["C5"] = c5
    out["timing"] = (f"every cell: median of {reps} timed regions of {INNER} back-to-back launches on the launching stream (CUDA events), "
                     "divided by the launch count; inputs far larger than L2")
    return out


def workload_config(chunk, n_gpus):
    return {
        "workload": "C3 (BASELINE.json configs[2]): WEST-style 640x512 uint16 movie, full per-frame pipeline, "
                    "frame-sharded; one step = one chunk per GPU",
        "frame": [W, H], "frames_per_step_per_gpu": chunk, "global_frames_per_step": chunk * n_gpus, "gop": GOP,
        "sigma": SIGMA, "translate": "per-frame shifts U(-3,3), nearest border", "precoder": "temporal delta + byte-plane split (+ min/max/histogram of the same frames)",
        "sharding": f"contiguous GOP-aligned frame ranges over {n_gpus} rank(s)",
        "l2": "inputs larger than L2 (each stage streams >= 2.7 GB per step)",
    }


DUMP_FRAMES = 8  # 5 outputs x 8 frames x 640x512 x 4 bytes: 52 MB per dump


def dump_outputs(path, outs, stats):
    """Write a fixed sample of frames of each array process_chunk returned (corrected, smoothed, registered, lo, hi) as
    float32, the sampled frame indices, and the step's statistics (min / max, histogram) as float64, to path/<name>.npy.
    The sample is frame 0, a key frame of the pre-coder (the chunk starts on a GOP boundary), and seeded others."""
    import numpy as np
    import torch

    os.makedirs(path, exist_ok=True)
    n = outs[0].shape[0]
    rest = np.random.default_rng(2024).choice(np.arange(1, n), min(n, DUMP_FRAMES) - 1, replace=False)
    idx = np.concatenate(([0], np.sort(rest)))
    sel = torch.from_numpy(idx).to(outs[0].device)
    arrays = {"frame_index": idx.astype(np.float64)}
    for name, t in zip(("corrected", "smoothed", "registered", "lo", "hi"), outs):
        if t.dtype == torch.uint16:  # read the bits as signed, then back to unsigned: few torch ops take uint16
            t = t.view(torch.int16).index_select(0, sel).to(torch.int32) & 0xFFFF
        else:
            t = t.index_select(0, sel)
        arrays[name] = t.to(torch.float32).cpu().numpy()
    arrays["stats_minmax"] = np.array([stats.min(), stats.max()], dtype=np.float64)
    arrays["stats_histogram"] = stats.histogram().astype(np.float64)
    for name, a in arrays.items():
        np.save(os.path.join(path, name + ".npy"), a)


# ------------------------------------------------------------------------------------------------
# GPU arm
# ------------------------------------------------------------------------------------------------
def run_ours(args, out):
    import numpy as np
    import torch
    import torch.distributed as dist

    from librir_b200 import _lib, movie

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device -- librir_b200 has no CPU path to time (use --impl reference)")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=dev)
    if world != args.gpus and rank == 0:
        print(f"bench.py: note: WORLD_SIZE={world} but --gpus {args.gpus}; using {world}", file=sys.stderr)

    chunk = args.chunk
    cfg = movie.PipelineConfig(width=W, height=H, sigma=SIGMA, strategy="nearest", gop=GOP, delta=True, chunk_frames=chunk,
                               fuse_stats=not args.unfused_stats)
    pipe = movie.FramePipeline(cfg, dev)
    # this rank's shard of the (virtual) movie: chunk frames per step, GOP-aligned
    shard = movie.shard_frames(chunk * world, world, rank, GOP)
    frames = synth_movie_torch(chunk, shard.start, dev)
    first = synth_movie_torch(1, 0, dev)[0] if rank != 0 else frames[0]
    pipe.set_first_frame(first)  # every rank derives the bad-pixel map from the movie's frame 0
    g = torch.Generator(device=dev).manual_seed(777 + rank)
    dx = torch.rand(chunk, generator=g, device=dev) * 6 - 3
    dy = torch.rand(chunk, generator=g, device=dev) * 6 - 3

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    nst = len(pipe.STAGES)
    for _ in range(args.warmup):
        pipe.process_chunk(frames, dx, dy, shard.start)
    ev = [[torch.cuda.Event(enable_timing=True) for _ in range(nst + 1)] for _ in range(args.steps)]
    t_start, t_stop = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    sampler = ClockSampler(local)
    barrier()
    if rank == 0:
        sampler.start()
    launches0 = _lib.launch_count()
    t_start.record()
    for k in range(args.steps):
        # a dump's statistics are the last step's alone, not a fold of every pass over the same chunk (one launch more)
        if args.dump_outputs and k == args.steps - 1:
            pipe.stats.reset()
        outs = pipe.process_chunk(frames, dx, dy, shard.start, events=ev[k])
    t_stop.record()
    barrier()
    launches = _lib.launch_count() - launches0
    clocks = sampler.stop() if rank == 0 else None
    ms = t_start.elapsed_time(t_stop)
    per_stage = [sum(ev[k][i].elapsed_time(ev[k][i + 1]) for k in range(args.steps)) / args.steps for i in range(nst)]
    if args.dump_outputs and rank == 0:  # before the later passes reuse the pipeline's buffers and statistics
        dump_outputs(args.dump_outputs, outs, pipe.stats)

    # the only collective of the path: statistics all-reduce (once per movie; timed for the record)
    warm = movie.MovieStats(dev)  # the first NCCL call of a shape pays its set-up: not what a movie pays per reduction
    warm.all_reduce()
    c0, c1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    c0.record()
    pipe.stats.all_reduce()
    c1.record()
    torch.cuda.synchronize()
    allreduce_ms = c0.elapsed_time(c1)

    # ---- e2e: same pipeline through the public API with pinned host buffers ---------------------
    e2e_n = min(args.e2e_frames, chunk)
    sub = args.e2e_sub
    host_in = torch.empty((e2e_n, H, W), dtype=torch.uint16).pin_memory()
    host_in.copy_(frames[:e2e_n])
    host_dx, host_dy = dx[:e2e_n].cpu().pin_memory(), dy[:e2e_n].cpu().pin_memory()
    host_lo = torch.empty((e2e_n, H, W), dtype=torch.uint8).pin_memory()
    host_hi = torch.empty((e2e_n, H, W), dtype=torch.uint8).pin_memory()
    e2e_steps = max(3, min(args.steps, 10))
    if args.e2e_api == "cabi":  # ONE call of the C ABI with host pointers: rirb_process_movie_host
        def e2e_call():
            movie.process_movie_host(pipe.bad_pixels, host_in, host_dx, host_dy, SIGMA, "nearest", 0, GOP, True, shard.start,
                                     host_lo, host_hi)
        e2e_what = ("rirb_process_movie_host (one C-ABI call): pinned host u16 frames + shifts -> bad-pixel correct -> gaussian "
                    "(kept on the device) -> translate -> delta pre-coder -> pinned host byte planes (lo, hi); sub-chunks of whole "
                    "GOPs (~64 MB) rotating over three streams")
    else:                       # the same chain driven from Python (torch copies + device-pointer C-ABI calls)
        def e2e_call():
            pipe.process_host(host_in, host_dx, host_dy, shard.start, host_lo, host_hi, sub)
        e2e_what = ("FramePipeline.process_host: pinned host u16 frames + shifts -> GPU pipeline -> pinned host byte planes (lo, hi), "
                    f"sub-chunks of {sub} frames rotating over three streams")
    for _ in range(2):
        e2e_call()
    barrier()
    t0 = time.perf_counter()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(e2e_steps):
        e2e_call()
    e1.record()
    barrier()
    e2e_ms = e0.elapsed_time(e1)  # device-timed; the events bracket uploads, kernels and downloads
    e2e_wall_ms = 1e3 * (time.perf_counter() - t0)
    # sanity: the e2e result equals the device-resident result
    ok = bool(torch.equal(host_lo[:64], pipe.process_chunk(frames[:e2e_n], dx[:e2e_n], dy[:e2e_n], shard.start,
                                                           with_stats=False)[3][:64].cpu()))

    # ---- what the host links carry with every rank copying at once, both directions (the e2e path's own roofline) ----
    link_gbs = None
    try:
        nb = 256 << 20
        lh_in = torch.empty(nb, dtype=torch.uint8).pin_memory()
        lh_out = torch.empty(nb, dtype=torch.uint8).pin_memory()
        ld_in = torch.empty(nb, dtype=torch.uint8, device=dev)
        ld_out = torch.empty(nb, dtype=torch.uint8, device=dev)
        ls1, ls2 = torch.cuda.Stream(device=dev), torch.cuda.Stream(device=dev)
        for timed_pass in (False, True):
            barrier()
            t_l = time.perf_counter()
            for _ in range(3):
                with torch.cuda.stream(ls1):
                    ld_in.copy_(lh_in, non_blocking=True)
                with torch.cuda.stream(ls2):
                    lh_out.copy_(ld_out, non_blocking=True)
            torch.cuda.synchronize()
            if timed_pass:
                link_gbs = 3 * nb / (time.perf_counter() - t_l) / 1e9  # per direction, this rank
        del lh_in, lh_out, ld_in, ld_out
    except Exception:
        link_gbs = None

    # ---- e2e with EVERY output returned (the smoothed float32 frames as well: 4 more bytes per pixel down) ----
    e2e_all = None
    if not args.no_e2e_all:
        host_sm = torch.empty((e2e_n, H, W), dtype=torch.float32).pin_memory()

        def e2e_all_call():
            movie.process_movie_host(pipe.bad_pixels, host_in, host_dx, host_dy, SIGMA, "nearest", 0, GOP, True, shard.start,
                                     host_lo, host_hi, host_sm)
        e2e_all_call()
        barrier()
        a0, a1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a0.record()
        for _ in range(e2e_steps):
            e2e_all_call()
        a1.record()
        barrier()
        e2e_all = a0.elapsed_time(a1)
        del host_sm

    # ---- C3 as named: 100,000 DISTINCT frames streamed through the chunk ring (device-resident, generated on the device) ----
    stream = None
    if args.stream_frames > 0:
        try:
            per_rank = max(chunk, (args.stream_frames // world) // chunk * chunk)
            nchunks = per_rank // chunk
            chunks = [frames] + [synth_movie_torch(chunk, shard.start + k * chunk, dev) for k in range(1, nchunks)]
            pipe.stats.reset()
            barrier()
            s0, s1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            s0.record()
            for k, ch in enumerate(chunks):
                pipe.process_chunk(ch, dx, dy, shard.start + k * chunk)
            s1.record()
            barrier()
            stream = (s0.elapsed_time(s1), per_rank)
            del chunks
            torch.cuda.empty_cache()
        except Exception as e:  # e.g. not enough free HBM next to another tenant: reported, not fatal
            stream = (None, str(e)[:200])

    configs = None
    if not args.no_configs:
        peak_all, _src = hbm_peak()
        configs = measure_configs(dev, rank, world, dist, peak_all)

    # ---- reduce over ranks ------------------------------------------------------------------------
    vals = torch.tensor([ms, e2e_ms, e2e_all or 0.0, (stream[0] if stream and stream[0] else 0.0)] + per_stage, dtype=torch.float64, device=dev)
    cnt = torch.tensor([launches], dtype=torch.int64, device=dev)
    link = torch.tensor([link_gbs or 0.0], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(vals, op=dist.ReduceOp.MAX)
        dist.all_reduce(cnt, op=dist.ReduceOp.SUM)
        dist.all_reduce(link, op=dist.ReduceOp.SUM)
    ms, e2e_ms, e2e_all_ms, stream_ms = float(vals[0]), float(vals[1]), float(vals[2]), float(vals[3])
    per_stage = [float(v) for v in vals[4:]]
    if rank == 0:
        peak, peak_src = hbm_peak()
        npx = W * H
        kernels = {}
        for name, t_ms in zip(pipe.STAGES, per_stage):
            gbs = BYTES_PER_PX[name] * npx * chunk / (t_ms * 1e-3) / 1e9
            kernels[name] = {"ms_per_launch": t_ms, "algorithmic_bytes_per_launch": BYTES_PER_PX[name] * npx * chunk,
                             "ncu_dram_bytes_per_launch": ncu_traffic(name, chunk),
                             "achieved_gbs": gbs, "frac_of_peak": gbs / peak, "share_of_step": t_ms / sum(per_stage)}
        dom = max(kernels, key=lambda k: kernels[k]["ms_per_launch"])
        value = chunk * world * args.steps / (ms * 1e-3)
        line = {
            "metric": METRIC, "value": value, "unit": "frames/s", "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": ms / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "u16",
            "data": "synthetic", "config": workload_config(chunk, world),
            "roofline": {"bound": "hbm", "kernel": dom, "achieved": kernels[dom]["achieved_gbs"], "peak": peak, "unit": "GB/s",
                         "frac": kernels[dom]["frac_of_peak"], "nominal_peak": 8000.0,
                         "frac_of_nominal": kernels[dom]["achieved_gbs"] / 8000.0,  # SURVEY.md 8d also quotes the 8 TB/s data-sheet figure
                         "traffic": ncu_traffic(dom, chunk),
                         "traffic_source": "profiles/ncu_traffic.json (ncu --set full, one launch, scaled per frame)",
                         "algorithmic_bytes": kernels[dom]["algorithmic_bytes_per_launch"], "peak_source": peak_src,
                         "pipeline_achieved": sum(BYTES_PER_PX[k] for k in pipe.STAGES) * npx * chunk / (sum(per_stage) * 1e-3) / 1e9},
            "kernels": kernels,
            "e2e": {"value": e2e_n * world * e2e_steps / (e2e_ms * 1e-3), "unit": "frames/s",
                    "h2d_bytes_per_step": e2e_n * (npx * 2 + 8), "d2h_bytes_per_step": e2e_n * npx * 2,
                    "frames_per_step_per_gpu": e2e_n, "steps": e2e_steps, "matches_device_path": ok,
                    "wall_ms_rank0": e2e_wall_ms,
                    "api": args.e2e_api, "what": e2e_what,
                    "note": "the Gaussian output stays on the device in this figure; `e2e_all_outputs` returns it as well"},
            "gpu_launches": int(cnt[0]), "clocks": clocks, "stats_allreduce_ms": allreduce_ms,
        }
        if float(link[0]) > 0:
            cap = float(link[0]) * 1e9 / (npx * 2)  # frames/s the links carry: 2 B/px up and 2 B/px down, both directions busy
            line["e2e"]["host_link"] = {"both_directions_gbs_per_direction_all_ranks": float(link[0]), "cap_frames_per_s": cap,
                                        "frac_of_cap": line["e2e"]["value"] / cap,
                                        "what": "pinned H2D + D2H copies of 256 MB by every rank at the same time, measured in this run: the "
                                                "end-to-end path's own roofline (profiles/r2_hostlink.md: this box's host side carries 47 / "
                                                "52 / 51 / 77 GB/s per direction at 1 / 2 / 4 / 8 GPUs, so the e2e figure cannot scale with N)"}
        if e2e_all:
            line["e2e_all_outputs"] = {"value": e2e_n * world * e2e_steps / (e2e_all_ms * 1e-3), "unit": "frames/s",
                                       "h2d_bytes_per_step": e2e_n * (npx * 2 + 8), "d2h_bytes_per_step": e2e_n * npx * 6,
                                       "what": "the same call with the smoothed float32 frames downloaded too (lo, hi, smoothed)"}
        if stream:
            if stream[0]:
                line["c3_stream"] = {"value": stream[1] * world / (stream_ms * 1e-3), "unit": "frames/s", "distinct_frames": stream[1] * world,
                                     "frames_per_gpu": stream[1], "ms": stream_ms,
                                     "what": "config 3 as named: that many DISTINCT device-resident frames through the reused chunk buffers, one pass"}
            else:
                line["c3_stream"] = {"unavailable": stream[1]}
        if configs is not None:
            line["configs"] = configs
        if world == 1 and not args.no_cpu:
            ncpu = args.cpu_frames
            mov = frames[:ncpu].cpu().view(torch.int16).numpy().view(np.uint16)
            fps, kind, el = time_cpu(mov, dx[:ncpu].cpu().numpy(), dy[:ncpu].cpu().numpy(), 1)
            line["cpu_baseline"] = {"value": fps, "unit": "frames/s", "cores": 1, "kind": kind,
                                    "sample": f"first {ncpu} frames of the step's chunk, {el:.1f} s, stock single-threaded "
                                              f"build (what librir ships: its OpenMP pragmas are never enabled)"}
        out.emit(line)
    if world > 1:
        dist.destroy_process_group()


class JsonOnlyStdout:
    """The driver reads ONE JSON line from stdout.  Native libraries (NCCL prints its version
    banner there) write to file descriptor 1 behind Python's back, so fd 1 is pointed at stderr
    for the duration of the run and the JSON line goes to the saved descriptor."""

    def __enter__(self):
        sys.stdout.flush()
        self.saved = os.dup(1)
        os.dup2(2, 1)
        return self

    def emit(self, obj):
        os.write(self.saved, (json.dumps(obj) + "\n").encode())

    def __exit__(self, *exc):
        sys.stdout.flush()
        os.dup2(self.saved, 1)
        os.close(self.saved)
        return False


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--chunk", type=int, default=4000, help="frames per step per GPU (multiple of the GOP)")
    ap.add_argument("--e2e-frames", type=int, default=1000)
    ap.add_argument("--e2e-api", default="cabi", choices=["cabi", "torch"],
                    help="host path: one rirb_process_movie_host call, or the Python-driven FramePipeline.process_host")
    ap.add_argument("--e2e-sub", type=int, default=100, help="frames per sub-chunk of the host path (rounded to whole GOPs)")
    ap.add_argument("--cpu-frames", type=int, default=300)
    ap.add_argument("--no-cpu", action="store_true")
    ap.add_argument("--unfused-stats", action="store_true", help="statistics as their own kernel instead of inside the pre-coder's pass")
    ap.add_argument("--no-configs", action="store_true", help="skip the per-kernel figures of the other BASELINE configs (C1, C2, C4, C5)")
    ap.add_argument("--no-e2e-all", action="store_true", help="skip the host-path figure that also downloads the smoothed frames")
    ap.add_argument("--stream-frames", type=int, default=100000,
                    help="distinct frames (all GPUs together) streamed once through the chunk ring: config 3 as named; 0 = skip")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write a sample of the last timed step's outputs to DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs writes what the GPU path computed: it needs --impl ours")
    args.warmup = max(args.warmup, 3) if args.impl == "ours" else args.warmup
    with JsonOnlyStdout() as out:
        if args.impl == "reference":
            run_reference(args, out)
        else:
            run_ours(args, out)


if __name__ == "__main__":
    main()
