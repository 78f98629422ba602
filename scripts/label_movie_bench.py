"""Throughput of rirb_label_movie (events of the (t, y, x) volume + statistics) on one GPU, against label_batch on the same
frames and against scipy.ndimage.label on the volume on one host core.

Workloads, at 640x512 and 1024x1024, connectivity 6, 18 and 26:
  ir     -- the IR movie of tests/conftest.py (32 distinct frames, repeated) above 9900: the background's hot centre, the
            drifting spot and the stuck-pixel specks, each one event through time;
  noise  -- uniform 3-D noise at the site-percolation density of the connectivity (0.31 for 6, 0.14 for 18, 0.10 for
            26), where events are largest and most tangled;
  full   -- every voxel foreground: one event holds the whole movie (the links' and statistics' worst contention).
Each timed pass is one call over --frames frames in HBM (more bytes than the 126 MB L2), CUDA events, median of --passes
after a warm-up call.  label_batch_frames_per_s is label_batch at the in-plane connectivity (4 for 6, else 8) without
statistics on the same frames in the same run: what the 2-D half costs.  scipy runs on the first --host-frames frames
as one volume, reported per frame.  Writes one JSON line per cell to --out and prints it.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

DENSITY = {6: 0.31, 18: 0.14, 26: 0.10}


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                       capture_output=True, text=True)
    return q.stdout.strip()


def workload(torch, name, n, h, w, conn, distinct=32):
    """uint16 frames [n, h, w] on the device and the threshold."""
    if name == "ir":
        from tests.conftest import ir_movie

        base = torch.from_numpy(ir_movie(distinct, h, w).view(np.int16)).cuda()
        reps = (n + distinct - 1) // distinct
        return base.repeat(reps, 1, 1)[:n].contiguous().view(torch.uint16), 9900
    g = torch.Generator(device="cuda").manual_seed(5)
    if name == "noise":
        f = (torch.rand((n, h, w), generator=g, device="cuda") < DENSITY[conn]).to(torch.int16) * 1000
        return f.view(torch.uint16), 500
    return torch.full((n, h, w), 1000, dtype=torch.int16, device="cuda").view(torch.uint16), 500


def time_gpu(torch, fn, passes):
    fn()
    torch.cuda.synchronize()
    ts = []
    for _ in range(passes):
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        out = fn()
        b.record()
        torch.cuda.synchronize()
        ts.append(a.elapsed_time(b) / 1e3)
    return float(np.median(ts)), ts, out


def time_scipy(frames_np, thr, conn):
    from scipy import ndimage

    st = ndimage.generate_binary_structure(3, {6: 1, 18: 2, 26: 3}[conn])
    mask = frames_np > thr
    t0 = time.perf_counter()
    ndimage.label(mask, structure=st)
    return (time.perf_counter() - t0) / len(frames_np) * 1e3


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--frames", type=int, default=4000)
    ap.add_argument("--passes", type=int, default=5)
    ap.add_argument("--cap", type=int, default=256)
    ap.add_argument("--sizes", default="512x640,1024x1024")
    ap.add_argument("--host-frames", type=int, default=20)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    import torch

    if not torch.cuda.is_available():
        sys.exit("label_movie_bench: needs a CUDA device")
    from librir_b200 import signal_processing as sp

    torch.cuda.set_device(0)
    info = card()
    lines = []
    for size in a.sizes.split(","):
        h, w = (int(v) for v in size.split("x"))
        for conn in (6, 18, 26):
            for name in ("ir", "noise", "full"):
                frames, thr = workload(torch, name, a.frames, h, w, conn)
                labels = torch.empty(frames.shape, dtype=torch.int32, device="cuda")
                med, ts, out = time_gpu(torch, lambda: sp.label_movie(frames, thr, conn, a.cap, labels=labels), a.passes)
                plane = 4 if conn == 6 else 8
                med2d, _, counts = time_gpu(torch, lambda: sp.label_batch(frames, thr, plane, 0, labels=labels)[1], a.passes)
                host_ms = time_scipy(frames[:a.host_frames].cpu().view(torch.int16).numpy().view(np.uint16), thr, conn)
                rec = dict(bench="label_movie", card=info, h=h, w=w, connectivity=conn, workload=name, frames=a.frames,
                           max_events=a.cap, median_s=med, passes_s=ts, frames_per_s=a.frames / med, events=out[1],
                           components_2d=int(counts.long().sum().item()), label_batch_frames_per_s=a.frames / med2d,
                           time_over_label_batch=med / med2d, host_frames=a.host_frames, scipy_3d_ms_per_frame=host_ms,
                           host_frames_per_s_scipy=1e3 / host_ms)
                print(json.dumps(rec), flush=True)
                lines.append(rec)
                del frames, labels, out, counts
                torch.cuda.empty_cache()
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            for rec in lines:
                f.write(json.dumps(rec) + "\n")


if __name__ == "__main__":
    main()
