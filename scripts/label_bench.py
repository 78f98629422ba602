"""Throughput of rirb_label_batch (labels + counts + statistics) on one GPU, against scipy and OpenCV on one host core.

Workloads, at 640x512 and 1024x1024, connectivity 4 and 8:
  ir     -- the IR movie of tests/conftest.py thresholded above its background (the hot spot and the stuck-pixel specks);
  noise  -- uniform noise at the site-percolation density of the connectivity (0.59 for 4, 0.41 for 8), where components
            are largest and most tangled: long union chains across tiles;
  full   -- every pixel foreground: one component holds the whole frame (the statistics' worst contention).
Each timed pass is one call over --frames frames (more bytes than the 126 MB L2), CUDA events, median of --passes after a
warm-up call.  The bound is the compulsory traffic, 2 B/px read + 4 B/px of labels written = 6 B/px, at 7.7 TB/s.
Writes one JSON line per cell to --out and prints it.
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

HBM_BYTES_PER_S = 7.7e12
BYTES_PER_PX = 6


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
        d = 0.59 if conn == 4 else 0.41
        f = (torch.rand((n, h, w), generator=g, device="cuda") < d).to(torch.int16) * 1000
        return f.view(torch.uint16), 500
    return torch.full((n, h, w), 1000, dtype=torch.int16, device="cuda").view(torch.uint16), 500


def time_gpu(torch, sp, frames, thr, conn, cap, passes):
    labels = torch.empty(frames.shape, dtype=torch.int32, device="cuda")
    sp.label_batch(frames, thr, conn, cap, labels=labels)
    torch.cuda.synchronize()
    ts = []
    for _ in range(passes):
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        _, counts, _ = sp.label_batch(frames, thr, conn, cap, labels=labels)
        b.record()
        torch.cuda.synchronize()
        ts.append(a.elapsed_time(b) / 1e3)
    return float(np.median(ts)), ts, counts


def time_host(frames_np, thr, conn, reps=10):
    from scipy import ndimage

    out = {}
    st = ndimage.generate_binary_structure(2, 1 if conn == 4 else 2)
    masks = [f > thr for f in frames_np]
    t0 = time.perf_counter()
    for i in range(reps):
        ndimage.label(masks[i % len(masks)], structure=st)
    out["scipy_label_ms"] = (time.perf_counter() - t0) / reps * 1e3
    try:
        import cv2

        m8 = [m.astype(np.uint8) for m in masks]
        t0 = time.perf_counter()
        for i in range(reps):
            cv2.connectedComponentsWithStats(m8[i % len(m8)], connectivity=conn, ltype=cv2.CV_32S)
        out["cv2_ccstats_ms"] = (time.perf_counter() - t0) / reps * 1e3
    except ImportError:
        out["cv2_ccstats_ms"] = None
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--frames", type=int, default=4000)
    ap.add_argument("--passes", type=int, default=5)
    ap.add_argument("--cap", type=int, default=256)
    ap.add_argument("--sizes", default="512x640,1024x1024")
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    import torch

    if not torch.cuda.is_available():
        sys.exit("label_bench: needs a CUDA device")
    try:  # host baselines on one core, as a user's one-frame-at-a-time loop runs
        import cv2

        cv2.setNumThreads(1)
    except ImportError:
        pass
    from librir_b200 import signal_processing as sp

    torch.cuda.set_device(0)
    info = card()
    lines = []
    for size in a.sizes.split(","):
        h, w = (int(v) for v in size.split("x"))
        for conn in (4, 8):
            for name in ("ir", "noise", "full"):
                frames, thr = workload(torch, name, a.frames, h, w, conn)
                med, ts, counts = time_gpu(torch, sp, frames, thr, conn, a.cap, a.passes)
                px = a.frames * h * w
                host = time_host(frames[:10].cpu().view(torch.int16).numpy().view(np.uint16), thr, conn)
                rec = dict(bench="label_batch", card=info, h=h, w=w, connectivity=conn, workload=name, frames=a.frames,
                           max_components=a.cap, median_s=med, passes_s=ts, frames_per_s=a.frames / med,
                           bytes_per_px_bound=BYTES_PER_PX, fraction_of_bound=BYTES_PER_PX * px / med / HBM_BYTES_PER_S,
                           mean_components=float(counts.double().mean().item()), **host)
                rec["host_frames_per_s_scipy"] = 1e3 / rec["scipy_label_ms"]
                print(json.dumps(rec), flush=True)
                lines.append(rec)
                del frames
                torch.cuda.empty_cache()
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            for rec in lines:
                f.write(json.dumps(rec) + "\n")


if __name__ == "__main__":
    main()
