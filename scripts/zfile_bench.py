#!/usr/bin/env python
"""scripts/zfile_bench.py -- write / read throughput of the zstd movie file (SURVEY.md 8f-3): the product's
thread-pooled container (rirb_z_write_images / rirb_z_read_images) next to the compiled reference's ZFile
(oracle/_ref, one frame per call on one thread -- what z_write_image / z_read_image do).  Host work; the GPU
only appears in the `device` rows, where the frames start / end in HBM.  Evidence for profiles/.

    python scripts/zfile_bench.py [--frames 400] [--coder host|gpu|gpu-lz|both|all] [--decoder host|gpu|auto|both] > zfile_bench.jsonl

--coder picks the entropy coder of the method 1/2/3 rows: host zstd at --clevel (the default), the device coder
(rirb_z_set_coder 1), the device coder with LZ matches (gpu-lz, rirb_z_set_coder 1 and rirb_z_set_lz 1), host and gpu (both), or all three.
With a device coder the first rows give its device time per frame (CUDA events around rirb_zstd_encode_batch and, with
gpu-lz, rirb_zstd_encode_batch_lz, alternated in one call on 600 frames of method-2 and method-3 planes, larger than L2),
next to the card's name and power limit.

--decoder sets the "zstd_decoder" switch around the read rows: host libzstd (0), the device decoder wherever a read ends
on the device (2), the library's default selection (auto, 1), or all three, run alternately --reps times in the same call
(each row then reports the best time and all of them).  With the
device decoder, rows give its device time per frame on 600 frames of 640x512 (output larger than L2) for three inputs:
device-coder method-3 planes, host zstd level-2 method-3 planes and host zstd level-2 method-1 frames.
"""
import argparse
import json
import os
import sys
import tempfile
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--frames", type=int, default=400)
    ap.add_argument("--clevel", type=int, default=2)
    ap.add_argument("--coder", choices=("host", "gpu", "gpu-lz", "both", "all"), default="host")
    ap.add_argument("--decoder", choices=("host", "gpu", "auto", "both"), default="auto")
    ap.add_argument("--reps", type=int, default=3)
    args = ap.parse_args()
    coders = {"both": ("host", "gpu"), "all": ("host", "gpu", "gpu-lz")}.get(args.coder, (args.coder,))
    decoders = ("host", "gpu", "auto") if args.decoder == "both" else (args.decoder,)
    switch = {"host": 0, "auto": 1, "gpu": 2}
    from librir_b200 import _lib, tools
    from oracle import container as oc  # checker / baseline only
    from tests.conftest import ir_movie

    n, h, w = args.frames, 512, 640
    mov = ir_movie(n, h, w)
    ts = np.arange(n, dtype=np.int64) * 20_000_000
    cores = os.cpu_count() or 1
    tmp = tempfile.mkdtemp(prefix="zfile_bench_")
    rows = []

    def rec(name, impl, threads, secs, extra=None):
        row = {"op": name, "impl": impl, "threads": threads, "frames": n, "frame": [w, h], "seconds": round(secs, 4),
               "frames_per_s": round(n / secs, 1), "MB_per_s": round(mov.nbytes / secs / 1e6, 1)}
        row.update(extra or {})
        rows.append(row)
        print(json.dumps(row), flush=True)

    def timed_reads(name, impl, threads, read, extra=None):
        """read(): one read of the whole file; alternates the decoders, args.reps times each."""
        times = {dec: [] for dec in decoders}
        for _ in range(args.reps):
            for dec in decoders:
                _lib.set_parameter("zstd_decoder", switch[dec])
                t0 = time.perf_counter()
                read()
                times[dec].append(time.perf_counter() - t0)
        _lib.set_parameter("zstd_decoder", 1)
        for dec in decoders:
            rec(name, impl, threads, min(times[dec]), dict(extra or {}, decoder=dec, all_seconds=[round(t, 4) for t in times[dec]]))

    if "gpu" in coders or "gpu-lz" in coders:
        coder_device_time(mov, ("gpu", "gpu-lz") if "gpu-lz" in coders else ("gpu",))
    if "host" not in decoders or len(decoders) > 1:
        decoder_device_time(mov)
    have_ref = oc.have_ref()
    if have_ref:
        p = os.path.join(tmp, "ref.bin")
        t0 = time.perf_counter()
        oc.ref_write_zfile(p, mov, ts, clevel=args.clevel)
        rec("write", "reference", 1, time.perf_counter() - t0, {"file_MB": round(os.path.getsize(p) / 1e6, 1)})
        t0 = time.perf_counter()
        frames, _ = oc.ref_read_zfile(p)
        rec("read", "reference", 1, time.perf_counter() - t0)
        assert np.array_equal(frames, mov)
    for threads in (1, 0):
        p = os.path.join(tmp, f"prod{threads}.bin")
        t0 = time.perf_counter()
        with tools.ZFileWriter(p, w, h, clevel=args.clevel, threads=threads) as wr:
            wr.add_images(mov, ts)
        rec("write", "product", threads or cores, time.perf_counter() - t0, {"file_MB": round(os.path.getsize(p) / 1e6, 1)})
        if have_ref:
            assert open(p, "rb").read() == open(os.path.join(tmp, "ref.bin"), "rb").read(), "files differ from the reference's"
        t0 = time.perf_counter()
        with tools.ZFileReader(p, threads=threads) as rd:
            frames = rd.read_images()
        rec("read", "product", threads or cores, time.perf_counter() - t0)
        assert np.array_equal(frames, mov)
    try:
        import torch

        if torch.cuda.is_available():
            d = torch.from_numpy(mov.view(np.int16)).cuda().view(torch.uint16)
            p = os.path.join(tmp, "dev.bin")
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            with tools.ZFileWriter(p, w, h, clevel=args.clevel, threads=0) as wr:
                wr.add_images(d, ts)
            rec("write", "product, frames in HBM", cores, time.perf_counter() - t0)
            out = torch.empty_like(d)

            def read_hbm(p=p):
                with tools.ZFileReader(p, threads=0) as rd:
                    rd.read_images(0, n, out=out)
                torch.cuda.synchronize()
                assert torch.equal(out.view(torch.int16), d.view(torch.int16))

            timed_reads("read", "product, frames to HBM", cores, read_hbm)
            # methods 2 / 3 (video_io.h:298-305): the GPU pre-coder in front of zstd; host frames and frames in HBM
            for method, coder in [(m, c) for c in coders for m in (1, 2, 3)]:
                for where, src in (("host", mov), ("HBM", d)):
                    p = os.path.join(tmp, f"m{method}{where}.bin")
                    torch.cuda.synchronize()
                    t0 = time.perf_counter()
                    with tools.ZFileWriter(p, w, h, method=method, clevel=args.clevel, threads=0, gop=50, coder=coder) as wr:
                        wr.add_images(src, ts)
                    rec("write", f"product, method {method}, frames in {where}", cores, time.perf_counter() - t0,
                        {"file_MB": round(os.path.getsize(p) / 1e6, 1), "coder": coder,
                         "ratio": round(mov.nbytes / (os.path.getsize(p) - 256), 3)})
                    def read(p=p, where=where):
                        with tools.ZFileReader(p, threads=0) as rd:
                            if where == "host":
                                back = rd.read_images()
                            else:
                                rd.read_images(0, n, out=out)
                        torch.cuda.synchronize()
                        if where == "host":
                            assert np.array_equal(back, mov)
                        else:
                            assert torch.equal(out.view(torch.int16), d.view(torch.int16))

                    timed_reads("read", f"product, method {method}, frames to {where}", cores, read, {"coder": coder})
    except ImportError:
        pass
    for f in os.listdir(tmp):
        os.remove(os.path.join(tmp, f))
    os.rmdir(tmp)


def coder_device_time(mov, coders, frames=600, reps=5):
    """Device time per frame of the device coders (gpu: rirb_zstd_encode_batch, gpu-lz: rirb_zstd_encode_batch_lz) on the
    method-2 and method-3 planes of `frames` frames (> L2): CUDA events, the coders alternated, best of reps each."""
    import torch

    from librir_b200 import _lib
    from tests import zcoder_cases as K

    n, h, w = len(mov), mov.shape[1], mov.shape[2]
    stride = 9 + 3 * 2 * ((h * w + 131071) // 131072) + 2 * h * w
    dst = torch.empty((frames, stride), dtype=torch.uint8, device="cuda")
    sizes = torch.empty(frames, dtype=torch.int64, device="cuda")
    _lib.use_torch_stream()
    lib = _lib.load()
    entry = {"gpu": lib.rirb_zstd_encode_batch, "gpu-lz": lib.rirb_zstd_encode_batch_lz}
    q = card()
    for method in (2, 3):
        planes = torch.from_numpy(K.planes(mov, method)).cuda()
        src = planes[torch.arange(frames) % n].contiguous()  # [frames, 2*h*w]

        def run(coder):
            assert entry[coder](src.data_ptr(), frames, 2 * h * w, h * w, dst.data_ptr(), stride, sizes.data_ptr()) == 0, _lib.last_error()

        ratio = {}
        for coder in coders:
            run(coder)
            torch.cuda.synchronize()
            ratio[coder] = src.numel() / float(sizes.sum())
        best = {}
        for _ in range(reps):
            for coder in coders:
                a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                a.record()
                run(coder)
                b.record()
                b.synchronize()
                best[coder] = min(best.get(coder, 1e30), a.elapsed_time(b))
        for coder in coders:
            row = {"op": f"device coder, method-{method} planes", "coder": coder, "gpu": torch.cuda.get_device_name(),
                   "nvidia_smi": q, "frames": frames, "frame": [w, h], "input_MB": round(src.numel() / 1e6, 1),
                   "ms_best_of_%d" % reps: round(best[coder], 3), "us_per_frame": round(1000 * best[coder] / frames, 2),
                   "input_GB_per_s": round(src.numel() / best[coder] / 1e6, 1), "ratio": round(ratio[coder], 3)}
            print(json.dumps(row), flush=True)
        del planes, src
        torch.cuda.empty_cache()


def card():
    import subprocess

    try:
        return subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                              capture_output=True, text=True, timeout=30).stdout.strip().splitlines()[0]
    except (OSError, IndexError, subprocess.SubprocessError):
        return "unknown"


def decoder_device_time(mov, frames=600, reps=5):
    """Device time of rirb_zstd_decode_batch per frame over `frames` records of 640x512 (output > L2), CUDA events, best of
    reps after a warm-up: device-coder method-3 planes, host zstd level-2 method-3 planes, host zstd level-2 method-1."""
    import torch

    from librir_b200 import _lib
    from librir_b200 import entropy as E
    from tests import zcoder_cases as K

    n, h, w = len(mov), mov.shape[1], mov.shape[2]
    fbytes = 2 * h * w
    lib = _lib.load()
    _lib.use_torch_stream()
    planes = K.planes(mov, 3)
    dplanes = torch.from_numpy(planes).cuda()
    stride = 9 + 3 * 2 * ((h * w + 131071) // 131072) + fbytes
    enc = torch.empty((n, stride), dtype=torch.uint8, device="cuda")
    sizes = torch.empty(n, dtype=torch.int64, device="cuda")
    assert lib.rirb_zstd_encode_batch(dplanes.data_ptr(), n, fbytes, h * w, enc.data_ptr(), stride, sizes.data_ptr()) == 0
    e, sz = enc.cpu().numpy(), sizes.cpu().numpy()
    inputs = {
        "device-coder method-3 planes": [e[i, :sz[i]].tobytes() for i in range(n)],
        "host zstd level-2 method-3 planes": [E.zstd_compress(planes[i], 2) for i in range(n)],
        "host zstd level-2 method-1 frames": [E.zstd_compress(mov[i].reshape(-1).view(np.uint8), 2) for i in range(n)],
    }
    q = card()
    for name, recs in inputs.items():
        pick = [recs[i % n] for i in range(frames)]
        offs = np.cumsum([0] + [len(r) for r in pick[:-1]]).astype(np.int64)
        src = torch.from_numpy(np.frombuffer(b"".join(pick), np.uint8).copy()).cuda()
        off = torch.from_numpy(offs).cuda()
        size = torch.from_numpy(np.array([len(r) for r in pick], np.uint32).view(np.int32)).cuda()
        dst = torch.empty((frames, fbytes), dtype=torch.uint8, device="cuda")
        status = torch.empty(frames, dtype=torch.int64, device="cuda")

        def run():
            assert lib.rirb_zstd_decode_batch(src.data_ptr(), off.data_ptr(), size.data_ptr(), frames, dst.data_ptr(), fbytes,
                                              fbytes, status.data_ptr()) == 0, _lib.last_error()

        run()
        torch.cuda.synchronize()
        assert bool((status == fbytes).all()), name
        best = None
        for _ in range(reps):
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record()
            run()
            b.record()
            b.synchronize()
            best = a.elapsed_time(b) if best is None else min(best, a.elapsed_time(b))
        row = {"op": "device decoder, " + name, "gpu": torch.cuda.get_device_name(), "nvidia_smi": q, "frames": frames,
               "frame": [w, h], "input_MB": round(src.numel() / 1e6, 1), "output_MB": round(frames * fbytes / 1e6, 1),
               "ms_best_of_%d" % reps: round(best, 3), "us_per_frame": round(1000 * best / frames, 2),
               "output_GB_per_s": round(frames * fbytes / best / 1e6, 1)}
        print(json.dumps(row), flush=True)


if __name__ == "__main__":
    main()
