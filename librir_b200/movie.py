"""Device-resident movie shards: the per-frame pipeline in batched launches, frame-range
sharding across ranks, and the all-reduce of per-movie statistics.

One process per GPU (``torch.distributed``, NCCL over NVLink).  Frames are independent on this
path (SURVEY.md 8e), so a movie is cut into contiguous frame ranges, one per rank, with every
range starting on a key frame of the writer (a multiple of the GOP) so that the temporal-delta
pre-coder never needs a frame owned by another rank.  The only exchange step is the reduction
of min / max / histogram (``ncclMin`` / ``ncclMax`` / ``ncclSum``) and, optionally, the broadcast
of frame 0 to the ranks that need it for bad-pixel detection.

PyTorch is used for device memory, streams and the process group only; every pixel is touched
by the kernels of ``libsignal_processing_b200.so``.
"""
from __future__ import annotations

import ctypes as ct
from dataclasses import dataclass

import numpy as np

from . import _lib
from . import signal_processing as sp
from . import video_io as vio


# ----------------------------------------------------------------------------------------
# sharding
# ----------------------------------------------------------------------------------------
@dataclass(frozen=True)
class FrameShard:
    rank: int
    world: int
    start: int  # first frame (inclusive), a multiple of the GOP
    stop: int   # last frame (exclusive)

    @property
    def nframes(self) -> int:
        return self.stop - self.start


def shard_frames(nframes: int, world: int, rank: int, gop: int = vio.DEFAULT_GOP) -> FrameShard:
    """Contiguous, GOP-aligned frame range of ``rank``: GOPs are dealt out as evenly as possible
    (the first ``ngop % world`` ranks get one more), so shard starts are key frames."""
    if world < 1 or not (0 <= rank < world) or nframes < 0 or gop < 1:
        raise ValueError("shard_frames: bad arguments")
    ngop = -(-nframes // gop)
    base, extra = divmod(ngop, world)
    g0 = rank * base + min(rank, extra)
    g1 = g0 + base + (1 if rank < extra else 0)
    return FrameShard(rank, world, min(nframes, g0 * gop), min(nframes, g1 * gop))


# ----------------------------------------------------------------------------------------
# statistics
# ----------------------------------------------------------------------------------------
class MovieStats:
    """min / max / 65,536-bin histogram of a movie shard, kept on the device and reduced across
    ranks in place.  ``quantile`` follows ``find_median_pixel`` (Filters.cpp:56-72) and
    ``background`` follows ``get_background`` (h264.cpp:1955-1991) on the reduced histogram.

    Layout: one int64 buffer ``[hist[65536] | count]`` so that the reduction is ONE ``SUM``
    all-reduce, and ``minmax`` = ``[min, max]`` reduced as ONE ``MIN`` all-reduce of ``[min, -max]``;
    nothing in ``update`` / ``all_reduce`` waits for the device."""

    def __init__(self, device):
        import torch

        self.device = torch.device(device)
        self.minmax = torch.empty(2, dtype=torch.int32, device=self.device)   # viewed as uint32 by the kernel
        self._sums = torch.zeros(65537, dtype=torch.int64, device=self.device)  # hist (viewed as uint64) + pixel count
        self.hist = self._sums[:65536]
        self._fresh = True

    @property
    def count(self) -> int:
        return int(self._sums[65536].item())

    @count.setter
    def count(self, v: int) -> None:
        self._sums[65536] = int(v)

    def reset(self) -> None:
        """Start a new movie: the next ``update`` initialises the statistics instead of folding into them."""
        self._fresh = True

    def update(self, frames) -> None:
        """Fold a chunk of uint16 frames (torch CUDA tensor) into the statistics."""
        lib = _lib.load()
        sp._prepare_device_call(frames)
        frames = sp._operand(frames, "movie_stats", "frames", dtype=np.uint16, copy=True)
        n = frames.numel()
        if self._fresh:
            self._sums[65536] = 0
        r = lib.rirb_movie_stats(sp._ptr(frames), n, ct.c_void_p(self.minmax.data_ptr()), ct.c_void_p(self.hist.data_ptr()),
                                 0 if self._fresh else 1)
        _lib.check(r, "movie_stats")
        self._fresh = False
        self._sums[65536] += n

    def all_reduce(self, group=None) -> None:
        """The path's only collective: min (MIN), max (MAX), histogram and count (SUM) -- two NCCL calls."""
        import torch
        import torch.distributed as dist

        if not (dist.is_available() and dist.is_initialized()) or dist.get_world_size(group) == 1:
            return
        if self._fresh:  # an empty shard contributes the identities
            self.minmax[0], self.minmax[1] = 65535, 0
            self._sums.zero_()
            self._fresh = False
        mm = torch.stack((self.minmax[0], -self.minmax[1]))  # max(x) = -min(-x): one MIN reduction for both
        dist.all_reduce(mm, op=dist.ReduceOp.MIN, group=group)
        dist.all_reduce(self._sums, op=dist.ReduceOp.SUM, group=group)
        self.minmax[0] = mm[0]
        self.minmax[1] = -mm[1]

    # host-side views -------------------------------------------------------------------
    def min(self) -> int:
        return int(self.minmax[0].item())

    def max(self) -> int:
        return int(self.minmax[1].item())

    def histogram(self) -> np.ndarray:
        return self.hist.cpu().numpy().astype(np.uint64)

    def quantile(self, percent: float = 0.5) -> int:
        lib = _lib.load()
        _lib.use_torch_stream()
        r = lib.rirb_hist_quantile(ct.c_void_p(self.hist.data_ptr()), self.count, float(percent))
        return _lib.check(r, "hist_quantile")

    def background(self) -> int:
        h4 = self.hist.view(16384, 4).sum(dim=1)
        return (int(h4.argmax().item()) << 2) + 1


# ----------------------------------------------------------------------------------------
# the per-frame pipeline on a shard
# ----------------------------------------------------------------------------------------
@dataclass
class PipelineConfig:
    width: int = 640
    height: int = 512
    sigma: float = 1.0                 # registration default is 0.5 (masked_registration_ecc.py:44)
    strategy: str = "nearest"          # border mode of the registration translate
    gop: int = vio.DEFAULT_GOP
    delta: bool = True                 # temporal delta in the pre-coder
    chunk_frames: int = 4096           # frames per batched launch (buffers are reused per chunk)
    fuse_stats: bool = True            # statistics ride along in the pre-coder's pass instead of their own


class FramePipeline:
    """bad-pixel correct -> Gaussian (u16 -> f32, the registration's input) -> translate
    (registration's resampling) -> lossless pre-coder, on chunks of device-resident frames.

    Buffers for one chunk are allocated once and reused: at 640x512x4096 that is 2.7 GB in,
    2.7 GB corrected, 5.4 GB smoothed, 2.7 GB registered, 2.7 GB of byte planes."""

    def __init__(self, cfg: PipelineConfig, device="cuda"):
        import torch

        self.cfg = cfg
        self.device = torch.device(device)
        n, h, w = cfg.chunk_frames, cfg.height, cfg.width
        self.corrected = torch.empty((n, h, w), dtype=torch.uint16, device=self.device)
        self.smoothed = torch.empty((n, h, w), dtype=torch.float32, device=self.device)
        self.registered = torch.empty((n, h, w), dtype=torch.uint16, device=self.device)
        self.lo = torch.empty((n, h, w), dtype=torch.uint8, device=self.device)
        self.hi = torch.empty((n, h, w), dtype=torch.uint8, device=self.device)
        self.bad_pixels = None
        self.stats = MovieStats(self.device)

    def set_first_frame(self, first_frame) -> None:
        """Bad-pixel detection on the movie's frame 0 (every rank is handed the same frame)."""
        self.bad_pixels = sp.BadPixels(first_frame)

    @property
    def STAGES(self):
        if self.cfg.fuse_stats:
            return ("bp_correct", "gaussian_u16_f32", "translate_u16", "precode_delta_split_stats")
        return ("bp_correct", "gaussian_u16_f32", "translate_u16", "precode_delta_split", "stats_minmax_hist")

    def process_chunk(self, frames, dx, dy, first_frame: int, with_stats: bool = True, events=None):
        """Run the stages on ``frames[n, h, w]`` (torch CUDA uint16, n <= chunk_frames).
        ``dx``/``dy``: per-frame float32 CUDA tensors or scalars; ``first_frame``: index of
        frames[0] in the movie (a multiple of the GOP when delta is on).  ``events``: optional list
        of ``len(STAGES)+1`` torch CUDA events recorded around the stages (per-kernel timing).
        Returns views of the reused buffers: ``(corrected, smoothed, registered, lo, hi)``."""
        import torch

        if self.bad_pixels is None:
            raise RuntimeError("FramePipeline: call set_first_frame() first")
        n = frames.shape[0]
        c, s, r = self.corrected[:n], self.smoothed[:n], self.registered[:n]
        lo, hi = self.lo[:n], self.hi[:n]
        mark = (lambda i: events[i].record(torch.cuda.current_stream())) if events is not None else (lambda i: None)
        mark(0)
        self.bad_pixels.correct_batch(frames, out=c)
        mark(1)
        sp.gaussian_filter_batch(c, self.cfg.sigma, out=s)
        mark(2)
        sp.translate_batch(c, dx, dy, self.cfg.strategy, background=0, out=r)
        mark(3)
        if self.cfg.fuse_stats:
            vio.precode_movie(r, self.cfg.gop, self.cfg.delta, first_frame, out=(lo, hi), stats=self.stats if with_stats else None)
            mark(4)
        else:
            vio.precode_movie(r, self.cfg.gop, self.cfg.delta, first_frame, out=(lo, hi))
            mark(4)
            if with_stats:
                self.stats.update(r)
            mark(5)
        return c, s, r, lo, hi

    def process_host(self, frames_host, dx_host, dy_host, first_frame: int, lo_host, hi_host, sub_frames: int = 256,
                     slots: int = 3):
        """End-to-end call on HOST buffers (pinned torch CPU tensors): the chunk is cut into
        sub-chunks that rotate over `slots` streams, so that the upload of one, the kernels of
        another and the download of a third overlap (PCIe is full duplex).  ``lo_host``/``hi_host``
        receive the pre-coded byte planes -- what the host codec / zstd stage consumes.  Returns
        after everything has landed in the host buffers."""
        import torch

        if self.bad_pixels is None:
            raise RuntimeError("FramePipeline: call set_first_frame() first")
        n = frames_host.shape[0]
        gop = self.cfg.gop
        sub = max(gop, sub_frames // gop * gop) if self.cfg.delta else sub_frames  # sub-chunks start on key frames
        ns = len(self._e2e) if hasattr(self, "_e2e") else slots
        if ns * sub > self.cfg.chunk_frames:  # each slot's window of the chunk buffers must hold a whole sub-chunk
            raise RuntimeError(f"process_host: {ns} slots of {sub} frames do not fit the {self.cfg.chunk_frames}-frame chunk buffers; "
                               "lower sub_frames or slots, or raise chunk_frames")
        if not hasattr(self, "_e2e"):
            h, w = self.cfg.height, self.cfg.width
            self._e2e = [dict(stream=torch.cuda.Stream(device=self.device),
                              inp=torch.empty((sub, h, w), dtype=torch.uint16, device=self.device),
                              dx=torch.empty(sub, dtype=torch.float32, device=self.device),
                              dy=torch.empty(sub, dtype=torch.float32, device=self.device)) for _ in range(slots)]
            self._e2e_sub = sub
        if self._e2e_sub != sub:
            raise RuntimeError("process_host: sub_frames changed between calls")
        main = torch.cuda.current_stream()
        k = 0
        for a in range(0, n, sub):
            b = min(n, a + sub)
            m = b - a
            ns = len(self._e2e)
            slot = self._e2e[k % ns]
            st = slot["stream"]
            st.wait_stream(main)
            with torch.cuda.stream(st):
                slot["inp"][:m].copy_(frames_host[a:b], non_blocking=True)
                slot["dx"][:m].copy_(dx_host[a:b], non_blocking=True)
                slot["dy"][:m].copy_(dy_host[a:b], non_blocking=True)
                # the chunk buffers are shared: give each stream its own window of them
                off = (k % ns) * sub
                c = self.corrected[off:off + m]
                s = self.smoothed[off:off + m]
                r = self.registered[off:off + m]
                lo, hi = self.lo[off:off + m], self.hi[off:off + m]
                self.bad_pixels.correct_batch(slot["inp"][:m], out=c)
                sp.gaussian_filter_batch(c, self.cfg.sigma, out=s)
                sp.translate_batch(c, slot["dx"][:m], slot["dy"][:m], self.cfg.strategy, background=0, out=r)
                vio.precode_movie(r, gop, self.cfg.delta, first_frame + a, out=(lo, hi))
                lo_host[a:b].copy_(lo, non_blocking=True)
                hi_host[a:b].copy_(hi, non_blocking=True)
            k += 1
        for slot in self._e2e:
            main.wait_stream(slot["stream"])
        main.synchronize()


def process_movie_host(bad_pixels, frames, dx, dy, sigma=1.0, strategy="nearest", background=0, gop=vio.DEFAULT_GOP, delta=True,
                       first_frame=0, lo=None, hi=None, smoothed=None):
    """The whole per-frame path on HOST buffers through ONE C-ABI call (``rirb_process_movie_host``):
    ``frames`` uint16 ``[n, h, w]`` (numpy array or CPU torch tensor, ideally pinned) -> ``(lo, hi)`` uint8
    byte planes of the corrected, registered, pre-coded frames.  ``smoothed``: optional float32 ``[n, h, w]``
    host buffer for the Gaussian output (otherwise it stays on the device).  ``lo`` / ``hi``: uint8 of ``frames``' shape.
    A strided numpy ``frames`` is copied first; strided outputs are refused."""
    lib = _lib.load()
    what = "process_movie_host"

    def host_ptr(x):
        if sp._is_torch(x) and x.is_cuda:
            raise RuntimeError("process_movie_host: contiguous host buffers expected")
        return sp._ptr(x)

    if len(frames.shape) != 3:
        raise RuntimeError("process_movie_host: wrong input dimension")
    frames = sp._operand(frames, what, "frames", dtype=np.uint16, copy=True)
    n, h, w = frames.shape
    if lo is None:
        lo = np.empty((n, h, w), np.uint8)
    if hi is None:
        hi = np.empty((n, h, w), np.uint8)
    lo = sp._operand(lo, what, "lo", frames.shape, np.uint8)
    hi = sp._operand(hi, what, "hi", frames.shape, np.uint8)
    if smoothed is not None:
        smoothed = sp._operand(smoothed, what, "smoothed", frames.shape, np.float32)
    if not sp._is_torch(dx):
        dx = np.ascontiguousarray(np.broadcast_to(np.asarray(dx, dtype=np.float32), (n,)))
        dy = np.ascontiguousarray(np.broadcast_to(np.asarray(dy, dtype=np.float32), (n,)))
    dx = sp._operand(dx, what, "dx", (n,), np.float32, copy=True)
    dy = sp._operand(dy, what, "dy", (n,), np.float32, copy=True)
    r = lib.rirb_process_movie_host(bad_pixels.handle, host_ptr(frames), n, w, h, float(sigma), host_ptr(dx), host_ptr(dy),
                                    sp.toCharP(strategy), int(background), int(gop), int(bool(delta)), int(first_frame),
                                    host_ptr(lo), host_ptr(hi), host_ptr(smoothed) if smoothed is not None else None)
    _lib.check(r, "process_movie_host")
    return lo, hi


def broadcast_first_frame(frame, src: int = 0, group=None):
    """Hand frame 0 (owned by the rank holding the movie's first shard) to every rank."""
    import torch
    import torch.distributed as dist

    if dist.is_available() and dist.is_initialized() and dist.get_world_size(group) > 1:
        dist.broadcast(frame.view(torch.uint8), src=src, group=group)  # uint16 has no NCCL datatype: ship the bytes
    return frame


__all__ = ["FrameShard", "shard_frames", "MovieStats", "PipelineConfig", "FramePipeline", "process_movie_host",
           "broadcast_first_frame"]
