"""State carried across frames, launches and calls, over movies as long as the ones the design quotes numbers for
(tests/long_movie_cases.py).  Everything else pins the stateless kernels; here a fault that shows only after the second
run, the 41st spread, the 65th ring write, a cache hit or a chunk boundary must fail.

* Lossy pre-conditioner (csrc/lossy.cu): 1,000-3,000-frame movies at small sizes and a 300-frame 640 x 512 one, cut into
  calls of 1 / 63 / 64 / 65 / 127 / 128 / 129 / random frames, the driver switched between calls, host and device frames
  mixed, two handles fed alternately -- every output frame, both bounds of every frame and MIN_T bit for bit against the
  restatement (oracle.Port.lossy_*).
* ECC tracker (rirb_ecc_track): 420-frame movies with seven flares (14 replacements of the reference image) and
  failing frames inside queued runs -- the same bits, iteration counts, threshold and median from every way of feeding
  it; each driver against the restated class (oracle/ecc.py) up to the first replacement, and the same replacements.
* FramePipeline: multi-chunk movies through process_chunk with a short last chunk, MovieStats folded over the chunks,
  reset and a second movie; process_host with all three slots rotating.

``RIRB_FUZZ_SEED`` / ``RIRB_FUZZ_SCALE`` as in test_gpu_fuzz.py."""
import ctypes as ct
import os

import numpy as np
import pytest

from oracle import ecc as oe
from oracle import oracle as O
from tests import gauss_exact as G
from tests import long_movie_cases as LM
from tests import vio_cases as C
from tests.conftest import ir_movie

pytestmark = pytest.mark.gpu

torch = pytest.importorskip("torch")
if not torch.cuda.is_available():  # pragma: no cover
    pytest.skip("needs a CUDA device", allow_module_level=True)

from librir_b200 import _lib, movie, registration as rg, video_io as vio  # noqa: E402
from tests.test_gpu_lossy_extremes import assert_same, fuzz_movie, to_dev, to_host  # noqa: E402

SEED = int(os.environ.get("RIRB_FUZZ_SEED", "0"))
SCALE = max(1, int(os.environ.get("RIRB_FUZZ_SCALE", "1")))


@pytest.fixture
def switches_restored():
    yield
    for k in ("lossy_run", "ecc_queue", "ecc_fused"):
        _lib.set_parameter(k, 1)


# ---- lossy pre-conditioner ---------------------------------------------------------------------------------------------
def port_lossy(port, mov, stop, cfg, door):
    """The restatement frame by frame: outputs, (BackgroundError, ForegroundError) per frame, MIN_T."""
    t = len(mov)
    st = port.lossy_open(mov.shape[2], mov.shape[1], stop, variant=1 if door == "add_loss" else 0, **C.lossy_params(cfg))
    outs, errs = np.empty_like(mov), np.empty((t, 2), np.int64)
    for i in range(t):
        o, e = port.lossy_add(st, mov[i])
        if door == "add_loss":
            o[stop:] = mov[i][stop:]  # addLoss copies back the lossy rows only
        outs[i], errs[i] = o, e
    m = port.lossy_get_min(st)
    port.lossy_close(st)
    return outs, errs, m


def lossy_min(pre):
    v = ct.c_int(-1)
    _lib.check(_lib.load().rirb_lossy_get_min(pre.handle, ct.addressof(v)), "lossy_get_min")
    return v.value


class GpuLossy:
    """One LossyPreconditioner fed a movie call by call."""

    def __init__(self, mov, stop, cfg, door):
        t, h, w = mov.shape
        self.mov, self.pre, self.a = mov, vio.LossyPreconditioner(w, h, stop, variant=door, **cfg), 0
        self.outs, self.errs, self.mins = [], [], []

    def feed(self, c, run, device):
        _lib.set_parameter("lossy_run", run)
        part = np.ascontiguousarray(self.mov[self.a:self.a + c])
        o, e = self.pre.add_images(to_dev(part) if device else part)
        self.outs.append(to_host(o))
        self.errs.append(e)
        self.mins.append(lossy_min(self.pre))
        self.a += c

    def check(self, want, what):
        want_o, want_e, want_min = want
        assert self.a == len(self.mov)
        assert_same(np.concatenate(self.outs), np.concatenate(self.errs), want_o, want_e, what)
        assert self.mins == [want_min] * len(self.mins), f"{what}: MIN_T {sorted(set(self.mins))} != {want_min}"


def run_schedule(mov, stop, cfg, door, sched):
    g = GpuLossy(mov, stop, cfg, door)
    for c, run, dev in sched:
        g.feed(c, run, dev)
    return g


# (id, frames, h, w, stop_lossy_height, saver parameters, door, lossy_movie arguments)
WIDE = dict(stdFactor=0.5, lowValueError=3000, highValueError=1500)
LOSSY_CASES = [
    ("ra0", 1500, 40, 48, 40, dict(runningAverage=0), "add_image_lossy", dict(blink=(46341,), bad_frames=LM.nan_frames(1500))),
    ("ra1_meta_rows", 2000, 33, 64, 30, dict(runningAverage=1), "add_image_lossy",
     dict(meta_rows=3, blink=(65535,), bad_frames=LM.nan_frames(2000, 8002))),
    ("ra39_subtract_min", 2500, 40, 48, 40, dict(runningAverage=39, subtractMin=1), "add_image_lossy",
     dict(blink=(46341, 65535), bad_frames=LM.nan_frames(2500))),
    ("ra40_bad_pixels_meta_rows", 1200, 64, 136, 61, dict(runningAverage=40, removeBadPixels=1), "add_image_lossy",
     dict(meta_rows=3, blink=(65535,), bad_frames=LM.nan_frames(1200, 8001))),
    ("ra41_add_loss", 3000, 33, 64, 33, dict(runningAverage=41), "add_loss", dict(blink=(46341,), bad_frames=LM.nan_frames(3000))),
    ("ra63_bp_subtract_min_add_loss", 1500, 40, 48, 37, dict(runningAverage=63, removeBadPixels=1, subtractMin=1), "add_loss",
     dict(meta_rows=3, bad_frames=LM.nan_frames(1500, 8003))),
    ("ra64_wide", 2000, 33, 64, 33, dict(WIDE, runningAverage=64), "add_image_lossy",
     dict(blink=(65535,), bad_frames=LM.nan_frames(2000))),
    ("ra100_clamped_to_64", 1000, 40, 48, 40, dict(runningAverage=100, subtractMin=1), "add_image_lossy",
     dict(bad_frames=LM.nan_frames(1000))),
    ("640x512", 300, 512, 640, 509, dict(runningAverage=32, removeBadPixels=1), "add_image_lossy",
     dict(meta_rows=3, blink=(46341,), bad_frames={50: 65535, 130: 8002, 251: 65535})),
]


@pytest.mark.parametrize("case", LOSSY_CASES, ids=[c[0] for c in LOSSY_CASES])
def test_lossy_long_movies(port, case, switches_restored):
    name, t, h, w, stop, cfg, door, kw = case
    mov = LM.lossy_movie(t, h, w, seed=len(name) * 1000 + t, **kw)
    want = port_lossy(port, mov, stop, cfg, door)
    assert len(np.unique(want[1][:, 0])) > 3  # the bounds move
    rng = np.random.default_rng(SEED * 7919 + t + h)
    for kind in ("one", "edges", "random"):
        sched = LM.schedule(t, kind, rng)
        run_schedule(mov, stop, cfg, door, sched).check(want, f"{name} {kind} {[s[0] for s in sched][:12]}")
    # one call per frame through the per-frame driver, then the rest as single launches of 64
    sched = [(1, 0, True)] * 70 + [(LM.LOSSY_RUN, 1, False)] * ((t - 70) // LM.LOSSY_RUN)
    sched.append((t - sum(s[0] for s in sched), 1, True))
    run_schedule(mov, stop, cfg, door, [s for s in sched if s[0] > 0]).check(want, f"{name} single frames then launches")


def test_lossy_two_handles_interleaved(port, switches_restored):
    """Two handles with different sizes and configurations fed alternately from one thread: they share its stream and
    staging buffers, nothing else."""
    rng = np.random.default_rng(99 + SEED)
    specs = [(LM.lossy_movie(1400, 40, 48, seed=1, blink=(65535,), bad_frames=LM.nan_frames(1400)), 40,
              dict(runningAverage=39, subtractMin=1), "add_image_lossy"),
             (LM.lossy_movie(1100, 33, 64, seed=2, meta_rows=3, bad_frames=LM.nan_frames(1100, 8002)), 30,
              dict(runningAverage=64, removeBadPixels=1), "add_loss")]
    wants = [port_lossy(port, *s) for s in specs]
    gpus = [GpuLossy(*s) for s in specs]
    k = 0
    while any(g.a < len(g.mov) for g in gpus):
        g = gpus[k % 2]
        k += 1
        if g.a < len(g.mov):
            c = int(rng.choice([1, 64, 65, int(rng.integers(1, 140))]))
            g.feed(min(c, len(g.mov) - g.a), int(rng.integers(0, 2)), bool(rng.integers(0, 2)))
    for i, (g, want) in enumerate(zip(gpus, wants)):
        g.check(want, f"handle {i} of two")


def test_fuzz_lossy_long_movies(port, switches_restored):
    rng = np.random.default_rng(4242 + SEED)
    for case in range(2 * SCALE):
        w = int(rng.choice([16, 33, 40, 64, 136]))
        h = int(rng.integers(8, 48))
        t = int(rng.integers(1000, 3001))
        stop = int(rng.choice([h, h - 3, int(rng.integers(0, h + 1))]))
        cfg = dict(runningAverage=int(rng.choice([0, 1, 39, 40, 41, 63, 64])), subtractMin=int(rng.integers(0, 2)),
                   removeBadPixels=int(rng.integers(0, 2)) if stop >= 3 else 0)
        if rng.integers(0, 2):
            cfg.update(WIDE)
        door = ("add_image_lossy", "add_loss")[int(rng.integers(0, 2))]
        if rng.integers(0, 2):
            mov = fuzz_movie(rng, t, h, w)
        else:
            mov = LM.lossy_movie(t, h, w, seed=int(rng.integers(0, 1 << 20)), meta_rows=h - stop if h - stop <= 3 else 0,
                                 blink=tuple(rng.choice([46341, 65535], int(rng.integers(0, 3)))),
                                 bad_frames=LM.nan_frames(t, int(rng.choice([65535, 8000 + int(rng.integers(0, 4))]))))
        want = port_lossy(port, mov, stop, cfg, door)
        sched = LM.schedule(t, "random", rng)
        run_schedule(mov, stop, cfg, door, sched).check(want, f"case {case}: {t}x{h}x{w} stop {stop} {door} {cfg}")


# ---- ECC tracker ---------------------------------------------------------------------------------------------------------
ECC_FRAMES = 420
FAIL_AT = (100, 262)  # failing frames inserted here: inside queued runs, after several replacements


@pytest.fixture(scope="module")
def ecc_movies():
    mov, _sx, _sy = LM.ecc_long_movie(ECC_FRAMES)
    return dict(clean=mov, failures=LM.with_failures(mov, FAIL_AT))


@pytest.fixture(scope="module")
def restated_run(ecc_movies):
    """The restated class (oracle/ecc.py) over the clean movie."""
    reg = oe.MaskedRegistratorECC(O.Port())
    mov = ecc_movies["clean"]
    reg.start(mov[0])
    for t in range(1, len(mov)):
        reg.compute(mov[t])
    return np.array([reg.x, reg.y, reg.confidences], dtype=np.float64), list(reg.iterations), reg.conf_thresh


def tracked(reg):
    return dict(xyc=np.array([reg.x, reg.y, reg.confidences], dtype=np.float64), iterations=list(reg.iterations),
                conf_thresh=reg.conf_thresh, median=reg.median)


def assert_same_track(a, b, what):
    bad = np.nonzero((a["xyc"] != b["xyc"]).any(axis=0))[0] if a["xyc"].shape == b["xyc"].shape else [-1]
    assert len(bad) == 0, f"{what}: frames {list(bad[:8])} differ"
    assert a["iterations"] == b["iterations"], f"{what}: iteration counts differ"
    assert a["conf_thresh"] == b["conf_thresh"] and a["median"] == b["median"], what


def splits(n, cuts):
    a, out = 0, []
    for c in list(cuts) + [n]:
        if c > a:
            out.append((a, c))
            a = c
    return out


def feed_calls(frames, cuts, kw=None, max_try=0):
    reg = rg.MaskedRegistratorECC(**(kw or {}))
    for a, b in splits(len(frames), cuts):
        reg.compute_movie(frames[a:b], max_try=max_try)
    return tracked(reg)


def feed_frames(frames, kw=None, step=None):
    reg = rg.MaskedRegistratorECC(**(kw or {}))
    reg.start(frames[0])
    for t in range(1, len(frames)):
        step(frames[t], reg)
    return tracked(reg)


def ecc_modes(mov, kw, rng, frame_step, max_try):
    """(name, run) for every way of feeding the tracker one movie."""
    d = to_dev(mov)
    r = int(rng.integers(23, 60))
    cuts = np.cumsum(rng.integers(1, 3 * LM.ECC_RUN, len(mov) // 8))
    out = [("whole, device float32", lambda: feed_calls(torch.from_numpy(mov.astype(np.float32)).cuda(), [], kw, max_try)),
           ("whole, host numpy", lambda: feed_calls(mov, [], kw, max_try))]
    for k in (15, 16, 17, 20, 21, 22, r):
        out.append((f"split at {k}", lambda k=k: feed_calls(d, [k], kw, max_try)))
    out.append(("random cuts", lambda: feed_calls(d, cuts[cuts < len(mov)], kw, max_try)))
    out.append(("frame by frame, device", lambda: feed_frames(d, kw, frame_step)))
    out.append(("frame by frame, host", lambda: feed_frames(mov, kw, frame_step)))
    return out


def check_every_mode(mov, kw, frame_step, max_try, what):
    """Every mode against the whole movie in one call of device u16 frames; frame_step (compute, or
    manage_computation_and_tries) and max_try (0, or 5) say what a failing frame does."""
    rng = np.random.default_rng(31 + SEED)
    base = feed_calls(to_dev(mov), [], kw, max_try)
    assert base["xyc"].shape == (3, len(mov)), f"{what}: {base['xyc'].shape[1]} of {len(mov)} frames tracked"
    for name, run in ecc_modes(mov, kw, rng, frame_step, max_try):
        assert_same_track(run(), base, f"{what}: {name}")
    _lib.set_parameter("ecc_queue", 0)
    assert_same_track(feed_calls(to_dev(mov), [], kw, max_try), base, f"{what}: ecc_queue 0")
    assert_same_track(feed_calls(to_dev(mov), [17, 21], kw, max_try), base, f"{what}: ecc_queue 0, split")
    _lib.set_parameter("ecc_queue", 1)
    return base


def compute_step(img, reg):
    reg.compute(img)


def test_ecc_long_movie_every_mode_same_bits(ecc_movies, switches_restored):
    base = check_every_mode(ecc_movies["clean"], None, compute_step, 0, "clean movie")
    c = base["xyc"][2]
    assert (c < base["conf_thresh"]).sum() >= 10  # the reference is replaced many times


def test_ecc_long_movie_failures_every_mode_same_bits(ecc_movies, switches_restored):
    base = check_every_mode(ecc_movies["failures"], None, rg.manage_computation_and_tries, 5, "movie with failing frames")
    assert base["iterations"].count(-1) >= 1  # a frame ran out of tries and repeated the previous estimate
    assert (base["xyc"][2] < base["conf_thresh"]).sum() >= 10


def _static_mask(shape):
    m = np.ones(shape, np.uint8)
    m[:, :140] = 0
    return m


def _fixed_ref(mov):
    probe = rg.MaskedRegistratorECC()
    return mov[0][probe.startY:probe.startY + probe.subH, probe.startX:probe.startX + probe.subW]


QUEUE_OFF = [("mask", lambda mov: dict(mask=_static_mask(mov.shape[1:]))),
             ("median_0.9", lambda mov: dict(median=0.9)),
             ("sigma_0_u16", lambda mov: dict(sigma=0)),
             ("fixed_ref", lambda mov: dict(ref=_fixed_ref(mov)))]


@pytest.mark.parametrize("cfg", QUEUE_OFF, ids=[c[0] for c in QUEUE_OFF])
def test_ecc_configurations_every_mode_same_bits(ecc_movies, cfg, switches_restored):
    """A mask, median < 1 (quantile thresholds, no queue), sigma = 0 on u16 frames (the converted-frame cache) and a fixed
    reference (no replacements), over the first 200 frames (two flares)."""
    mov = ecc_movies["clean"][:200]
    check_every_mode(mov, cfg[1](mov), compute_step, 0, cfg[0])


@pytest.mark.parametrize("fused", [1, 0], ids=["one cooperative launch", "launch per iteration"])
def test_ecc_long_movie_against_restated_class(ecc_movies, restated_run, fused, switches_restored):
    want, want_its, want_th = restated_run
    _lib.set_parameter("ecc_fused", fused)
    got = feed_calls(to_dev(ecc_movies["clean"]), [], None)
    a = got["xyc"]
    resets = np.nonzero(want[2] < want_th)[0]
    assert len(resets) >= 10
    r = int(resets[0]) + 1  # up to and including the frame that triggers the first replacement
    assert np.max(np.abs(a[:2, :r] - want[:2, :r])) < 5e-5 and np.max(np.abs(a[2, :r] - want[2, :r])) < 5e-7
    assert got["iterations"][:r - 1] == want_its[:r - 1]
    assert abs(got["conf_thresh"] - want_th) < 1e-6
    assert np.array_equal(np.nonzero(a[2] < got["conf_thresh"])[0], resets), "the reference is replaced on other frames"


# ---- FramePipeline -------------------------------------------------------------------------------------------------------
def oracle_chain(port, mov, dx, dy):
    oxy, _thr, oclamp = port.bad_pixels_detect(mov[0])
    c = np.stack([port.bad_pixels_correct_with(oxy, oclamp, f) for f in mov])
    r = np.stack([port.translate(c[t], dx[t], dy[t], "nearest", 0) for t in range(len(mov))])
    return c, r


def f32_dev(a):
    return torch.from_numpy(np.ascontiguousarray(a, np.float32)).cuda()


def pipe_movie(n, h, w, seed):
    mov = ir_movie(n, h, w, seed=seed, drift=0.3)
    rng = np.random.default_rng(seed)
    return mov, rng.uniform(-3, 3, n).astype(np.float32), rng.uniform(-3, 3, n).astype(np.float32)


def check_chunked_movie(port, pipe, mov, dx, dy, what):
    cfg = pipe.cfg
    d = to_dev(mov)
    pipe.set_first_frame(d[0])
    pipe.stats.reset()
    got = {k: [] for k in ("c", "s", "r", "lo", "hi")}
    n, chunk = len(mov), cfg.chunk_frames
    for a in range(0, n, chunk):
        b = min(n, a + chunk)
        outs = pipe.process_chunk(d[a:b], f32_dev(dx[a:b]), f32_dev(dy[a:b]), first_frame=a)
        for k, o in zip(("c", "s", "r", "lo", "hi"), outs):
            got[k].append(o.cpu().view(torch.int16).numpy().view(np.uint16) if o.dtype == torch.uint16 else o.cpu().numpy())
    got = {k: np.concatenate(v) for k, v in got.items()}
    want_c, want_r = oracle_chain(port, mov, dx, dy)
    for k, want in (("c", want_c), ("r", want_r)):
        bad = np.nonzero((got[k] != want).reshape(n, -1).any(axis=1))[0]
        assert bad.size == 0, f"{what}: {k} frames {bad[:8]} differ"
    for a in range(0, n, 32):
        G.assert_gauss_exact(got["s"][a:a + 32], want_c[a:a + 32], cfg.sigma, f"{what}: smoothed frames {a}..")
    olo, ohi = port.precode_movie(want_r, cfg.gop, cfg.delta)
    assert np.array_equal(got["lo"], olo) and np.array_equal(got["hi"], ohi), f"{what}: byte planes"
    lo, hi, hist = port.movie_stats(want_r)
    st = pipe.stats
    assert (st.min(), st.max()) == (lo, hi), what
    assert np.array_equal(st.histogram(), hist), f"{what}: histogram"
    assert st.count == want_r.size, f"{what}: count {st.count} != {want_r.size}"
    for p in (0.001, 0.25, 0.5, 0.9, 0.999):
        assert st.quantile(p) == port.quantile_from_hist(hist, p), f"{what}: quantile {p}"
    assert st.background() == port.get_background(want_r.ravel()), f"{what}: background"


# (id, h, w, gop, chunk_frames, frames of the first movie, of the second, delta, fuse_stats): 7 and 6 chunks at 64 x 96, 3 at
# 640 x 512 (the benchmark's pairing and the other extreme), each with a short last chunk
CHUNKED = [(f"64x96-{d}-{f}", 64, 96, 10, 40, 6 * 40 + 17, 5 * 40 + 3, d == "delta", f == "fused")
           for d in ("delta", "no_delta") for f in ("fused", "separate")]
CHUNKED += [("640x512-delta-fused", 512, 640, 10, 20, 2 * 20 + 7, 2 * 20 + 13, True, True),
            ("640x512-no_delta-separate", 512, 640, 10, 20, 2 * 20 + 7, 2 * 20 + 13, False, False)]


@pytest.mark.parametrize("case", CHUNKED, ids=[c[0] for c in CHUNKED])
def test_process_chunk_multi_chunk_movies(port, case):
    name, h, w, gop, chunk, n1, n2, delta, fuse_stats = case
    cfg = movie.PipelineConfig(width=w, height=h, sigma=1.0, gop=gop, delta=delta, chunk_frames=chunk, fuse_stats=fuse_stats)
    pipe = movie.FramePipeline(cfg)
    check_chunked_movie(port, pipe, *pipe_movie(n1, h, w, seed=h + n1), f"{name} first movie")
    # a second, different movie through the same object: nothing of the first may leak into it
    mov2, dx2, dy2 = pipe_movie(n2, h, w, seed=h + n2 + 1)
    mov2 = (mov2.astype(np.int64) + 3000).clip(0, 65535).astype(np.uint16)
    check_chunked_movie(port, pipe, mov2, dx2, dy2, f"{name} second movie")


def pinned(a):
    t = torch.from_numpy(a.view(np.int16)).view(torch.uint16) if a.dtype == np.uint16 else torch.from_numpy(a)
    return t.pin_memory()


@pytest.mark.parametrize("delta", [True, False], ids=["delta", "no delta"])
def test_process_host_rotates_slots(port, delta):
    """process_host: sub-chunks over all three slots and round again, a ragged last one, first_frame != 0, a second call on
    the same object; against process_chunk and the oracle chain."""
    h, w, gop = 48, 80, 10
    sub_frames = 20 if delta else 23
    sub = 20 if delta else 23
    cfg = movie.PipelineConfig(width=w, height=h, sigma=1.0, gop=gop, delta=delta, chunk_frames=3 * sub)
    pipe = movie.FramePipeline(cfg)
    ref = movie.FramePipeline(movie.PipelineConfig(width=w, height=h, sigma=1.0, gop=gop, delta=delta, chunk_frames=400))
    for call, (n, first) in enumerate(((7 * sub + 13, 30), (2 * sub + 1, 60 if delta else 7))):
        mov, dx, dy = pipe_movie(n, h, w, seed=call + 5)
        d = to_dev(mov)
        pipe.set_first_frame(d[0])
        ref.set_first_frame(d[0])
        lo = torch.empty((n, h, w), dtype=torch.uint8).pin_memory()
        hi = torch.empty((n, h, w), dtype=torch.uint8).pin_memory()
        lo.fill_(0xAA)
        hi.fill_(0x55)
        pipe.process_host(pinned(mov), pinned(dx), pinned(dy), first, lo, hi, sub_frames)
        _c, _s, _r, rlo, rhi = ref.process_chunk(d, f32_dev(dx), f32_dev(dy), first_frame=first, with_stats=False)
        assert torch.equal(lo, rlo.cpu()) and torch.equal(hi, rhi.cpu()), f"call {call}: process_host != process_chunk"
        _want_c, want_r = oracle_chain(port, mov, dx, dy)
        olo, ohi = port.precode_movie(want_r, gop, delta)
        assert np.array_equal(lo.numpy(), olo) and np.array_equal(hi.numpy(), ohi), f"call {call}: against the oracle chain"


def test_process_host_refuses_slots_beyond_the_chunk_buffers(port):
    """slots x sub-chunk frames must fit chunk_frames: each slot works in its own window of the shared buffers."""
    h, w = 16, 32
    pipe = movie.FramePipeline(movie.PipelineConfig(width=w, height=h, gop=10, delta=True, chunk_frames=50))
    mov = ir_movie(60, h, w)
    pipe.set_first_frame(to_dev(mov[:1])[0])
    lo = torch.empty((60, h, w), dtype=torch.uint8)
    hi = torch.empty_like(lo)
    z = torch.zeros(60)
    with pytest.raises(RuntimeError, match="do not fit"):
        pipe.process_host(pinned(mov), z, z, 0, lo, hi, sub_frames=20)  # 3 x 20 > 50
    pipe.process_host(pinned(mov), z, z, 0, lo, hi, sub_frames=10)  # 3 x 10 fits
    assert np.array_equal(lo.numpy(), port.precode_movie(oracle_chain(port, mov, np.zeros(60), np.zeros(60))[1], 10, True)[0])
