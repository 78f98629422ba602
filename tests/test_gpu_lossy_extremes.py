"""The lossy pre-conditioner's kernels (csrc/lossy.cu) on the content where the reference's arithmetic wraps: the int square
of stdDev for |diff| >= 46,341 and x86's conversion of a NaN or out-of-range bound (tests/lossy_extreme_cases.py; the
restatement is pinned against the compiled statements by tests/test_lossy_extremes.py).  Bit for bit against the
restatement: outputs and per-frame (BackgroundError, ForegroundError), through both drivers switching on one handle, runs
that cross the 40-frame window and the 64-frame launch limit, host and device frames, and the drop-in saver entries of
libvideo_io_b200.so.  Then two sizes (640 x 512, and 2048 x 2048 = 2^22 lossy pixels, the largest at which the kernels'
exact integer sum of wrapped squares equals the reference's sequential double sum) and a seeded fuzzer
(``RIRB_FUZZ_SEED`` / ``RIRB_FUZZ_SCALE``, as in test_gpu_fuzz.py).

Also the same conversion class in the ECC front end: rirb_ecc_quantile casts its float window like numpy's
astype(uint16) on x86-64, where NaN, +-inf and values beyond int range become 0."""
import ctypes as ct
import os

import numpy as np
import pytest

from tests import lossy_extreme_cases as L
from tests.conftest import ir_movie
from tests.ecc_cases import hash_noise
from tests.test_oracle_vs_refvio import run_port_lossy

pytestmark = pytest.mark.gpu

torch = pytest.importorskip("torch")
if not torch.cuda.is_available():  # pragma: no cover
    pytest.skip("needs a CUDA device", allow_module_level=True)

from librir_b200 import _lib, video_io as vio  # noqa: E402

SEED = int(os.environ.get("RIRB_FUZZ_SEED", "0"))
SCALE = max(1, int(os.environ.get("RIRB_FUZZ_SCALE", "1")))
CHUNKS = (1, 39, 1, 64, 70)  # single frames, the window filling up, a full launch, one over the launch limit
# (frames per call, lossy_run per call (cycled), device frames): the one-launch driver, the per-frame one, and the two
# alternating on one handle; a whole movie or a 70-frame call is split into launches of at most 64 frames
MODES = [(CHUNKS, (1,), True), ((), (0,), False), ((2, 70), (1, 0), True), (CHUNKS, (0, 1), False), ((), (1,), False)]


@pytest.fixture
def lossy_run_restored():
    yield
    _lib.set_parameter("lossy_run", 1)


def to_dev(a):
    return torch.from_numpy(a.view(np.int16)).cuda().view(torch.uint16)


def to_host(t):
    return t if isinstance(t, np.ndarray) else t.cpu().view(torch.int16).numpy().view(np.uint16)


def chunking(t, pattern=CHUNKS):
    out, a = [], 0
    for c in pattern:
        if a + c >= t:
            break
        out.append(c)
        a += c
    return out + [t - a]


def gpu_lossy(mov, stop, cfg, door, chunks, drivers, device):
    t, h, w = mov.shape
    pre = vio.LossyPreconditioner(w, h, stop, variant=door, **cfg)
    outs, errs, a = [], [], 0
    for k, c in enumerate(chunks):
        _lib.set_parameter("lossy_run", drivers[k % len(drivers)])
        part = np.ascontiguousarray(mov[a:a + c])
        o, e = pre.add_images(to_dev(part) if device else part)
        outs.append(to_host(o))
        errs.append(e)
        a += c
    assert a == t
    return np.concatenate(outs), np.concatenate(errs)


def assert_same(outs, errs, want_o, want_e, what):
    bad_e = np.nonzero((errs != want_e).any(axis=1))[0]
    assert bad_e.size == 0, f"{what}: bounds differ from frame {bad_e[:6]}: {errs[bad_e[:3]].tolist()} != {want_e[bad_e[:3]].tolist()}"
    bad_o = np.nonzero((outs != want_o).reshape(len(outs), -1).any(axis=1))[0]
    assert bad_o.size == 0, f"{what}: frames {bad_o[:6]} differ"


# ---- the cases ----------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("door", L.DOORS)
@pytest.mark.parametrize("case", L.CASES, ids=[c[0] for c in L.CASES])
def test_lossy_extremes_equal_the_restatement(port, case, door, lossy_run_restored):
    name, mov, stop, cfg = case
    want_o, want_e = run_port_lossy(port, mov, stop, cfg, door)
    for pattern, drivers, device in MODES:
        outs, errs = gpu_lossy(mov, stop, cfg, door, chunking(len(mov), pattern), drivers, device)
        assert_same(outs, errs, want_o, want_e, f"{name} {door} lossy_run {drivers} device {device}")


def _vio():
    lib = ct.CDLL(os.path.join(os.path.dirname(_lib.lib_path()), "libvideo_io_b200.so"))
    lib.h264_open_file.restype = ct.c_int
    lib.h264_open_file.argtypes = [ct.c_char_p, ct.c_int, ct.c_int, ct.c_int]
    lib.h264_set_parameter.argtypes = [ct.c_int, ct.c_char_p, ct.c_char_p]
    lib.h264_add_image_lossy.argtypes = [ct.c_int, ct.c_void_p, ct.c_int64, ct.c_int, ct.c_void_p, ct.c_void_p, ct.c_void_p, ct.c_void_p]
    lib.h264_add_loss.argtypes = [ct.c_int, ct.c_void_p]
    for f in (lib.h264_get_low_errors, lib.h264_get_high_errors):
        f.argtypes = [ct.c_int, ct.c_void_p, ct.POINTER(ct.c_int)]
    lib.h264_close_file.restype = None
    lib.h264_close_file.argtypes = [ct.c_int]
    lib.open_camera_file.argtypes = [ct.c_char_p, ct.POINTER(ct.c_int)]
    lib.load_image.argtypes = [ct.c_int, ct.c_int, ct.c_int, ct.c_void_p]
    return lib


def saver_errors(lib, fn, handle, t):
    out = []
    for f in (lib.h264_get_low_errors, lib.h264_get_high_errors):
        e, size = np.zeros(t, np.uint16), ct.c_int(t)
        assert f(handle, e.ctypes.data, ct.byref(size)) == 0 and size.value == t
        out.append(e)
    return np.stack(out, axis=1)


@pytest.mark.parametrize("door", L.DOORS)
@pytest.mark.parametrize("case", L.CASES, ids=[c[0] for c in L.CASES])
def test_dropin_saver_entries_give_the_restated_bounds(port, tmp_path, case, door):
    """h264_add_image_lossy / h264_add_loss, one frame per call, and h264_get_low_errors / h264_get_high_errors."""
    name, mov, stop, cfg = case
    t, h, w = mov.shape
    want_o, want_e = run_port_lossy(port, mov, stop, cfg, door)
    lib = _vio()
    fn = str(tmp_path / "m.bin").encode()
    s = lib.h264_open_file(fn, w, h, stop)
    assert s > 0
    for k, v in cfg.items():
        assert lib.h264_set_parameter(s, k.encode(), str(v).encode()) == 0
    outs = []
    for i in range(t):
        img = np.ascontiguousarray(mov[i])
        if door == "add_loss":
            assert lib.h264_add_loss(s, img.ctypes.data) == 0
            outs.append(img)
        else:
            assert lib.h264_add_image_lossy(s, img.ctypes.data, 1000 * i, 0, None, None, None, None) == 0
    errs = saver_errors(lib, fn, s, t)
    lib.h264_close_file(s)
    assert np.array_equal(errs, want_e.astype(np.uint16)), f"{name} {door}: first differing frame {np.nonzero((errs != want_e).any(1))[0][:5]}"
    if door == "add_loss":
        assert np.array_equal(np.stack(outs), want_o)
    elif not cfg.get("subtractMin"):  # the reader adds MIN_T back on a subtractMin file
        fmt = ct.c_int(0)
        cam = lib.open_camera_file(fn, ct.byref(fmt))
        assert cam > 0
        img = np.empty((h, w), np.uint16)
        for i in range(t):
            assert lib.load_image(cam, i, 0, img.ctypes.data) == 0
            assert np.array_equal(img, want_o[i]), f"{name}: frame {i}"
        lib.close_camera(cam)


# ---- sizes --------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("shape", [(52, 512, 640), (50, 2048, 2048)], ids=["640x512", "2048x2048"])
def test_full_range_sizes(port, shape, lossy_run_restored):
    t, h, w = shape
    mov = np.random.default_rng(h).integers(0, 65536, shape, dtype=np.uint16)
    cfg = dict(L.WIDE, runningAverage=4)
    for door in L.DOORS:
        want_o, want_e = run_port_lossy(port, mov, h, cfg, door)
        assert len(np.unique(want_e[:, 0])) > 3  # the bounds move: the sums decide them
        for drivers, device in (((1,), True), ((0, 1), False)):
            outs, errs = gpu_lossy(mov, h, cfg, door, chunking(t), drivers, device)
            assert_same(outs, errs, want_o, want_e, f"{h}x{w} {door} lossy_run {drivers}")


# ---- fuzz ---------------------------------------------------------------------------------------------------------------
def fuzz_movie(rng, t, h, w):
    """ir_movie content with the extreme classes mixed in at random places."""
    mov = ir_movie(t, h, w, seed=int(rng.integers(0, 1 << 20)), drift=0.7).astype(np.int64)
    for _ in range(int(rng.integers(1, 4))):
        kind = int(rng.integers(0, 6))
        if kind == 0:  # blinking pixels
            idx = rng.choice(h * w, int(rng.integers(1, 6)), replace=False)
            level = int(rng.choice([46340, 46341, int(rng.integers(46341, 65536)), 65535]))
            mov.reshape(t, -1)[:, idx] = np.where(np.arange(t)[:, None] % 2 == int(rng.integers(0, 2)), 0, level)
        elif kind == 1:  # dead / saturated pixels
            m = rng.random((h, w))
            mov[:, m < 0.03] = 0
            mov[:, m > 0.97] = 65535
        elif kind == 2:  # saturated or flat frames, some of them on the first split
            frames = rng.choice(np.arange(35, t), int(rng.integers(1, 4)), replace=False) if t > 35 else [t - 1]
            mov[frames] = int(rng.choice([65535, 4 * int(rng.integers(1000, 16000)) + int(rng.integers(0, 4))]))
        elif kind == 3:  # a band of full-range noise
            r0 = int(rng.integers(0, h))
            band = mov[:, r0:r0 + int(rng.integers(1, 4))]
            band[...] = rng.integers(0, 65536, band.shape)
        elif kind == 4:  # the scene crosses integration-time ranges
            mov += 8192 * (np.arange(t)[:, None, None] // int(rng.integers(3, 20)) % 8)
        else:  # a step down (below the first frame's minimum)
            mov[int(rng.integers(1, t)):] -= int(rng.integers(500, 9000))
    return mov.clip(0, 65535).astype(np.uint16)


def test_fuzz_lossy_extremes(port, lossy_run_restored):
    rng = np.random.default_rng(606 + SEED)
    for case in range(6 * SCALE):
        w = int(rng.choice([8, 16, 33, 40, 64, 136]))
        h = int(rng.integers(4, 40))
        t = int(rng.integers(42, 120))
        stop = int(rng.choice([0, 1, h, int(rng.integers(0, h + 1))]))
        wide = bool(rng.integers(0, 2))
        cfg = dict(lowValueError=int(rng.choice([6, 3000])) if wide else int(rng.integers(0, 12)),
                   highValueError=int(rng.choice([2, 1500])) if wide else int(rng.integers(0, 6)),
                   stdFactor=float(rng.choice([0.5, 5.0, 1e10])), runningAverage=int(rng.choice([0, 1, 4, 32, 63, 64, 70])),
                   subtractMin=int(rng.integers(0, 2)), removeBadPixels=int(rng.integers(0, 2)) if stop >= 3 else 0)
        mov = fuzz_movie(rng, t, h, w)
        door = L.DOORS[int(rng.integers(0, 2))]
        want_o, want_e = run_port_lossy(port, mov, stop, cfg, door)
        cuts = np.sort(rng.choice(np.arange(1, t), int(rng.integers(0, 5)), replace=False))
        chunks = np.diff(np.concatenate([[0], cuts, [t]])).tolist()
        drivers = [int(v) for v in rng.integers(0, 2, len(chunks))]
        outs, errs = gpu_lossy(mov, stop, cfg, door, chunks, drivers, device=bool(rng.integers(0, 2)))
        assert_same(outs, errs, want_o, want_e, f"case {case}: {t}x{h}x{w} stop {stop} {door} {cfg} chunks {chunks} drivers {drivers}")


# ---- the ECC quantile's cast --------------------------------------------------------------------------------------------
ECC_SPECIAL = np.array([2.0 ** 31, 3e9, 1e20, np.inf, -np.inf, np.nan, 2147483520.0, -2147483648.0, -3e9, 70000.5, 65535.9,
                        -1.0, 0.25], dtype=np.float32)


@pytest.mark.parametrize("frac", [0.05, 0.3, 0.7])
def test_ecc_quantile_casts_like_numpy(port, frac):
    """find_median_pixel(window.astype(np.uint16), percent) of the reference on float windows with values numpy's cast
    sends to 0 (NaN, +-inf, >= 2^31), next to values just inside int range."""
    lib = _lib.load()
    h, w = 24, 40
    win = (8000 + 40 * hash_noise((h, w), 31)).astype(np.float32)
    m = hash_noise((h, w), 32) + 0.5
    pick = (7 * np.arange(h * w).reshape(h, w)) % len(ECC_SPECIAL)
    win[m < frac] = ECC_SPECIAL[pick[m < frac]]
    with np.errstate(invalid="ignore"):
        q16 = win.astype(np.uint16)
    hd = lib.rirb_ecc_open(w, h)
    assert hd > 0
    try:
        for which in (0, 1):
            assert lib.rirb_ecc_set_image(hd, which, win.ctypes.data_as(ct.c_void_p), w) == 0
            for pc in (0.02, 0.3, 0.5, 0.9, 0.99):
                assert lib.rirb_ecc_quantile(hd, which, pc, 0) == port.find_median_pixel(q16, pc), (which, pc)
    finally:
        lib.rirb_ecc_close(hd)
