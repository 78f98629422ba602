"""The ECC solver (csrc/ecc.cu) bit for bit against the restatement of its own arithmetic (tests/ecc_kernel.py).

The kernel's roundings are all fixed by its source (explicit _rn intrinsics, products of floats exact in fp64, sums added
in a fixed order with no atomics), so (status, rho, tx, ty, iterations) must be the same bits as the restatement's, with
the grid each driver runs on this device.  No tolerance anywhere.  How close the restatement is to OpenCV's iteration is
tests/test_ecc_kernel.py's business.  RIRB_FUZZ_SEED / RIRB_FUZZ_SCALE draw more random windows and starts.

The module's name sorts it after the modules that read kernel names from torch.profiler (tests/test_gpu_dispatch.py,
tests/test_gpu_gauss_exact.py): in one process, ECC solves and tracker runs after a profiler session have been seen to
leave later profiler sessions without any kernel record on a B200 (the ECC tests of tests/test_gpu_long_movies.py do the
same when run ahead of those modules), which fails their dispatch checks rather than anything here.
"""
import ctypes as ct
import os

import numpy as np
import pytest

from tests import ecc_cases as ec
from tests import ecc_kernel as ek

pytestmark = pytest.mark.gpu

torch = pytest.importorskip("torch")
if not torch.cuda.is_available():  # pragma: no cover
    pytest.skip("needs a CUDA device", allow_module_level=True)

from librir_b200 import _lib  # noqa: E402

SEED = int(os.environ.get("RIRB_FUZZ_SEED", "0"))
SCALE = max(1, int(os.environ.get("RIRB_FUZZ_SCALE", "1")))
SMS = torch.cuda.get_device_properties(0).multi_processor_count
INF, NAN = float("inf"), float("nan")


@pytest.fixture(params=[True, False], ids=["cooperative solve", "launch per iteration"])
def fused(request):
    _lib.set_parameter("ecc_fused", request.param)
    yield request.param
    _lib.set_parameter("ecc_fused", 1)


class Window:
    """A solver handle with its two images (and mask) set from inside wider frames, so that the row stride of
    rirb_ecc_set_image is not the window's width; the pixels around the window are huge and would show if read."""

    def __init__(self, ref, cur, mask=None, pad=13):
        self.lib = _lib.load()
        self.h, self.w = ref.shape
        self.hd = self.lib.rirb_ecc_open(self.w, self.h)
        assert self.hd > 0, _lib.last_error()
        self.keep = []
        for which, img in ((0, ref), (1, cur)):
            wide = np.full((self.h + 1, self.w + pad), 3e38, np.float32)
            wide[1:, pad // 2:pad // 2 + self.w] = img
            self.keep.append(wide)
            ptr = wide.ctypes.data + ((self.w + pad) + pad // 2) * 4
            assert self.lib.rirb_ecc_set_image(self.hd, which, ct.c_void_p(ptr), self.w + pad) == 0
        self.use_mask = mask is not None
        if self.use_mask:
            m8 = np.ascontiguousarray(mask, dtype=np.uint8)
            assert self.lib.rirb_ecc_set_mask(self.hd, 0, m8.ctypes.data_as(ct.c_void_p)) == 0

    def solve(self, tx0, ty0, max_it=500, thresh=INF, eps=1e-3):
        shift = np.array([tx0, ty0], np.float32)
        rho, its = ct.c_double(0), ct.c_int(0)
        st = self.lib.rirb_ecc_compute(self.hd, thresh, int(self.use_mask), max_it, eps, shift.ctypes.data_as(ct.c_void_p), ct.byref(rho),
                                       ct.byref(its))
        assert st >= 0, _lib.last_error()
        return st, rho.value, float(shift[0]), float(shift[1]), its.value

    def close(self):
        self.lib.rirb_ecc_close(self.hd)


def restated(ref, cur, mask, tx0, ty0, fused, max_it=500, thresh=INF, prepared=None):
    """ek.solve as rirb_ecc_compute reports it: the start is handed back when the solve fails."""
    p = prepared or ek.prepare(ref, cur, mask, thresh)
    st, rho, tx, ty, it = ek.solve(p, tx0, ty0, ek.grid(ref.size, SMS, fused), max_it=max_it)
    if st != 0:
        tx, ty = float(np.float32(tx0)), float(np.float32(ty0))
    return st, rho, tx, ty, it


def bits(r):
    st, rho, tx, ty, it = r
    return st, np.float64(rho).view(np.uint64) if not np.isnan(rho) else "nan", np.float32(tx).view(np.uint32), np.float32(ty).view(np.uint32), it


def assert_same(got, want, what):
    assert bits(got) == bits(want), f"{what}: library {got} != restatement {want}"


def check(ref, cur, mask, starts, fused, max_it=500, thresh=INF, what=""):
    win = Window(ref, cur, mask)
    try:
        p = ek.prepare(ref, cur, mask, thresh)
        for tx0, ty0 in starts:
            want = restated(ref, cur, mask, tx0, ty0, fused, max_it, thresh, prepared=p)
            assert_same(win.solve(tx0, ty0, max_it, thresh), want, f"{what} start ({tx0!r}, {ty0!r}) max_it {max_it}")
    finally:
        win.close()


# ---- one step from many starts: every iteration the solver can take, on its own ------------------------------------
def out_starts(h, w):
    """Starts that push most of the window out of the image, and starts beyond it (empty warped mask: status 1)."""
    return [(w - 2.5, 0.25), (0.0, -(h - 1.75)), (-(w - 3.0), h - 2.0), (w - 0.6, h - 0.6), (w + 5.0, 0.0), (0.0, -h - 3.5),
            (-w - 10.0, h + 10.0), (3.0 * w, -2.0 * h)]


def test_one_step_from_every_kind_of_start(fused):
    ref, cur = ec.ir_window_pair(3)
    s = ec.boundary_starts()
    starts = [(tx, s[(k * 7) % len(s)]) for k, tx in enumerate(s)] + [(tx, tx) for tx in s[::3]] + out_starts(*ref.shape)
    check(ref, cur, None, starts, fused, max_it=1, what="ir window, one step")
    sm_t, sm_i = ec.small_pair(1.2, 0.7, k=9)
    mask = np.zeros(sm_t.shape, np.uint8)
    mask[10:100, 20:150] = 1
    check(sm_t, sm_i, mask, [(tx, -tx) for tx in s[::2]] + out_starts(*sm_t.shape), fused, max_it=1, what="small masked, one step")


# ---- whole solves: against the chain of one-step calls (the library against itself) and against the restatement -----
def chained(win, tx0, ty0, max_it=500, eps=1e-3):
    """The whole solve as one-step calls, with ecc.cu's stopping rule applied here."""
    tx, ty, rho, last, it = float(np.float32(tx0)), float(np.float32(ty0)), -1.0, -eps, 0
    while True:
        st, r, ntx, nty, one = win.solve(tx, ty, 1)
        assert one == 1
        it += 1
        if st != 0:
            return st, None, float(np.float32(tx0)), float(np.float32(ty0)), it
        last, rho, tx, ty = rho, r, ntx, nty
        if it >= max_it or not abs(rho - last) >= eps:
            return 0, rho, tx, ty, it


@pytest.mark.parametrize("case", ["ir 1", "ir 3", "ir 6", "small", "small masked", "small warm"])
def test_whole_solve_is_the_chain_of_its_steps(case, fused):
    if case.startswith("ir"):
        ref, cur = ec.ir_window_pair(int(case[3:]))
        mask, start = None, (0.0, 0.0)
    else:
        ref, cur = ec.small_pair(1.2, 0.7, k=9) if case != "small" else ec.small_pair(-2.5, 3.25, k=2)
        mask = None
        if case == "small masked":
            mask = np.zeros(ref.shape, np.uint8)
            mask[10:100, 20:150] = 1
        start = (1.0, 0.5) if case == "small warm" else (0.0, 0.0)
    win = Window(ref, cur, mask)
    try:
        whole = win.solve(*start)
        chain = chained(win, *start)
    finally:
        win.close()
    assert whole[0] == 0 and whole[4] > 1, whole
    assert_same(whole, chain, f"{case}: whole solve against its one-step chain")
    assert_same(whole, restated(ref, cur, mask, *start, fused), f"{case}: whole solve")


# ---- windows: tiny, around one CTA, around each driver's grid, and large ----------------------------------------------
def shape_of(n):
    """A window of n pixels (both sides >= 2, as square as possible); a prime n takes the next composite size, which
    still puts one more pixel than threads on the grid."""
    while True:
        f = [d for d in range(2, int(n ** 0.5) + 1) if n % d == 0]
        if f:
            return f[-1], n // f[-1]
        n += 1


def window_shapes():
    shapes = [(2, 2), (2, 37), (37, 2), (2, 300), (300, 2)]
    for g in (1, SMS, min(2 * SMS, ek.MAX_SLOTS)):
        shapes += [shape_of(g * ek.THREADS - 1), shape_of(g * ek.THREADS), shape_of(g * ek.THREADS + 1)]
    return sorted(set(shapes)) + [(358, 448), (512, 640), (1024, 1024), (2048, 2048)]


@pytest.mark.parametrize("h,w", window_shapes())
def test_windows(h, w, fused):
    ref, cur = ec.small_pair(1.3, -0.6, h=h, w=w, k=h + w)
    steps = 500 if h * w <= 400_000 else (2 if h * w <= 1 << 20 else 1)
    starts = [(0.0, 0.0), (0.7, -0.4)] if steps == 500 else [(0.3, -0.2)]
    check(ref, cur, None, starts, fused, max_it=steps, what=f"{h} x {w}")
    if h * w <= 400_000:
        check(ref, cur, None, [(0.3, -0.2), (-1.45, 2.55)], fused, max_it=1, what=f"{h} x {w}, one step")


# ---- masks, clamps, content ------------------------------------------------------------------------------------------
def masks(h, w, rng):
    ring = np.ones((h, w), np.uint8)
    ring[3:-3, 3:-3] = 0
    single = np.zeros((h, w), np.uint8)
    single[h // 2, w // 3] = 1
    return {"none": None, "full": np.ones((h, w), np.uint8), "empty": np.zeros((h, w), np.uint8), "single pixel": single,
            "border ring": ring, "checkerboard": ((np.arange(h)[:, None] + np.arange(w)[None, :]) % 2).astype(np.uint8),
            "random 50 %": (rng.random((h, w)) < 0.5).astype(np.uint8) * np.uint8(rng.integers(1, 256))}


def test_masks(fused):
    ref, cur = ec.small_pair(1.37, -0.62, k=0)
    for name, mask in masks(*ref.shape, np.random.default_rng(5)).items():
        check(ref, cur, mask, [(0.0, 0.0), (1.0, -1.0)], fused, what=f"mask {name}")


def test_clamps(fused):
    t, i = ec.ir_window_pair(2)
    lo = float(min(t.min(), i.min()))
    for thresh in (INF, NAN, float(np.quantile(t, 0.1)), float(np.quantile(i, 0.6)), float(np.nextafter(np.float32(lo), np.float32(-1)))):
        check(t, i, None, [(0.0, 0.0)], fused, thresh=thresh, what=f"thresh {thresh!r}")


def test_content(fused):
    t, i = ec.ir_window_pair(4)
    const = np.full_like(i, 8000.0)
    inverted = (20000.0 - i).astype(np.float32)
    cases = {"ir frame 4": (t, i), "constant image": (t, const), "constant template": (const, i), "contrast-inverted": (t, inverted)}
    for v, name in ((np.nan, "NaN"), (np.inf, "+inf"), (-np.inf, "-inf")):
        bad = i.copy()
        bad[100, 200] = v
        cases[f"a {name} pixel"] = (t, bad)
        cases[f"a {name} pixel in the template"] = (bad, i)
    for k, (dx, dy) in enumerate(ec.SMALL_CASES):
        cases[f"scene {k}"] = ec.small_pair(dx, dy, k=k)
    seen = set()
    for name, (a, b) in cases.items():
        win = Window(a, b)
        try:
            got = win.solve(0.0, 0.0)
        finally:
            win.close()
        assert_same(got, restated(a, b, None, 0.0, 0.0, fused), name)
        seen.add(got[0])
    assert seen == {0, 1, 2}


def test_random_windows_and_starts(fused):
    rng = np.random.default_rng(905 + SEED)
    for case in range(8 * SCALE):
        h, w = int(rng.integers(2, 260)), int(rng.integers(2, 330))
        dx, dy = float(rng.uniform(-4, 4)), float(rng.uniform(-4, 4))
        t, i = ec.small_pair(dx, dy, h=h, w=w, k=int(rng.integers(0, 1000)))
        scale, offset = float(rng.choice([1.0, 5000.0])), float(rng.choice([0.0, 8000.0]))
        t, i = (t * scale + offset).astype(np.float32), (i * np.float32(scale * rng.uniform(0.8, 1.2)) + np.float32(offset)).astype(np.float32)
        mask = list(masks(h, w, rng).values())[int(rng.integers(0, 7))] if h > 6 and w > 6 else None
        thresh = [INF, NAN, float(np.quantile(t, rng.uniform(0.05, 0.95)))][int(rng.integers(0, 3))]
        starts = [(float(np.float32(dx + rng.uniform(-1, 1))), float(np.float32(dy + rng.uniform(-1, 1)))), (0.0, 0.0)]
        check(t, i, mask, starts, fused, max_it=int(rng.choice([1, 2, 500])), thresh=thresh, what=f"case {case}: {h} x {w}")


# ---- queued runs: the tracker on frames in device memory ------------------------------------------------------------
@pytest.mark.parametrize("sigma,median", [(0.0, 1.0), (0.5, 1.0), (0.5, 0.9)])
def test_tracker_is_the_chain_of_restated_solves(sigma, median, fused):
    """rirb_ecc_track over 12 frames (under the 21 confidences after which the class may replace its reference): every
    frame's (x, y, conf, iterations) is the restated solve from the previous frame's shift, on windows of the library's
    own full-frame Gaussian -- so the region the tracker filters is exact inside the window -- and, for median < 1, with
    the quantile clamp restated."""
    from librir_b200 import registration as rg
    from librir_b200 import signal_processing as sp
    from oracle import oracle as O

    mov, _, _ = ec.movie(12)
    d = torch.from_numpy(mov.view(np.int16)).cuda().view(torch.uint16)
    reg = rg.MaskedRegistratorECC(sigma=sigma, median=median)
    assert reg.compute_movie(d, max_try=0) == len(mov)
    full = sp.gaussian_filter_batch(d, sigma).cpu().numpy() if sigma > 0 else mov.astype(np.float32)
    wins = full[:, reg.startY:reg.startY + reg.subH, reg.startX:reg.startX + reg.subW]
    port = O.Port()
    tx, ty = 0.0, 0.0
    assert (reg.x[0], reg.y[0], reg.confidences[0]) == (0, 0, 1)
    for t in range(1, len(mov)):
        thresh = INF
        if median < 1:
            thresh = float(max(port.find_median_pixel(wins[t].astype(np.uint16), median), port.find_median_pixel(wins[0].astype(np.uint16), median)))
        p = ek.prepare(wins[0], wins[t], None, thresh)
        st, rho, tx, ty, it = ek.solve(p, tx, ty, ek.grid(wins[0].size, SMS, fused))
        assert st == 0
        got = (0, reg.confidences[t], float(reg.x[t]), float(reg.y[t]), reg.iterations[t - 1])
        assert_same(got, (st, rho, tx, ty, it), f"frame {t}")
