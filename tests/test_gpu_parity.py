"""Parity of the CUDA path with the oracle, THROUGH THE C ABI (numpy in -> ctypes -> CUDA ->
numpy out for the per-frame entries; torch CUDA tensors for the batched ones).

Bars (BASELINE.json north_star): bit-exact for bad pixels, pre-coder, statistics -- and, since
the blend is evaluated in the reference's fp64 order, for integer translate as well (the
allowed +-1 LSB is not used); float32 Gaussian output within the rounding bound of the float64 operation on every
pixel (tests/gauss_exact.py).
"""
import os

import numpy as np
import pytest

from tests.conftest import ir_frame, ir_movie
from tests.gauss_exact import assert_gauss_exact, assert_reference_exact
from tests.golden.make_golden import DTYPES, STRATEGIES, typed_image

pytestmark = pytest.mark.gpu

torch = pytest.importorskip("torch")

from librir_b200 import _lib, signal_processing as sp, video_io as vio  # noqa: E402
from oracle import oracle as O  # noqa: E402


@pytest.fixture(scope="module")
def best():
    return O.best()


def to_dev(a):
    """numpy (u)int/float array -> torch CUDA tensor of the same dtype."""
    if a.dtype == np.uint16:
        return torch.from_numpy(a.view(np.int16)).cuda().view(torch.uint16)
    return torch.from_numpy(a).cuda()


# One-off fuzzing on the GPU box: RIRB_FUZZ_SEED shifts the seeds of the randomised tests, RIRB_FUZZ_SCALE multiplies
# their case counts (defaults: the committed, deterministic cases).
FUZZ_SEED = int(os.environ.get("RIRB_FUZZ_SEED", "0"))
FUZZ_SCALE = max(1, int(os.environ.get("RIRB_FUZZ_SCALE", "1")))


def rand_u16(shape, seed, high=16384):
    """Random uint16 CUDA tensor (values < 2**15, built through int16: same bits)."""
    g = torch.Generator(device="cuda").manual_seed(seed)
    return torch.randint(0, high, shape, generator=g, device="cuda", dtype=torch.int32).to(torch.int16).view(torch.uint16)


def as_int(t):
    """uint16 CUDA tensor (values < 2**15) -> int32, via the int16 view."""
    return t.view(torch.int16).to(torch.int32)


def to_host(t):
    if t.dtype == torch.uint16:
        return t.cpu().view(torch.int16).numpy().view(np.uint16)
    return t.cpu().numpy()


# ---------------------------------------------------------------------------------------------
# the library really is the thing that runs
# ---------------------------------------------------------------------------------------------
def test_device_present_and_kernels_launch():
    assert _lib.device_available()
    before = _lib.launch_count()
    sp.gaussian_filter(np.ones((8, 8), np.float32), 1.0)
    assert _lib.launch_count() > before


# ---------------------------------------------------------------------------------------------
# translate
# ---------------------------------------------------------------------------------------------
@pytest.mark.parametrize("dt", DTYPES)
def test_translate_golden_all_dtypes(golden, dt):
    img = golden[f"tr_{dt}_in"]
    for si, st in enumerate(STRATEGIES):
        for k, (dx, dy) in enumerate(golden["tr_shifts"]):
            got = sp.translate(img, dx, dy, st, background=1)
            want = golden[f"tr_{dt}_{si}_{k}"]
            assert got.dtype == want.dtype
            np.testing.assert_array_equal(got, want, err_msg=f"{dt} {st!r} dx={dx} dy={dy}")


def test_translate_golden_ir_frame(golden):
    f = golden["tr_ir_in"]
    for si, st in enumerate(STRATEGIES):
        np.testing.assert_array_equal(sp.translate(f, 1.3, -2.7, st, background=7), golden[f"tr_ir_{si}"])
    np.testing.assert_array_equal(sp.translate(f, 1.3, -2.7, "constant", background=7), golden["tr_ir_1"])


@pytest.mark.parametrize("strategy", ["", "background", "wrap", "nearest"])
def test_translate_u16_full_frame_many_shifts(best, strategy):
    f = ir_frame(512, 640, 21)
    shifts = [(1.3, -2.7), (0.0, 0.0), (3.0, -2.0), (-0.5, 0.5), (0.3, 0.7), (-0.3, -0.7), (2.9999998, 511.5),
              (639.25, 0.0), (-640.0, 3.0), (1e-30, -1e-30), (0.99999994, 0.99999994), (100.125, -200.0625), (700.0, 3.0)]
    for dx, dy in shifts:
        got = sp.translate(f, dx, dy, strategy, background=123)
        want = best.translate(f, dx, dy, strategy, background=123)
        np.testing.assert_array_equal(got, want, err_msg=f"{strategy!r} dx={dx} dy={dy}")


@pytest.mark.parametrize("shape", [(37, 53), (5, 7), (1, 1), (2, 9), (64, 66)])
def test_translate_u16_odd_shapes(best, shape):
    rng = np.random.default_rng(3)
    f = rng.integers(0, 65536, shape, dtype=np.uint16)
    for st in ["", "background", "wrap", "nearest"]:
        for dx, dy in [(1.3, -2.7), (0.5, 0.5), (-0.25, 0.75), (0, 0)]:
            np.testing.assert_array_equal(sp.translate(f, dx, dy, st, 9), best.translate(f, dx, dy, st, 9))


def test_kernel_variant_switches():
    """rirb_set_parameter: the register-only kernels behind "translate_tma" / "gauss_tma" = 0 give the same
    results as the TMA-tiled ones (bit-exact translate; Gaussian within the bound of the float64 operation)."""
    f = ir_frame(96, 128, 5)
    want_t = sp.translate(f, 1.3, -2.7, "nearest", 0)
    assert_gauss_exact(sp.gaussian_filter(f, 1.0), f, 1.0, "default")
    try:
        _lib.set_parameter("translate_tma", 0)
        _lib.set_parameter("gauss_tma", 0)
        np.testing.assert_array_equal(sp.translate(f, 1.3, -2.7, "nearest", 0), want_t)
        assert_gauss_exact(sp.gaussian_filter(f, 1.0), f, 1.0, "gauss_tma = 0")
    finally:
        _lib.set_parameter("translate_tma", 1)
        _lib.set_parameter("gauss_tma", 1)
    with pytest.raises(RuntimeError):
        _lib.set_parameter("no_such_switch", 1)


@pytest.mark.parametrize("shape", [(8, 8), (1, 8), (3, 16), (64, 128), (65, 136), (129, 256), (130, 264), (200, 320), (70, 1032)])
def test_translate_u16_tiled_shapes(best, shape):
    """Widths that are multiples of 8 take the TMA-tiled kernel: tile / stage boundaries (128 columns,
    64 rows), images smaller than one box, every residual column offset 0..7 and both signs of shift."""
    rng = np.random.default_rng(31)
    f = rng.integers(0, 65536, shape, dtype=np.uint16)
    shifts = [(0.0, 0.0), (1.3, -2.7), (-2.6, 1.4), (7.5, 0.25), (-8.0, -8.0), (3.999999, 63.5), (-65.25, 64.0), (130.5, -129.75),
              (0.5, 1e-7), (5.0000005, -0.99999994)]
    shifts += [tuple(rng.uniform(-9, 9, 2).astype(np.float32)) for _ in range(6)]
    for st in ["nearest", "background", "wrap", ""]:
        for dx, dy in shifts:
            np.testing.assert_array_equal(sp.translate(f, dx, dy, st, 77), best.translate(f, dx, dy, st, 77),
                                          err_msg=f"{shape} {st!r} dx={dx} dy={dy}")


def test_translate_u16_random_shifts_full_size(best):
    """Many random sub-pixel shifts on the shapes of configs 3 and 4 (per-frame shifts, one launch)."""
    rng = np.random.default_rng(32)
    for h, w, n in [(512, 640, 12), (1024, 1024, 4)]:
        mov = np.stack([ir_frame(h, w, 100 + t) for t in range(n)])
        dx = rng.uniform(-3, 3, n).astype(np.float32)
        dy = rng.uniform(-3, 3, n).astype(np.float32)
        got = to_host(sp.translate_batch(to_dev(mov), to_dev(dx), to_dev(dy), "nearest", 0))
        for t in range(n):
            np.testing.assert_array_equal(got[t], best.translate(mov[t], dx[t], dy[t], "nearest", 0), err_msg=f"{h}x{w} frame {t}")


def reference_reads_past_the_buffer(h, w, dx, dy):
    """Pixels for which the reference's in-range branch indexes past the end of the image (Filters.h:300-310 with
    px + 1.0f or py + 1.0f rounded up beyond the clamp): undefined in the reference, last-pixel reads here."""
    px = np.broadcast_to(np.arange(w, dtype=np.float32)[None, :] - np.float32(dx), (h, w))
    py = np.broadcast_to(np.arange(h, dtype=np.float32)[:, None] - np.float32(dy), (h, w))
    inr = (px >= 0) & (px < w) & (py >= 0) & (py < h)
    rt = np.where(inr, px + np.float32(1), np.float32(0)).astype(np.int64)
    b = np.where(inr, py + np.float32(1), np.float32(0)).astype(np.int64)
    rt = np.where(rt == w, w - 1, rt)  # clamped onto l
    b = np.where(b == h, h - 1, b)     # clamped onto t
    return inr & (b * w + rt >= h * w)


def test_translate_u16_randomized(best, port):
    """150 random (shape, shift, strategy) cases: widths on and off the TMA path, shifts from sub-ulp to beyond the
    image, exact integers, halves and values one float ulp away from an integer."""
    rng = np.random.default_rng(2026 + FUZZ_SEED)
    specials = [0.0, 1.0, -1.0, 0.5, -0.5, 8.0, -8.0, 7.9999995, -7.9999995, 1.0000001, 127.5, -128.0, 1e-20, -1e-20, 0.25, 63.75]
    for case in range(150 * FUZZ_SCALE):
        w = int(rng.choice([8, 16, 24, 40, 64, 96, 128, 136, 200, 264, 7, 33, 130]))
        h = int(rng.integers(1, 150))
        f = rng.integers(0, 65536, (h, w), dtype=np.uint16)
        if case % 3 == 0:
            f = (f >> 6).astype(np.uint16)  # small values: exact-integer results are common
        def pick(extent):
            k = rng.integers(0, 4)
            if k == 0:
                return float(rng.choice(specials))
            if k == 1:
                return float(np.float32(rng.uniform(-3, 3)))
            if k == 2:
                return float(np.float32(rng.uniform(-extent - 5, extent + 5)))
            return float(np.float32(rng.integers(-extent, extent + 1)) + np.float32(rng.choice([0, 2 ** -20, -2 ** -20, 0.5])))
        dx, dy = pick(w), pick(h)
        st = ["nearest", "background", "wrap", ""][case % 4]
        got, want = sp.translate(f, dx, dy, st, 321), best.translate(f, dx, dy, st, 321)
        undefined = reference_reads_past_the_buffer(h, w, dx, dy)
        if undefined.any():  # there the compiled reference returns whatever follows its buffer: the restatement decides
            want = np.where(undefined, port.translate(f, dx, dy, st, 321), want)
        np.testing.assert_array_equal(got, want, err_msg=f"case {case}: {h}x{w} {st!r} dx={dx!r} dy={dy!r}")


@pytest.mark.parametrize("h,w,st,dx,dy", [
    (46, 16, "nearest", -4.999999046325684, -14.0), (121, 8, "nearest", -7.9999995, 0.0),
    (33, 16, "wrap", -6.999999046325684, -2.654136896133423), (40, 136, "background", -7.9999995, -15.999999),
    (64, 128, "", 0.25, -31.999998), (70, 264, "nearest", -127.99999, -5.9999995), (9, 7, "nearest", -2.9999998, -3.9999998)])
def test_translate_source_index_one_past_the_clamp(best, port, h, w, st, dx, dy):
    """px (py) within half a float ulp below w (h): px + 1.0f rounds up to w + 1, the reference's `== w` clamp does not
    fire and it reads the first pixels of the NEXT row (found by fuzzing: the staged box holds zeros there).  Defined
    pixels must equal the compiled reference; the ones whose read leaves the buffer follow the restatement's clamp."""
    rng = np.random.default_rng(h * 1000 + w)
    f = rng.integers(0, 65536, (h, w), dtype=np.uint16)
    undefined = reference_reads_past_the_buffer(h, w, dx, dy)
    want = np.where(undefined, port.translate(f, dx, dy, st, 321), best.translate(f, dx, dy, st, 321))
    np.testing.assert_array_equal(sp.translate(f, dx, dy, st, 321), want)
    mov = np.stack([f, f[::-1].copy(), f])  # batched: every frame keeps its own "last pixel"
    got = sp.translate_batch(mov, dx, dy, st, 321)
    for k in range(3):
        und_k = port.translate(mov[k], dx, dy, st, 321)
        np.testing.assert_array_equal(got[k], np.where(undefined, und_k, best.translate(mov[k], dx, dy, st, 321)))
    # the reader's motion variant takes the same route (u16 -> float -> u16)
    moved = vio.remove_motion(mov, [-dx] * 3, [-dy] * 3, meta_rows=0)
    for k in range(3):
        want_k = port.loader_remove_motion(mov[k], -dx, -dy)
        np.testing.assert_array_equal(moved[k][~undefined], want_k[~undefined])


@pytest.mark.parametrize("w,h", [(640, 136), (2048, 72), (1288, 200)])
def test_translate_shifts_half_an_ulp_from_an_integer(best, port, w, h):
    """-dx (-dy) within half a float ulp below an integer: in the upper float binades of a row (column) px rounds up to
    the next integer and the reference blends that column with weight 1 -- a different (l, u) than in the lower binades
    of the same row.  The tiled kernel keeps such pixels on its fast path as `regular taps, u = 1` (they used to go
    through the per-pixel routine: one such frame in 200 made a 2048 x 2048 launch 2.3x slower,
    profiles/r2_translate_seed_probe.md); values must not move."""
    rng = np.random.default_rng(w + h)
    shifts = [(-0.99997, 0.4), (3e-05, -1.25), (2.00002, 2.00002), (-1.999985, -0.99997), (0.75, 3e-05), (-0.99997, -1.999985),
              (1.0000001, -2.0000002), (-3.0, 2.0), (0.0, 0.0), (-0.9999999, 0.9999999)]
    mov = rng.integers(0, 65536, (len(shifts), h, w), dtype=np.uint16)
    dx = np.array([s[0] for s in shifts], np.float32)
    dy = np.array([s[1] for s in shifts], np.float32)
    for st in ("nearest", "background"):
        got = to_host(sp.translate_batch(to_dev(mov), to_dev(dx), to_dev(dy), st, 77))
        for k in range(len(shifts)):
            undefined = reference_reads_past_the_buffer(h, w, float(dx[k]), float(dy[k]))
            want = best.translate(mov[k], dx[k], dy[k], st, 77)
            np.testing.assert_array_equal(got[k][~undefined], want[~undefined], err_msg=f"{st} shift {shifts[k]}")
    moved = vio.remove_motion(mov, (-dx).astype(np.float64), (-dy).astype(np.float64), meta_rows=3)
    for k in range(len(shifts)):
        want_k = port.loader_remove_motion(mov[k][: h - 3], -float(dx[k]), -float(dy[k]))
        undefined = reference_reads_past_the_buffer(h - 3, w, float(dx[k]), float(dy[k]))
        np.testing.assert_array_equal(moved[k][: h - 3][~undefined], want_k[~undefined], err_msg=f"motion, shift {shifts[k]}")
        np.testing.assert_array_equal(moved[k][h - 3:], mov[k][h - 3:])


def test_translate_batch_per_frame_shifts_device(best):
    mov = ir_movie(9, 96, 128)
    rng = np.random.default_rng(777)
    dx = rng.uniform(-3, 3, len(mov)).astype(np.float32)
    dy = rng.uniform(-3, 3, len(mov)).astype(np.float32)
    d = to_dev(mov)
    got = to_host(sp.translate_batch(d, to_dev(dx), to_dev(dy), "nearest", 0))
    for t in range(len(mov)):
        np.testing.assert_array_equal(got[t], best.translate(mov[t], dx[t], dy[t], "nearest", 0), err_msg=f"frame {t}")
    # host arrays of shifts, host movie, uniform shift
    got2 = sp.translate_batch(mov, dx, dy, "nearest", 0)
    np.testing.assert_array_equal(got2, got)
    got3 = sp.translate_batch(mov, 1.3, -2.7, "wrap", 0)
    for t in range(len(mov)):
        np.testing.assert_array_equal(got3[t], best.translate(mov[t], 1.3, -2.7, "wrap", 0))


def test_translate_float_dtypes_live(best):
    rng = np.random.default_rng(5)
    for dt in ["float32", "float64", "int32", "uint8", "int64"]:
        img = typed_image(dt, 61, 83, rng)
        for st in STRATEGIES:
            np.testing.assert_array_equal(sp.translate(img, 2.37, -1.61, st, 1), best.translate(img, 2.37, -1.61, st, 1))


def test_translate_identity_and_integer_shift_properties():
    f = ir_frame(512, 640, 33)
    np.testing.assert_array_equal(sp.translate(f, 0, 0, "nearest"), f)
    got = sp.translate(f, 5, -3, "background", background=0)
    want = np.zeros_like(f)
    want[:-3, 5:] = f[3:, :-5]
    np.testing.assert_array_equal(got, want)


# ---------------------------------------------------------------------------------------------
# gaussian
# ---------------------------------------------------------------------------------------------
def test_gaussian_golden(golden):
    """The compiled reference's outputs (the goldens) are within the reference's own rounding bound of the float64
    operation -- that pins the operation to the reference -- and the kernel is within the kernel's bound of it."""
    g = golden["ga_in"]
    for k, s in enumerate(golden["ga_sigmas"]):
        assert_reference_exact(golden[f"ga_{k}"], g, float(s), f"golden sigma {s}")
        assert_gauss_exact(sp.gaussian_filter(g, float(s)), g, float(s), f"sigma {s}")


@pytest.mark.parametrize("sigma", [0.5, 1.0, 2.0])
def test_gaussian_full_frame(sigma):
    f = ir_frame(512, 640, 41)
    assert_gauss_exact(sp.gaussian_filter(f, sigma), f, sigma)
    pair = np.stack([f, f[::-1].copy()])
    d = to_dev(pair)
    got = sp.gaussian_filter_batch(d, sigma).cpu().numpy()  # fused uint16 -> float32 path
    assert_gauss_exact(got, pair, sigma)
    gotf = sp.gaussian_filter_batch(d.view(torch.int16).to(torch.float32), sigma).cpu().numpy()
    np.testing.assert_array_equal(gotf, got)


@pytest.mark.parametrize("shape,sigma", [((37, 53), 1.0), ((5, 7), 1.0), ((3, 3), 2.0), ((40, 56), 4.2), ((64, 128), 3.0),
                                         ((33, 132), 0.5), ((16, 260), 1.5)])
def test_gaussian_odd_shapes_and_large_sigma(shape, sigma):
    rng = np.random.default_rng(6)
    img = (rng.random(shape) * 4000).astype(np.float32)
    assert_gauss_exact(sp.gaussian_filter(img, sigma), img, sigma)


@pytest.mark.parametrize("shape", [(8, 8), (1, 8), (64, 128), (65, 136), (130, 264), (63, 120), (200, 320)])
@pytest.mark.parametrize("sigma", [0.5, 1.0, 1.7, 2.4])
def test_gaussian_tiled_shapes_u16_and_f32(shape, sigma):
    """TMA-tiled kernel (16-byte aligned rows), radius 1..4, uint16 and float32 input, tile edges."""
    rng = np.random.default_rng(61)
    f = rng.integers(0, 16384, shape, dtype=np.uint16)
    assert_gauss_exact(sp.gaussian_filter(f, sigma), f, sigma)
    assert_gauss_exact(sp.gaussian_filter(f.astype(np.float32), sigma), f, sigma, "float32 input")
    got = sp.gaussian_filter_batch(to_dev(np.stack([f, f])), sigma).cpu().numpy()
    assert_gauss_exact(got, np.stack([f, f]), sigma, "batch")


def test_gaussian_randomized():
    """60 random (shape, sigma, dtype) cases through both input types."""
    rng = np.random.default_rng(77 + FUZZ_SEED)
    for case in range(60 * FUZZ_SCALE):
        w = int(rng.choice([8, 12, 16, 40, 64, 128, 132, 136, 200, 264, 7, 33]))
        h = int(rng.integers(1, 140))
        sigma = float(rng.choice([0.3, 0.5, 0.8, 1.0, 1.3, 1.7, 2.0, 2.49, 3.1]))
        if case % 2:
            img = rng.integers(0, 16384, (h, w), dtype=np.uint16)
        else:
            img = (rng.random((h, w)) * 5000 - 1000).astype(np.float32)
        assert_gauss_exact(sp.gaussian_filter(img, sigma), img, sigma, f"case {case}: {h}x{w} {img.dtype}")


def test_gaussian_constant_image_stays_constant():
    img = np.full((512, 640), 1234.0, dtype=np.float32)
    out = sp.gaussian_filter(img, 1.0)
    np.testing.assert_allclose(out, 1234.0, rtol=2e-6)


# ---------------------------------------------------------------------------------------------
# bad pixels
# ---------------------------------------------------------------------------------------------
@pytest.mark.parametrize("k", range(5))
def test_bad_pixels_golden(golden, k):
    first, other = golden[f"bp_{k}_first"], golden[f"bp_{k}_other"]
    bp = sp.BadPixels(first)
    xy, _clamp = sp.bad_pixels_list(bp.handle)
    np.testing.assert_array_equal(xy, golden[f"bp_{k}_xy"])
    np.testing.assert_array_equal(bp.correct(first), golden[f"bp_{k}_first_out"])
    np.testing.assert_array_equal(bp.correct(other), golden[f"bp_{k}_other_out"])


@pytest.mark.parametrize("k", range(5))
def test_bad_pixels_beyond_the_int_product_range(k):
    """Saturated / dead pixels more than 46,340 counts from the median (found by fuzzing): the reference's int product
    wraps; list, clamp and corrected frames must equal the compiled reference's (tests/golden/bp_extreme_golden.npz)."""
    from tests import bp_extreme_cases as bc

    g = np.load(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "bp_extreme_golden.npz"))
    first = bc.frames()[k]
    bp = sp.BadPixels(first)
    xy, _clamp = sp.bad_pixels_list(bp.handle)
    np.testing.assert_array_equal(xy, g[f"xy_{k}"])
    np.testing.assert_array_equal(bp.correct(first), g[f"first_out_{k}"])
    np.testing.assert_array_equal(bp.correct(bc.second_frame(first, k)), g[f"other_out_{k}"])


@pytest.mark.parametrize("shape", [(512, 640), (256, 320), (100, 101), (1, 1), (2, 2), (7, 40)])
def test_bad_pixels_live(port, shape):
    h, w = shape
    first = ir_frame(h, w, 51)
    oxy, _thr, oclamp = port.bad_pixels_detect(first)
    handle = sp.bad_pixels_create(first)
    assert handle > 0
    xy, clamp = sp.bad_pixels_list(handle)
    np.testing.assert_array_equal(xy, oxy)
    assert clamp == oclamp
    mov = np.stack([ir_frame(h, w, 60 + i) for i in range(4)])
    want = np.stack([port.bad_pixels_correct_with(oxy, oclamp, f) for f in mov])
    for t in range(len(mov)):
        np.testing.assert_array_equal(sp.bad_pixels_correct(handle, mov[t]), want[t])
    np.testing.assert_array_equal(to_host(sp.bad_pixels_correct_batch(handle, to_dev(mov))), want)
    np.testing.assert_array_equal(sp.bad_pixels_correct_batch(handle, mov), want)
    sp.bad_pixels_destroy(handle)
    with pytest.raises(RuntimeError):
        sp.bad_pixels_correct(handle, first)


def test_bad_pixels_handles_are_lowest_free_slot():
    f = ir_frame(16, 16, 1)
    a, b, c = (sp.bad_pixels_create(f) for _ in range(3))
    assert len({a, b, c}) == 3 and min(a, b, c) > 0
    sp.bad_pixels_destroy(b)
    assert sp.bad_pixels_create(f) == b
    for h in (a, b, c):
        sp.bad_pixels_destroy(h)


def test_bad_pixels_in_place_is_sequential_like_the_reference(port):
    first = ir_frame(48, 64, 71, n_bad_frac=0.15)  # dense enough that bad pixels touch each other
    oxy, _thr, oclamp = port.bad_pixels_detect(first)
    handle = sp.bad_pixels_create(first)
    lib = _lib.load()
    img = ir_frame(48, 64, 72, n_bad_frac=0.15)
    want = port.bad_pixels_correct_inplace(oxy, oclamp, img)
    assert not np.array_equal(want, port.bad_pixels_correct_with(oxy, oclamp, img)), "case too sparse to tell the two apart"
    got = img.copy()
    assert lib.bad_pixels_correct(handle, sp._ptr(got), sp._ptr(got)) == 0
    np.testing.assert_array_equal(got, want)
    sp.bad_pixels_destroy(handle)


def test_loader_bad_pixels_variant(port):
    mov = np.stack([ir_frame(67, 80, 80 + i) for i in range(3)])
    lb = vio.LoaderBadPixels(mov[0])
    oxy, _, _ = port.bad_pixels_detect(mov[0][:64])
    want = mov.copy()
    for t in range(3):
        want[t, :64] = port.loader_remove_bad_pixels(mov[t, :64], oxy)
    got = lb.remove(mov.copy())
    np.testing.assert_array_equal(got, want)
    np.testing.assert_array_equal(to_host(lb.remove(to_dev(mov))), want)


# ---------------------------------------------------------------------------------------------
# motion-correction variant
# ---------------------------------------------------------------------------------------------
def test_remove_motion_golden_and_live(golden, best, port):
    for k in range(5):
        first = golden[f"bp_{k}_first"]
        h, w = first.shape
        got = vio.remove_motion(first, 1.3, -2.7, meta_rows=0)
        np.testing.assert_array_equal(got, golden[f"bp_{k}_motion"])
    mov = np.stack([ir_frame(67, 80, 90 + i) for i in range(4)])
    sx = np.array([1.3, -0.5, 0.0, 7.25])
    sy = np.array([-2.7, 0.5, 0.0, -3.125])
    want = mov.copy()
    for t in range(4):
        want[t, :64] = best.loader_remove_motion(mov[t, :64], sx[t], sy[t])
    np.testing.assert_array_equal(vio.remove_motion(mov, sx, sy), want)
    d = to_dev(mov)
    np.testing.assert_array_equal(to_host(vio.remove_motion(d, sx, sy, out=d)), want)  # in place


# ---------------------------------------------------------------------------------------------
# statistics
# ---------------------------------------------------------------------------------------------
@pytest.fixture(params=[0, 1], ids=["two_pass", "fused"])
def loader_mode(request):
    """rirb_loader_read_movie as merge pass + motion pass, and as the one-pass fused kernel."""
    _lib.set_parameter("loader_fused", request.param)
    yield request.param
    _lib.set_parameter("loader_fused", 0)


@pytest.mark.parametrize("shape", [(12, 67, 96), (5, 131, 80), (3, 40, 37), (4, 259, 640), (2, 5, 3)])
def test_loader_read_movie_chain(port, best, shape, loader_mode):
    """The reader's post-decode chain in one call (merge -> +min_T -> removeBadPixels -> removeMotion)
    against the restated reference chain, with each stage switched on and off."""
    n, h, w = shape
    rng = np.random.default_rng(91)
    mov = ir_movie(n, h, w, seed=7)
    mov[:, -3:] = rng.integers(0, 65536, (n, 3, w), dtype=np.uint16)  # metadata rows: arbitrary bits
    lo, hi = (mov & 0xFF).astype(np.uint8), (mov >> 8).astype(np.uint8)
    sx = rng.uniform(-3, 3, n)
    sy = rng.uniform(-3, 3, n)
    bp = vio.LoaderBadPixels(mov[0]) if h - 3 >= 1 else None
    xy = sp.bad_pixels_list(bp.handle)[0] if bp is not None else None
    cases = [dict(bad=False, min_T=0, rows=0, motion=False), dict(bad=True, min_T=0, rows=0, motion=False),
             dict(bad=True, min_T=273, rows=h - 3, motion=True), dict(bad=False, min_T=60000, rows=h // 2, motion=True),
             dict(bad=True, min_T=-5, rows=h, motion=False),
             dict(bad=False, min_T=300, rows=0, motion=False)]  # MIN_T_HEIGHT absent: height - 3 (IRFileLoader.cpp:918-921)
    for c in cases:
        if c["bad"] and bp is None:
            continue
        got = vio.read_movie(lo, hi, bp if c["bad"] else None, c["min_T"], c["rows"], sx if c["motion"] else None,
                             sy if c["motion"] else None)
        for t in range(n):
            want = port.loader_read_image(lo[t], hi[t], xy if c["bad"] else None, c["min_T"], c["rows"] if c["rows"] else max(h - 3, 0),
                                          (sx[t], sy[t]) if c["motion"] else None)
            np.testing.assert_array_equal(got[t], want, err_msg=f"{shape} {c} frame {t}")
    # device-resident planes give the same frames
    c = cases[2]
    if bp is not None:
        got_d = to_host(vio.read_movie(to_dev(lo), to_dev(hi), bp, c["min_T"], c["rows"], sx, sy))
        np.testing.assert_array_equal(got_d, vio.read_movie(lo, hi, bp, c["min_T"], c["rows"], sx, sy))


@pytest.mark.parametrize("shape", [(5, 64, 80), (3, 35, 48), (4, 130, 264)])
def test_loader_finish_frames_chain(port, shape):
    """The chain behind load_image of libvideo_io_b200.so (frames already uint16): += min_T -> removeBadPixels -> removeMotion
    in place, host and device frames, every stage on and off -- the same oracle as the plane-fed reader.  (The motion step
    once staged its shifts into the scratch slot that held the frames' copy: the first pixels of frame 0 came back as the
    bits of a float.)"""
    n, h, w = shape
    rng = np.random.default_rng(5)
    mov = ir_movie(n, h, w, seed=11)
    mov[:, -3:] = rng.integers(0, 65536, (n, 3, w), dtype=np.uint16)
    lo, hi = (mov & 0xFF).astype(np.uint8), (mov >> 8).astype(np.uint8)
    sx = rng.uniform(-3, 3, n)
    sy = rng.uniform(-3, 3, n)
    sx[0] = sy[0] = 0.0
    bp = vio.LoaderBadPixels(mov[0])
    xy = sp.bad_pixels_list(bp.handle)[0]
    for c in [dict(bad=False, min_T=0, rows=0, motion=True), dict(bad=True, min_T=273, rows=h - 3, motion=True),
              dict(bad=True, min_T=0, rows=0, motion=False), dict(bad=False, min_T=300, rows=0, motion=False)]:
        want = np.stack([port.loader_read_image(lo[t], hi[t], xy if c["bad"] else None, c["min_T"], c["rows"] if c["rows"] else h - 3,
                                                (sx[t], sy[t]) if c["motion"] else None) for t in range(n)])
        args = (bp if c["bad"] else None, c["min_T"], c["rows"], sx if c["motion"] else None, sy if c["motion"] else None)
        np.testing.assert_array_equal(vio.finish_frames(mov.copy(), *args), want, err_msg=f"{shape} {c} host")
        np.testing.assert_array_equal(to_host(vio.finish_frames(to_dev(mov.copy()), *args)), want, err_msg=f"{shape} {c} device")
        one = mov[1].copy()  # a single frame, as load_image calls it
        args1 = (bp if c["bad"] else None, c["min_T"], c["rows"], sx[1:2] if c["motion"] else None, sy[1:2] if c["motion"] else None)
        np.testing.assert_array_equal(vio.finish_frames(one[None], *args1)[0], want[1], err_msg=f"{shape} {c} one frame")


def test_loader_read_movie_fused_large_shifts_and_edges(port, loader_mode):
    """Fused reader kernel (w % 16 == 0): shifts far beyond the staged box (clamped reads rebuilt from the
    planes, including flagged source pixels), integer shifts, image smaller than a tile, many flagged pixels."""
    rng = np.random.default_rng(17)
    for (n, h, w) in [(6, 70, 160), (4, 35, 16), (3, 200, 272)]:
        mov = ir_movie(n, h, w, seed=3)
        bad = rng.choice(h * w, h * w // 40, replace=False)  # 2.5 % stuck pixels, some adjacent, some on the borders
        mov.reshape(n, -1)[:, bad] = 0
        mov[:, 0, :8] = 0
        mov[:, :, 0] = 16000
        lo, hi = (mov & 0xFF).astype(np.uint8), (mov >> 8).astype(np.uint8)
        bp = vio.LoaderBadPixels(mov[0])
        xy = sp.bad_pixels_list(bp.handle)[0]
        sx = np.array([0.0, 25.5, -30.25, 3.0, -2.0, 1e-7][:n])
        sy = np.array([0.0, -40.75, 19.5, -3.0, 70.0, 0.99999][:n])
        got = vio.read_movie(lo, hi, bp, 1000, h - 3, sx, sy)
        for t in range(n):
            want = port.loader_read_image(lo[t], hi[t], xy, 1000, h - 3, (sx[t], sy[t]))
            np.testing.assert_array_equal(got[t], want, err_msg=f"{(n, h, w)} frame {t} shift {(sx[t], sy[t])}")


def test_loader_read_movie_is_inverse_of_the_writer_split():
    """decode side of the lossless round trip the reference's tests pin (test_IRMovie.py:46-49): planes
    written by the pre-coder, read back by the loader chain with every correction off = the frames."""
    mov = ir_movie(20, 64, 96)
    lo, hi = vio.precode_movie(mov, gop=5, delta=False)
    np.testing.assert_array_equal(vio.read_movie(lo, hi, None), mov)


def test_find_median_pixel_golden(golden):
    f, m = golden["mp_in"], golden["mp_mask"]
    for p, want, want_m in zip(golden["mp_percents"], golden["mp_out"], golden["mp_out_mask"]):
        assert sp.find_median_pixel(f, float(p)) == want
        assert sp.find_median_pixel(f, float(p), m) == want_m


def test_stats_live(port):
    import ctypes as ct

    lib = _lib.load()
    mov = ir_movie(6, 96, 128)
    mov[2, 5, 5] = 60000  # exercises the global-atomic range above the shared-memory bins
    d = to_dev(mov)
    mm = torch.zeros(2, dtype=torch.int32, device="cuda")
    hist = torch.zeros(65536, dtype=torch.int64, device="cuda")
    _lib.use_torch_stream()
    assert lib.rirb_movie_stats(sp._ptr(d[:3]), d[:3].numel(), ct.c_void_p(mm.data_ptr()), ct.c_void_p(hist.data_ptr()), 0) == 0
    assert lib.rirb_movie_stats(sp._ptr(d[3:]), d[3:].numel(), ct.c_void_p(mm.data_ptr()), ct.c_void_p(hist.data_ptr()), 1) == 0
    lo, hi, ohist = port.movie_stats(mov)
    assert (int(mm[0]), int(mm[1])) == (lo, hi)
    np.testing.assert_array_equal(hist.cpu().numpy().astype(np.uint64), ohist)
    for pc in [0.0, 0.1, 0.5, 0.9, 1.0]:
        assert lib.rirb_hist_quantile(ct.c_void_p(hist.data_ptr()), mov.size, pc) == port.quantile_from_hist(ohist, pc)
    for t in range(3):
        assert lib.rirb_get_background(sp._ptr(mov[t]), mov[t].size) == port.get_background(mov[t])
    # host-pointer variant
    mmh = np.zeros(2, np.uint32)
    hh = np.zeros(65536, np.uint64)
    assert lib.rirb_movie_stats(sp._ptr(mov), mov.size, sp._ptr(mmh), sp._ptr(hh), 0) == 0
    assert tuple(mmh) == (lo, hi)
    np.testing.assert_array_equal(hh, ohist)


# ---------------------------------------------------------------------------------------------
# pre-coder
# ---------------------------------------------------------------------------------------------
def test_split_merge_layouts(port):
    rng = np.random.default_rng(5)
    for shape in [(13, 37), (64, 96), (512, 640)]:
        img = rng.integers(0, 65536, shape, dtype=np.uint16)
        it = rng.integers(0, 256, shape, dtype=np.uint8)
        h, w = shape
        for got, want in zip(vio.split_yuv444(img, it), port.split_444(img, it)):
            w_ = want.copy()
            w_[:, w:] = 0  # the oracle marks untouched padding with 0xAA, ours starts from zeros
            np.testing.assert_array_equal(got, w_)
        y, u, v = vio.split_yuv444(img)
        assert not y.any()
        back, _ = vio.merge_yuv444(y, u, v, w)
        np.testing.assert_array_equal(back, img)
        p = vio.split_yuv420(img)
        np.testing.assert_array_equal(p[:h, :w], img & 0xFF)
        np.testing.assert_array_equal(p[h:, :w], img >> 8)
        np.testing.assert_array_equal(vio.merge_yuv420(p, w), img)
        p2, u2 = vio.split_yuv420(img, it)
        np.testing.assert_array_equal(p2, p)
        np.testing.assert_array_equal(u2[:, :w], it)
        back, it_back = vio.merge_yuv420(p2, w, u2)
        np.testing.assert_array_equal(back, img)
        np.testing.assert_array_equal(it_back, it)


def test_split_preserves_row_padding():
    import ctypes as ct

    lib = _lib.load()
    img = np.arange(5 * 7, dtype=np.uint16).reshape(5, 7) * 300
    planes = [np.full((5, 32), 0xAA, np.uint8) for _ in range(3)]
    assert lib.rirb_split_yuv444(sp._ptr(img), None, 7, 5, *(sp._ptr(p) for p in planes), 32, 32, 32) == 0
    for p in planes:
        assert (p[:, 7:] == 0xAA).all()
    np.testing.assert_array_equal(planes[1][:, :7], img & 0xFF)
    np.testing.assert_array_equal(planes[2][:, :7], img >> 8)


@pytest.mark.parametrize("shape", [(23, 20, 28), (12, 64, 96), (7, 5, 3), (120, 32, 48)])
@pytest.mark.parametrize("delta", [False, True])
def test_precode_movie_vs_oracle(port, shape, delta):
    mov = ir_movie(*shape) if shape[1] >= 16 else np.random.default_rng(1).integers(0, 65536, shape, dtype=np.uint16)
    for gop in (5, 50):
        lo, hi = vio.precode_movie(mov, gop, delta)
        olo, ohi = port.precode_movie(mov, gop, delta)
        np.testing.assert_array_equal(lo, olo)
        np.testing.assert_array_equal(hi, ohi)
        np.testing.assert_array_equal(vio.decode_movie(lo, hi, gop, delta), mov)
        d = to_dev(mov)
        dlo, dhi = vio.precode_movie(d, gop, delta)
        np.testing.assert_array_equal(dlo.cpu().numpy(), olo)
        np.testing.assert_array_equal(dhi.cpu().numpy(), ohi)
        assert torch.equal(vio.decode_movie(dlo, dhi, gop, delta).view(torch.int16), d.view(torch.int16))


@pytest.mark.parametrize("shape", [(23, 20, 32), (120, 64, 96), (7, 5, 3), (260, 16, 16)])
@pytest.mark.parametrize("delta", [False, True])
def test_precode_movie_fused_with_stats(port, shape, delta):
    """rirb_precode_movie_stats: the planes of the plain pre-coder and the statistics of rirb_movie_stats, from one
    pass; accumulation over two calls; values above the shared-memory histogram's range; odd sizes (fallback)."""
    from librir_b200 import movie

    rng = np.random.default_rng(12)
    mov = ir_movie(*shape)
    mov[0, 0, 0] = 65535
    mov[-1, -1, -1] = 50000          # beyond the 49,152 shared bins
    mov.reshape(-1)[rng.choice(mov.size, 5, replace=False)] = 0
    d = to_dev(mov)
    st = movie.MovieStats("cuda")
    half = (shape[0] // 2) // 5 * 5
    if half:
        lo_a, hi_a = vio.precode_movie(d[:half], 5, delta, 0, stats=st)
        lo_b, hi_b = vio.precode_movie(d[half:], 5, delta, half, stats=st)
        lo = torch.cat([lo_a, lo_b]).cpu().numpy()
        hi = torch.cat([hi_a, hi_b]).cpu().numpy()
    else:
        lo, hi = (x.cpu().numpy() for x in vio.precode_movie(d, 5, delta, 0, stats=st))
    wlo, whi = port.precode_movie(mov, gop=5, delta=delta)
    np.testing.assert_array_equal(lo, wlo)
    np.testing.assert_array_equal(hi, whi)
    mn, mx, hist = port.movie_stats(mov)
    assert (st.min(), st.max(), st.count) == (mn, mx, mov.size)
    np.testing.assert_array_equal(st.histogram(), hist)


def test_precode_delta_needs_key_frame_aligned_shards():
    mov = ir_movie(10, 16, 16)
    with pytest.raises(RuntimeError):
        vio.precode_movie(mov, gop=5, delta=True, first_frame=3)
    lo, hi = vio.precode_movie(mov, gop=5, delta=True, first_frame=10)
    lo0, hi0 = vio.precode_movie(mov, gop=5, delta=True, first_frame=0)
    np.testing.assert_array_equal(lo, lo0)
    np.testing.assert_array_equal(hi, hi0)


def test_lossless_precoder_frame_by_frame(port):
    mov = ir_movie(7, 32, 40)
    pre = vio.LosslessPrecoder(40, 32, gop=3)
    keys = []
    for f in mov:
        key, y, u, v = pre.add_image(f)
        keys.append(key)
        img, _ = vio.merge_yuv444(y, u, v, 40)  # what the reader gets back: the writer's identity guarantee
        np.testing.assert_array_equal(img, f)
    assert keys == [bool(k) for k in port.key_frames(7, 3)]


# ---------------------------------------------------------------------------------------------
# BASELINE.json full sizes: size-independent properties
# ---------------------------------------------------------------------------------------------
def test_process_movie_host_one_call_equals_the_staged_calls(port, best):
    """rirb_process_movie_host (host frames in, host byte planes out, one C-ABI call, three streams)
    against the per-stage entries and the oracle chain."""
    from librir_b200 import movie

    n, h, w = 230, 64, 96  # several sub-chunks would need a bigger movie; GOP 7 makes ragged tails
    mov = ir_movie(n, h, w)
    rng = np.random.default_rng(5)
    dx = rng.uniform(-3, 3, n).astype(np.float32)
    dy = rng.uniform(-3, 3, n).astype(np.float32)
    bp = sp.BadPixels(mov[0])
    smoothed = np.empty((n, h, w), np.float32)
    for delta in (False, True):
        lo, hi = movie.process_movie_host(bp, mov, dx, dy, 1.0, "nearest", 0, gop=7, delta=delta, first_frame=14, smoothed=smoothed)
        corr = bp.correct_batch(mov)
        reg = sp.translate_batch(corr, dx, dy, "nearest", 0)
        wlo, whi = vio.precode_movie(reg, gop=7, delta=delta, first_frame=14)
        np.testing.assert_array_equal(lo, wlo)
        np.testing.assert_array_equal(hi, whi)
        np.testing.assert_array_equal(smoothed, sp.gaussian_filter_batch(corr, 1.0))
    # against the oracle, frame by frame (delta off: planes are the registered frame's bytes)
    lo, hi = movie.process_movie_host(bp, mov[:6], dx[:6], dy[:6], 1.0, "background", 5, gop=50, delta=False)
    xy, clamp = sp.bad_pixels_list(bp.handle)
    for t in range(6):
        want = best.translate(port.bad_pixels_correct_with(xy, clamp, mov[t]), dx[t], dy[t], "background", 5)
        np.testing.assert_array_equal(lo[t].astype(np.uint16) | (hi[t].astype(np.uint16) << 8), want)
    with pytest.raises(RuntimeError):
        movie.process_movie_host(bp, mov[:2], dx[:2], dy[:2], strategy="noborder")


def test_more_frames_than_one_grid_dimension(port, best):
    """66,000 tiny frames in one call: the translate grid carries the frame index in gridDim.y (<= 65,535),
    so long movies go in several launches; every other kernel folds frames into a 1-D grid."""
    n, h, w = 66000, 8, 16
    rng = np.random.default_rng(8)
    mov = rng.integers(0, 16384, (n, h, w), dtype=np.uint16)
    dx = rng.uniform(-3, 3, n).astype(np.float32)
    dy = rng.uniform(-3, 3, n).astype(np.float32)
    d = to_dev(mov)
    reg = to_host(sp.translate_batch(d, to_dev(dx), to_dev(dy), "nearest", 0))
    sm = sp.gaussian_filter_batch(d, 1.0).cpu().numpy()
    bp = sp.BadPixels(mov[0])
    xy, clamp = sp.bad_pixels_list(bp.handle)
    cor = to_host(bp.correct_batch(d))
    lo, hi = vio.precode_movie(d, gop=50, delta=True)
    back = to_host(vio.decode_movie(lo, hi, gop=50, delta=True))
    np.testing.assert_array_equal(back, mov)
    for t in [0, 1, 65534, 65535, 65536, 65537, n - 1]:
        np.testing.assert_array_equal(reg[t], best.translate(mov[t], dx[t], dy[t], "nearest", 0), err_msg=f"translate frame {t}")
        assert_gauss_exact(sm[t], mov[t], 1.0, f"gaussian frame {t}")
        np.testing.assert_array_equal(cor[t], port.bad_pixels_correct_with(xy, clamp, mov[t]), err_msg=f"bad pixels frame {t}")


def test_lossless_chain_with_host_zstd_round_trip_and_ratio():
    """frames -> GPU pre-coder -> host zstd -> host zstd^-1 -> GPU inverse = frames (the lossless guarantee the
    reference's tests pin, tests/python/test_IRMovie.py:46-49), and the pre-coder earns its keep: byte planes
    compress better than raw frames, the temporal delta better still (SURVEY.md 8c)."""
    from librir_b200 import entropy

    mov = ir_movie(100, 128, 160)
    sizes = {}
    for delta in (False, True):
        chunks = entropy.compress_movie(mov, gop=50, delta=delta, level=3)
        np.testing.assert_array_equal(entropy.decompress_movie(chunks, 128, 160, gop=50, delta=delta), mov)
        sizes[delta] = sum(len(c[2]) + len(c[3]) for c in chunks)
    raw = sum(len(entropy.zstd_compress(mov[a:a + 50], 3)) for a in range(0, 100, 50))
    assert sizes[True] < sizes[False] < raw, (raw, sizes)


def lossy_movie(n, h, w, seed=0):
    """IR-like movie for the lossy pre-conditioner: static background + noise (pixels that freeze), a hot spot
    that moves (pixels that restart), integration-time bits (>> 13) that flip in a patch, metadata rows."""
    rng = np.random.default_rng(seed)
    mov = ir_movie(n, h, w, seed=seed + 1, drift=0.7).astype(np.int64)
    mov[n // 3:, 5:12, 5:20] += 8192          # integration time changes at frame n/3 in a patch
    mov[:, : h // 2] += rng.integers(-1, 2, (n, h // 2, w))
    mov[:, -3:] = rng.integers(0, 65536, (n, 3, w))
    return np.clip(mov, 0, 65535).astype(np.uint16)


@pytest.fixture(params=["one launch per run of frames", "three launches per frame"])
def lossy_driver(request):
    _lib.set_parameter("lossy_run", request.param == "one launch per run of frames")
    yield request.param
    _lib.set_parameter("lossy_run", 1)


@pytest.mark.parametrize("cfg", [dict(), dict(runningAverage=0), dict(runningAverage=5, subtractMin=True),
                                 dict(removeBadPixels=True, lowValueError=12, highValueError=5),
                                 dict(runningAverage=64, subtractMin=True, removeBadPixels=True, stdFactor=2.0)])
@pytest.mark.parametrize("variant", ["add_image_lossy", "add_loss"])
def test_lossy_preconditioner_matches_restated_reference(port, cfg, lossy_driver, variant):
    """rirb_lossy_* against the restatement of addImageLossyNoCamera / addLoss (itself bit-equal to the compiled
    reference, tests/test_oracle_vs_refvio.py), frame by frame and with the state carried across calls: the frozen /
    restarted pixels, the running average ring wrapping, the switch to background-split spreads after 40 frames, the
    smeared window entry, the per-frame error attributes."""
    n, h, w = 90, 43, 64
    mov = lossy_movie(n, h, w)
    stop = h - 3
    st = port.lossy_open(w, h, stop, cfg.get("lowValueError", 6), cfg.get("highValueError", 2), cfg.get("stdFactor", 5.0),
                         cfg.get("runningAverage", 32), cfg.get("subtractMin", False), cfg.get("removeBadPixels", False),
                         variant=int(variant == "add_loss"))
    want, werr = [], []
    for t in range(n):
        o, e = port.lossy_add(st, mov[t])
        want.append(o)
        werr.append(e)
    port.lossy_close(st)
    want, werr = np.stack(want), np.array(werr)
    pre = vio.LossyPreconditioner(w, h, stop, variant=variant, **cfg)
    got_a, err_a = pre.add_images(mov[:37])            # host frames, several calls
    got_b, err_b = pre.add_images(to_dev(mov[37:]))    # device frames
    got = np.concatenate([got_a, to_host(got_b)])
    err = np.concatenate([err_a, err_b])
    np.testing.assert_array_equal(err, werr)
    for t in range(n):
        np.testing.assert_array_equal(got[t], want[t], err_msg=f"{cfg} frame {t}")
    assert (got != mov).any() and (got[:, -3:] == mov[:, -3:]).all()  # something was frozen; metadata rows untouched


def test_full_size_c2_round_trip_and_checksums():
    """640x512x1000 (configs[1]): decode(precode(x)) == x with and without delta, and the byte
    planes carry exactly the movie's bytes (checksum of checksums)."""
    mov = rand_u16((1000, 512, 640), 1234)
    for delta in (False, True):
        lo, hi = vio.precode_movie(mov, 50, delta)
        back = vio.decode_movie(lo, hi, 50, delta)
        assert torch.equal(back.view(torch.int16), mov.view(torch.int16))
        if not delta:
            total = lo.to(torch.int64).sum() + 256 * hi.to(torch.int64).sum()
            assert int(total) == int(as_int(mov).to(torch.int64).sum())
        else:  # key frames are raw, the rest are differences
            raw = (lo[::50].to(torch.int32) | (hi[::50].to(torch.int32) << 8))
            assert torch.equal(raw, as_int(mov[::50]))


def test_full_size_c4_translate_properties():
    """1024x1024 with per-frame shifts (configs[3]): zero shift is the identity, integer shifts
    move pixels exactly, and min/max of a nearest-border translate stay inside the source's."""
    mov = rand_u16((64, 1024, 1024), 777)
    n = mov.shape[0]
    zero = torch.zeros(n, device="cuda")
    assert torch.equal(sp.translate_batch(mov, zero, zero, "nearest", 0).view(torch.int16), mov.view(torch.int16))
    dx = torch.arange(n, device="cuda", dtype=torch.float32) - 32
    out = sp.translate_batch(mov, dx, zero, "background", 0)
    for t in (0, 17, 32, 63):
        s = int(dx[t])
        src = as_int(mov[t])
        want = torch.zeros_like(src)
        if s > 0:
            want[:, s:] = src[:, :-s]
        elif s < 0:
            want[:, :s] = src[:, -s:]
        else:
            want = src
        assert torch.equal(as_int(out[t]), want), f"frame {t} shift {s}"
    fr = torch.rand(n, device="cuda") * 6 - 3
    o2 = as_int(sp.translate_batch(mov, fr, -fr, "nearest", 0))
    assert int(o2.min()) >= int(as_int(mov).min()) and int(o2.max()) <= int(as_int(mov).max())


def test_full_size_pipeline_matches_oracle_on_sampled_frames(port):
    """configs[0]/[2] shape (640x512): the four stages chained on the device, a few frames of the
    chunk checked end to end against the oracle."""
    from librir_b200 import movie

    mov = ir_movie(60, 512, 640)
    cfg = movie.PipelineConfig(chunk_frames=60, gop=50, delta=True, sigma=1.0)
    pipe = movie.FramePipeline(cfg)
    d = to_dev(mov)
    pipe.set_first_frame(d[0])
    rng = np.random.default_rng(777)
    dx = rng.uniform(-3, 3, 60).astype(np.float32)
    dy = rng.uniform(-3, 3, 60).astype(np.float32)
    c, s, r, lo, hi = pipe.process_chunk(d, to_dev(dx), to_dev(dy), first_frame=0)
    oxy, _thr, oclamp = port.bad_pixels_detect(mov[0])
    for t in (0, 1, 49, 50, 59):
        oc = port.bad_pixels_correct_with(oxy, oclamp, mov[t])
        np.testing.assert_array_equal(to_host(c[t]), oc)
        assert_gauss_exact(s[t].cpu().numpy(), oc, 1.0, f"smoothed frame {t}")
        np.testing.assert_array_equal(to_host(r[t]), port.translate(oc, dx[t], dy[t], "nearest", 0))
    reg = to_host(r)
    olo, ohi = port.precode_movie(reg, 50, True)
    np.testing.assert_array_equal(lo.cpu().numpy(), olo)
    np.testing.assert_array_equal(hi.cpu().numpy(), ohi)
    glo, ghi, ghist = port.movie_stats(reg)
    assert (pipe.stats.min(), pipe.stats.max()) == (glo, ghi)
    np.testing.assert_array_equal(pipe.stats.histogram(), ghist)
    assert pipe.stats.quantile(0.5) == port.quantile_from_hist(ghist, 0.5)


def test_handles_refuse_another_device():
    """Handles own memory on the device they were created on; a call from a thread that moved to another device must be
    refused with a message, not fault.  Needs two GPUs (skipped on the single-GPU box)."""
    lib = _lib.load()
    if lib.rirb_device_count() < 2:
        pytest.skip("needs two CUDA devices")
    img = ir_frame(64, 96, 5)
    assert lib.rirb_set_device(0) == 0
    bp = sp.BadPixels(img)
    ecc = lib.rirb_ecc_open(64, 48)
    assert ecc > 0
    try:
        assert lib.rirb_set_device(1) == 0
        with pytest.raises(RuntimeError) as e:
            bp.correct(img)
        assert "belongs to CUDA device 0" in _lib.last_error() or "device" in str(e.value)
        f = np.zeros((48, 64), np.float32)
        assert lib.rirb_ecc_set_image(ecc, 0, sp._ptr(f), 64) == -1 and "belongs to CUDA device 0" in _lib.last_error()
        other = sp.BadPixels(img)  # a handle made here works here
        np.testing.assert_array_equal(other.correct(img), (lib.rirb_set_device(0), bp.correct(img), lib.rirb_set_device(1))[1])
    finally:
        lib.rirb_set_device(0)
        lib.rirb_ecc_close(ecc)


def test_entries_are_reentrant_across_threads(best):
    """ctypes releases the GIL, so the reference's callers may be in several entries at once (SURVEY.md 8b, threading):
    eight threads hammer the per-frame calls -- one shared bad-pixel handle, per-thread scratch -- and every result must
    equal the single-threaded one."""
    import threading

    mov = ir_movie(16, 96, 136)
    bp = sp.BadPixels(mov[0])
    want_c = [bp.correct(f) for f in mov]
    want_t = [sp.translate(f, 1.3 + 0.1 * i, -0.7, "nearest") for i, f in enumerate(mov)]
    want_g = [sp.gaussian_filter(f, 1.0) for f in mov]
    want_q = [sp.find_median_pixel(f, 0.5) for f in mov]
    errors = []

    def work(k):
        try:
            for rep in range(6):
                for i in range(k, len(mov), 4):
                    assert np.array_equal(bp.correct(mov[i]), want_c[i])
                    assert np.array_equal(sp.translate(mov[i], 1.3 + 0.1 * i, -0.7, "nearest"), want_t[i])
                    assert np.array_equal(sp.gaussian_filter(mov[i], 1.0), want_g[i])
                    assert sp.find_median_pixel(mov[i], 0.5) == want_q[i]
                    lo, hi = vio.precode_movie(mov[i:i + 2], gop=1)
                    assert np.array_equal(lo.astype(np.uint16) | (hi.astype(np.uint16) << 8), mov[i:i + 2])
        except Exception as e:  # noqa: BLE001
            errors.append(repr(e))

    threads = [threading.Thread(target=work, args=(k % 4,)) for k in range(8)]
    for t in threads:
        t.start()
    for t in threads:
        t.join()
    assert not errors, errors[:3]


def test_scratch_is_safe_across_a_change_of_stream():
    """Device-pointer calls return without synchronising and the scratch slots belong to the calling thread: a call on
    another stream right behind one that is still running must not overwrite its scratch (in-place motion removal keeps a
    copy of the movie there).  rirb_set_stream makes the new stream wait for the old one."""
    n, h, w = 300, 256, 320
    a = ir_movie(n, h, w, seed=1)
    b = ir_movie(n, h, w, seed=2)
    sx = np.linspace(-2.5, 2.5, n)
    sy = np.linspace(1.5, -1.5, n)
    want_a = to_host(vio.remove_motion(to_dev(a), sx, sy))
    want_b = to_host(vio.remove_motion(to_dev(b), sy, sx))
    s1, s2 = torch.cuda.Stream(), torch.cuda.Stream()
    for _ in range(3):
        da, db = to_dev(a), to_dev(b)
        torch.cuda.synchronize()
        with torch.cuda.stream(s1):
            vio.remove_motion(da, sx, sy, out=da)  # in place: the input's copy lives in the thread's scratch
        with torch.cuda.stream(s2):
            vio.remove_motion(db, sy, sx, out=db)  # same scratch slot, other stream, no synchronisation in between
        torch.cuda.synchronize()
        np.testing.assert_array_equal(to_host(da), want_a)
        np.testing.assert_array_equal(to_host(db), want_b)


def test_short_lived_threads_give_their_device_memory_back():
    """Every calling thread owns a stream, staging buffers and (for the one-call host path) three pipeline slots.  They are
    released when the thread ends -- or on demand with rirb_release_thread_resources() -- so a service that calls from
    short-lived worker threads does not grow (round-1 review: they were never freed)."""
    import threading

    from librir_b200 import movie

    lib = _lib.load()
    mov = ir_movie(40, 256, 320)
    bp = sp.BadPixels(mov[0])
    dx = np.zeros(len(mov), np.float32)
    errors = []

    def work(release_explicitly):
        try:
            sp.gaussian_filter(mov[0], 1.0)
            sp.translate(mov[1], 0.5, 0.25, "nearest")
            movie.process_movie_host(bp, mov, dx, dx, 1.0, "nearest", 0, gop=10, delta=True, first_frame=0)
            if release_explicitly:
                lib.rirb_release_thread_resources()
        except Exception as e:  # noqa: BLE001
            errors.append(repr(e))

    def burst(n, release_explicitly):
        for _ in range(n):
            t = threading.Thread(target=work, args=(release_explicitly,))
            t.start()
            t.join()

    burst(3, False)  # one-time allocations of the process (CUDA context, pools) out of the way
    torch.cuda.synchronize()
    free0 = torch.cuda.mem_get_info()[0]
    burst(12, False)
    burst(12, True)
    torch.cuda.synchronize()
    free1 = torch.cuda.mem_get_info()[0]
    assert not errors, errors[:3]
    per_thread = 3 * 12 * 320 * 256 * 10  # what one thread's host pipeline holds, at the very least
    assert free0 - free1 < 4 * per_thread, f"device memory shrank by {(free0 - free1) / 1e6:.1f} MB over 24 short-lived threads"


@pytest.mark.parametrize("shape", [(5, 64, 128), (3, 200, 264), (4, 70, 136), (2, 5, 8), (3, 130, 640), (2, 33, 20), (2, 64, 127)])
@pytest.mark.parametrize("sigma", [0.5, 1.0, 1.7, 2.2])
def test_bad_pixels_correct_gaussian_fused(port, shape, sigma):
    """rirb_bad_pixels_correct_gaussian_batch = the two separate calls, bit for bit (corrected frames AND filter output):
    tile seams, images smaller than a tile, flagged pixels on borders / in halos / adjacent to each other, a clamp level
    that really clamps, widths off the tiled path (fallback), host and device buffers."""
    n, h, w = shape
    rng = np.random.default_rng(h * w)
    mov = ir_movie(n, h, w, seed=5)
    bad = rng.choice(h * w, max(3, h * w // 25), replace=False)      # 4 % stuck pixels: clusters are common
    mov.reshape(n, -1)[:, bad[: len(bad) // 2]] = 0
    mov.reshape(n, -1)[:, bad[len(bad) // 2:]] = 16000
    mov[:, 0, :] = 0                                                   # a dead first row
    mov[1:, h // 2, : w // 2] = 3000                                   # below the clamp level in later frames
    bp = sp.BadPixels(mov[0])
    want_c = bp.correct_batch(mov)
    want_g = sp.gaussian_filter_batch(want_c, sigma)
    got_c, got_g = bp.correct_gaussian_batch(mov, sigma)
    np.testing.assert_array_equal(got_c, want_c)
    np.testing.assert_array_equal(got_g, want_g)
    oxy, _thr, oclamp = port.bad_pixels_detect(mov[0])
    np.testing.assert_array_equal(got_c[-1], port.bad_pixels_correct_with(oxy, oclamp, mov[-1]))
    d = to_dev(mov)
    dc, dg = bp.correct_gaussian_batch(d, sigma)
    np.testing.assert_array_equal(to_host(dc), want_c)
    np.testing.assert_array_equal(dg.cpu().numpy(), want_g)
