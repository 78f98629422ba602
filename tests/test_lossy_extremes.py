"""The lossy pre-conditioner's restatement (oracle.c, f-2) where the reference's arithmetic is undefined C++: the wrapping
int square of stdDev (h264.cpp:1993-2036) and `error -= (int)round(x)` with x NaN or beyond int range (:2367-2368,
:2559-2563).  Cases: tests/lossy_extreme_cases.py.

* Pinned by compilation: tests/lossy_ref_excerpt.cpp holds those statements in functions of the reference's shape; it is
  compiled here with the reference's flags (g++ -std=c++14 -O3 -DNDEBUG, no -march) and run next to the restatement's
  helpers on edge inputs.  What the compiled code did is printed (pytest -s).
* Live against the compiled saver (oracle/_ref/libs/libvideo_io.so) for every case and both doors, where it is built.
* The counterfactuals -- exact squares, a saturating conversion with NaN -> 0 -- change the bounds of these cases, so a
  later return to either is seen.

No golden file: the project's goldens are written by the compiled reference only, and these cases have not been run
through it yet; the live tests do that wherever oracle/_ref exists."""
import ctypes as ct
import math
import shutil
import subprocess

import numpy as np
import pytest

from oracle import refvio as rv
from tests import lossy_extreme_cases as L
from tests import vio_cases as C
from tests.test_oracle_vs_refvio import run_port_lossy

EXCERPT = __file__.replace("test_lossy_extremes.py", "lossy_ref_excerpt.cpp")
INT_MIN = -(2 ** 31)
CASE_IDS = [c[0] for c in L.CASES]


def case(name):
    return next(c for c in L.CASES if c[0] == name)


@pytest.fixture(scope="module")
def excerpt(tmp_path_factory):
    gxx = shutil.which("g++")
    if gxx is None:
        pytest.skip("g++ not found")
    so = tmp_path_factory.mktemp("excerpt") / "libexcerpt.so"
    subprocess.check_call([gxx, "-std=c++14", "-O3", "-DNDEBUG", "-fPIC", "-shared", EXCERPT, "-o", str(so)])
    lib = ct.CDLL(str(so))
    lib.excerpt_std_dev.restype = None
    lib.excerpt_std_dev.argtypes = [ct.c_void_p, ct.c_void_p, ct.c_int, ct.c_void_p, ct.c_uint, ct.c_void_p]
    for f in (lib.excerpt_bounds_add_image_lossy, lib.excerpt_bounds_add_loss):
        f.restype = None
        f.argtypes = [ct.c_void_p, ct.c_void_p, ct.c_double, ct.c_void_p]
    lib.excerpt_square.restype = ct.c_int
    lib.excerpt_square.argtypes = [ct.POINTER(ct.c_int)]
    lib.excerpt_round_to_int.restype = ct.c_int
    lib.excerpt_round_to_int.argtypes = [ct.POINTER(ct.c_double)]
    return lib


def excerpt_std_dev(lib, prev, img, img_dl=None, back=0):
    prev, img = np.ascontiguousarray(prev, np.uint16), np.ascontiguousarray(img, np.uint16)
    dl = None if img_dl is None else np.ascontiguousarray(img_dl, np.uint16)
    out = np.zeros(2)
    lib.excerpt_std_dev(prev.ctypes.data, img.ctypes.data, img.size, None if dl is None else dl.ctypes.data, back, out.ctypes.data)
    return float(out[0]), float(out[1])


def excerpt_bounds(lib, variant, sd0, sd1, m0, m1, f, low, high):
    e = np.array([low, high], np.int32)
    sd, m = np.array([sd0, sd1]), np.array([m0, m1])
    fn = lib.excerpt_bounds_add_loss if variant else lib.excerpt_bounds_add_image_lossy
    fn(sd.ctypes.data, m.ctypes.data, f, e.ctypes.data)
    return int(e[0]), int(e[1])


def wrapped_square(d):
    """diff * diff modulo 2^32, as a signed 32-bit value"""
    return (d * d + 2 ** 31) % 2 ** 32 - 2 ** 31


def x86_round_to_int(x):
    """(int)round(x) through cvttsd2si: INT_MIN for NaN and for anything outside int range"""
    if math.isnan(x) or math.isinf(x):
        return INT_MIN
    r = math.floor(abs(x) + 0.5) * (1 if x >= 0 else -1)  # round(): half away from zero (exact for doubles this size)
    return int(r) if -(2 ** 31) <= r <= 2 ** 31 - 1 else INT_MIN


def kernel_std_dev(prev, img, img_dl=None, back=0):
    """What the CUDA kernels compute: wrapped squares summed exactly in 64-bit integers, converted to double once."""
    d = np.abs(img.astype(np.int64) - prev.astype(np.int64)).ravel()
    w = (d * d).astype(np.uint32).view(np.int32).astype(np.int64)

    def sd(mask):
        s, s2, n = float(d[mask].sum()), float(w[mask].sum()), int(mask.sum())
        with np.errstate(invalid="ignore", divide="ignore"):
            return float(np.float64(math.sqrt(s * s - s2) if s * s - s2 >= 0 else math.nan) / np.float64(n))

    if img_dl is None:
        v = sd(np.ones(d.size, bool))
        return v, v
    fore = img_dl.ravel().astype(np.int64) > back
    return sd(~fore), sd(fore)


def same(a, b):
    return all((x == y) or (math.isnan(x) and math.isnan(y)) for x, y in zip(a, b))


# ---- pinned by compilation --------------------------------------------------------------------------------------------
def test_compiled_int_square_wraps(excerpt):
    for d in (0, 1, 46339, 46340, 46341, 46342, 50000, 65534, 65535):
        got = excerpt.excerpt_square(ct.byref(ct.c_int(d)))
        print(f"int {d} * {d}: compiled {got}, restatement {wrapped_square(d)}")
        assert got == wrapped_square(d)


def test_compiled_round_to_int_is_cvttsd2si(excerpt):
    xs = [0.0, 2.5, -2.5, 2147483647.0, 2147483647.4, 2147483647.5, 2147483648.0, 2 ** 31 + 1e6, 1e300, math.inf, -math.inf,
          math.nan, -2147483648.0, -2147483648.4, -2147483648.5, -1e300, 4.5e15]
    for x in xs:
        got = excerpt.excerpt_round_to_int(ct.byref(ct.c_double(x)))
        print(f"(int)round({x!r}): compiled {got}, restatement {x86_round_to_int(x)}")
        assert got == x86_round_to_int(x)


def std_dev_inputs():
    z = np.zeros
    yield "one 65535", z(1), np.full(1, 65535), None, 0
    yield "46340 x 9 (exact sums cross 2^31 nine times)", z(9), np.full(9, 46340), None, 0
    yield "46341 x 9 (each square wraps)", z(9), np.full(9, 46341), None, 0
    yield "65535 x 100,000 (the wrapped sum crosses -2^31 and back)", z(100000), np.full(100000, 65535), None, 0
    alt = np.where(np.arange(4000) % 2 == 0, 65535, 46340)
    yield "65535 / 46340 alternating (partial sums swing across +-2^31)", z(4000), alt, None, 0
    noise = np.floor((C.hash_noise((1, 20000), 77)[0] + 0.5) * 65536).clip(0, 65535)
    yield "full-range noise", np.roll(noise, 1), noise, None, 0
    yield "full-range noise, split", np.roll(noise, 1), noise, noise, 32769
    yield "split, foreground empty", z(50), np.full(50, 65535), np.full(50, 8000), 8001
    yield "split, background empty", z(50), np.full(50, 65535), np.full(50, 8002), 8001
    yield "no pixels", z(0), z(0), None, 0


@pytest.mark.parametrize("k", range(10))
def test_compiled_std_dev_equals_the_restatement_and_the_kernel_sums(excerpt, port, k):
    name, prev, img, dl, back = list(std_dev_inputs())[k]
    prev, img = prev.astype(np.uint16), img.astype(np.uint16)
    dl = None if dl is None else dl.astype(np.uint16)
    got = excerpt_std_dev(excerpt, prev, img, dl, back)
    want = port.lossy_std_dev(prev, img, dl, back)
    kern = kernel_std_dev(prev, img, dl, back)
    print(f"stdDev {name}: compiled {got}, restatement {want}, exact 64-bit sum of wrapped squares {kern}")
    assert same(got, want) and same(got, kern)


def bound_inputs():
    nan, inf = math.nan, math.inf
    for sd0, m0 in ((3.0, 1.0), (nan, 2.0), (2.0, nan), (inf, 1.0), (1.0, inf), (-inf, 0.0), (1e10, 0.0), (0.0, 1e10),
                    (5e8, 1.0), (429496729.6, 0.0), (4.3e8, 0.0)):
        for sd1, m1 in ((1.0, 0.5), (nan, 0.0), (2.5, 1.0), (1e10, 0.0)):
            for f in (5.0, 0.5, 1e12, -5.0):
                for low, high in ((6, 2), (40, 20), (0, 0), (2 ** 31 - 1, 2 ** 31 - 2), (-7, -3)):
                    yield sd0, sd1, m0, m1, f, low, high


@pytest.mark.parametrize("variant", [0, 1], ids=list(L.DOORS))
def test_compiled_bound_update_equals_the_restatement(excerpt, port, variant):
    n = 0
    for sd0, sd1, m0, m1, f, low, high in bound_inputs():
        got = excerpt_bounds(excerpt, variant, sd0, sd1, m0, m1, f, low, high)
        want = port.lossy_bounds(variant, sd0, sd1, m0, m1, f, low, high)
        if n < 40 or got != want:
            print(f"{L.DOORS[variant]} sd ({sd0}, {sd1}) mean ({m0}, {m1}) stdFactor {f} errors ({low}, {high}): "
                  f"compiled {got}, restatement {want}")
        assert got == want
        n += 1
    assert n > 800


def test_nan_spread_gives_the_wrapped_bounds(port):
    """x86: NaN -> INT_MIN, so lowError - INT_MIN wraps negative and the bounds close to (0, 0) or (high, high)."""
    nan = math.nan
    assert port.lossy_bounds(0, nan, nan, 1.0, 1.0, 5.0, 6, 2) == (0, 0)
    assert port.lossy_bounds(0, nan, 1.0, 1.0, 1.0, 5.0, 6, 2) == (2, 2)
    assert port.lossy_bounds(1, 1.0, nan, 1.0, 1.0, 5.0, 6, 2) == (6, 0)


# ---- the cases through the restatement --------------------------------------------------------------------------------
def restated(port, name, door, **kw):
    _n, mov, stop, cfg = case(name)
    return run_port_lossy(port, mov, stop, cfg, door, **kw)


EXACT_SQUARES_MATTER = ["blink_46341_default", "blink_46341_no_average", "blink_46341_sub_min", "blink_65535_default",
                        "blink_65535_no_average", "blink_65535_sub_min", "running_average_63", "full_range", "dead_and_saturated_bp"]
NAN_MATTERS = ["saturated_frames", "saturated_frames_bp", "flat_frames_4k0", "flat_frames_4k1", "flat_frames_4k2", "flat_frames_4k3",
               "flat_on_first_split", "flat_movie", "stop_0", "stop_1", "stop_20", "running_average_0"]


@pytest.mark.parametrize("name", EXACT_SQUARES_MATTER)
def test_exact_squares_would_change_the_bounds(port, name):
    changed = 0
    for door in L.DOORS:
        _o, e = restated(port, name, door)
        _o2, e2 = restated(port, name, door, exact_squares=True)
        changed += int((e != e2).any(axis=1).sum())
    assert changed > 0


@pytest.mark.parametrize("name", NAN_MATTERS)
def test_nan_to_zero_would_change_the_bounds(port, name):
    for door in L.DOORS:
        _o, e = restated(port, name, door)
        _o2, e2 = restated(port, name, door, saturating_round=True)
        assert (e != e2).any(axis=1).sum() > 0, door


def test_below_the_wrap_nothing_changes(port):
    """0 <-> 46,340: every square fits an int, so exact squares give the same frames."""
    for door in L.DOORS:
        o, e = restated(port, "blink_46340_default", door)
        o2, e2 = restated(port, "blink_46340_default", door, exact_squares=True)
        assert np.array_equal(e, e2) and np.array_equal(o, o2)


def test_huge_std_factor_closes_the_bounds_either_way(port):
    """|sd - mean| * stdFactor >= 2^31 but finite: x86 (INT_MIN, then a wrap) and a saturating conversion agree on (0, 0)."""
    for name in ("huge_std_factor", "huge_std_factor_noise"):
        for door in L.DOORS:
            o, e = restated(port, name, door)
            o2, e2 = restated(port, name, door, saturating_round=True)
            assert np.array_equal(e, e2) and np.array_equal(o, o2)
            closed = (e[2:] == 0).all(axis=1)  # frame 1: its spread is its own mean
            if door == "add_image_lossy":
                assert closed.all()
            else:  # addLoss leaves a bound at its default when its spread is below the mean; a closed low is raised to high
                low, high = e[2:, 0], e[2:, 1]
                assert closed.any() and ((high == 0) | (high == e[0, 1])).all() and ((low == high) | (low == e[0, 0])).all()


def test_cases_cover_the_window_and_stay_small():
    names = set(CASE_IDS)
    assert len(names) == len(L.CASES)
    for name, mov, stop, cfg in L.CASES:
        t, h, w = mov.shape
        assert 50 <= t <= 120 and h * w <= 64 * 136 and 0 <= stop <= h, name


# ---- live: the compiled saver -----------------------------------------------------------------------------------------
needs_ref = pytest.mark.skipif(not rv.have_ref_vio(), reason="oracle/_ref/libs/libvideo_io.so not built")


@needs_ref
@pytest.mark.parametrize("name", CASE_IDS)
def test_live_extremes_both_doors(port, tmp_path, name):
    _n, mov, stop, cfg = case(name)
    t, h, w = mov.shape
    for door in L.DOORS:
        s = rv.Saver(tmp_path / "l.bin", w, h, stop, **cfg)
        if door == "add_loss":
            ref = np.stack([s.add_loss(f) for f in mov])
        else:
            for i, f in enumerate(mov):
                s.add_image_lossy(f, i)
        lo_e, hi_e = s.low_errors(), s.high_errors()
        s.close()
        if door != "add_loss":
            d = rv.read_stub_file(tmp_path / "l.bin")
            ref = np.stack([r["planes"][1].astype(np.uint16) | (r["planes"][2].astype(np.uint16) << 8) for r in d["records"]])
        outs, errs = run_port_lossy(port, mov, stop, cfg, door)
        assert np.array_equal(errs[:, 0], lo_e) and np.array_equal(errs[:, 1], hi_e), door
        assert np.array_equal(outs, ref), door
