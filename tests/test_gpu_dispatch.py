"""Every kernel the launchers can dispatch to, against the oracle -- and proof of which kernel ran.

Each public entry picks one of several kernels from a ``rirb_set_parameter`` switch, the pointer alignment, the width,
the Gaussian radius and the grid limits.  Freshly allocated buffers are 256-byte aligned and the switches sit at their
defaults, so without this file several instantiations that ship in the library would never run under test.  Every
case here names the kernel it expects (``kernels_run`` reads the launched kernels back from ``torch.profiler``),
checks that the kernel of the other path did NOT run, and compares the result with the oracle and with the default
route (Gaussian: with the float64 operation of tests/gauss_exact.py, within its rounding bound on every pixel).  The
last test checks that the cases together reached every instantiation in ``ALL_KERNELS``.
"""
import contextlib
import re

import numpy as np
import pytest

from tests.conftest import ir_movie
from tests.gauss_exact import assert_gauss_exact
from tests.test_gpu_parity import reference_reads_past_the_buffer, to_dev, to_host

pytestmark = pytest.mark.gpu

torch = pytest.importorskip("torch")

from librir_b200 import _lib, movie, signal_processing as sp, video_io as vio  # noqa: E402
from oracle import oracle as O  # noqa: E402

U16 = "unsigned short"
# the kernel instantiations of libsignal_processing_b200.so that the launchers below choose between (names as
# `cuobjdump -elf` lists them, after kernel_name's normalisation)
ALL_KERNELS = (
    ["bp_correct_kernel<0>", "bp_correct_kernel<1>"]
    + [f"gauss_sep_kernel<{r},{t}>" for r in range(1, 5) for t in ("float", U16)]
    + [f"gauss_tile_kernel<{r},{t},0>" for r in range(1, 5) for t in ("float", U16)]
    + [f"gauss_tile_kernel<{r},{U16},1>" for r in range(1, 5)]
    + [f"gauss_tile_wide_kernel<{r},{t}>" for r in (3, 4) for t in ("float", U16)]
    + ["gauss_generic_kernel<float>", f"gauss_generic_kernel<{U16}>"]
    + ["translate_u16_rows_kernel<0>", "translate_u16_rows_kernel<1>", "translate_u16_tma_kernel<0,0>",
       "translate_u16_tma_kernel<1,0>", "translate_u16_kernel<0>", "translate_u16_kernel<1>", "translate_order_kernel"]
    + ["loader_merge_kernel<0>", "loader_merge_kernel<1>"]
    + ["split_flat_kernel", "split_scalar_kernel", "merge_flat_kernel", "merge_scalar_kernel", "delta_split_kernel",
       "delta_split_scalar_kernel", "delta_merge_kernel", "delta_merge_scalar_kernel", "split_stats_kernel<0>",
       "split_stats_kernel<1>", "movie_stats_kernel<1>"]
)
SEEN = set()  # every kernel any case of this module saw launched


@pytest.fixture(scope="module")
def best():
    return O.best()


# ---------------------------------------------------------------------------------------------
# kernel-name probe
# ---------------------------------------------------------------------------------------------
def kernel_name(name):
    """Demangled kernel name -> `base<args>`: no namespace, return type or parameter list; template arguments without
    spaces after commas, casts such as `(int)3` dropped, booleans as 0 / 1."""
    n = name.replace("(anonymous namespace)::", "")
    depth, end = 0, len(n)
    for i, c in enumerate(n):
        if c == "<":
            depth += 1
        elif c == ">":
            depth -= 1
        elif c == "(" and depth == 0:
            end = i
            break
    base, sep, args = n[:end].strip().partition("<")
    base = base.split()[-1].split("::")[-1] if base.split() else base
    args = re.sub(r"\((?:int|bool|unsigned int|unsigned short|long long)\)", "", args)
    args = re.sub(r"\btrue\b", "1", re.sub(r"\bfalse\b", "0", args))
    args = re.sub(r"\s*,\s*", ",", args).strip()
    return base + (sep + args if sep else "")


def kernels_run(fn):
    """Run fn under the CUDA profiler; return (fn's result, set of normalised kernel names it launched)."""
    from torch.profiler import ProfilerActivity, profile

    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        result = fn()
        torch.cuda.synchronize()
    names = {kernel_name(e.name) for e in prof.events()}
    names = {k for k in names if re.match(r"\w+_kernel(<|$)", k)}
    if not names:
        pytest.fail("the profiler recorded no kernel at all for a launch that runs at least one: the dispatch checks of "
                    "this module would be empty")
    SEEN.update(names)
    return result, names


def expect(names, want, family, what=""):
    """`want` (one name or several) ran, and no other kernel whose name starts with one of `family` did."""
    want = {want} if isinstance(want, str) else set(want)
    fam = {k for k in names if k.startswith(tuple(family))}
    assert want <= names and fam <= want, f"{what}: expected {sorted(want)}, launched {sorted(names)}"


GAUSS = ("gauss_",)
TRANSLATE = ("translate_u16_", "translate_order_kernel")
PRECODE = ("split_", "merge_", "delta_", "movie_stats_kernel")


@pytest.fixture
def switch():
    """switch(name, value) for one case; the defaults (gauss_tma, translate_tma, translate_rows = 1, loader_fused = 0)
    are back when the case ends, whatever happened in it."""
    def set_(name, value):
        _lib.set_parameter(name, value)

    try:
        yield set_
    finally:
        for name in ("gauss_tma", "translate_tma", "translate_rows"):
            _lib.set_parameter(name, 1)
        _lib.set_parameter("loader_fused", 0)


@contextlib.contextmanager
def switched(set_, name, value, default=1):
    set_(name, value)
    try:
        yield
    finally:
        set_(name, default)


# ---------------------------------------------------------------------------------------------
# buffers at a chosen byte offset from an aligned allocation, inside a sentinel-filled backing store
# ---------------------------------------------------------------------------------------------
SENTINEL = 0xA5
TDT = {np.uint8: torch.uint8, np.uint16: torch.uint16, np.float32: torch.float32}


class Placed:
    """A contiguous [n, h, w] view that starts `offset` bytes into a 0xA5-filled device buffer."""

    def __init__(self, shape, dtype, offset, fill=None):
        esz = np.dtype(dtype).itemsize
        assert offset % esz == 0
        self.nbytes = int(np.prod(shape)) * esz
        self.offset = offset
        self.buf = torch.full((offset + self.nbytes + 64,), SENTINEL, dtype=torch.uint8, device="cuda")
        self.t = self.buf[offset: offset + self.nbytes].view(TDT[dtype]).view(*shape)
        if fill is not None:  # byte for byte: no dtype-specific copy kernel involved
            raw = np.ascontiguousarray(fill, dtype=dtype).reshape(-1).view(np.uint8)
            self.buf[offset: offset + self.nbytes].copy_(torch.from_numpy(raw).cuda())
        assert self.t.data_ptr() % 256 == offset % 256

    def untouched_outside(self):
        b = self.buf.cpu().numpy()
        return bool((b[: self.offset] == SENTINEL).all() and (b[self.offset + self.nbytes:] == SENTINEL).all())

    def host(self):
        return to_host(self.t)


def aligned(t, n):
    return t.data_ptr() % n == 0


def tma_ok(t, row_bytes, frame_bytes):
    """tma_compatible (tma.cuh): 16-byte aligned base and strides."""
    return aligned(t, 16) and row_bytes % 16 == 0 and frame_bytes % 16 == 0


def test_profiler_sees_the_library_kernels():
    """Canary: a launch the library certainly makes shows up, under its normalised name."""
    d = to_dev(np.ones((2, 16, 16), np.float32))
    _, names = kernels_run(lambda: sp.gaussian_filter_batch(d, 1.0))
    assert "gauss_tile_kernel<2,float,0>" in names, names
    assert kernel_name("void rirb::gauss_sep_kernel<(int)3, float>(float const*, float*, int)") == "gauss_sep_kernel<3,float>"
    assert kernel_name("void rirb::gauss_tile_kernel<4, unsigned short, (bool)1>(CUtensorMap_st)") == f"gauss_tile_kernel<4,{U16},1>"
    assert kernel_name("rirb::split_flat_kernel(unsigned short const*, unsigned char*)") == "split_flat_kernel"
    assert kernel_name("void rirb::translate_u16_tma_kernel<true, false>(CUtensorMap_st)") == "translate_u16_tma_kernel<1,0>"


# ---------------------------------------------------------------------------------------------
# Gaussian: every instantiation
# ---------------------------------------------------------------------------------------------
def gauss_route(dt, r, w, src, dst, route):
    """The kernel launch_gaussian (gaussian.cu) picks: route = "default", "tile" (gauss_tma = 2) or "sep" (gauss_tma = 0)."""
    t = U16 if dt == np.uint16 else "float"
    esz = np.dtype(dt).itemsize
    if r > 4 or w % 4 or not aligned(dst, 16) or not aligned(src, 16):
        return f"gauss_generic_kernel<{t}>"
    if route == "sep" or (w * esz) % 16:
        return f"gauss_sep_kernel<{r},{t}>"
    if r >= 3 and route == "default":
        return f"gauss_tile_wide_kernel<{r},{t}>"
    return f"gauss_tile_kernel<{r},{t},0>"


GAUSS_SHAPES = [(3, 130, 264), (2, 65, 136), (2, 1, 8), (2, 5, 12), (2, 3, 16), (2, 33, 132), (2, 6, 20), (2, 9, 30)]


@pytest.mark.parametrize("dt", [np.uint16, np.float32], ids=["u16", "f32"])
@pytest.mark.parametrize("sigma", [0.5, 1.0, 1.5, 2.0, 2.6])
@pytest.mark.parametrize("shape", GAUSS_SHAPES, ids=lambda s: "x".join(map(str, s)))
def test_gaussian_every_kernel(dt, sigma, shape):
    """R = max(1, int(2 sigma)) = 1..5 on tile seams, below one tile and below 2R+1 rows; every kernel the launcher
    can pick for the shape: tile, wide, sep (gauss_tma = 0, and uint16 rows that are 8 but not 16 bytes), the first-
    generation tile kernel at R = 3, 4 (gauss_tma = 2) and the generic kernel (misaligned input or output, R > 4)."""
    n, h, w = shape
    r = max(1, int(2 * sigma))
    rng = np.random.default_rng(h * w + r)
    mov = (rng.integers(0, 16384, shape) if dt == np.uint16 else rng.random(shape) * 5000 - 1000).astype(dt)
    d = to_dev(mov)
    esz = np.dtype(dt).itemsize
    default, names = kernels_run(lambda: sp.gaussian_filter_batch(d, sigma))
    expect(names, gauss_route(dt, r, w, d, default, "default"), GAUSS, "default")
    assert_gauss_exact(default.cpu().numpy(), mov, sigma, "default")

    def check(got, what):
        assert_gauss_exact(got, mov, sigma, what)

    for name, value, route in [("gauss_tma", 0, "sep"), ("gauss_tma", 2, "tile")]:
        _lib.set_parameter(name, value)
        try:
            got, names = kernels_run(lambda: sp.gaussian_filter_batch(d, sigma))
        finally:
            _lib.set_parameter(name, 1)
        expect(names, gauss_route(dt, r, w, d, got, route), GAUSS, f"{name}={value}")
        check(got.cpu().numpy(), f"{name}={value}")
    src = Placed(shape, dt, esz, fill=mov)                     # misaligned input
    got, names = kernels_run(lambda: sp.gaussian_filter_batch(src.t, sigma))
    expect(names, gauss_route(dt, r, w, src.t, got, "default"), GAUSS, "misaligned src")
    check(got.cpu().numpy(), "misaligned src")
    out = Placed(shape, np.float32, 4)                         # misaligned output
    _, names = kernels_run(lambda: sp.gaussian_filter_batch(d, sigma, out=out.t))
    expect(names, gauss_route(dt, r, w, d, out.t, "default"), GAUSS, "misaligned out")
    check(out.t.cpu().numpy(), "misaligned out")
    assert out.untouched_outside(), "the filter wrote outside its output view"


def bp_movie(n, h, w, seed):
    rng = np.random.default_rng(seed)
    mov = ir_movie(n, h, w, seed=seed)
    bad = rng.choice(h * w, max(3, h * w // 25), replace=False)
    mov.reshape(n, -1)[:, bad[: len(bad) // 2]] = 0
    mov.reshape(n, -1)[:, bad[len(bad) // 2:]] = 16000
    mov[:, 0, :] = 0
    return mov


@pytest.mark.parametrize("sigma", [0.5, 1.0, 1.5, 2.0])
@pytest.mark.parametrize("shape", [(3, 70, 136), (2, 5, 8), (2, 130, 264)], ids=lambda s: "x".join(map(str, s)))
def test_bad_pixels_correct_gaussian_every_radius(shape, sigma):
    """Fused bad-pixel + Gaussian at R = 1..4 (gauss_tile_kernel<R, u16, 1>), and its fallback when `corrected` or the
    filter output is misaligned: both equal the two separate calls on the same buffers, bit for bit, and the fallback's
    corrected frames equal the fused ones."""
    n, h, w = shape
    r = max(1, int(2 * sigma))
    mov = bp_movie(n, h, w, h * w)
    bp = sp.BadPixels(mov[0])
    d = to_dev(mov)
    (fc, fg), names = kernels_run(lambda: bp.correct_gaussian_batch(d, sigma))
    expect(names, f"gauss_tile_kernel<{r},{U16},1>", GAUSS + ("bp_correct_kernel",), "fused")
    want_c = bp.correct_batch(d)
    want_g = sp.gaussian_filter_batch(want_c, sigma)
    assert torch.equal(fc.view(torch.int16), want_c.view(torch.int16))
    assert torch.equal(fg, want_g)
    assert_gauss_exact(fg.cpu().numpy(), to_host(want_c), sigma, "fused")
    for c_off, g_off in [(2, 0), (0, 4), (16 + 2, 8)]:
        cor, sm = Placed(shape, np.uint16, c_off), Placed(shape, np.float32, g_off)
        _, names = kernels_run(lambda: bp.correct_gaussian_batch(d, sigma, out=cor.t, smoothed=sm.t))
        vec = aligned(cor.t, 32) and (h * w) % 16 == 0
        expect(names, {f"bp_correct_kernel<{int(vec)}>", gauss_route(np.uint16, r, w, cor.t, sm.t, "default")},
               GAUSS + ("bp_correct_kernel",), f"fallback corrected+{c_off} smoothed+{g_off}")
        sep_c, sep_g = Placed(shape, np.uint16, c_off), Placed(shape, np.float32, g_off)
        bp.correct_batch(d, out=sep_c.t)
        sp.gaussian_filter_batch(sep_c.t, sigma, out=sep_g.t)
        assert torch.equal(cor.t.view(torch.int16), sep_c.t.view(torch.int16))
        assert torch.equal(sm.t, sep_g.t)
        assert torch.equal(cor.t.view(torch.int16), want_c.view(torch.int16))
        assert_gauss_exact(sm.t.cpu().numpy(), to_host(want_c), sigma, f"fallback corrected+{c_off} smoothed+{g_off}")
        assert cor.untouched_outside() and sm.untouched_outside(), "a fallback kernel wrote outside its view"


# ---------------------------------------------------------------------------------------------
# uint16 translate: every instantiation
# ---------------------------------------------------------------------------------------------
HARD_SHIFTS = [(0.0, 0.0), (1.3, -2.7), (-2.6, 1.4), (7.5, 0.25), (-8.0, -8.0), (3.999999, 63.5), (-65.25, 64.0),
               (130.5, -129.75), (0.5, 1e-7), (5.0000005, -0.99999994),
               (-4.999999046325684, -14.0), (-7.9999995, 0.0), (-6.999999046325684, -2.654136896133423),
               (-7.9999995, -15.999999), (0.25, -31.999998), (-127.99999, -5.9999995), (-2.9999998, -3.9999998),
               (-0.99997, 0.4), (3e-05, -1.25), (2.00002, 2.00002), (-1.999985, -0.99997), (0.75, 3e-05),
               (1.0000001, -2.0000002), (-0.9999999, 0.9999999)]
TR_SHAPES = [(8, 8), (1, 8), (3, 16), (65, 136), (130, 264), (46, 16), (121, 8), (33, 16), (40, 136), (70, 264), (9, 7),
             (33, 20)]


def translate_want(best, port, mov, dx, dy, st, bg):
    out = []
    for k in range(len(mov)):
        h, w = mov[k].shape
        undefined = reference_reads_past_the_buffer(h, w, float(dx[k]), float(dy[k]))
        want = best.translate(mov[k], dx[k], dy[k], st, bg)
        if undefined.any():  # the reference reads past its buffer there: the restatement's clamp decides
            want = np.where(undefined, port.translate(mov[k], dx[k], dy[k], st, bg), want)
        out.append(want)
    return np.stack(out)


@pytest.mark.parametrize("strategy", ["nearest", "background", "wrap", ""])
@pytest.mark.parametrize("shape", TR_SHAPES, ids=lambda s: "x".join(map(str, s)))
def test_translate_u16_every_kernel(best, port, switch, shape, strategy):
    """Plain translate, one frame per hard shift: the row kernel (default), the row kernel behind the order kernel
    (translate_rows = 2), the first-generation tiled kernel (translate_rows = 0) and the register kernel
    (translate_tma = 0, a misaligned output).  Each equals the oracle, and the default kernel on every pixel."""
    h, w = shape
    rng = np.random.default_rng(h * 7 + w)
    mov = rng.integers(0, 65536, (len(HARD_SHIFTS), h, w), dtype=np.uint16)
    dx = np.array([s[0] for s in HARD_SHIFTS], np.float32)
    dy = np.array([s[1] for s in HARD_SHIFTS], np.float32)
    d, ddx, ddy = to_dev(mov), to_dev(dx), to_dev(dy)
    want = translate_want(best, port, mov, dx, dy, strategy, 77)
    run = lambda **kw: kernels_run(lambda: sp.translate_batch(d, ddx, ddy, strategy, 77, **kw))  # noqa: E731
    default, names = run()
    tiled = w % 8 == 0
    expect(names, "translate_u16_rows_kernel<0>" if tiled else "translate_u16_kernel<0>", TRANSLATE, "default")
    default = to_host(default)
    np.testing.assert_array_equal(default, want, err_msg="default kernel")
    routes = [("translate_rows", 2, {"translate_order_kernel", "translate_u16_rows_kernel<0>"} if tiled else "translate_u16_kernel<0>"),
              ("translate_rows", 0, "translate_u16_tma_kernel<0,0>" if tiled else "translate_u16_kernel<0>"),
              ("translate_tma", 0, "translate_u16_kernel<0>")]
    for name, value, kern in routes:
        with switched(switch, name, value):
            got, names = run()
        expect(names, kern, TRANSLATE, f"{name}={value}")
        np.testing.assert_array_equal(to_host(got), default, err_msg=f"{name}={value} against the default kernel")
    out = Placed(mov.shape, np.uint16, 2, fill=mov if strategy == "" else None)   # "noborder" keeps unwritten pixels
    _, names = run(out=out.t)
    expect(names, "translate_u16_kernel<0>", TRANSLATE, "misaligned out")
    np.testing.assert_array_equal(out.host(), default, err_msg="misaligned out against the default kernel")
    assert out.untouched_outside(), "translate wrote outside its output view"


@pytest.mark.parametrize("shape", [(8, 8), (11, 16), (67, 136), (133, 264), (73, 264), (49, 16), (9, 7), (12, 20)], ids=lambda s: "x".join(map(str, s)))
def test_translate_u16_motion_every_kernel(best, port, switch, shape):
    """The reader's motion variant (u16 -> float -> u16; vio.remove_motion, 3 metadata rows): the row kernel<1>
    (default), the first-generation tiled kernel<1, 0> (translate_rows = 0) and the register kernel<1>
    (translate_tma = 0).  Defined pixels equal the compiled reference, the rest the restatement, every kernel equals
    the default one on every pixel, and the metadata rows pass through."""
    h, w = shape
    hb = h - 3
    rng = np.random.default_rng(h + 11 * w)
    mov = rng.integers(0, 65536, (len(HARD_SHIFTS), h, w), dtype=np.uint16)
    dx = np.array([s[0] for s in HARD_SHIFTS], np.float32)
    dy = np.array([s[1] for s in HARD_SHIFTS], np.float32)
    sx, sy = -dx.astype(np.float64), -dy.astype(np.float64)  # remove_motion translates by (-sx, -sy) in float
    want = mov.copy()
    for k in range(len(mov)):
        undefined = reference_reads_past_the_buffer(hb, w, float(dx[k]), float(dy[k]))
        want[k, :hb] = np.where(undefined, port.loader_remove_motion(mov[k, :hb], sx[k], sy[k]),
                                best.loader_remove_motion(mov[k, :hb], sx[k], sy[k]))
    d = to_dev(mov)
    run = lambda **kw: kernels_run(lambda: vio.remove_motion(d, sx, sy, meta_rows=3, **kw))  # noqa: E731
    default, names = run()
    tiled = w % 8 == 0
    expect(names, {"translate_order_kernel", "translate_u16_rows_kernel<1>"} if tiled else "translate_u16_kernel<1>",
           TRANSLATE, "default")
    default = to_host(default)
    np.testing.assert_array_equal(default, want, err_msg="default kernel")
    for name, value, kern in [("translate_rows", 0, "translate_u16_tma_kernel<1,0>" if tiled else "translate_u16_kernel<1>"),
                              ("translate_tma", 0, "translate_u16_kernel<1>")]:
        with switched(switch, name, value):
            got, names = run()
        expect(names, kern, TRANSLATE, f"{name}={value}")
        np.testing.assert_array_equal(to_host(got), default, err_msg=f"{name}={value} against the default kernel")
    out = Placed(mov.shape, np.uint16, 4)
    _, names = run(out=out.t)
    expect(names, "translate_u16_kernel<1>", TRANSLATE, "misaligned out")
    np.testing.assert_array_equal(out.host(), default)
    assert out.untouched_outside()


# ---------------------------------------------------------------------------------------------
# alignment matrix of the streaming entries
# ---------------------------------------------------------------------------------------------
ALIGN_SHAPES = [(3, 64, 640), (6, 32, 48), (3, 5, 7)]
SHAPE_IDS = ["3x64x640", "6x32x48", "3x5x7"]
U16_OFFSETS = [(0, 0), (2, 0), (4, 0), (8, 0), (16, 0), (0, 2), (0, 4), (0, 8), (0, 16), (2, 16), (16, 8), (4, 2)]
# (movie, lo plane, hi plane) byte offsets: every plane offset 1..15 for lo and for hi, movie offsets cycling
PLANE_OFFSETS = [(0, 0, 0), (2, 0, 0), (16, 0, 0)] + [((0, 2, 4, 8, 16)[k % 5], k, (5 * k) % 16) for k in range(1, 16)]


def pid(o):
    return "+".join(map(str, o))


@pytest.mark.parametrize("shape", ALIGN_SHAPES, ids=SHAPE_IDS)
def test_bad_pixels_and_gaussian_alignment(port, shape):
    """correct_batch, correct_gaussian_batch, gaussian_filter_batch on inputs and outputs misaligned independently:
    bit-identical to the aligned call (Gaussian: within the bound of the float64 operation), the vector kernel exactly
    when the layout allows it, and nothing written outside the output views."""
    n, h, w = shape
    mov = bp_movie(n, h, w, 3 * h + w)
    bp = sp.BadPixels(mov[0])
    oxy, _thr, oclamp = port.bad_pixels_detect(mov[0])
    want_c = np.stack([port.bad_pixels_correct_with(oxy, oclamp, f) for f in mov])
    d = to_dev(mov)
    ref_c = to_host(bp.correct_batch(d))
    np.testing.assert_array_equal(ref_c, want_c)
    for io, oo in U16_OFFSETS:
        src = Placed(shape, np.uint16, io, fill=mov)
        what = f"in+{io} out+{oo}"
        out = Placed(shape, np.uint16, oo)
        _, names = kernels_run(lambda: bp.correct_batch(src.t, out=out.t))
        vec = aligned(src.t, 32) and aligned(out.t, 32) and (h * w) % 16 == 0
        expect(names, f"bp_correct_kernel<{int(vec)}>", ("bp_correct_kernel",), f"correct_batch {what}")
        np.testing.assert_array_equal(out.host(), ref_c, err_msg=f"correct_batch {what}")
        assert out.untouched_outside(), f"correct_batch {what}"

        csrc = Placed(shape, np.uint16, io, fill=want_c)
        gout = Placed(shape, np.float32, oo * 2)
        _, names = kernels_run(lambda: sp.gaussian_filter_batch(csrc.t, 1.0, out=gout.t))
        expect(names, gauss_route(np.uint16, 2, w, csrc.t, gout.t, "default"), GAUSS, f"gaussian {what}")
        assert_gauss_exact(gout.t.cpu().numpy(), want_c, 1.0, f"gaussian {what}")
        assert gout.untouched_outside(), f"gaussian {what}"

        cor, sm = Placed(shape, np.uint16, oo), Placed(shape, np.float32, 2 * io + (4 if oo else 0))
        _, names = kernels_run(lambda: bp.correct_gaussian_batch(src.t, 1.0, out=cor.t, smoothed=sm.t))
        fused = w % 8 == 0 and aligned(sm.t, 16) and aligned(cor.t, 16) and tma_ok(src.t, 2 * w, 2 * h * w)
        if fused:
            kern = {f"gauss_tile_kernel<2,{U16},1>"}
        else:
            kern = {f"bp_correct_kernel<{int(aligned(src.t, 32) and aligned(cor.t, 32) and (h * w) % 16 == 0)}>",
                    gauss_route(np.uint16, 2, w, cor.t, sm.t, "default")}
        expect(names, kern, GAUSS + ("bp_correct_kernel",), f"correct_gaussian {what}")
        np.testing.assert_array_equal(cor.host(), ref_c, err_msg=f"correct_gaussian {what}")
        assert_gauss_exact(sm.t.cpu().numpy(), want_c, 1.0, f"correct_gaussian {what}")
        assert cor.untouched_outside() and sm.untouched_outside(), f"correct_gaussian {what}"


@pytest.mark.parametrize("shape", ALIGN_SHAPES, ids=SHAPE_IDS)
def test_translate_alignment(best, port, shape):
    """translate_batch with input and output misaligned independently: the tiled kernel only on a 16-byte aligned
    input and output, bit-identical to the aligned call and to the oracle."""
    n, h, w = shape
    mov = ir_movie(n, h, w, seed=h + w)
    rng = np.random.default_rng(w)
    dx = rng.uniform(-3, 3, n).astype(np.float32)
    dy = rng.uniform(-3, 3, n).astype(np.float32)
    ddx, ddy = to_dev(dx), to_dev(dy)
    want = translate_want(best, port, mov, dx, dy, "nearest", 0)
    np.testing.assert_array_equal(to_host(sp.translate_batch(to_dev(mov), ddx, ddy, "nearest", 0)), want)
    for io, oo in U16_OFFSETS:
        src, out = Placed(shape, np.uint16, io, fill=mov), Placed(shape, np.uint16, oo)
        _, names = kernels_run(lambda: sp.translate_batch(src.t, ddx, ddy, "nearest", 0, out=out.t))
        tiled = w % 8 == 0 and aligned(out.t, 16) and tma_ok(src.t, 2 * w, 2 * h * w)
        expect(names, "translate_u16_rows_kernel<0>" if tiled else "translate_u16_kernel<0>", TRANSLATE, f"in+{io} out+{oo}")
        np.testing.assert_array_equal(out.host(), want, err_msg=f"in+{io} out+{oo}")
        assert out.untouched_outside(), f"in+{io} out+{oo}"


def split_kernels(mov, lo, hi, npx, nframes, delta):
    """What launch_precode_movie (precode.cu) launches."""
    if delta:
        vec = npx % 16 == 0 and aligned(mov, 32) and aligned(lo, 16) and aligned(hi, 16)
        return {"delta_split_kernel" if vec else "delta_split_scalar_kernel"}
    n = npx * nframes
    if aligned(mov, 32) and aligned(lo, 16) and aligned(hi, 16) and n >= 16:
        return {"split_flat_kernel"} | ({"split_scalar_kernel"} if n % 16 else set())
    return {"split_scalar_kernel"}


def merge_kernels(lo, hi, mov, npx, nframes, delta):
    return {k.replace("split", "merge") for k in split_kernels(mov, lo, hi, npx, nframes, delta)}


@pytest.mark.parametrize("delta", [False, True], ids=["plain", "delta"])
@pytest.mark.parametrize("shape", ALIGN_SHAPES, ids=SHAPE_IDS)
def test_precode_decode_stats_alignment(port, shape, delta):
    """precode_movie with and without stats=, decode_movie and MovieStats.update with the movie and each byte plane
    at its own offset (plane offsets 1..15): planes bit-identical to the aligned call and to the oracle, the round trip
    the identity, the statistics the oracle's; the vector / fused kernel exactly when the layout allows it."""
    n, h, w = shape
    npx = h * w
    gop = 2
    rng = np.random.default_rng(npx)
    mov = rng.integers(0, 65536, shape, dtype=np.uint16)
    mov[0, 0, 0], mov[-1, -1, -1] = 65535, 50000
    wlo, whi = port.precode_movie(mov, gop=gop, delta=delta)
    mn, mx, whist = port.movie_stats(mov)
    d = to_dev(mov)
    alo, ahi = (x.cpu().numpy() for x in vio.precode_movie(d, gop, delta))
    np.testing.assert_array_equal(alo, wlo)
    np.testing.assert_array_equal(ahi, whi)
    for mo, lo_o, hi_o in PLANE_OFFSETS:
        what = f"movie+{mo} lo+{lo_o} hi+{hi_o}"
        src = Placed(shape, np.uint16, mo, fill=mov)
        for with_stats in (False, True):
            lo, hi = Placed(shape, np.uint8, lo_o), Placed(shape, np.uint8, hi_o)
            st = movie.MovieStats("cuda") if with_stats else None
            _, names = kernels_run(lambda: vio.precode_movie(src.t, gop, delta, out=(lo.t, hi.t), stats=st))
            kern = split_kernels(src.t, lo.t, hi.t, npx, n, delta)
            if with_stats:
                if npx % 16 == 0 and aligned(src.t, 32) and aligned(lo.t, 16) and aligned(hi.t, 16):
                    kern = {f"split_stats_kernel<{int(delta)}>"}
                else:
                    kern |= {"movie_stats_kernel<1>"}
            expect(names, kern, PRECODE + ("split_stats_kernel",), f"precode stats={with_stats} {what}")
            np.testing.assert_array_equal(lo.host(), alo, err_msg=f"lo stats={with_stats} {what}")
            np.testing.assert_array_equal(hi.host(), ahi, err_msg=f"hi stats={with_stats} {what}")
            assert lo.untouched_outside() and hi.untouched_outside(), f"precode wrote outside its planes: {what}"
            if with_stats:
                assert (st.min(), st.max(), st.count) == (mn, mx, mov.size), what
                np.testing.assert_array_equal(st.histogram(), whist, err_msg=what)
        # the inverse, planes at the same offsets, movie out at the movie's offset
        plo, phi = Placed(shape, np.uint8, lo_o, fill=wlo), Placed(shape, np.uint8, hi_o, fill=whi)
        back = Placed(shape, np.uint16, mo)
        _, names = kernels_run(lambda: vio.decode_movie(plo.t, phi.t, gop, delta, out=back.t))
        expect(names, merge_kernels(plo.t, phi.t, back.t, npx, n, delta), PRECODE, f"decode {what}")
        np.testing.assert_array_equal(back.host(), mov, err_msg=f"decode {what}")
        assert back.untouched_outside(), f"decode wrote outside its movie: {what}"
        if not delta:  # MovieStats.update once per movie offset is enough
            st = movie.MovieStats("cuda")
            _, names = kernels_run(lambda: st.update(src.t))
            expect(names, "movie_stats_kernel<1>", PRECODE, f"MovieStats.update {what}")
            assert (st.min(), st.max(), st.count) == (mn, mx, mov.size), what
            np.testing.assert_array_equal(st.histogram(), whist, err_msg=what)


@pytest.mark.parametrize("fused", [0, 1], ids=["two_pass", "fused"])
@pytest.mark.parametrize("shape", [(3, 64, 640), (6, 32, 48), (3, 7, 7)], ids=["3x64x640", "6x32x48", "3x7x7"])
def test_read_movie_alignment(port, switch, shape, fused):
    """read_movie (bad pixels, min_T, with and without motion) with lo / hi planes at offsets 1..15 and the output
    misaligned: equal to the restated reader chain; loader_merge_kernel<1> / the one-pass kernel exactly when the
    layout allows them."""
    switch("loader_fused", fused)
    n, h, w = shape
    hb = h - 3
    fpx = h * w
    rng = np.random.default_rng(fpx + fused)
    mov = ir_movie(n, h, w, seed=w)
    mov[:, -3:] = rng.integers(0, 65536, (n, 3, w), dtype=np.uint16)
    wlo, whi = (mov & 0xFF).astype(np.uint8), (mov >> 8).astype(np.uint8)
    bp = vio.LoaderBadPixels(mov[0])
    xy = sp.bad_pixels_list(bp.handle)[0]
    sx, sy = rng.uniform(-3, 3, n), rng.uniform(-3, 3, n)
    want_still = np.stack([port.loader_read_image(wlo[t], whi[t], xy, 273, hb, None) for t in range(n)])
    want_moved = np.stack([port.loader_read_image(wlo[t], whi[t], xy, 273, hb, (sx[t], sy[t])) for t in range(n)])
    for oo, lo_o, hi_o in PLANE_OFFSETS:
        what = f"out+{oo} lo+{lo_o} hi+{hi_o}"
        lo, hi = Placed(shape, np.uint8, lo_o, fill=wlo), Placed(shape, np.uint8, hi_o, fill=whi)
        planes_vec = w % 16 == 0 and aligned(lo.t, 16) and aligned(hi.t, 16) and fpx % 16 == 0
        out = Placed(shape, np.uint16, oo)
        _, names = kernels_run(lambda: vio.read_movie(lo.t, hi.t, bp, 273, hb, out=out.t))
        vec = planes_vec and aligned(out.t, 32)
        expect(names, f"loader_merge_kernel<{int(vec)}>", ("loader_merge_kernel", "translate_u16_"), f"still {what}")
        np.testing.assert_array_equal(out.host(), want_still, err_msg=f"still {what}")
        assert out.untouched_outside(), f"still {what}"

        out = Placed(shape, np.uint16, oo)
        _, names = kernels_run(lambda: vio.read_movie(lo.t, hi.t, bp, 273, hb, sx, sy, out=out.t))
        if fused and planes_vec and hb >= 3 and aligned(out.t, 16):
            kern = {"translate_u16_tma_kernel<1,1>"}
        else:  # merge into an aligned scratch movie, then the motion pass into out
            tiled = w % 8 == 0 and aligned(out.t, 16) and fpx % 8 == 0
            kern = {f"loader_merge_kernel<{int(planes_vec)}>", "translate_u16_rows_kernel<1>" if tiled else "translate_u16_kernel<1>"}
        expect(names, kern, ("loader_merge_kernel", "translate_u16_"), f"moved {what}")
        np.testing.assert_array_equal(out.host(), want_moved, err_msg=f"moved {what}")
        assert out.untouched_outside(), f"moved {what}"


# ---------------------------------------------------------------------------------------------
# more GOPs than one grid dimension
# ---------------------------------------------------------------------------------------------
@pytest.mark.parametrize("with_stats", [False, True], ids=["precode", "precode_stats"])
@pytest.mark.parametrize("offset", [0, 2], ids=["aligned", "misaligned"])
def test_more_gops_than_one_grid_dimension(port, offset, with_stats):
    """140,000 frames of 8 x 16 at GOP 2 with delta on: 70,000 GOPs, more than gridDim.y holds.  The delta split and
    merge go in launches of at most 65,535 GOPs, so every path accepts the movie the fused one does: the planes equal
    the oracle's around GOP 65,535, and decode_movie gives the movie back."""
    n, h, w, gop = 140_000, 8, 16, 2
    rng = np.random.default_rng(140)
    mov = rng.integers(0, 65536, (n, h, w), dtype=np.uint16)
    src = Placed(mov.shape, np.uint16, offset, fill=mov)
    lo, hi = Placed(mov.shape, np.uint8, offset), Placed(mov.shape, np.uint8, offset)
    st = movie.MovieStats("cuda") if with_stats else None
    _, names = kernels_run(lambda: vio.precode_movie(src.t, gop, True, out=(lo.t, hi.t), stats=st))
    if offset == 0:
        kern = {"split_stats_kernel<1>"} if with_stats else {"delta_split_kernel"}
    else:
        kern = {"delta_split_scalar_kernel"} | ({"movie_stats_kernel<1>"} if with_stats else set())
    expect(names, kern, PRECODE + ("split_stats_kernel",), "precode")
    assert lo.untouched_outside() and hi.untouched_outside()
    glo, ghi = lo.host(), hi.host()
    for a, b in [(0, 6), (2 * 65534 - 4, 2 * 65536 + 6), (n - 6, n)]:
        wlo, whi = port.precode_movie(mov[a:b], gop=gop, delta=True)
        np.testing.assert_array_equal(glo[a:b], wlo, err_msg=f"lo frames {a}..{b}")
        np.testing.assert_array_equal(ghi[a:b], whi, err_msg=f"hi frames {a}..{b}")
    if with_stats:
        assert (st.min(), st.max(), st.count) == (int(mov.min()), int(mov.max()), mov.size)
        np.testing.assert_array_equal(st.histogram(), np.bincount(mov.reshape(-1), minlength=65536).astype(np.uint64))
    back = Placed(mov.shape, np.uint16, offset)
    _, names = kernels_run(lambda: vio.decode_movie(lo.t, hi.t, gop, True, out=back.t))
    expect(names, "delta_merge_kernel" if offset == 0 else "delta_merge_scalar_kernel", PRECODE, "decode")
    np.testing.assert_array_equal(back.host(), mov)
    assert back.untouched_outside()


def test_every_dispatched_kernel_was_seen():
    """Runs last: the cases above together launched every instantiation in ALL_KERNELS, so dropping or re-routing a
    case cannot leave a kernel untested without this failing."""
    missing = [k for k in ALL_KERNELS if k not in SEEN]
    assert not missing, f"never launched by this module: {missing}"
