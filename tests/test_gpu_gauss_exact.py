"""Every Gaussian instantiation held to the float64 operation of tests/gauss_exact.py, pixel by pixel.

Each launch names the kernel it expects (``kernels_run`` / ``gauss_route`` of tests/test_gpu_dispatch.py read it back
from ``torch.profiler``), and every output pixel must lie within ``gamma_c S + c 2**-149 / N`` of the exact value,
c(R) = 4(2R + 1) + 8: a bar that sees one count of one input pixel, where the former frame-relative tolerance did
not.  Cases: sigma around every radius threshold and up to radius 64, images no larger than the kernel, tile and strip
edges, widths off the vector paths, misaligned buffers, the frame sizes of the benchmark, many frames per launch,
IR / uniform / mixed-sign / wide-range / zero / subnormal / non-finite content, the fused correction + Gaussian with
flagged pixels in the tile halos, and the pipeline's smoothed frames.  The last test fails if one of the 26 Gaussian
instantiations never ran, and prints the worst error each one made, in units of u S.
"""
import numpy as np
import pytest

from tests import gauss_exact as G
from tests.conftest import ir_frame, ir_movie
from tests.test_gpu_dispatch import ALL_KERNELS, GAUSS, U16, Placed, expect, gauss_route, kernels_run
from tests.test_gpu_parity import FUZZ_SCALE, FUZZ_SEED, to_dev, to_host

pytestmark = pytest.mark.gpu

torch = pytest.importorskip("torch")

from librir_b200 import _lib, movie, signal_processing as sp  # noqa: E402

GAUSS_KERNELS = [k for k in ALL_KERNELS if k.startswith("gauss_")]
SEEN = set()
WORST = {}  # kernel -> largest error seen, in units of u S
ROUTES = {"default": 1, "sep": 0, "tile": 2}  # "gauss_tma" switch value of each route


# ---------------------------------------------------------------------------------------------
# contents
# ---------------------------------------------------------------------------------------------
def ir_stack(n, h, w, seed):
    """IR frames with pixels stuck at 0 and at 65535."""
    rng = np.random.default_rng(seed)
    mov = np.stack([ir_frame(h, w, seed + i) for i in range(n)])
    idx = rng.choice(h * w, min(h * w, max(2, h * w // 200)), replace=False)
    mov.reshape(n, -1)[:, idx[: len(idx) // 2]] = 0
    mov.reshape(n, -1)[:, idx[len(idx) // 2:]] = 65535
    return mov


def content(kind, shape, seed):
    """[n, h, w] frames of one kind of content: uint16 for "ir" / "uniform", float32 otherwise."""
    rng = np.random.default_rng(seed)
    n, h, w = shape
    if kind == "ir":
        return ir_stack(n, h, w, seed)
    if kind == "uniform":
        return rng.integers(0, 65536, shape).astype(np.uint16)
    if kind == "mixed":
        return (rng.normal(0, 1000, shape) + rng.choice([-4000.0, 4000.0], shape)).astype(np.float32)
    if kind == "wide":
        return (np.exp(rng.uniform(np.log(1e-3), np.log(1e5), shape)) * rng.choice([-1.0, 1.0], shape)).astype(np.float32)
    if kind == "zeros":
        return np.zeros(shape, np.float32)
    if kind == "blocks":  # 8 x 8 blocks of zeros next to blocks of 1e5
        y, x = np.mgrid[0:h, 0:w]
        return np.broadcast_to((((y // 8 + x // 8 + seed) % 2) * 1e5).astype(np.float32), shape).copy()
    if kind == "subnormal":  # subnormals, some next to normal values of the same and of much larger size
        x = rng.uniform(-1, 1, shape) * 2.0 ** -126 * np.exp2(-rng.integers(0, 24, shape))
        x[rng.random(shape) < 0.05] = 1.0
        return x.astype(np.float32)
    raise ValueError(kind)


U16_KINDS = ["ir", "uniform"]
F32_KINDS = ["mixed", "wide", "blocks", "subnormal"]


def kinds(dt):
    return U16_KINDS if dt == np.uint16 else F32_KINDS


# ---------------------------------------------------------------------------------------------
# launching and checking
# ---------------------------------------------------------------------------------------------
def note(kernel, worst):
    WORST[kernel] = max(WORST.get(kernel, 0.0), worst)


def filter_all(cases, sigma, route="default"):
    """cases: [(what, device frames [n, h, w], host frames, output tensor or None)].  The cases are grouped by the
    kernel gauss_route expects and each group runs under one profiler session with "gauss_tma" set for `route`; every
    output is held to the bound.  Returns [(what, kernel, host output)]."""
    groups = {}
    for what, src, img, out in cases:
        if out is None:
            out = torch.empty(tuple(src.shape), dtype=torch.float32, device="cuda")
        dt = np.uint16 if src.dtype == torch.uint16 else np.float32
        kern = gauss_route(dt, G.radius(sigma), src.shape[2], src, out, route)
        groups.setdefault(kern, []).append((what, src, img, out))
    done = []
    for kern, grp in groups.items():
        _lib.set_parameter("gauss_tma", ROUTES[route])
        try:
            _, names = kernels_run(lambda: [sp.gaussian_filter_batch(src, float(sigma), out=out) for _, src, _, out in grp])
        finally:
            _lib.set_parameter("gauss_tma", 1)
        SEEN.update(names)
        expect(names, kern, GAUSS, f"sigma {sigma!r} route {route}: {[g[0] for g in grp]}")
        for what, _src, img, out in grp:
            got = out.cpu().numpy()
            note(kern, G.assert_gauss_exact(got, img, sigma, f"{kern}, {what}, sigma {sigma!r}, route {route}"))
            done.append((what, kern, got))
    return done


def every_route(cases, sigma, misaligned=True):
    """The cases through each route the launcher has at this radius, then with the input and with the output one
    element off a 16-byte boundary (generic kernel; nothing written outside the output view)."""
    r = G.radius(sigma)
    for route in (("default", "sep", "tile") if r <= 4 else ("default",)):
        filter_all(cases, sigma, route)
    if not misaligned:
        return
    shifted, outs = [], []
    for what, src, img, _out in cases:
        dt = np.uint16 if src.dtype == torch.uint16 else np.float32
        s = Placed(tuple(src.shape), dt, np.dtype(dt).itemsize, fill=img)
        o = Placed(tuple(src.shape), np.float32, 4)
        outs.append(o)
        shifted += [(f"{what}, src+{np.dtype(dt).itemsize}", s.t, img, None), (f"{what}, out+4", src, img, o.t)]
    filter_all(shifted, sigma)
    assert all(o.untouched_outside() for o in outs), "the filter wrote outside its output view"


def dev_cases(shapes, dt, seed, n=2):
    cases = []
    for i, (h, w) in enumerate(shapes):
        kind = kinds(dt)[i % len(kinds(dt))]
        img = content(kind, (n, h, w), seed + 7 * i)
        cases.append((f"{kind} {n}x{h}x{w}", to_dev(img), img, None))
    return cases


# ---------------------------------------------------------------------------------------------
# sigma grid: radius thresholds, large radii, images no larger than the kernel
# ---------------------------------------------------------------------------------------------
@pytest.mark.parametrize("dt", [np.uint16, np.float32], ids=["u16", "f32"])
@pytest.mark.parametrize("sigma", G.SIGMAS)
def test_sigma_grid_small_images(dt, sigma):
    """h, w in {1, 2, 2R, 2R + 1, 2R + 2} and two medium frames, at every sigma of the grid (one float32 ulp either
    side of each radius threshold k / 2 included, so that both kernels of an R -> R + 1 step run), every route."""
    r = G.radius(sigma)
    sizes = sorted({1, 2, 2 * r, 2 * r + 1, 2 * r + 2})
    shapes = [(h, w) for h in sizes for w in sizes] + [(70, 136), (33, 132)]
    every_route(dev_cases(shapes, dt, seed=r * 100), sigma)


def test_radius_65_is_refused():
    d = to_dev(np.ones((1, 8, 8), np.float32))
    sp.gaussian_filter_batch(d, 32.499998)  # radius 64: the largest there is
    with pytest.raises(RuntimeError, match="radius 65"):
        sp.gaussian_filter_batch(d, 32.5)


# ---------------------------------------------------------------------------------------------
# tile and strip edges, widths off the vector paths
# ---------------------------------------------------------------------------------------------
EDGE_W = [127, 128, 129, 255, 256, 257]
EDGE_H = [31, 32, 33, 63, 64, 65, 127, 128, 129]


@pytest.mark.parametrize("dt", [np.uint16, np.float32], ids=["u16", "f32"])
@pytest.mark.parametrize("sigma", [0.5, 1.0, 1.7, 2.49])
def test_tile_and_strip_edges(dt, sigma):
    """128-column tiles and strips, 64- and 128-row tiles at R = 1..4; widths with w % 4 != 0 (generic) and
    w % 8 == 4 (uint16 rows of 8 but not 16 bytes: the strip kernel)."""
    shapes = [(h, w) for w in EDGE_W for h in EDGE_H] + [(h, w) for w in (6, 12, 20, 130, 132, 260) for h in (33, 65)]
    every_route(dev_cases(shapes, dt, seed=int(sigma * 10)), sigma, misaligned=False)


# ---------------------------------------------------------------------------------------------
# float32 contents, non-finite values
# ---------------------------------------------------------------------------------------------
@pytest.mark.parametrize("sigma", [0.5, 1.0, 1.7, 2.49, 5.0])
def test_float_contents(sigma):
    """Mixed sign, |x| from 1e-3 to 1e5, zeros (exactly 0 out), 8 x 8 blocks of 0 next to 1e5, subnormals."""
    cases = []
    for kind in F32_KINDS + ["zeros"]:
        for shape in [(3, 130, 264), (2, 33, 20)]:
            img = content(kind, shape, seed=len(cases))
            cases.append((f"{kind} {shape}", to_dev(img), img, None))
    every_route(cases, sigma)
    for route in ROUTES:
        for what, _kern, got in filter_all([c for c in cases if c[0].startswith("zeros")], sigma, route):
            assert not got.any(), f"{what}: zeros in, not zeros out"


def non_finite_frames(h, w, seed):
    """Mixed-sign frames with NaN / +Inf / -Inf at the borders, the tile and strip seams and inside; the third frame
    puts +Inf and -Inf into one window."""
    img = content("mixed", (3, h, w), seed)
    spots = [(0, 0), (0, w - 1), (h - 1, 5), (h // 2, 0), (h // 2, w - 1), (h - 1, w - 1), (63, 127), (64, 128),
             (127, 40), (128, 131), (40, 255), (90, 256), (33, 33)]
    for k, (y, x) in enumerate(spots):
        if y < h and x < w:
            img[0, y, x] = np.inf
            img[1, y, x] = (np.nan, -np.inf)[k % 2]
            img[2, y, x] = (np.inf, -np.inf)[k % 2]
    img[2, 20, 20], img[2, 21, 22] = np.inf, -np.inf
    return img


@pytest.mark.parametrize("sigma", [0.05, 0.5, 1.0, 1.7, 2.49, 5.0])
def test_non_finite(sigma):
    """The non-finite output pixels and the sign of each infinity equal the float64 operation's (sigma 0.05: the outer
    taps are 0, and 0 * Inf = NaN); the finite ones are within the bound."""
    cases = []
    for h, w in [(130, 264), (70, 136)]:
        img = non_finite_frames(h, w, h + w)
        cases.append((f"non-finite {h}x{w}", to_dev(img), img, None))
    every_route(cases, sigma)


# ---------------------------------------------------------------------------------------------
# benchmark frame sizes, many frames per launch
# ---------------------------------------------------------------------------------------------
@pytest.mark.parametrize("sigma", [1.0, 2.49])
def test_benchmark_frame_sizes(sigma):
    """640 x 512 and the frame-size sweep's sizes, 320 x 256 to 2048 x 2048, a few frames each."""
    cases = []
    for n, h, w in [(4, 512, 640), (3, 256, 320), (2, 1024, 1024), (2, 1024, 1280), (2, 2048, 2048)]:
        img = ir_stack(n, h, w, seed=h + w)
        cases.append((f"ir {n}x{h}x{w}", to_dev(img), img, None))
    f = content("mixed", (2, 512, 640), 5)
    cases.append(("mixed 2x512x640", to_dev(f), f, None))
    filter_all(cases, sigma)
    filter_all(cases[:2], sigma, "sep")


@pytest.mark.parametrize("route", ["default", "sep", "tile"])
def test_many_frames_per_launch(route):
    cases = []
    for n, h, w, kind in [(3000, 8, 16, "ir"), (400, 33, 132, "uniform"), (1500, 12, 24, "mixed"), (200, 65, 136, "wide")]:
        img = content(kind, (n, h, w), n)
        cases.append((f"{kind} {n}x{h}x{w}", to_dev(img), img, None))
    for sigma in (1.0, 1.7):
        filter_all(cases, sigma, route)


# ---------------------------------------------------------------------------------------------
# randomised cases (RIRB_FUZZ_SEED / RIRB_FUZZ_SCALE)
# ---------------------------------------------------------------------------------------------
def test_random_cases():
    """Random shape, sigma (the grid and uniform ones), content, route and alignment."""
    rng = np.random.default_rng(4242 + FUZZ_SEED)
    for case in range(40 * FUZZ_SCALE):
        dt = (np.uint16, np.float32)[case % 2]
        sigma = float(np.float32(rng.choice(G.SIGMAS[:-1]) if rng.random() < 0.5 else rng.uniform(0.2, 6.0)))
        h, w = int(rng.integers(1, 200)), int(rng.choice([int(rng.integers(1, 300)), 8 * int(rng.integers(1, 40))]))
        n = int(rng.integers(1, 5))
        kind = kinds(dt)[int(rng.integers(0, len(kinds(dt))))]
        img = content(kind, (n, h, w), int(rng.integers(0, 1 << 30)))
        what = f"case {case}: {kind} {n}x{h}x{w}"
        if rng.random() < 0.25:
            src = Placed((n, h, w), dt, np.dtype(dt).itemsize, fill=img).t
            what += " misaligned src"
        else:
            src = to_dev(img)
        filter_all([(what, src, img, None)], sigma, str(rng.choice(list(ROUTES))))


# ---------------------------------------------------------------------------------------------
# fused bad-pixel correction + Gaussian
# ---------------------------------------------------------------------------------------------
def halo_movie(n, h, w, r, seed):
    """IR frames whose first frame flags pixels in the halo rows and columns of the 128 x 64 tiles (single pixels at
    distance 0..R of every seam, fully flagged 3 x 3 clusters on the seams and in the image's corners) and whose later
    frames put pixels below the clamp level into the same halos."""
    rng = np.random.default_rng(seed)
    mov = ir_movie(n, h, w, seed=seed)
    stuck = np.zeros((h, w), bool)
    seams_x = [x for x in range(128, w, 128)]
    seams_y = [y for y in range(64, h, 64)]
    for sx in seams_x:
        for d in range(-r - 1, r + 1):
            stuck[rng.integers(0, h, 3), sx + d] = True
    for sy in seams_y:
        for d in range(-r - 1, r + 1):
            stuck[sy + d, rng.integers(0, w, 3)] = True
    ys, xs = np.nonzero(stuck)
    mov[:, ys, xs] = np.where(rng.random(len(ys)) < 0.5, 0, 16000).astype(np.uint16)
    centres = [(sy, sx) for sy in seams_y for sx in seams_x] + [(sy - 1, 127) for sy in seams_y] + [(1, 1), (h - 2, w - 2)]
    for cy, cx in centres:  # dead clusters: below the frame's global threshold, so flagged in full
        stuck[max(0, cy - 1): cy + 2, max(0, cx - 1): cx + 2] = True
        mov[:, max(0, cy - 1): cy + 2, max(0, cx - 1): cx + 2] = 0
    for sy in seams_y:  # below the clamp level, not flagged (frame 0 keeps its background there)
        mov[1:, sy - r: sy + r, : w // 2] = np.where(stuck[sy - r: sy + r, : w // 2], mov[1:, sy - r: sy + r, : w // 2], 3000)
    return mov, centres


@pytest.mark.parametrize("sigma", [0.5, 1.0, 1.7, 2.49])
def test_fused_correction_gaussian_halos(port, sigma):
    """gauss_tile_kernel<R, u16, 1>: `corrected` equals the oracle's correction bit for bit, `smoothed` is within the
    bound of the operation on the oracle-corrected frames.  A slightly wrong median or a missing clamp in a tile's halo
    moves the smoothed output by a fraction of a count, which this bar sees."""
    r = G.radius(sigma)
    n, h, w = 3, 200, 392
    mov, centres = halo_movie(n, h, w, r, seed=r)
    oxy, _thr, oclamp = port.bad_pixels_detect(mov[0])
    assert oclamp > 3000, "the case needs a clamp level that clamps"
    flagged = {(int(x), int(y)) for x, y in np.asarray(oxy).reshape(-1, 2)}
    for cy, cx in centres:  # every 3 x 3 cluster is flagged in full
        assert all((x, y) in flagged for x in range(max(0, cx - 1), cx + 2) for y in range(max(0, cy - 1), cy + 2)), (cy, cx)
    want_c = np.stack([port.bad_pixels_correct_with(oxy, oclamp, f) for f in mov])
    assert (want_c == oclamp).sum() > 50, "the clamp must act on the case"
    bp = sp.BadPixels(mov[0])
    d = to_dev(mov)
    (c, s), names = kernels_run(lambda: bp.correct_gaussian_batch(d, sigma))
    SEEN.update(names)
    kern = f"gauss_tile_kernel<{r},{U16},1>"
    expect(names, kern, GAUSS + ("bp_correct_kernel",), "fused")
    np.testing.assert_array_equal(to_host(c), want_c)
    note(kern, G.assert_gauss_exact(s.cpu().numpy(), want_c, sigma, f"{kern} smoothed"))


# ---------------------------------------------------------------------------------------------
# the bar sees a one-count error on the kernels' own output
# ---------------------------------------------------------------------------------------------
@pytest.mark.parametrize("sigma", [1.0, 1.7, 2.49])
def test_resolving_power_on_device_output(sigma):
    img = ir_frame(70, 136, 9)[None]
    y, x = 12, 20
    assert 7900 < img[0, y, x] < 8100
    moved = img.astype(np.float64)
    moved[0, y, x] += 1
    for route in ROUTES:
        (_what, kern, got), = filter_all([("ir", to_dev(img), img, None)], sigma, route)
        with pytest.raises(AssertionError, match="outside the bound"):
            G.assert_gauss_exact(got, moved, sigma, f"{kern} against the frame with one count added")


# ---------------------------------------------------------------------------------------------
# the pipeline's smoothed frames
# ---------------------------------------------------------------------------------------------
def test_pipeline_chunk_every_frame(port):
    """FramePipeline.process_chunk: every smoothed frame of a 200-frame 640 x 512 chunk against the operation on
    the oracle-corrected frame."""
    n, h, w = 200, 512, 640
    mov = ir_movie(n, h, w)
    cfg = movie.PipelineConfig(chunk_frames=n, gop=50, delta=True, sigma=1.0)
    pipe = movie.FramePipeline(cfg)
    d = to_dev(mov)
    pipe.set_first_frame(d[0])
    dx = torch.zeros(n, device="cuda")
    c, s, _r, _lo, _hi = pipe.process_chunk(d, dx, dx, first_frame=0)
    oxy, _thr, oclamp = port.bad_pixels_detect(mov[0])
    got_c, got_s = to_host(c), s.cpu().numpy()
    for a in range(0, n, 25):
        want_c = np.stack([port.bad_pixels_correct_with(oxy, oclamp, f) for f in mov[a:a + 25]])
        np.testing.assert_array_equal(got_c[a:a + 25], want_c)
        G.assert_gauss_exact(got_s[a:a + 25], want_c, 1.0, f"process_chunk frames {a}..{a + 24}")


def test_process_movie_host_smoothed(port):
    n, h, w = 60, 256, 320
    mov = ir_movie(n, h, w, seed=3)
    bp = sp.BadPixels(mov[0])
    smoothed = np.empty((n, h, w), np.float32)
    dx = np.zeros(n, np.float32)
    movie.process_movie_host(bp, mov, dx, dx, 1.7, "nearest", 0, gop=10, delta=True, first_frame=0, smoothed=smoothed)
    oxy, _thr, oclamp = port.bad_pixels_detect(mov[0])
    want_c = np.stack([port.bad_pixels_correct_with(oxy, oclamp, f) for f in mov])
    G.assert_gauss_exact(smoothed, want_c, 1.7, "process_movie_host smoothed")


# ---------------------------------------------------------------------------------------------
def test_every_gaussian_kernel_was_seen():
    """Runs last: the cases above launched all 26 Gaussian instantiations.  Prints the worst error of each."""
    assert len(GAUSS_KERNELS) == 26
    print()
    for k in GAUSS_KERNELS:
        bound = "c(R) = 4(2R+1)+8" if "generic" in k else f"c(R) = {G.c_of(int(k.split('<')[1].split(',')[0]))}"
        print(f"{k:40s} worst {WORST.get(k, float('nan')):6.2f} u S   ({bound})")
    missing = [k for k in GAUSS_KERNELS if k not in SEEN]
    assert not missing, f"never launched by this module: {missing}"
