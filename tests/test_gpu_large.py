"""Parity at the large frame sizes of BASELINE.json's config 5 (1280x1024, 2048x2048), every kernel of the path, through
the C ABI against the compiled reference (oracle/_ref) where it has the function and the C restatement otherwise: a few
frames bit for bit (Gaussian: within the rounding bound of the float64 operation, tests/gauss_exact.py), plus size-independent properties on a longer stack (round trips, identity shifts,
statistics against torch)."""
import numpy as np
import pytest

from tests.conftest import ir_frame
from tests.gauss_exact import assert_gauss_exact

pytestmark = pytest.mark.gpu

torch = pytest.importorskip("torch")

from librir_b200 import movie, signal_processing as sp, video_io as vio  # noqa: E402
from oracle import oracle as O  # noqa: E402

SIZES = [(1024, 1280), (2048, 2048)]  # (h, w)


def to_dev(a):
    if a.dtype == np.uint16:
        return torch.from_numpy(a.view(np.int16)).cuda().view(torch.uint16)
    return torch.from_numpy(a).cuda()


def to_host(t):
    return t.cpu().view(torch.int16).numpy().view(np.uint16) if t.dtype == torch.uint16 else t.cpu().numpy()


@pytest.fixture(scope="module", params=SIZES, ids=[f"{w}x{h}" for h, w in SIZES])
def stack(request):
    h, w = request.param
    rng = np.random.default_rng(h + w)
    base = ir_frame(h, w, seed=h)
    frames = np.stack([np.clip(base.astype(np.int32) + rng.integers(-6, 7, base.shape), 0, 65535).astype(np.uint16) for _ in range(3)])
    stuck = base == 0
    frames[:, stuck] = 0
    frames[:, base == 16000] = 16000
    return frames


def test_bad_pixels_detect_and_correct(stack, port):
    best = O.best()
    bp = sp.BadPixels(stack[0])
    xy, clamp = sp.bad_pixels_list(bp.handle)
    oxy, _thr, oclamp = port.bad_pixels_detect(stack[0])
    assert np.array_equal(xy, oxy) and clamp == oclamp
    if isinstance(best, O.Ref):  # the compiled badPixels<u16> itself
        assert np.array_equal(xy, best.bad_pixels_list(stack[0]))
    got = to_host(bp.correct_batch(to_dev(stack)))
    h = best.bad_pixels_create(stack[0])
    for t in range(len(stack)):
        assert np.array_equal(got[t], best.bad_pixels_correct(h, stack[t])), t
    best.bad_pixels_destroy(h)


@pytest.mark.parametrize("sigma", [0.5, 1.0, 2.0])
def test_gaussian(stack, sigma):
    got = to_host(sp.gaussian_filter_batch(to_dev(stack[:2]), sigma))
    assert_gauss_exact(got, stack[:2], sigma)


@pytest.mark.parametrize("strategy", ["nearest", "background", "wrap", ""])
def test_translate(stack, strategy):
    best = O.best()
    dx = np.array([1.3, -2.7, 117.25], dtype=np.float32)
    dy = np.array([-2.7, 0.5, -63.75], dtype=np.float32)
    src = to_dev(stack)
    got = to_host(sp.translate_batch(src, torch.from_numpy(dx).cuda(), torch.from_numpy(dy).cuda(), strategy, background=77))
    for t in range(3):
        want = best.translate(stack[t], dx[t], dy[t], strategy, background=77)
        assert np.array_equal(got[t], want), (strategy, t, int((got[t] != want).sum()))


def test_translate_motion_variant(stack, port):
    sx = np.array([0.37, -3.6, 12.5])
    sy = np.array([-1.9, 2.25, -0.01])
    got = to_host(vio.remove_motion(to_dev(stack), sx, sy, meta_rows=3))
    best = O.best()
    for t in range(3):
        want = stack[t].copy()
        h = stack.shape[1]
        want[: h - 3] = (best if hasattr(best, "loader_remove_motion") else port).loader_remove_motion(stack[t][: h - 3], sx[t], sy[t])
        assert np.array_equal(got[t], want), t


def test_precoder_statistics_and_reader_chain(stack, port):
    n = 101  # three GOPs of 50 with a partial last one
    h, w = stack.shape[1:]
    reps = -(-n // 3)
    mov = np.concatenate([stack] * reps)[:n].copy()
    mov[:, 5, 7] = (np.arange(n) * 611) % 65536  # something that changes from frame to frame
    d = to_dev(mov)
    for delta in (False, True):
        lo, hi = vio.precode_movie(d, 50, delta)
        olo, ohi = port.precode_movie(mov[:52], 50, delta)
        assert np.array_equal(lo[:52].cpu().numpy(), olo) and np.array_equal(hi[:52].cpu().numpy(), ohi)
        back = vio.decode_movie(lo, hi, 50, delta)
        assert torch.equal(back.view(torch.int16), d.view(torch.int16))
    st = movie.MovieStats("cuda")
    st.update(d)
    assert st.min() == int(mov.min()) and st.max() == int(mov.max())
    assert np.array_equal(st.histogram(), np.bincount(mov.ravel(), minlength=65536).astype(np.uint64))
    # the reader's chain on the planes of the first frames: merge -> += MIN_T -> bad pixels -> motion
    lo, hi = (mov[:3] & 0xFF).astype(np.uint8), (mov[:3] >> 8).astype(np.uint8)
    bp = vio.LoaderBadPixels(mov[0])
    xy = sp.bad_pixels_list(bp.handle)[0]
    sx, sy = np.array([1.5, -0.25, 3.0]), np.array([-2.0, 0.75, 0.0])
    got = to_host(vio.read_movie(to_dev(lo), to_dev(hi), bp, 273, 0, sx, sy))
    for t in range(3):
        assert np.array_equal(got[t], port.loader_read_image(lo[t], hi[t], xy, 273, h - 3, (sx[t], sy[t]))), t


def test_whole_path_on_host_buffers(stack):
    """rirb_process_movie_host against the same stages called one by one on the device."""
    n = 60
    mov = np.concatenate([stack] * 20)[:n].copy()
    h, w = mov.shape[1:]
    rng = np.random.default_rng(3)
    dx = rng.uniform(-3, 3, n).astype(np.float32)
    dy = rng.uniform(-3, 3, n).astype(np.float32)
    bp = sp.BadPixels(mov[0])
    lo, hi = movie.process_movie_host(bp, mov, dx, dy, 1.0, "nearest", 0, 50, True, 0)
    c = bp.correct_batch(to_dev(mov))
    r = sp.translate_batch(c, torch.from_numpy(dx).cuda(), torch.from_numpy(dy).cuda(), "nearest", background=0)
    wlo, whi = vio.precode_movie(r, 50, True)
    assert np.array_equal(lo, wlo.cpu().numpy()) and np.array_equal(hi, whi.cpu().numpy())
