"""Deterministic inputs of the registration tests (no RNG stream involved): shared by
tests/golden/make_ecc_golden.py, which runs the reference's own MaskedRegistratorECC class (with OpenCV) on them, and
tests/test_ecc.py."""
import numpy as np


def hash_noise(shape_t, t):
    """Zero-mean pseudo-noise in [-0.5, 0.5), a pure function of (t, y, x)."""
    h, w = shape_t
    y, x = np.mgrid[0:h, 0:w].astype(np.uint64)
    v = (x * np.uint64(73856093)) ^ (y * np.uint64(19349663)) ^ (np.uint64(t + 1) * np.uint64(83492791))
    v = (v * np.uint64(2654435761)) % np.uint64(1 << 32)
    return ((v >> np.uint64(12)) % np.uint64(4096)).astype(np.float64) / 4096.0 - 0.5


def trajectory(n):
    """Camera shift of frame t (pixels): a slow drift plus a wobble, sub-pixel steps."""
    t = np.arange(n, dtype=np.float64)
    sx = 0.35 * t + 1.5 * np.sin(t / 3.0)
    sy = -0.2 * t + 1.1 * np.cos(t / 4.0) - 1.1
    return sx, sy


BLOBS = [(200, 150, 2500, 30), (420, 300, 1800, 45), (320, 250, 1200, 18), (150, 380, 2100, 38), (500, 120, 1500, 25),
         (260, 330, 900, 12), (380, 180, 1100, 22)]


def frame(t, sx, sy, h=512, w=640, noise=6.0, flare=0.0):
    y, x = np.mgrid[0:h, 0:w].astype(np.float64)
    xs, ys = x - sx, y - sy
    f = 8000.0 + 40.0 * np.sin(xs / 23.0) * np.cos(ys / 31.0)
    for cx, cy, a, sg in BLOBS:
        f += a * np.exp(-(((xs - cx) / sg) ** 2 + ((ys - cy) / sg) ** 2))
    if flare:
        f += flare * np.exp(-(((x - 330) / 60.0) ** 2 + ((y - 240) / 50.0) ** 2))  # does not move with the scene
    f += noise * hash_noise((h, w), t)
    return np.clip(np.rint(f), 0, 65535).astype(np.uint16)


def movie(n, flare_from=None, flare=0.0):
    sx, sy = trajectory(n)
    return np.stack([frame(t, sx[t], sy[t], flare=(flare if flare_from is not None and t >= flare_from else 0.0)) for t in range(n)]), sx, sy


def small_pair(dx, dy, h=120, w=160, k=0):
    """A normalised float32 template / image pair for the solver alone."""
    y, x = np.mgrid[0:h, 0:w].astype(np.float64)

    def scene(ox, oy, t):
        s = np.zeros((h, w))
        for cx, cy, a, sg in [(40, 30, 1.0, 9), (110, 70, 0.7, 14), (80, 100, 0.5, 6), (20, 90, 0.8, 11)]:
            s += a * np.exp(-(((x - cx - ox) / sg) ** 2 + ((y - cy - oy) / sg) ** 2))
        return (s + 0.02 * hash_noise((h, w), t)).astype(np.float32)

    def norm(a):
        return (a - a.min()) / (a.max() - a.min())

    return norm(scene(0, 0, 2 * k)), norm(scene(dx, dy, 2 * k + 1))


FLARE = 1200.0        # lowers the confidence below the reset threshold, ECC still converges
SMALL_CASES = [(1.37, -0.62), (0.1, 0.05), (-2.5, 3.25), (4.8, -3.9), (0.0, 0.0), (7.3, 5.1)]


def ir_window_pair(t=3, h=358, w=448):
    """The class's default window (448 x 358 of a 640 x 512 frame) of frames 0 and t of the movie, as float32."""
    sx, sy = trajectory(t + 1)
    y0, x0 = (512 - h) // 2, (640 - w) // 2
    crop = (slice(y0, y0 + h), slice(x0, x0 + w))
    return frame(0, sx[0], sy[0])[crop].astype(np.float32), frame(t, sx[t], sy[t])[crop].astype(np.float32)


def ulps(v):
    """v and the float32 values one ulp either side of it."""
    v = np.float32(v)
    return [float(np.nextafter(v, np.float32(-np.inf))), float(v), float(np.nextafter(v, np.float32(np.inf)))]


def boundary_starts():
    """Starts on and one float ulp either side of every (2k+1)/64 px boundary (bilinear fraction), every (2k+1)/2 px
    boundary (nearest), ties tx * 1024 = m + 1/2 (round half to even), negative starts included."""
    s = []
    for k in range(-5, 5):
        s += ulps((2 * k + 1) / 64.0) + ulps((2 * k + 1) / 2.0) + ulps(k + (2 * k + 1) / 64.0)
    for m in (-1537, -512, -17, -16, -15, -1, 0, 1, 15, 16, 17, 511, 512, 1535):
        s += ulps((m + 0.5) / 1024.0)
    return sorted(set(s))


def failing_frames():
    """Second frames on which findTransformECC raises: contrast-inverted (correlation about to be minimised) and flat (NaN)."""
    sx, sy = trajectory(6)
    f5 = frame(5, sx[5], sy[5])
    return [(20000 - f5.astype(np.int32)).astype(np.uint16), np.full_like(f5, 8000)]
