"""Movies that reach the two places where the lossy pre-conditioner's arithmetic leaves ordinary ground (SURVEY.md 8f-2):

* stdDev's `diff * diff` is an int product (h264.cpp:1993-2036): a pixel that changes by 46,341 counts or more between two
  frames -- blinking, dead next to saturated, 16-bit noise -- makes it wrap modulo 2^32;
* from frame 41 on the spreads are split by img > background; when every pixel falls on one side -- a saturated or flat
  frame, or no lossy rows at all -- the other side's spread is 0 / 0 = NaN, and `lowError -= (int)round(NaN * f)` takes
  x86's conversion of NaN (INT_MIN) and wraps.

Each case is (name, movie, stop_lossy_height, saver parameters).  Deterministic (no RNG stream, like
tests/bp_extreme_cases.py); frames are at most 64 x 136 and movies 50-120 frames, so every case crosses the 40-frame window
of spreads."""
import numpy as np

from tests.ecc_cases import hash_noise
from tests.vio_cases import movie as ir_like

# 0 <-> J across the wrap of the int square: 46,340^2 < 2^31 <= 46,341^2
BLINK_LEVELS = (46340, 46341, 65535)


def blink(t, h, w, level, seed, npix=3):
    """An IR-like movie with `npix` pixels alternating between 0 and `level` from frame to frame."""
    mov = ir_like(t, h, w, seed=seed)
    idx = np.argsort(hash_noise((1, h * w), seed + 17)[0], kind="stable")[:npix]
    flat = mov.reshape(t, -1)
    flat[0::2, idx] = 0
    flat[1::2, idx] = level
    return mov


def dead_and_saturated(t, h, w, seed):
    """Ordinary background with 4 % dead (0) and 4 % saturated (65,535) pixels whose sets move every few frames, so that a
    dead pixel meets a saturated one across two frames."""
    mov = ir_like(t, h, w, seed=seed).astype(np.int64)
    for i in range(t):
        m = hash_noise((h, w), seed * 100 + i // 3) + 0.5
        mov[i][m < 0.04] = 0
        mov[i][m > 0.96] = 65535
    return mov.astype(np.uint16)


def full_range(t, h, w, seed):
    """Uniform 16-bit noise, a new draw every frame."""
    return np.stack([np.floor((hash_noise((h, w), seed * 1000 + i) + 0.5) * 65536).clip(0, 65535) for i in range(t)]).astype(np.uint16)


def with_frames(mov, frames, value):
    """`mov` with the given frames replaced by one flat value (65,535: saturated; else a flat field, e.g. a shutter frame)."""
    mov = mov.copy()
    mov[list(frames)] = value
    return mov


def below_first_min(t, h, w, seed):
    """For subtractMin: from frame 30 on the scene drops 3,000 counts below the first frame and some pixels go to 0."""
    mov = ir_like(t, h, w, seed=seed).astype(np.int64)
    mov[30:] -= 3000
    m = hash_noise((h, w), seed + 5) + 0.5
    mov[45:, m < 0.05] = 0
    return mov.clip(0, 65535).astype(np.uint16)


def itime_bits(t, h, w, seed):
    """Values whose three top bits (v >> 13, the integration-time tag) change: every pixel steps through the eight 8,192-count
    ranges, some by one count across a boundary, others by a whole range."""
    base = ir_like(t, h, w, seed=seed).astype(np.int64) - 8000  # about [0, 3,500)
    out = np.empty((t, h, w), np.int64)
    m = hash_noise((h, w), seed + 9) + 0.5
    for i in range(t):
        rng_k = (np.floor(m * 8).astype(np.int64) + i // 7) % 8
        v = rng_k * 8192 + base[i] % 8192
        edge = (m > 0.5) & (m < 0.6)  # these sit on a boundary and cross it by one count every other frame
        v[edge] = ((rng_k[edge] + 1) % 8) * 8192 - (i & 1)
        out[i] = v
    return out.clip(0, 65535).astype(np.uint16)


WIDE = dict(stdFactor=0.5, lowValueError=3000, highValueError=1500)  # bounds that stay open on wide-range content


def _cases():
    out = []
    t, h, w = 64, 24, 40
    for j in BLINK_LEVELS:
        for cname, cfg in (("default", {}), ("no_average", dict(runningAverage=0)), ("sub_min", dict(subtractMin=1))):
            out.append((f"blink_{j}_{cname}", blink(t, h, w, j, seed=j % 97), h - 3, cfg))
    out.append(("blink_65535_many_bp", blink(80, 32, 48, 65535, seed=5, npix=40), 32, dict(removeBadPixels=1)))
    out.append(("dead_and_saturated", dead_and_saturated(70, 32, 40, seed=3), 29, WIDE))
    out.append(("dead_and_saturated_bp", dead_and_saturated(70, 32, 40, seed=4), 29, dict(WIDE, removeBadPixels=1, subtractMin=1)))
    out.append(("full_range", full_range(60, 17, 64, seed=6), 17, WIDE))
    out.append(("full_range_136", full_range(52, 9, 136, seed=7), 6, dict(WIDE, runningAverage=1)))
    sat = with_frames(ir_like(70, 32, 40, seed=8), (44, 45, 46), 65535)
    out.append(("saturated_frames", sat, 32, {}))
    out.append(("saturated_frames_bp", sat, 32, dict(removeBadPixels=1)))
    for r in range(4):  # 4k + r: background = 4k + 1, so r <= 1 empties the foreground, r >= 2 the background
        out.append((f"flat_frames_4k{r}", with_frames(ir_like(70, 32, 40, seed=9), (44, 45, 46), 8000 + r), 29, {}))
    out.append(("flat_on_first_split", with_frames(ir_like(60, 20, 40, seed=10), (41,), 8002), 20, {}))
    out.append(("flat_movie", np.full((55, 16, 24), 8003, np.uint16), 16, {}))
    base = ir_like(56, 20, 32, seed=11)
    for stop in (0, 1, 20):
        out.append((f"stop_{stop}", with_frames(base, (45,), 65535), stop, {}))
    out.append(("below_first_min", below_first_min(72, 24, 40, seed=12), 24, dict(subtractMin=1)))
    out.append(("itime_bits", itime_bits(70, 24, 40, seed=13), 24, dict(WIDE, runningAverage=4)))
    sat_blink = with_frames(blink(90, 20, 40, 65535, seed=14), (60,), 65535)
    for ra in (0, 1, 63, 64, 70):
        out.append((f"running_average_{ra}", sat_blink, 20, dict(runningAverage=ra)))
    # |sd - mean| * stdFactor >= 2^31: finite but beyond int range; x86 (INT_MIN, then a wrap) and a saturating conversion
    # both end at (0, 0) here
    out.append(("huge_std_factor", blink(60, 20, 32, 46341, seed=15), 20, dict(stdFactor=1e12)))
    out.append(("huge_std_factor_noise", full_range(50, 8, 24, seed=16), 8, dict(stdFactor=3e9, lowValueError=40, highValueError=20)))
    return out


CASES = _cases()
DOORS = ("add_image_lossy", "add_loss")
