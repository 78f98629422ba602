"""Long movies for the stateful paths (tests/test_gpu_long_movies.py): the lossy pre-conditioner's runs, spread window and
running-average ring, the ECC tracker's queued runs and filtered-frame cache, and call schedules that cut a movie into
host calls of the lengths where those states turn over.  Every generator is a pure function of its arguments."""
import numpy as np

from tests import ecc_cases as ec
from tests.conftest import ir_movie

LOSSY_RUN = 64     # LOSSY_MAX_RUN: frames per cooperative launch of the lossy pre-conditioner
SPREADS = 40       # the window of spreads; from frame 41 on the spreads are split by img > background
ECC_RUN = 16       # ECC_BATCH: solves queued in one launch
ECC_THRESH = 21    # the confidence threshold is fixed when the 21st confidence arrives
EDGE_CALLS = (1, 63, 64, 65, 127, 128, 129)


def lossy_movie(t, h, w, seed, meta_rows=0, blink=(), bad_frames=(), itime=True):
    """IR background with a drifting hot spot and noise, a slow global drift, and
    * ``itime``: integration-time bit flips, +8,192 on a patch for a few stretches of frames;
    * ``blink``: levels (46,341 / 65,535 wrap the reference's int square) of pixels alternating with 0 over a stretch;
    * ``bad_frames``: ``{frame: value}``, saturated (65,535) or flat frames; placed beyond frame 40 they put a NaN spread
      into the window, which leaves it 40 frames later;
    * ``meta_rows``: the last rows carry a frame counter and a constant, like a camera's metadata lines."""
    rng = np.random.default_rng(seed)
    mov = ir_movie(t, h, w, seed=seed, drift=0.01).astype(np.int64)
    mov[mov == 0] = 300  # dead pixels above 0, so that subtractMin's MIN_T is not 0
    i = np.arange(t)
    mov += np.rint(250 * np.sin(i / 97.0) + 120 * np.sin(i / 13.0)).astype(np.int64)[:, None, None]
    if itime:
        for _ in range(max(1, t // 400)):
            a = int(rng.integers(1, t - 1))
            b = min(t, a + int(rng.integers(1, 30)))
            y0, x0 = int(rng.integers(0, max(1, h - 6))), int(rng.integers(0, max(1, w - 8)))
            mov[a:b, y0:y0 + 6, x0:x0 + 8] += 8192
    for level in blink:
        idx = rng.choice(h * w, 3, replace=False)
        a = int(rng.integers(0, t // 2))
        b = int(rng.integers(a + 1, t + 1))
        flat = mov.reshape(t, -1)
        flat[a:b, idx] = np.where((np.arange(a, b) % 2 == 0)[:, None], 0, level)
    for f, v in dict(bad_frames).items():
        if f < t:
            mov[f] = v
    if meta_rows:
        mov[:, h - meta_rows:] = 1234
        mov[:, h - meta_rows, :4] = (i % 65536)[:, None]
    return mov.clip(0, 65535).astype(np.uint16)


def nan_frames(t, value=65535):
    """Saturated or flat frames placed so that NaN spreads enter the 40-frame window, leave it, and land again after
    several turns of it: two next to each other early, then single ones at odd distances."""
    out = {}
    for f in (45, 46, 45 + 3 * SPREADS + 7, 45 + 10 * SPREADS + 13, 45 + 24 * SPREADS + 1, 45 + 50 * SPREADS + 29):
        if f < t:
            out[f] = value
    return out


def schedule(t, kind, rng=None):
    """A movie of t frames cut into calls: a list of ``(frames, lossy_run, device_frames)``.
    one: one call; edges: calls of the lengths around the launch limit, cycled, the driver switched between calls and host /
    device frames mixed; random: random lengths (1 .. 3 launches), drivers and frame locations."""
    if kind == "one":
        return [(t, 1, True)]
    out, a, k = [], 0, 0
    while a < t:
        if kind == "edges":
            c, run, dev = EDGE_CALLS[k % len(EDGE_CALLS)], (1, 1, 0)[k % 3], k % 2 == 0
        else:
            c = int(rng.choice([1, int(rng.integers(1, 3 * LOSSY_RUN + 2))]))
            run, dev = int(rng.integers(0, 2)), bool(rng.integers(0, 2))
        c = min(c, t - a)
        out.append((c, run, dev))
        a += c
        k += 1
    return out


# ---- ECC --------------------------------------------------------------------------------------------------------------------
FLARES = ((60, 63), (110, 111), (150, 158), (231, 232), (300, 306), (340, 342), (371, 374))  # [first, last): a static flare
NOISY = (4, 11, 17)  # frames among the first 21 with 10x the noise


def ecc_frame(t, sx, sy, flare=0.0, h=512, w=640, noise=6.0):
    """The scene of ecc_cases.frame (same blobs, texture, flare and noise) written with separable factors, which is several
    times faster on a long movie; the values differ from ecc_cases.frame by float rounding only."""
    x = np.arange(w, dtype=np.float64) - sx
    y = np.arange(h, dtype=np.float64) - sy
    f = 8000.0 + 40.0 * np.outer(np.cos(y / 31.0), np.sin(x / 23.0))
    for cx, cy, a, sg in ec.BLOBS:
        f += a * np.outer(np.exp(-((y - cy) / sg) ** 2), np.exp(-((x - cx) / sg) ** 2))
    if flare:
        f += flare * np.outer(np.exp(-((np.arange(h) - 240) / 50.0) ** 2), np.exp(-((np.arange(w) - 330) / 60.0) ** 2))
    f += noise * ec.hash_noise((h, w), t)
    return np.clip(np.rint(f), 0, 65535).astype(np.uint16)


def ecc_long_movie(n, flares=FLARES, amplitude=ec.FLARE):
    """ecc_cases frames on a bounded wobble (the scene stays in the registration window however long the movie) with a
    flare that does not move with the scene switched on in several stretches: each stretch and its end replace the
    reference image, so a long movie has many replacements and queued runs that stop inside.  The NOISY frames spread the
    first 21 confidences, whose min - 2 std is the replacement threshold: only the flares' edges then fall below it, by
    1e-1 against margins of 3e-4 for every other frame (with a uniformly quiet start the threshold sits within 1e-7 of
    most confidences, and rounding decides where the reference is replaced)."""
    t = np.arange(n, dtype=np.float64)
    sx = 5.0 * np.sin(t / 19.0) + 1.5 * np.sin(t / 3.0)
    sy = 4.0 * np.cos(t / 27.0) + 1.1 * np.cos(t / 4.0) - 1.1
    on = np.zeros(n, bool)
    for a, b in flares:
        on[a:min(b, n)] = True
    return np.stack([ecc_frame(k, sx[k], sy[k], flare=amplitude if on[k] else 0.0, noise=60.0 if k in NOISY else 6.0)
                     for k in range(n)]), sx, sy


def with_failures(mov, at):
    """``mov`` with ec.failing_frames() inserted before the given frame indices (cycled through the two kinds)."""
    bad = ec.failing_frames()
    parts, a = [], 0
    for k, f in enumerate(sorted(at)):
        parts += [mov[a:f], bad[k % len(bad)][None]]
        a = f
    return np.concatenate(parts + [mov[a:]])
