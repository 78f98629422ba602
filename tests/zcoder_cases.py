"""Payloads for the device zstd coder (librir_b200/csrc/zcoder.cu) and its restatement (oracle/zcoder.py), shared by the CPU
and GPU tests.  Each case is (name, payload bytes as uint8, segment)."""
import numpy as np

from tests import vio_cases as C

LENGTHS = (1, 2, 5, 6, 1023, 1024, 131072, 131073, 655360)


def fibonacci_bytes(n, seed):
    """Symbol k appears F(k) times (F = 1, 1, 2, 3, 5, ...): the unlimited Huffman code would need ~24 bits."""
    f = [1, 1]
    while len(f) < 25:
        f.append(f[-1] + f[-2])
    x = np.repeat(np.arange(25, dtype=np.uint8), f)
    np.random.default_rng(seed).shuffle(x)
    return np.resize(x, n)


def planes(mov, method, gop=50):
    """Record payloads of methods 2 / 3: per frame [low-byte plane | high-byte plane] of the frame or its temporal residual."""
    m = mov.astype(np.uint16)
    if method == 3:
        d = m.copy()
        for t in range(1, len(m)):
            if t % gop:
                d[t] = m[t] - m[t - 1]
        m = d
    t = len(m)
    return np.concatenate([(m & 0xFF).astype(np.uint8).reshape(t, -1), (m >> 8).astype(np.uint8).reshape(t, -1)], axis=1)


def cases():
    rng = np.random.default_rng(7)
    out = []
    for n in LENGTHS:
        out.append((f"geometric{n}", np.minimum(rng.geometric(0.05, n), 255).astype(np.uint8), 0))
    out.append(("constant", np.full(300000, 7, np.uint8), 0))
    out.append(("two_symbols", rng.choice(np.array([3, 200], np.uint8), 40000), 0))
    out.append(("all_256", np.concatenate([np.arange(256, dtype=np.uint8), np.minimum(rng.geometric(0.02, 200000), 255).astype(np.uint8)]), 0))
    out.append(("direct_weights", np.minimum(rng.geometric(0.1, 30000), 128).astype(np.uint8), 0))
    out.append(("length_limited", fibonacci_bytes(300000, 1), 0))
    out.append(("random", rng.integers(0, 256, 300000).astype(np.uint8), 0))
    out.append(("segments", np.minimum(rng.geometric(0.05, 100000), 255).astype(np.uint8), 30000))
    mov = C.movie(4, 96, 128, seed=3)
    for method in (2, 3):
        for t, p in enumerate(planes(mov, method, gop=2)):
            out.append((f"planes_m{method}_{t}", p, 96 * 128))
    return out
