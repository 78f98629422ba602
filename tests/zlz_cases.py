"""Payloads for coder 2, the device zstd coder with LZ matches (librir_b200/csrc/zcoder.cu, the zl_* kernels) and its
restatement (oracle/zlz.py, encode_frame_lz), shared by the CPU and GPU tests.  Each case is (name, payload bytes as
uint8, segment).  tests/test_zlz.py checks that the corpus reaches every sequence feature it names."""
import numpy as np

from tests import vio_cases as C
from tests import zcoder_cases as K


def runs(n, seed, lo=9, hi=200):
    """Runs of one byte value: every match is an overlap at offset 1."""
    rng = np.random.default_rng(seed)
    vals = rng.integers(0, 256, n // lo + 1).astype(np.uint8)
    return np.repeat(vals, rng.integers(lo, hi, len(vals)))[:n]


def repeated_rows(h, w, seed):
    """Rows that repeat the row above with a few bytes changed: matches at offset w, LL = 0 between them."""
    rng = np.random.default_rng(seed)
    rows = [rng.integers(0, 256, w).astype(np.uint8)]
    for _ in range(h - 1):
        r = rows[-1].copy()
        r[rng.integers(0, w, 3)] = rng.integers(0, 256, 3)
        rows.append(r)
    return np.concatenate(rows)


def cases():
    rng = np.random.default_rng(11)
    out = [(f"c1_{name}", data, seg) for name, data, seg in K.cases()]  # coder 1's corpus and its lengths
    out.append(("runs", runs(200000, 1), 0))
    out.append(("runs_only_block", np.repeat(np.array([5, 9], np.uint8), [70000, 61072]), 0))
    out.append(("rows_w640", repeated_rows(300, 640, 2), 0))
    out.append(("rows_segments", repeated_rows(250, 96, 3), 96 * 50))
    head = rng.integers(0, 256, 1000).astype(np.uint8)
    out.append(("match_to_block_end", np.concatenate([head, head[:500]]), 0))
    out.append(("ml_code_52", np.concatenate([head, np.zeros(100000, np.uint8)]), 0))  # one match of ML 99 999
    out.append(("one_sequence", np.concatenate([head[:40], head[:40], rng.integers(0, 256, 30).astype(np.uint8)]), 0))
    out.append(("at_block_edge", np.tile(head[:100], 1400), 0))  # 140 000 bytes: the match runs to the block's end
    for n in (7, 8, 9, 15, 16, 17, 300):
        out.append((f"short{n}", np.tile(np.array([1, 2, 3], np.uint8), n)[:n], 0))
    out.append(("random_with_copies", np.concatenate([rng.integers(0, 256, 20000).astype(np.uint8)] * 3), 0))
    tail = rng.integers(0, 256, 100000).astype(np.uint8)
    out.append(("ll_code_35", np.concatenate([tail, tail[:20]]), 0))  # the one sequence (LL 100 000, ML 20, offset 100 000)
    mov = C.movie(3, 120, 160, seed=4)
    for method in (1, 2):
        p = mov.reshape(3, -1).view(np.uint8) if method == 1 else K.planes(mov, method)
        out.append((f"movie_m{method}", p[1], 0 if method == 1 else 120 * 160))
    return out
