"""The device zstd decoder's per-frame code (librir_b200/csrc/zdecoder.cu) compiled for the host through
tests/zdecoder_host_shim.cu, against libzstd on random frames: random payloads (uniform, small alphabets, runs, periodic
data with sparse noise, geometric bytes, IR movie frames and the byte planes of methods 2 / 3) compressed by libzstd
with random parameters (level, window log, strategy, minimum match, search log, target length, long-distance matching,
content size flag, checksum, forced raw or Huffman literals, small target block sizes), then mutated and truncated.
A valid frame decodes to its payload; a mutated frame the decoder accepts is one libzstd accepts with the same bytes;
nothing is written past the capacity.  CPU only: the same code runs without a device.  The committed case counts are
small; ``RIRB_FUZZ_SEED=<n> RIRB_FUZZ_SCALE=<k>`` runs k times as many cases from other seeds.
tests/test_gpu_zstd_fuzz.py runs the same generators through the kernels and holds them to this harness."""
import ctypes as ct
import os
import shutil
import subprocess

import numpy as np
import pytest

from tests import zcoder_cases as K
from tests import zdecoder_cases as D
from tests.conftest import ir_movie
from tests.test_zdecoder import FEATURES

SEED = int(os.environ.get("RIRB_FUZZ_SEED", "0"))
SCALE = max(1, int(os.environ.get("RIRB_FUZZ_SCALE", "1")))
HERE = os.path.dirname(os.path.abspath(__file__))
GUARD = 0xA5

# ZSTD_cParameter values (zstd.h); literalCompressionMode and targetCBlockSize are experimental parameters
P_LEVEL, P_WINDOW_LOG, P_SEARCH_LOG, P_MIN_MATCH, P_TARGET_LENGTH, P_STRATEGY = 100, 101, 104, 105, 106, 107
P_LDM, P_CONTENT_SIZE, P_CHECKSUM, P_LITERAL_MODE = 160, 200, 201, 1002


def p_target_block():
    """ZSTD_c_targetCBlockSize: experimental parameter 1003 before zstd 1.5.6, a stable one (130) from then on."""
    z = D.libzstd()
    z.ZSTD_versionNumber.restype = ct.c_uint
    return 130 if z.ZSTD_versionNumber() >= 10506 else 1003


def nvcc():
    for c in (os.environ.get("NVCC"), shutil.which("nvcc"), "/usr/local/cuda/bin/nvcc"):
        if c and os.path.exists(c):
            return c
    return None


def build_host_decoder(out_dir):
    """Compiles tests/zdecoder_host_shim.cu with the library's nvcc line into out_dir -> decode(frame, cap) that
    returns (status, content bytes) and checks the guard bytes behind the capacity and the literal scratch."""
    exe = nvcc()
    if exe is None:
        pytest.skip("nvcc not found: the host build of the decoder needs it")
    so = os.path.join(str(out_dir), "libzdhost.so")
    subprocess.check_call([exe, "-gencode", "arch=compute_100a,code=sm_100a", "-O3", "-std=c++17", "-ccbin", "/usr/bin/g++",
                           "-Xcompiler", "-fPIC,-fvisibility=hidden", "-shared", "-cudart", "static",
                           "-Xlinker", "--no-undefined", os.path.join(HERE, "zdecoder_host_shim.cu"), "-o", so])
    lib = ct.CDLL(so)
    lib.zd_host_decode.restype = ct.c_longlong
    lib.zd_host_decode.argtypes = [ct.c_void_p, ct.c_longlong, ct.c_void_p, ct.c_longlong, ct.c_void_p]

    def decode(frame, cap):
        src = np.frombuffer(frame, np.uint8).copy() if len(frame) else np.zeros(1, np.uint8)
        dst = np.full(cap + 64, GUARD, np.uint8)
        lits = np.full(cap + 64, GUARD, np.uint8)
        r = lib.zd_host_decode(src.ctypes.data, len(frame), dst.ctypes.data, cap, lits.ctypes.data)
        assert (dst[cap:] == GUARD).all() and (lits[cap:] == GUARD).all(), "write past the capacity"
        assert r >= -2, r
        return int(r), dst[:max(r, 0)].tobytes()

    return decode


@pytest.fixture(scope="module")
def host_decode(tmp_path_factory):
    return build_host_decoder(tmp_path_factory.mktemp("zdhost"))


# ---- generators ---------------------------------------------------------------------------------------------------------
def payload(rng, max_len=800_000):
    """One random payload: a length from the edges (0, 1, 5, a block +- 1, a 640x512 method-1 record) or at random, and
    one of the kinds of the module docstring (or a single byte value)."""
    n = int(rng.choice([0, 1, 5, 100, 1000, 4096, 70_000, 131_071, 131_072, 131_073, 300_000, 655_360,
                        int(rng.integers(0, max_len + 1)), int(rng.integers(0, 20_000))]))
    n = min(n, max_len)
    kind = int(rng.integers(0, 8))
    if kind == 7:  # one value: RLE blocks
        x = np.full(n, rng.integers(0, 256))
    elif kind == 0:
        x = rng.integers(0, 256, n)
    elif kind == 1:
        x = rng.integers(0, int(rng.integers(1, 40)), n)
    elif kind == 2:
        x = np.repeat(rng.integers(0, 256, n // 8 + 1), rng.integers(1, 16, n // 8 + 1))[:n]
    elif kind == 3:
        base = rng.integers(0, 256, int(rng.integers(1, 5000)))
        x = np.resize(base, n)
        noise = rng.random(n) < rng.choice([0, 0.001, 0.05])
        x[noise] = rng.integers(0, 256, int(noise.sum()))
    elif kind == 4:
        x = rng.geometric(rng.uniform(0.01, 0.9), n) % 256
    else:
        w = int(rng.choice([64, 256, 640]))
        h = max(1, -(-n // (2 * w)))
        mov = ir_movie(2, h, w, seed=int(rng.integers(0, 1000)))
        if kind == 5:
            x = mov[1].reshape(-1).view(np.uint8)[:n]
        else:  # the [lo | hi] planes of method 2 or of a method-3 residual frame
            x = K.planes(mov, int(rng.choice([2, 3])))[1]
    return np.ascontiguousarray(x, np.uint8)


def params(rng):
    """libzstd parameters for one frame, as {ZSTD_cParameter: value}."""
    p = {P_LEVEL: int(rng.integers(-7, 23)), P_CONTENT_SIZE: int(rng.random() < 0.7)}
    if rng.random() < 0.5:
        p[P_WINDOW_LOG] = int(rng.integers(10, 24))
    if rng.random() < 0.4:
        p[P_STRATEGY] = int(rng.integers(1, 10))
    if rng.random() < 0.4:
        p[P_MIN_MATCH] = int(rng.integers(3, 8))
    if rng.random() < 0.3:
        p[P_SEARCH_LOG] = int(rng.integers(1, 10))
    if rng.random() < 0.3:
        p[P_TARGET_LENGTH] = int(rng.integers(0, 1000))
    if rng.random() < 0.2:
        p[P_LDM] = 1
    if rng.random() < 0.3:
        p[P_LITERAL_MODE] = int(rng.integers(0, 3))  # auto, Huffman, raw
    if rng.random() < 0.3:
        p[p_target_block()] = int(rng.integers(1340, 10000))  # many small blocks
    if rng.random() < 0.08:
        p[P_CHECKSUM] = 1
    return p


def compress(data, p):
    """ZSTD_compress2 with the parameters p; every parameter must be taken."""
    z = D.libzstd()
    src = np.ascontiguousarray(data, np.uint8).reshape(-1)
    out = np.empty(z.ZSTD_compressBound(src.size) + 64, np.uint8)
    c = z.ZSTD_createCCtx()
    try:
        for k, v in p.items():
            assert not z.ZSTD_isError(z.ZSTD_CCtx_setParameter(c, k, v)), ("libzstd refused a parameter", k, v)
        n = z.ZSTD_compress2(c, out.ctypes.data, out.size, src.ctypes.data, src.size)
        assert not z.ZSTD_isError(n)
    finally:
        z.ZSTD_freeCCtx(c)
    return out[:n].tobytes()


def one_literal_value(rng):
    """Random 128 KiB, then copies of random pieces of it, each followed by the byte 0xAA: at level 19 the literals of
    the later blocks are all 0xAA, which libzstd writes as RLE literals."""
    r = rng.integers(0, 256, 131072).astype(np.uint8)
    n = int(rng.integers(8, 100))
    parts = [r]
    for s in rng.integers(0, len(r) - n, 131072 // (n + 1)):
        parts += [r[s:s + n], np.array([0xAA], np.uint8)]
    return np.concatenate(parts), {P_LEVEL: 19, P_CONTENT_SIZE: int(rng.integers(0, 2))}


def special_frame(rng, k):
    """Features that random libzstd parameters reach too rarely (RLE literals) or never (more than 0x7F00 sequences in
    a block, the three-byte count; RLE literals in a block without sequences): the hand-built frames of
    tests/zdecoder_cases.py with random content, and one_literal_value."""
    if k % 3 == 0:
        frame, data = D.long_count_frame(int(rng.integers(0, 1 << 30)))
        return frame, data, {}
    if k % 3 == 1:
        # at least 3 bytes: the block content (3 bytes) must fit the window, which is the content size (RFC 8878
        # 3.1.1.2.3); libzstd takes shorter ones, the decoder refuses them with -1 and the reader falls back to the host
        frame, data = D.rle_literals_frame(int(rng.integers(0, 256)), int(rng.integers(3, 32)))
        return frame, data, {}
    data, p = one_literal_value(rng)
    return compress(data, p), data.tobytes(), p


def valid_frame(rng, i, max_len=800_000):
    """Case i of a run -> (frame, payload, parameters).  Every 20th case is a special_frame."""
    if i % 20 == 19:
        return special_frame(rng, i // 20)
    data, p = payload(rng, max_len), params(rng)
    return compress(data, p), data.tobytes(), p


def mutate(rng, frame):
    """1-3 byte changes or bit flips, then (one time in five) a cut."""
    b = bytearray(frame)
    for _ in range(int(rng.integers(1, 4))):
        if not b:
            break
        i = int(rng.integers(0, len(b)))
        if rng.random() < 0.5:
            b[i] ^= 1 << int(rng.integers(0, 8))
        else:
            b[i] = int(rng.integers(0, 256))
    if rng.random() < 0.2:
        b = b[:int(rng.integers(0, len(b) + 1))]
    return bytes(b)


def expected_status(payload_bytes, p):
    return -2 if p.get(P_CHECKSUM) else len(payload_bytes)


# ---- tests --------------------------------------------------------------------------------------------------------------
def test_valid_frames_decode(host_decode):
    rng = np.random.default_rng(601 + SEED)
    seen = set()
    for i in range(600 * SCALE):
        frame, data, p = valid_frame(rng, i)
        seen |= D.walk(frame)
        cap = len(data) + int(rng.integers(0, 100))
        st, out = host_decode(frame, cap)
        assert st == expected_status(data, p), (i, len(data), st, p)
        if st >= 0:
            assert out == data, (i, p)
    # the random frames alone reach every format feature the fixed corpus of tests/zdecoder_cases.py reaches
    assert FEATURES <= seen, sorted(FEATURES - seen)


def test_capacity_one_short_is_refused(host_decode):
    rng = np.random.default_rng(602 + SEED)
    for i in range(150 * SCALE):
        frame, data, p = valid_frame(rng, i, max_len=200_000)
        if not data:
            continue
        st, _ = host_decode(frame, len(data) - 1)
        assert st == (-2 if p.get(P_CHECKSUM) else -1), (i, len(data), st, p)


def test_mutated_frames(host_decode):
    rng = np.random.default_rng(603 + SEED)
    accepted = 0
    for i in range(600 * SCALE):
        frame, data, _ = valid_frame(rng, i, max_len=200_000)
        bad = mutate(rng, frame)
        cap = len(data) + int(rng.integers(0, 64))
        st, out = host_decode(bad, cap)
        if st >= 0:  # accepted: then exactly what libzstd makes of the mutated frame
            accepted += 1
            assert out == D.decompress(bad, cap), (i, st)
        else:
            assert st in (-1, -2), (i, st)
    assert accepted > 0
