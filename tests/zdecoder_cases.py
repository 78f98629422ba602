"""Frames for the device zstd decoder (librir_b200/csrc/zdecoder.cu), shared by the CPU and GPU tests: what the device coder
writes (oracle/zcoder.py), what libzstd writes at several levels and parameters on movie payloads, edge payloads, and two
hand-built frames for the features libzstd never emits.  Each case is (name, frame bytes, payload bytes).  `walk` lists the
format features a frame uses, so that the tests can show the corpus covers all of them."""
import ctypes as ct
import ctypes.util

import numpy as np

from oracle import zcoder as Z
from tests import zcoder_cases as K
from tests.conftest import ir_movie

# ZSTD_cParameter values (zstd.h)
C_LEVEL, C_WINDOW_LOG, C_CONTENT_SIZE, C_CHECKSUM = 100, 101, 200, 201

_z = None


def libzstd():
    global _z
    if _z is None:
        z = ct.CDLL(ctypes.util.find_library("zstd") or "libzstd.so.1")
        z.ZSTD_createCCtx.restype = ct.c_void_p
        z.ZSTD_freeCCtx.argtypes = [ct.c_void_p]
        z.ZSTD_CCtx_setParameter.argtypes = [ct.c_void_p, ct.c_int, ct.c_int]
        z.ZSTD_CCtx_setParameter.restype = ct.c_size_t
        z.ZSTD_compress2.argtypes = [ct.c_void_p, ct.c_void_p, ct.c_size_t, ct.c_void_p, ct.c_size_t]
        z.ZSTD_compress2.restype = ct.c_size_t
        z.ZSTD_compressBound.argtypes = [ct.c_size_t]
        z.ZSTD_compressBound.restype = ct.c_size_t
        z.ZSTD_decompress.argtypes = [ct.c_void_p, ct.c_size_t, ct.c_void_p, ct.c_size_t]
        z.ZSTD_decompress.restype = ct.c_size_t
        z.ZSTD_isError.argtypes = [ct.c_size_t]
        z.ZSTD_isError.restype = ct.c_uint
        _z = z
    return _z


def compress(data, level, content_size=1, checksum=0, window_log=0):
    """ZSTD_compress2 with the given parameters (window_log 0 = the level's default)."""
    z = libzstd()
    src = np.ascontiguousarray(data, dtype=np.uint8).reshape(-1)
    out = np.empty(z.ZSTD_compressBound(src.size) + 64, np.uint8)
    c = z.ZSTD_createCCtx()
    try:
        for k, v in ((C_LEVEL, level), (C_CONTENT_SIZE, content_size), (C_CHECKSUM, checksum), (C_WINDOW_LOG, window_log)):
            assert not z.ZSTD_isError(z.ZSTD_CCtx_setParameter(c, k, v))
        n = z.ZSTD_compress2(c, out.ctypes.data, out.size, src.ctypes.data, src.size)
        assert not z.ZSTD_isError(n)
    finally:
        z.ZSTD_freeCCtx(c)
    return out[:n].tobytes()


def decompress(frame, capacity):
    """libzstd's one-shot decoder into `capacity` bytes: the content, or None when libzstd rejects the frame."""
    z = libzstd()
    dst = np.empty(max(capacity, 1), np.uint8)
    src = np.frombuffer(frame, np.uint8) if len(frame) else np.zeros(1, np.uint8)
    n = z.ZSTD_decompress(dst.ctypes.data, capacity, src.ctypes.data, len(frame))
    return None if z.ZSTD_isError(n) else dst[:n].tobytes()


def rle_literals_frame(value=0x5A, size=25):
    """One compressed block: RLE literals (header 0x01 | size << 3, one byte), no sequences."""
    block = bytes([0x01 | size << 3, value, 0])
    return Z.MAGIC + bytes([0x20, size]) + (1 | 2 << 1 | len(block) << 3).to_bytes(3, "little") + block, bytes([value]) * size


def long_count_frame(seed=3):
    """32,512 sequences (count 0xFF + 2 bytes), raw literals, LL/OF/ML tables all RLE (symbols 1, 0, 0), bitstream 0x01:
    every sequence is 1 literal and a match of 3 at repeat offset 1, so each literal comes out four times."""
    nseq = 32512
    lits = np.random.default_rng(seed).integers(0, 256, nseq).astype(np.uint8).tobytes()
    lh = bytes([0 | 3 << 2 | (nseq & 15) << 4, (nseq >> 4) & 0xFF, nseq >> 12])
    block = lh + lits + bytes([0xFF]) + (nseq - 0x7F00).to_bytes(2, "little") + bytes([0x54, 1, 0, 0, 0x01])
    payload = bytes(b for b in lits for _ in range(4))
    head = Z.MAGIC + bytes([0xA0]) + len(payload).to_bytes(4, "little")
    return head + (1 | 2 << 1 | len(block) << 3).to_bytes(3, "little") + block, payload


def method_payloads(t=3, h=200, w=256):
    """Record payloads of the three methods for a small IR movie: raw frames, and the [lo | hi] planes of methods 2 / 3."""
    mov = ir_movie(t, h, w, seed=11)
    raw = [mov[i].tobytes() for i in range(t)]
    return {1: raw, 2: [p.tobytes() for p in K.planes(mov, 2, gop=t)], 3: [p.tobytes() for p in K.planes(mov, 3, gop=t)]}


def cases():
    out = []
    for name, data, segment in K.cases():
        if data.size <= 140000:
            out.append(("coder_" + name, Z.encode_frame(data, segment), data.tobytes()))
    pay = method_payloads()
    for m in (1, 2, 3):
        for level in (-5, 1, 2, 3, 12, 19):
            p = pay[m][1]
            out.append((f"m{m}_level{level}", compress(np.frombuffer(p, np.uint8), level), p))
    two = pay[1][0] + pay[1][1]  # 200 KiB: blocks that reach back into earlier blocks
    out.append(("m1_two_frames_level3", compress(np.frombuffer(two, np.uint8), 3), two))
    rng = np.random.default_rng(5)
    for n in (0, 1, 131072, 131073):
        z = bytes(n)
        out.append((f"zeros{n}", compress(np.frombuffer(z, np.uint8) if n else np.zeros(0, np.uint8), 3), z))
    for n in (1, 131072, 131073):
        r = rng.integers(0, 256, n).astype(np.uint8).tobytes()
        out.append((f"random{n}", compress(np.frombuffer(r, np.uint8), 3), r))
    p = pay[1][2]
    out.append(("no_content_size", compress(np.frombuffer(p, np.uint8), 3, content_size=0), p))
    out.append(("checksum", compress(np.frombuffer(p, np.uint8), 3, checksum=1), p))
    out.append(("window_log10", compress(np.frombuffer(p, np.uint8), 3, window_log=10), p))
    text = b"".join(b"frame %d of the zstd movie file, offset %d\n" % (i, i * 37) for i in range(3000))
    out.append(("text_level19", compress(np.frombuffer(text, np.uint8), 19), text))
    out.append(("text_fcs2", compress(np.frombuffer(text[:300], np.uint8), 3), text[:300]))
    out.append(("rle_literals", *rle_literals_frame()))
    out.append(("long_sequence_count", *long_count_frame()))
    return out


def walk(frame):
    """The format features of one frame, as a set of strings (see tests/test_zdecoder.py for the list)."""
    f = frame
    feats = set()
    fhd = f[4]
    single, fcs_flag = (fhd >> 5) & 1, fhd >> 6
    feats.add("single_segment" if single else "window_descriptor")
    fcs_bytes = (1 if single else 0) if fcs_flag == 0 else (2, 4, 8)[fcs_flag - 1]
    feats.add(f"fcs{fcs_bytes}")
    if fhd & 4:
        feats.add("checksum")
    p = 5 + (0 if single else 1) + (0, 1, 2, 4)[fhd & 3] + fcs_bytes
    while True:
        h = int.from_bytes(f[p:p + 3], "little")
        last, kind, size = h & 1, (h >> 1) & 3, h >> 3
        p += 3
        feats.add(f"block{kind}")
        if kind == 2:
            b0 = f[p]
            lt, sf = b0 & 3, (b0 >> 2) & 3
            feats.add(f"literals{lt}")
            if lt < 2:
                hs = (1, 2, 1, 3)[sf]
                regen = b0 >> 3 if hs == 1 else int.from_bytes(f[p:p + hs], "little") >> 4
                cs = regen if lt == 0 else 1
            else:
                feats.add("streams1" if sf == 0 else "streams4")
                hs = (3, 3, 4, 5)[sf]
                v = int.from_bytes(f[p:p + hs], "little")
                bits = (10, 10, 14, 18)[sf]
                cs = (v >> (4 + bits)) & ((1 << bits) - 1)
                if lt == 2:
                    feats.add("weights_direct" if f[p + hs] >= 128 else "weights_fse")
            q = p + hs + cs
            b = f[q]
            if b == 0:
                feats.add("nseq0")
            else:
                feats.add("nseq1" if b < 128 else "nseq2" if b < 255 else "nseq3")
                q += 1 if b < 128 else 2 if b < 255 else 3
                modes = f[q]
                for i, t in enumerate(("LL", "OF", "ML")):
                    feats.add(f"{t}_mode{(modes >> (6 - 2 * i)) & 3}")
        p += 1 if kind == 1 else size
        if last:
            return feats
