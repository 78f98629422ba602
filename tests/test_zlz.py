"""Coder 2, the device zstd coder with LZ matches, as oracle/zlz.py restates it (encode_frame_lz), against an independent
decoder, the system libzstd: every frame decodes to its payload, the corpus reaches every sequence feature, the parse
replays to its block, and the block choice keeps coder 1's bytes wherever the LZ form does not win.  CPU only;
tests/test_gpu_zlz.py holds the kernels to the restatement byte for byte."""
import numpy as np
import pytest

from librir_b200 import _lib
from librir_b200 import entropy as E
from oracle import zcoder as Z1
from oracle import zlz as Z
from tests import zcoder_cases as K
from tests import zlz_cases as L
from tests.conftest import ir_movie

CASES = L.cases()


def split_blocks(frame):
    """The blocks of a frame of either coder, each with its 3-byte header."""
    assert frame[:4] == Z1.MAGIC and frame[4] == 0xA0
    p, out = 9, []
    while True:
        h = int.from_bytes(frame[p:p + 3], "little")
        end = p + 3 + (1 if (h >> 1) & 3 == 1 else h >> 3)
        out.append(frame[p:end])
        p = end
        if h & 1:
            assert p == len(frame)
            return out


def has_sequences(block):
    """Whether a compressed block's sequences section is not empty (its last byte is the count 0 otherwise)."""
    return (block[0] >> 1) & 3 == 2 and block[-1] != 0


def parsed_blocks(data, segment):
    return [Z.parse(data[a:a + n]) + (data[a:a + n],) for a, n in Z1.blocks_of(len(data), segment)]


@pytest.mark.parametrize("name,data,segment", CASES, ids=[c[0] for c in CASES])
def test_libzstd_decodes_coder2(name, data, segment):
    f = Z.encode_frame_lz(data, segment)
    assert E.zstd_decompress(f) == data.tobytes()
    assert len(f) <= len(Z1.encode_frame(data, segment)) <= Z1.frame_bound(len(data), segment)
    assert len(split_blocks(f)) == max(1, Z1.n_blocks(len(data), segment))


@pytest.mark.parametrize("name,data,segment", CASES, ids=[c[0] for c in CASES])
def test_parse_replays_to_the_block(name, data, segment):
    for seqs, lits, block in parsed_blocks(data, segment):
        assert np.array_equal(Z.replay(seqs, lits), block)
        for ll, ml, off in seqs:
            assert ml >= Z.MIN_MATCH and 1 <= off


def test_corpus_covers_every_feature():
    seen = set()
    for name, data, segment in CASES:
        f = Z.encode_frame_lz(data, segment)
        for (seqs, lits, block), b in zip(parsed_blocks(data, segment), split_blocks(f)):
            if not has_sequences(b):
                continue
            seen.add("lz_block")
            if any(off < ml for _, ml, off in seqs):
                seen.add("overlap")
            if any(off == 1 for _, _, off in seqs):
                seen.add("run")
            if any(ml >= 65539 for _, ml, _ in seqs):
                seen.add("ml_code_52")
            if any(ll == 0 for ll, _, _ in seqs):
                seen.add("ll_0")
            if any(ll >= 65536 for ll, _, _ in seqs):
                seen.add("ll_code_35")
            if len(seqs) == 1:
                seen.add("one_sequence")  # every table in mode RLE
            if len(seqs) >= 128:
                seen.add("two_byte_count")
            if sum(ll + ml for ll, ml, _ in seqs) == len(block):
                seen.add("no_trailing_literals")  # the last match ends at the block's end
            if any(off == 640 for _, _, off in seqs):
                seen.add("offset_w")
            if segment and len(data) > segment:
                seen.add("segments")
            mode = b[3 + len(Z.literals_section(lits)) + (1 if len(seqs) < 128 else 2)]
            seen.add("predefined" if mode != 0b01010100 else "all_rle")
            lit_kind = b[3] & 3
            seen.add(("raw", "rle", "huffman", "?")[lit_kind] + "_literals")
    # RLE literals cannot occur in a block that takes the LZ form: every byte value of a block is a literal once, so
    # literals of one value mean a block of one value, and that block is coder 1's RLE block
    assert seen >= {"lz_block", "overlap", "run", "ml_code_52", "ll_0", "ll_code_35", "one_sequence", "two_byte_count",
                    "no_trailing_literals", "offset_w", "segments", "predefined", "all_rle", "raw_literals",
                    "huffman_literals"}, seen


def test_frame_without_lz_blocks_is_coder1():
    for name, data, segment in CASES:
        f, f1 = Z.encode_frame_lz(data, segment), Z1.encode_frame(data, segment)
        if not any(has_sequences(b) for b in split_blocks(f)):
            assert f == f1, name
    assert Z.encode_frame_lz(K.cases()[0][1]) == Z1.encode_frame(K.cases()[0][1])


def test_ir_movie_ratios():
    """ir_movie(3, 512, 640), frame 1: method 2 reaches host zstd's ratio class, methods 1 and 3 never grow, and a block
    where the LZ form loses is coder 1's block byte for byte."""
    mov = ir_movie(3, 512, 640)
    npx = 512 * 640
    payload = {1: mov[1].reshape(-1).view(np.uint8), 2: K.planes(mov, 2)[1], 3: K.planes(mov, 3)[1]}
    ratio = {}
    for method, p in payload.items():
        seg = 0 if method == 1 else npx
        f, f1 = Z.encode_frame_lz(p, seg), Z1.encode_frame(p, seg)
        assert E.zstd_decompress(f) == p.tobytes()
        assert len(f) <= len(f1), method
        for b, b1 in zip(split_blocks(f), split_blocks(f1)):
            if not has_sequences(b):
                assert b == b1
        ratio[method] = len(p) / len(f)
    assert ratio[2] >= 1.9, ratio  # 1.997x (coder 1: 1.663x, host zstd level 1: 2.045x)
    assert ratio[1] >= 1.47 and ratio[3] >= 3.07, ratio


def test_set_lz_rejects_bad_values(tmp_path):
    lib = _lib.load()
    z = lib.rirb_z_open_file_write(str(tmp_path / "a.bin").encode(), 32, 16, 50, 1, 1)
    assert z > 0, _lib.last_error()
    assert lib.rirb_z_set_lz(z, 2) == -1 and "z_set_lz" in _lib.last_error()
    assert lib.rirb_z_set_lz(z, -1) == -1
    if _lib.device_available():
        assert lib.rirb_z_set_lz(z, 1) == 0
    else:
        assert lib.rirb_z_set_lz(z, 1) == -1 and "CUDA device" in _lib.last_error()
    assert lib.rirb_z_set_lz(z, 0) == 0
    lib.rirb_z_close_file(z)
    assert lib.rirb_z_set_lz(z, 0) == -1  # closed


@pytest.mark.skipif(_lib.device_available(), reason="checks behaviour WITHOUT a CUDA device")
def test_lz_coder_without_gpu_fails_cleanly(tmp_path):
    from librir_b200 import tools

    with pytest.raises(RuntimeError, match="device coder"):
        tools.ZFileWriter(tmp_path / "m1.bin", 32, 16, method=1, coder="gpu-lz")
    buf = np.zeros(64, np.uint8)
    lib = _lib.load()
    assert lib.rirb_zstd_encode_batch_lz(buf.ctypes.data, 1, 8, 0, buf.ctypes.data, 32, buf.ctypes.data) == -1
    assert "zstd_encode_batch_lz" in _lib.last_error()
