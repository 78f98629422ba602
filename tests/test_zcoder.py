"""The restatement of the device zstd coder (oracle/zcoder.py) against an independent decoder, the system libzstd: every
frame decodes to its payload, the block policy is what the format subset says, and the frame is never larger than raw
blocks plus headers.  CPU only; tests/test_gpu_zcoder.py holds the kernel to the restatement byte for byte."""
import numpy as np
import pytest

from librir_b200 import _lib
from librir_b200 import entropy as E
from oracle import zcoder as Z
from tests import zcoder_cases as K

CASES = K.cases()


def blocks(frame):
    """(block type, literals size format or None) of every block; checks the frame header on the way."""
    assert frame[:4] == Z.MAGIC and frame[4] == 0xA0
    p, out = 9, []
    while True:
        h = int.from_bytes(frame[p:p + 3], "little")
        last, kind, size = h & 1, (h >> 1) & 3, h >> 3
        p += 3
        if kind == 2:
            assert frame[p] & 3 == 2  # Huffman-coded literals with their own tree
            out.append((2, (frame[p] >> 2) & 3, frame[p + (3 if (frame[p] >> 2) & 3 < 2 else ((frame[p] >> 2) & 3) + 2)]))
            assert frame[p + size - 1] == 0  # no sequences
        else:
            out.append((kind, None, None))
        p += 1 if kind == 1 else size
        if last:
            assert p == len(frame)
            return out


@pytest.mark.parametrize("name,data,segment", CASES, ids=[c[0] for c in CASES])
def test_libzstd_decodes_the_restatement(name, data, segment):
    f = Z.encode_frame(data, segment)
    assert E.zstd_decompress_bound(f) == len(data)
    assert E.zstd_decompress(f) == data.tobytes()
    assert len(f) <= Z.frame_bound(len(data), segment)
    assert len(blocks(f)) == max(1, Z.n_blocks(len(data), segment))


def test_block_policy_covers_every_form():
    kinds = {}
    for name, data, segment in CASES:
        kinds[name] = blocks(Z.encode_frame(data, segment))
    assert all(k[0] == 1 for k in kinds["constant"])                       # RLE
    assert all(k[0] == 0 for k in kinds["random"])                         # raw: Huffman cannot win
    assert kinds["geometric1023"] == [(2, 0, kinds["geometric1023"][0][2])]  # one stream
    assert all(k[:2] in ((2, 2), (2, 3)) for k in kinds["geometric131072"])  # four streams, 4- and 5-byte headers
    assert kinds["direct_weights"][0][2] >= 128                             # weights as nibbles
    assert kinds["all_256"][0][2] < 128                                     # FSE-compressed weights
    assert all(k[0] == 2 for k in kinds["length_limited"])
    assert all(k[0] in (1, 2) for k in kinds["planes_m3_1"])


def test_code_lengths_limited_and_complete():
    for data in (K.fibonacci_bytes(300000, 2), np.arange(256, dtype=np.uint8), np.array([0, 0, 0, 9], np.uint8)):
        lens = Z.code_lengths(np.bincount(data, minlength=256))
        used = lens[lens > 0]
        assert used.max() <= Z.MAX_BITS and len(used) == len(np.unique(data))
        assert sum(2.0 ** -int(n) for n in used) == 1.0  # a complete prefix code
    assert Z.code_lengths(np.bincount(K.fibonacci_bytes(300000, 2), minlength=256)).max() == Z.MAX_BITS


def test_deterministic():
    data = CASES[-1][1]
    assert Z.encode_frame(data, 96 * 128) == Z.encode_frame(data.copy(), 96 * 128)


def test_set_coder_rejects_unknown_value(tmp_path):
    lib = _lib.load()
    z = lib.rirb_z_open_file_write(str(tmp_path / "a.bin").encode(), 32, 16, 50, 1, 1)
    assert z > 0, _lib.last_error()
    assert lib.rirb_z_set_coder(z, 2) == -1 and "coder" in _lib.last_error()
    assert lib.rirb_z_set_coder(z, -1) == -1
    assert lib.rirb_z_set_coder(z, 0) == 0
    lib.rirb_z_close_file(z)
    assert lib.rirb_z_set_coder(z, 0) == -1  # closed


@pytest.mark.skipif(_lib.device_available(), reason="checks behaviour WITHOUT a CUDA device")
def test_device_coder_without_gpu_fails_cleanly(tmp_path):
    from librir_b200 import tools

    lib = _lib.load()
    fn = tmp_path / "m1.bin"
    z = lib.rirb_z_open_file_write(str(fn).encode(), 32, 16, 50, 1, 1)
    assert z > 0
    assert lib.rirb_z_set_coder(z, 1) == -1 and "CUDA device" in _lib.last_error()
    img = np.arange(32 * 16, dtype=np.uint16)
    assert lib.rirb_z_write_images(z, img.ctypes.data, 1, np.zeros(1, np.int64).ctypes.data, 1) == 0  # still the host coder
    lib.rirb_z_close_file(z)
    with pytest.raises(RuntimeError, match="device coder"):
        tools.ZFileWriter(tmp_path / "m1b.bin", 32, 16, method=1, coder="gpu")
    with pytest.raises(ValueError):
        tools.ZFileWriter(tmp_path / "m1c.bin", 32, 16, method=1, coder="cuda")
    buf = np.zeros(64, np.uint8)
    assert lib.rirb_zstd_encode_batch(buf.ctypes.data, 1, 8, 0, buf.ctypes.data, 32, buf.ctypes.data) == -1
