"""The corpus of the device zstd decoder (tests/zdecoder_cases.py) against the system libzstd, its coverage of the format
features the decoder takes, and the decoder's C entry and switch without a device.  CPU only; tests/test_gpu_zdecoder.py
runs the kernels on the corpus."""
import numpy as np
import pytest

from librir_b200 import _lib
from tests import zdecoder_cases as D

CASES = D.cases()

FEATURES = {
    "single_segment", "window_descriptor", "fcs0", "fcs1", "fcs2", "fcs4", "block0", "block1", "block2",
    "literals0", "literals1", "literals2", "literals3", "streams1", "streams4", "weights_direct", "weights_fse",
    "nseq0", "nseq1", "nseq2", "nseq3", "checksum",
} | {f"{t}_mode{m}" for t in ("LL", "OF", "ML") for m in range(4)}


@pytest.mark.parametrize("name,frame,payload", CASES, ids=[c[0] for c in CASES])
def test_libzstd_decodes_every_corpus_frame(name, frame, payload):
    assert D.decompress(frame, len(payload)) == payload


def test_corpus_covers_every_feature():
    seen = set()
    for _, frame, _ in CASES:
        seen |= D.walk(frame)
    assert FEATURES <= seen, sorted(FEATURES - seen)


def test_hand_built_frames():
    f, p = D.rle_literals_frame(0x33, 20)
    assert D.walk(f) >= {"literals1", "nseq0"} and D.decompress(f, 20) == p == b"\x33" * 20
    f, p = D.long_count_frame()
    assert "nseq3" in D.walk(f) and len(p) == 4 * 32512 and D.decompress(f, len(p)) == p


@pytest.mark.skipif(_lib.device_available(), reason="checks behaviour WITHOUT a CUDA device")
def test_decode_batch_without_gpu_fails_cleanly():
    lib = _lib.load()
    buf = np.zeros(64, np.uint8)
    p = buf.ctypes.data
    assert lib.rirb_zstd_decode_batch(p, p, p, 1, p, 32, 32, p) == -1
    assert "CUDA device" in _lib.last_error()


def test_decode_batch_rejects_bad_arguments():
    lib = _lib.load()
    buf = np.zeros(64, np.uint8)
    p = buf.ctypes.data
    assert lib.rirb_zstd_decode_batch(p, p, p, -1, p, 32, 32, p) == -1
    assert lib.rirb_zstd_decode_batch(p, p, p, 1, p, 16, 32, p) == -1  # slots would overlap
    assert lib.rirb_zstd_decode_batch(None, p, p, 1, p, 32, 32, p) == -1


def test_zstd_decoder_switch():
    lib = _lib.load()
    for v in (b"0", b"2", b"1"):
        assert lib.rirb_set_parameter(b"zstd_decoder", v) == 0
