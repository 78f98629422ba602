"""The device zstd decoder (librir_b200/csrc/zdecoder.cu): every corpus frame of tests/zdecoder_cases.py decodes to its
payload, alone and in one mixed batch; malformed frames are rejected without touching anything outside their slot; and
the zstd movie file reads the same through the device decoder and through host libzstd (the "zstd_decoder" switch)."""
import os
import struct

import numpy as np
import pytest

from tests import container_cases as cc
from tests import vio_cases as C
from tests import zdecoder_cases as D
from tests.conftest import ir_movie

pytestmark = pytest.mark.gpu

torch = pytest.importorskip("torch")

from librir_b200 import _lib, tools  # noqa: E402
from oracle import container as oc  # noqa: E402

CASES = D.cases()
GUARD = 0xA5
GOLD = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")


def device_decode(frames, caps, stride=None):
    """rirb_zstd_decode_batch over a list of frames -> (statuses, [n, stride] output with guard bytes, stride)."""
    n = len(frames)
    cap = max(caps) if caps else 0
    stride = stride or cap + 64
    offs = np.zeros(n, np.int64)
    pos = 16  # guard bytes before the first frame too
    blob = bytearray(b"\xee" * 16)
    for i, f in enumerate(frames):
        offs[i] = pos
        blob += f + b"\xee" * 13
        pos += len(f) + 13
    src = torch.from_numpy(np.frombuffer(bytes(blob), np.uint8).copy()).cuda()
    off = torch.from_numpy(offs).cuda()
    size = torch.from_numpy(np.array([len(f) for f in frames], np.uint32).view(np.int32)).cuda()
    dst = torch.full((n + 2, stride), GUARD, dtype=torch.uint8, device="cuda")
    status = torch.full((n,), 7777, dtype=torch.int64, device="cuda")
    _lib.use_torch_stream()
    lib = _lib.load()
    # one capacity for the batch: the slots are cap bytes in a stride that leaves guard bytes behind each
    assert lib.rirb_zstd_decode_batch(src.data_ptr(), off.data_ptr(), size.data_ptr(), n, dst[1:].data_ptr(), stride, cap,
                                      status.data_ptr()) == 0, _lib.last_error()
    torch.cuda.synchronize()
    return status.cpu().numpy(), dst.cpu().numpy(), cap


@pytest.mark.parametrize("name,frame,payload", CASES, ids=[c[0] for c in CASES])
def test_corpus_frame(name, frame, payload):
    st, out, cap = device_decode([frame], [len(payload)])
    if name == "checksum":
        assert st[0] == -2
        return
    assert st[0] == len(payload)
    assert out[1, :len(payload)].tobytes() == payload
    assert (out[1, cap:] == GUARD).all() and (out[0] == GUARD).all() and (out[2] == GUARD).all()


def test_corpus_in_one_batch():
    frames = [f for _, f, _ in CASES]
    pays = [p for _, _, p in CASES]
    st, out, cap = device_decode(frames, [max(len(p) for p in pays)], stride=max(len(p) for p in pays) + 4096)
    for i, (name, _, p) in enumerate(CASES):
        if name == "checksum":
            assert st[i] == -2
            continue
        assert st[i] == len(p), name
        assert out[1 + i, :len(p)].tobytes() == p, name


def offset_past_output_frame():
    """One literal, then a match at offset 4: more than the one byte produced so far."""
    block = bytes([1 << 3, 0x41, 1, 0x54, 1, 2, 0, 0x07])
    return D.Z.MAGIC + bytes([0x20, 4]) + (1 | 2 << 1 | len(block) << 3).to_bytes(3, "little") + block


def test_malformed_frames_are_rejected():
    rng = np.random.default_rng(2024)
    names = [c[0] for c in CASES]
    _, good, good_pay = CASES[names.index("m1_level3")]
    cap = max(len(p) for _, _, p in CASES)
    frames, expect = [], []
    for name, f, p in CASES:
        muts = [f[:int(len(f) * c)] for c in (0.1, 0.5, 0.9, 0.999)]
        for _ in range(6):
            b = bytearray(f)
            if b:
                i = int(rng.integers(0, len(b)))
                b[i] = (b[i] + int(rng.integers(1, 256))) & 0xFF
            muts.append(bytes(b))
        for m in muts:
            frames += [m, good]
            expect.append(D.decompress(m, cap))
    frames.append(offset_past_output_frame())
    expect.append(D.decompress(frames[-1], cap))
    assert expect[-1] is None
    st, out, _ = device_decode(frames, [cap])
    for j, ref in enumerate(expect):
        i = 2 * j
        if st[i] >= 0:  # accepted: then exactly what libzstd makes of the mutated frame
            assert ref is not None and st[i] == len(ref) and out[1 + i, :st[i]].tobytes() == ref, j
        else:
            assert st[i] in (-1, -2), (j, st[i])
        assert (out[1 + i, cap:] == GUARD).all(), j
        if i + 1 < len(frames):  # the neighbour is intact
            assert st[i + 1] == len(good_pay) and out[2 + i, :len(good_pay)].tobytes() == good_pay, j
    assert (out[0] == GUARD).all() and (out[-1] == GUARD).all()
    # a capacity one byte short of the content
    for name, f, p in CASES:
        if len(p) and name != "checksum":
            st, out, c = device_decode([f], [len(p) - 1])
            assert st[0] == -1 and (out[1, c:] == GUARD).all() and (out[0] == GUARD).all() and (out[2] == GUARD).all(), name


def set_decoder(on):
    _lib.set_parameter("zstd_decoder", on)


def read_all(path, count=None, device=False, pos=0):
    with tools.ZFileReader(path) as r:
        n = count if count is not None else len(r) - pos
        if device:
            out = torch.empty((n, r.height, r.width), dtype=torch.int16, device="cuda")
            r.read_images(pos, n, out)
            torch.cuda.synchronize()
            return out.cpu().numpy().view(np.uint16)
        return r.read_images(pos, n)


def check_file(path, mov, gop=50):
    """Reads with every "zstd_decoder" setting (2: the device decoder wherever a read ends on the device, 1: the default
    selection, 0: host libzstd), to numpy and into HBM, whole and from GOP boundaries."""
    try:
        for on in (2, 1, 0):
            set_decoder(on)
            for device in (False, True):
                assert np.array_equal(read_all(path, device=device), mov), (on, device)
                for k in sorted({0, gop - 1, gop, min(len(mov) - 1, gop + 1), len(mov) - 1}):
                    if k < len(mov):
                        got = read_all(path, count=min(3, len(mov) - k), device=device, pos=k)
                        assert np.array_equal(got, mov[k:k + 3]), (on, device, k)
    finally:
        set_decoder(1)


@pytest.mark.parametrize("method", [1, 2, 3])
@pytest.mark.parametrize("coder", ["host1", "host2", "host12", "gpu"])
def test_file_reads_match(tmp_path, method, coder):
    mov = C.movie(60, 48, 64, seed=21)
    ts = np.arange(60, dtype=np.int64)
    p = tmp_path / f"m{method}_{coder}.bin"
    level = int(coder[4:]) if coder != "gpu" else 2
    with tools.ZFileWriter(p, 64, 48, method=method, clevel=level, gop=25, coder="gpu" if coder == "gpu" else "host") as w:
        w.add_images(mov, ts)
    check_file(p, mov, gop=25)


def test_golden_reference_file():
    check_file(os.path.join(GOLD, "zfile_ref.bin"), cc.golden_movie(), gop=3)


@pytest.mark.parametrize("method", [1, 3])
def test_large_read_spans_passes(tmp_path, method):
    mov = ir_movie(230, 512, 640, seed=5)
    p = tmp_path / f"big{method}.bin"
    with tools.ZFileWriter(p, 640, 512, method=method, clevel=2) as w:
        w.add_images(mov, np.arange(230, dtype=np.int64))
    try:
        for on in (2, 1):
            set_decoder(on)
            assert np.array_equal(read_all(p, device=True), mov)
    finally:
        set_decoder(1)


def test_mixed_coder_file(tmp_path):
    mov = C.movie(20, 32, 48, seed=2)
    ts = np.arange(20, dtype=np.int64)
    lib = _lib.load()
    z = lib.rirb_z_open_file_write(str(tmp_path / "mix.bin").encode(), 48, 32, 50, 1, 3)
    for a in range(0, 20, 5):
        assert lib.rirb_z_set_coder(z, (a // 5) % 2) == 0
        assert lib.rirb_z_write_images(z, mov[a:a + 5].ctypes.data, 5, ts[a:a + 5].ctypes.data, 0) == 0
    lib.rirb_z_close_file(z)
    check_file(tmp_path / "mix.bin", mov, gop=5)


def test_checksum_record_takes_the_host_path(tmp_path):
    mov = C.movie(6, 32, 48, seed=4)
    ts = np.arange(6, dtype=np.int64)
    body, positions, pos = b"", [], 256
    for i in range(6):
        c = D.compress(mov[i].reshape(-1).view(np.uint8), 3, checksum=int(i == 2))
        positions.append(pos)
        body += struct.pack("<qI", int(ts[i]), len(c)) + c
        pos += 12 + len(c)
    trailer = oc.build_trailer({b"positions": struct.pack("<6q", *positions)}, [{} for _ in range(6)], ts)
    p = tmp_path / "checksum.bin"
    p.write_bytes(oc.zfile_headers(48, 32, 50, 6) + body + trailer)
    assert "checksum" in D.walk(body[positions[2] - 256 + 12:positions[3] - 256])
    check_file(p, mov, gop=3)


def test_read_on_side_stream(tmp_path):
    mov = C.movie(30, 48, 64, seed=9)
    p = tmp_path / "side.bin"
    with tools.ZFileWriter(p, 64, 48, method=3, gop=10) as w:
        w.add_images(mov, np.arange(30, dtype=np.int64))
    s = torch.cuda.Stream()
    with torch.cuda.stream(s):
        out = torch.empty((30, 48, 64), dtype=torch.int16, device="cuda")
        with tools.ZFileReader(p) as r:
            r.read_images(0, 30, out)
        got = out.view(-1).cpu().numpy().view(np.uint16).reshape(30, 48, 64)
    s.synchronize()
    assert np.array_equal(got, mov)
