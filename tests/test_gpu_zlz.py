"""Coder 2, the device zstd coder with LZ matches (librir_b200/csrc/zcoder.cu, rirb_zstd_encode_batch_lz): byte for byte
what oracle/zlz.py (encode_frame_lz) writes, decoded by the device decoder and libzstd, and the zstd movie file written
with coder="gpu-lz" reads back through every decoder path, the drop-in saver and the reference's reader."""
import ctypes as ct
import os

import numpy as np
import pytest

from tests import vio_cases as C
from tests import zcoder_cases as K
from tests import zlz_cases as L

pytestmark = pytest.mark.gpu

torch = pytest.importorskip("torch")

from librir_b200 import _lib, tools  # noqa: E402
from librir_b200 import entropy as E  # noqa: E402
from oracle import container as oc  # noqa: E402
from oracle import zcoder as Z1  # noqa: E402
from oracle import zlz as Z  # noqa: E402
from tests.test_gpu_zcoder import records, to_dev  # noqa: E402
from tests.test_gpu_zdecoder import check_file, device_decode  # noqa: E402

CASES = L.cases()


def device_encode_lz(payloads, segment):
    """rirb_zstd_encode_batch_lz over n equal-length payloads [n, bytes] -> list of frames (bytes)."""
    payloads = np.ascontiguousarray(payloads, dtype=np.uint8)
    n, nbytes = payloads.shape
    stride = Z1.frame_bound(nbytes, segment)
    src = torch.from_numpy(payloads).cuda()
    dst = torch.zeros((n, stride), dtype=torch.uint8, device="cuda")
    sizes = torch.full((n,), -1, dtype=torch.int64, device="cuda")
    _lib.use_torch_stream()
    lib = _lib.load()
    assert lib.rirb_zstd_encode_batch_lz(src.data_ptr(), n, nbytes, segment, dst.data_ptr(), stride, sizes.data_ptr()) == 0, _lib.last_error()
    d, s = dst.cpu().numpy(), sizes.cpu().numpy()
    return [d[i, :s[i]].tobytes() for i in range(n)]


def check_frames(frames, payloads, segment):
    """Frames equal the restatement's, and the device decoder gives back the payloads with status = size."""
    for f, p in zip(frames, payloads):
        assert f == Z.encode_frame_lz(p, segment)
    st, out, _ = device_decode(frames, [payloads.shape[1]])
    assert (st == payloads.shape[1]).all(), st
    assert np.array_equal(out[1:1 + len(frames), :payloads.shape[1]], payloads)


@pytest.mark.parametrize("name,data,segment", CASES, ids=[c[0] for c in CASES])
def test_byte_identical_to_restatement(name, data, segment):
    got = device_encode_lz(data[None], segment)[0]
    assert got == Z.encode_frame_lz(data, segment)
    assert E.zstd_decompress(got) == data.tobytes()
    if len(data):
        check_frames([got], data[None], segment)


def test_batches_of_frames():
    mov = C.movie(12, 64, 80, seed=5)
    for method in (2, 3):
        p = K.planes(mov, method, gop=5)
        check_frames(device_encode_lz(p, 64 * 80), p, 64 * 80)
    raw = mov.reshape(len(mov), -1).view(np.uint8)
    check_frames(device_encode_lz(raw, 0), raw, 0)


def test_short_payloads():
    rng = np.random.default_rng(3)
    for n in range(1, 301):
        p = np.stack([np.tile(rng.integers(0, 256, 1 + k * 5).astype(np.uint8), n)[:n] for k in range(3)])
        check_frames(device_encode_lz(p, 0), p, 0)


@pytest.mark.parametrize("h,w", [(512, 640), (2048, 2048)])
def test_full_size_planes(h, w):
    mov = C.movie(2, h, w, seed=9)
    for method in (2, 3):
        p = K.planes(mov, method)
        check_frames(device_encode_lz(p, h * w), p, h * w)


def test_many_blocks_span_sort_chunks():
    """More than 512 blocks in one call: the candidate sort runs in several chunks."""
    mov = C.movie(100, 512, 640, seed=12)
    p = K.planes(mov, 2)
    got = device_encode_lz(p, 512 * 640)
    for i in (0, 57, 99):
        assert got[i] == Z.encode_frame_lz(p[i], 512 * 640), i
    for f, q in zip(got, p):
        assert E.zstd_decompress(f) == q.tobytes()


@pytest.mark.parametrize("method,gop", [(1, 50), (2, 50), (3, 7)])
def test_round_trip_in_pieces(tmp_path, method, gop):
    t, h, w = 60, 48, 64
    mov = C.movie(t, h, w, seed=method * 10 + gop)
    ts = np.arange(t, dtype=np.int64) * 1000 + 5
    fn = tmp_path / f"lz{method}.bin"
    wr = tools.ZFileWriter(fn, w, h, method=method, gop=gop, coder="gpu-lz")
    cuts = [0, 1, 2, 2 + gop + 3, min(t, 2 * gop + 9), t]  # pieces across GOP boundaries, host and device frames mixed
    for a, b in zip(cuts[:-1], cuts[1:]):
        if b > a:
            part = np.ascontiguousarray(mov[a:b])
            wr.add_images(to_dev(part) if a % 2 else part, ts[a:b])
    assert wr.close() > 256
    with tools.ZFileReader(fn) as r:
        assert np.array_equal(r.timestamps, ts)
    check_file(fn, mov, gop=gop)
    payload = mov.reshape(t, -1).view(np.uint8) if method == 1 else K.planes(mov, method, gop=gop)
    for i, (_ts, f) in enumerate(records(fn)):
        assert f == Z.encode_frame_lz(payload[i], 0 if method == 1 else h * w), i


@pytest.mark.parametrize("method", [1, 2])
def test_same_movie_twice_gives_identical_files(tmp_path, method):
    t, h, w = 120, 512, 640
    mov = C.movie(t, h, w, seed=method)
    ts = np.arange(t, dtype=np.int64)
    for k in range(2):
        with tools.ZFileWriter(tmp_path / f"{k}.bin", w, h, method=method, gop=50, coder="gpu-lz") as wr:
            wr.add_images(to_dev(mov) if k else mov, ts)
    a, b = open(tmp_path / "0.bin", "rb").read(), open(tmp_path / "1.bin", "rb").read()
    assert a == b
    with tools.ZFileReader(tmp_path / "0.bin") as r:
        assert np.array_equal(r.read_images(0, t), mov)


@pytest.mark.skipif(not oc.have_ref(), reason="oracle/_ref not built (no /root/reference here)")
def test_reference_reads_method1_lz_file(tmp_path):
    mov = C.movie(140, 48, 64, seed=8)
    ts = np.arange(140, dtype=np.int64) * 20_000_000
    p = tmp_path / "lz.bin"
    with tools.ZFileWriter(p, 64, 48, rate=50, coder="gpu-lz") as w:
        w.add_images(mov, ts)
    frames, times = oc.ref_read_zfile(p)
    assert np.array_equal(frames, mov) and np.array_equal(times, ts)


def test_dropin_saver_entropy_coder_gpu_lz(tmp_path):
    vio = ct.CDLL(os.path.join(os.path.dirname(_lib.lib_path()), "libvideo_io_b200.so"))
    mov = C.movie(12, 64, 96, seed=6)
    fn = str(tmp_path / "saver.bin").encode()
    s = vio.h264_open_file(fn, 96, 64, 64)
    assert s > 0
    assert vio.h264_set_parameter(s, b"entropyCoder", b"gpu-lz") == 0
    assert vio.h264_set_parameter(s, b"GOP", b"5") == 0
    for t in range(len(mov)):
        assert vio.h264_add_image_lossless(s, mov[t].ctypes.data_as(ct.c_void_p), ct.c_int64(1000 * t), 0, None, None, None, None) == 0
    vio.h264_close_file(s)
    fmt = ct.c_int(0)
    cam = vio.open_camera_file(fn, ct.byref(fmt))
    assert cam > 0 and vio.get_image_count(cam) == len(mov)
    img = np.empty((64, 96), dtype=np.uint16)
    for t in (len(mov) - 1, 0, 7):
        assert vio.load_image(cam, t, 0, img.ctypes.data_as(ct.c_void_p)) == 0 and np.array_equal(img, mov[t])
    vio.close_camera(cam)
    lo_hi = K.planes(mov, 3, gop=5)
    assert records(fn.decode())[1][1] == Z.encode_frame_lz(lo_hi[1], 64 * 96)


def test_lz_switch_mixes_in_one_file(tmp_path):
    """rirb_z_set_lz turns LZ matches on and off between writes of one file; every record is its coder's frame."""
    mov = C.movie(20, 32, 48, seed=2)
    ts = np.arange(20, dtype=np.int64)
    lib = _lib.load()
    z = lib.rirb_z_open_file_write(str(tmp_path / "mix.bin").encode(), 48, 32, 50, 1, 3)
    assert lib.rirb_z_set_coder(z, 1) == 0
    for a in range(0, 20, 5):
        assert lib.rirb_z_set_lz(z, (a // 5) % 2) == 0
        assert lib.rirb_z_write_images(z, mov[a:a + 5].ctypes.data, 5, ts[a:a + 5].ctypes.data, 0) == 0
    lib.rirb_z_close_file(z)
    raw = mov.reshape(20, -1).view(np.uint8)
    for i, (_ts, f) in enumerate(records(tmp_path / "mix.bin")):
        assert f == (Z.encode_frame_lz(raw[i]) if (i // 5) % 2 else Z1.encode_frame(raw[i])), i
    with tools.ZFileReader(tmp_path / "mix.bin") as r:
        assert np.array_equal(r.read_images(0, 20), mov)
