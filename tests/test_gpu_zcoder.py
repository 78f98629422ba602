"""The device zstd coder (librir_b200/csrc/zcoder.cu): byte for byte what oracle/zcoder.py writes, and the zstd movie file
written with it (coder="gpu") reads back as the movie, through this library, libzstd and the reference's reader."""
import ctypes as ct
import os

import numpy as np
import pytest

from tests import vio_cases as C
from tests import zcoder_cases as K

pytestmark = pytest.mark.gpu

torch = pytest.importorskip("torch")

from librir_b200 import _lib, tools  # noqa: E402
from librir_b200 import entropy as E  # noqa: E402
from oracle import container as oc  # noqa: E402
from oracle import zcoder as Z  # noqa: E402

CASES = K.cases()


def device_encode(payloads, segment):
    """rirb_zstd_encode_batch over n equal-length payloads [n, bytes] -> list of frames (bytes)."""
    payloads = np.ascontiguousarray(payloads, dtype=np.uint8)
    n, nbytes = payloads.shape
    stride = Z.frame_bound(nbytes, segment)
    src = torch.from_numpy(payloads).cuda()
    dst = torch.zeros((n, stride), dtype=torch.uint8, device="cuda")
    sizes = torch.full((n,), -1, dtype=torch.int64, device="cuda")
    _lib.use_torch_stream()
    lib = _lib.load()
    assert lib.rirb_zstd_encode_batch(src.data_ptr(), n, nbytes, segment, dst.data_ptr(), stride, sizes.data_ptr()) == 0, _lib.last_error()
    d, s = dst.cpu().numpy(), sizes.cpu().numpy()
    return [d[i, :s[i]].tobytes() for i in range(n)]


@pytest.mark.parametrize("name,data,segment", CASES, ids=[c[0] for c in CASES])
def test_byte_identical_to_restatement(name, data, segment):
    got = device_encode(data[None], segment)[0]
    assert got == Z.encode_frame(data, segment)
    assert E.zstd_decompress(got) == data.tobytes()


def test_batches_of_frames():
    mov = C.movie(12, 64, 80, seed=5)
    for method in (2, 3):
        p = K.planes(mov, method, gop=5)
        got = device_encode(p, 64 * 80)
        for i in range(len(p)):
            assert got[i] == Z.encode_frame(p[i], 64 * 80), (method, i)
    raw = mov.reshape(len(mov), -1).view(np.uint8)
    for i, f in enumerate(device_encode(raw, 0)):
        assert f == Z.encode_frame(raw[i]) and E.zstd_decompress(f) == raw[i].tobytes()


@pytest.mark.parametrize("h,w", [(512, 640), (2048, 2048)])
def test_full_size_planes(h, w):
    mov = C.movie(2, h, w, seed=9)
    p = K.planes(mov, 3)
    got = device_encode(p, h * w)
    for i in range(len(p)):
        assert got[i] == Z.encode_frame(p[i], h * w)
        assert E.zstd_decompress(got[i]) == p[i].tobytes()


def to_dev(a):
    return torch.from_numpy(a.view(np.int16)).cuda().view(torch.uint16)


def records(path):
    """(timestamp, zstd frame) of every record, walked from the headers on."""
    b = open(path, "rb").read()
    n = int.from_bytes(b[128 + 16:128 + 24], "little")
    p, out = 256, []
    for _ in range(n):
        ts = int.from_bytes(b[p:p + 8], "little", signed=True)
        c = int.from_bytes(b[p + 8:p + 12], "little")
        out.append((ts, b[p + 12:p + 12 + c]))
        p += 12 + c
    return out


@pytest.mark.parametrize("method,gop", [(1, 50), (2, 50), (3, 50), (3, 7), (3, 1)])
@pytest.mark.parametrize("shape", [(130, 40, 48), (33, 19, 24), (5, 64, 80)])
def test_round_trip_in_pieces(tmp_path, method, gop, shape):
    t, h, w = shape
    mov = C.movie(t, h, w, seed=method * 10 + gop)
    ts = np.arange(t, dtype=np.int64) * 1000 + 5
    files = {}
    for coder in ("gpu", "host"):
        fn = str(tmp_path / f"{coder}.bin")
        wr = tools.ZFileWriter(fn, w, h, method=method, clevel=3, gop=gop, coder=coder)
        # pieces that do not respect GOP boundaries, host and device pointers mixed
        cuts = [0, 1, 2, min(t, 2 + gop + 3), min(t, 2 * gop + 9), t]
        for a, b in zip(cuts[:-1], cuts[1:]):
            if b > a:
                part = np.ascontiguousarray(mov[a:b])
                wr.add_images(to_dev(part) if a % 2 else part, ts[a:b])
        assert wr.close() > 256
        files[coder] = fn
    r = tools.ZFileReader(files["gpu"])
    assert r.images == t and (r.height, r.width) == (h, w)
    assert np.array_equal(r.timestamps, ts)
    assert np.array_equal(r.read_images(0, t), mov)
    for i in (t - 1, 0, t // 2, min(t - 1, gop), min(t - 1, gop + 1), 1):
        assert np.array_equal(r.read_image(i), mov[i]), i
    out = torch.empty((min(t, 11), h, w), dtype=torch.uint16, device="cuda")
    assert _lib.load().rirb_z_read_images(r.handle, t - out.shape[0], out.shape[0], out.data_ptr(), None, 0) == 0
    assert np.array_equal(out.cpu().view(torch.int16).numpy().view(np.uint16), mov[t - out.shape[0]:])
    r.close()
    # every record decodes (libzstd) to what the host coder's record of the same frame decodes to
    g, hst = records(files["gpu"]), records(files["host"])
    assert len(g) == len(hst) == t
    for (tg, fg), (th, fh) in zip(g, hst):
        assert tg == th and E.zstd_decompress(fg) == E.zstd_decompress(fh)


@pytest.mark.parametrize("method", [1, 3])
def test_long_write_spans_passes_and_is_deterministic(tmp_path, method):
    t, h, w = 230, 512, 640
    rng = np.random.default_rng(method)
    base = C.movie(10, h, w, seed=method)
    mov = base[rng.integers(0, 10, t)] + rng.integers(0, 4, (t, 1, 1)).astype(np.uint16)
    ts = np.arange(t, dtype=np.int64)
    d = to_dev(mov)
    for k in range(2):
        with tools.ZFileWriter(tmp_path / f"{k}.bin", w, h, method=method, gop=50, coder="gpu") as wr:
            wr.add_images(d if k else mov, ts)  # device frames, then the same frames from the host
    a, b = open(tmp_path / "0.bin", "rb").read(), open(tmp_path / "1.bin", "rb").read()
    assert a == b
    with tools.ZFileReader(tmp_path / "0.bin") as r:
        assert np.array_equal(r.read_images(0, t), mov)
        out = torch.empty((t, h, w), dtype=torch.uint16, device="cuda")
        r.read_images(0, t, out=out)
        assert np.array_equal(out.cpu().view(torch.int16).numpy().view(np.uint16), mov)
    payload = K.planes(mov, 3) if method == 3 else mov.reshape(t, -1).view(np.uint8)
    for i, (_ts, f) in enumerate(records(tmp_path / "0.bin")[:3]):
        assert f == Z.encode_frame(payload[i], h * w if method == 3 else 0)
    os.remove(tmp_path / "0.bin")
    os.remove(tmp_path / "1.bin")


def test_coders_mix_in_one_file(tmp_path):
    mov = C.movie(20, 32, 48, seed=2)
    ts = np.arange(20, dtype=np.int64)
    lib = _lib.load()
    z = lib.rirb_z_open_file_write(str(tmp_path / "mix.bin").encode(), 48, 32, 50, 1, 3)
    for a in range(0, 20, 5):
        assert lib.rirb_z_set_coder(z, (a // 5) % 2) == 0
        assert lib.rirb_z_write_images(z, mov[a:a + 5].ctypes.data, 5, ts[a:a + 5].ctypes.data, 0) == 0
    lib.rirb_z_close_file(z)
    with tools.ZFileReader(tmp_path / "mix.bin") as r:
        assert np.array_equal(r.read_images(0, 20), mov)


@pytest.mark.skipif(not oc.have_ref(), reason="oracle/_ref not built (no /root/reference here)")
def test_reference_reads_method1_gpu_file(tmp_path):
    mov = C.movie(140, 48, 64, seed=8)
    ts = np.arange(140, dtype=np.int64) * 20_000_000
    p = tmp_path / "gpu.bin"
    with tools.ZFileWriter(p, 64, 48, rate=50, coder="gpu") as w:
        w.add_images(mov, ts)
    frames, times = oc.ref_read_zfile(p)
    assert np.array_equal(frames, mov) and np.array_equal(times, ts)


def test_dropin_saver_entropy_coder_gpu(tmp_path):
    vio = ct.CDLL(os.path.join(os.path.dirname(_lib.lib_path()), "libvideo_io_b200.so"))
    mov = C.movie(12, 64, 96, seed=6)
    fn = str(tmp_path / "saver.bin").encode()
    s = vio.h264_open_file(fn, 96, 64, 64)
    assert s > 0
    assert vio.h264_set_parameter(s, b"entropyCoder", b"cuda") == -1
    assert vio.h264_set_parameter(s, b"entropyCoder", b"gpu") == 0
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
    assert records(fn.decode())[1][1] == Z.encode_frame(lo_hi[1], 64 * 96)
