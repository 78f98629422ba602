"""Random write / read programs over the zstd movie file (tools.ZFileWriter / ZFileReader and the C ABI): method 1 / 2 / 3,
GOP 1-60, the host coder, "gpu" and "gpu-lz" switched between calls, random compression levels and thread counts, pieces
of random length from numpy arrays and device tensors; reads of random ranges and single frames in random order, to
numpy, into device tensors and on a side stream, each under a random "zstd_decoder" setting.  The programs run as the
sequences that move the work buffers between files: files of different frame sizes one after another (the parked set
grows and is handed on), two writers open at once and a reader next to an open writer, two host threads with a file
each, and with two GPUs a file written on one device and read on the other.  Every read is the movie; the headers and
timestamps are the movie's; method-1 files of the host coder are the bytes oracle/container.py writes, every method-1
file reads back through it, and every record of a method-2/3 file is, decoded by libzstd, the byte planes of its GOP.
``RIRB_FUZZ_SEED=<n> RIRB_FUZZ_SCALE=<k>`` runs k times as many programs from other seeds."""
import os
import threading

import numpy as np
import pytest

from tests import vio_cases as C
from tests import zcoder_cases as K

pytestmark = pytest.mark.gpu

torch = pytest.importorskip("torch")
if not torch.cuda.is_available():  # pragma: no cover
    pytest.skip("needs a CUDA device", allow_module_level=True)

from librir_b200 import _lib, tools  # noqa: E402
from librir_b200 import entropy as E  # noqa: E402
from oracle import container as oc  # noqa: E402
from tests.test_gpu_zcoder import records, to_dev  # noqa: E402

SEED = int(os.environ.get("RIRB_FUZZ_SEED", "0"))
SCALE = max(1, int(os.environ.get("RIRB_FUZZ_SCALE", "1")))
CODERS = ("host", "gpu", "gpu-lz")


class Program:
    """One file: a random movie written in random pieces with random coders, then read back at random."""

    def __init__(self, rng, path, t, h, w):
        self.rng, self.path = rng, str(path)
        self.method, self.gop, self.clevel = int(rng.integers(1, 4)), int(rng.integers(1, 61)), int(rng.integers(1, 10))
        self.mov = C.movie(t, h, w, seed=int(rng.integers(0, 1 << 20)))
        self.ts = np.cumsum(rng.integers(1, 40_000_000, t)).astype(np.int64)
        self.writer = tools.ZFileWriter(self.path, w, h, method=self.method, clevel=self.clevel, gop=self.gop)
        self.done, self.coders = 0, set()

    def write_piece(self):
        """One call of rirb_z_write_images with a piece that ignores GOP and pass boundaries; False once all is written."""
        rng, lib, t = self.rng, _lib.load(), len(self.mov)
        a = self.done
        b = min(t, a + int(rng.integers(1, 2 * self.gop + 3)))
        coder = CODERS[int(rng.integers(0, 3))]
        assert lib.rirb_z_set_coder(self.writer.handle, int(coder != "host")) == 0, _lib.last_error()
        assert lib.rirb_z_set_lz(self.writer.handle, int(coder == "gpu-lz")) == 0, _lib.last_error()
        self.writer.threads = int(rng.integers(0, 5))
        part = np.ascontiguousarray(self.mov[a:b])
        self.writer.add_images(to_dev(part) if rng.random() < 0.5 else part, self.ts[a:b])
        self.coders.add(coder)
        self.done = b
        return b < t

    def write(self):
        while self.done < len(self.mov):
            self.write_piece()
        assert self.writer.close() > 256

    def read(self, reader, n_reads):
        """Random reads of reader (this file), each under a random zstd_decoder setting."""
        rng, mov = self.rng, self.mov
        t, h, w = mov.shape
        try:
            for _ in range(n_reads):
                pos = int(rng.integers(0, t))
                count = 1 if rng.random() < 0.3 else int(rng.integers(1, t - pos + 1))
                _lib.set_parameter("zstd_decoder", int(rng.integers(0, 3)))
                where = int(rng.integers(0, 4))
                if where == 0:
                    got = reader.read_images(pos, count)
                elif where == 1:
                    got = reader.read_image(pos)[None]
                    count = 1
                else:
                    stream = torch.cuda.Stream() if where == 3 else torch.cuda.current_stream()
                    with torch.cuda.stream(stream):
                        out = torch.empty((count, h, w), dtype=torch.uint16, device="cuda")
                        reader.read_images(pos, count, out)
                    stream.synchronize()
                    _lib.use_torch_stream()  # back to the default stream for this thread
                    got = out.cpu().view(torch.int16).numpy().view(np.uint16)
                assert np.array_equal(got, mov[pos:pos + count]), (self.path, self.method, pos, count, where)
        finally:
            _lib.set_parameter("zstd_decoder", 1)

    def check(self, n_reads=6):
        t, h, w = self.mov.shape
        with tools.ZFileReader(self.path, threads=int(self.rng.integers(0, 5))) as r:
            assert len(r) == t and (r.height, r.width) == (h, w)
            assert _lib.load().rirb_z_method(r.handle) == self.method
            assert np.array_equal(r.timestamps, self.ts)
            self.read(r, n_reads)
        self.check_records()

    def check_records(self):
        t, h, w = self.mov.shape
        if self.method == 1:
            frames, times, _ = oc.read_zfile(self.path)
            assert np.array_equal(frames, self.mov) and np.array_equal(times, self.ts)
            if self.coders == {"host"}:
                ref = self.path + ".oracle"
                oc.write_zfile(ref, self.mov, self.ts, rate=50, clevel=self.clevel)
                assert open(ref, "rb").read() == open(self.path, "rb").read()
                os.remove(ref)
        else:
            planes = K.planes(self.mov, self.method, gop=self.gop)
            for i, (ts, f) in enumerate(records(self.path)):
                assert ts == self.ts[i] and E.zstd_decompress(f) == planes[i].tobytes(), (self.path, i)


def used_memory():
    torch.cuda.synchronize()
    torch.cuda.empty_cache()
    free, total = torch.cuda.mem_get_info()
    return total - free


def test_files_one_after_another(tmp_path):
    """Small, large, small frame sizes and random ones: the parked buffer set grows and is handed from file to file.  The
    rounds repeat the same programs, so the first one grows the parked set to all they need; after the later rounds the
    device memory in use is what it was after the first (nothing a file takes stays behind when it is closed)."""
    shapes = [(24, 32), (512, 640), (48, 64)]
    after_first = None
    for rnd in range(1 + 2 * SCALE):
        rng = np.random.default_rng(801 + SEED)
        extra = [(int(rng.integers(1, 300)), int(rng.integers(1, 300))) for _ in range(2)]
        for k, (h, w) in enumerate(shapes + extra):
            t = int(rng.integers(2, 13)) if h * w > 100_000 else int(rng.integers(1, 90))
            p = Program(rng, tmp_path / f"r{rnd}_{k}.bin", t, h, w)
            p.write()
            p.check()
            os.remove(p.path)
        if after_first is None:
            after_first = used_memory()
    assert used_memory() <= after_first + (64 << 20), (after_first, used_memory())


def test_two_writers_and_a_reader(tmp_path):
    """Two files written at once in interleaved pieces and closed in either order; a reader of the first open while the
    second is still being written."""
    rng = np.random.default_rng(802 + SEED)
    for case in range(3 * SCALE):
        shape = [(int(rng.integers(8, 120)), int(rng.integers(8, 160))) for _ in range(2)]
        a = Program(rng, tmp_path / f"a{case}.bin", int(rng.integers(1, 70)), *shape[0])
        b = Program(rng, tmp_path / f"b{case}.bin", int(rng.integers(1, 70)), *shape[1])
        progs = [a, b]
        busy = [True, True]
        while busy[0] and busy[1]:
            k = int(rng.integers(0, 2))
            busy[k] = progs[k].write_piece()
        first = progs[0] if not busy[0] else progs[1]
        other = progs[1] if first is progs[0] else progs[0]
        assert first.writer.close() > 256
        with tools.ZFileReader(first.path) as r:  # while the other writer is open
            first.read(r, 3)
            if other.done < len(other.mov):
                other.write_piece()
            first.read(r, 3)
        other.write()
        first.check(3)
        other.check(3)


def test_two_host_threads(tmp_path):
    """Two host threads, each running programs on its own files at the same time (the parked set is process-wide)."""
    errors = []

    def run(k):
        try:
            torch.cuda.set_device(0)
            rng = np.random.default_rng(803 + 10 * k + SEED)
            for i in range(3 * SCALE):
                h, w = [(24, 32), (256, 320), (40, 56)][i % 3]
                p = Program(rng, tmp_path / f"t{k}_{i}.bin", int(rng.integers(1, 40)), h, w)
                p.write()
                p.check(4)
        except BaseException as e:  # noqa: BLE001 -- reported by the main thread
            errors.append((k, e))
        finally:
            _lib.load().rirb_release_thread_resources()

    threads = [threading.Thread(target=run, args=(k,)) for k in range(2)]
    for th in threads:
        th.start()
    for th in threads:
        th.join()
    assert not errors, errors


def test_file_moves_between_devices(tmp_path):
    """A file written on device 0 and read on device 1, and a reader whose calls alternate devices: the buffer set follows
    the calling thread's device.  Needs two GPUs (skipped on a single-GPU machine)."""
    lib = _lib.load()
    if lib.rirb_device_count() < 2:
        pytest.skip("needs two CUDA devices")
    rng = np.random.default_rng(804 + SEED)
    try:
        for case in range(2 * SCALE):
            torch.cuda.set_device(0)
            assert lib.rirb_set_device(0) == 0
            p = Program(rng, tmp_path / f"d{case}.bin", int(rng.integers(1, 40)), 64, 80)
            p.write()
            with tools.ZFileReader(p.path) as r:
                for k in range(4):
                    dev = (k + 1) % 2
                    torch.cuda.set_device(dev)
                    assert lib.rirb_set_device(dev) == 0
                    _lib.use_torch_stream()
                    p.read(r, 2)
            p.check_records()
    finally:
        torch.cuda.set_device(0)
        lib.rirb_set_device(0)
        _lib.use_torch_stream()
