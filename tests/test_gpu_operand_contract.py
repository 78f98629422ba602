"""The operand contract on the device: wrong outputs, overlapping operands, every kind of memory, scratch slots under load.

* Facade entries given a torch CUDA output one frame / row / column short: the output is a view at the start of a
  0xA5-filled buffer as large as the correct output, so a write past the view lands in the guard inside the allocation.
  The call must be refused and every guard byte must survive.
* The C ABI with device operands that share one element, one row or one frame: -1, a ``rirb_last_error`` text, no
  launch, and not one byte of the backing buffer changed.  Equal pointers stay allowed where an entry is documented
  in place; overlapping host operands are staged and give the out-of-place answer.
* Every C-ABI entry with pointer operands, each operand in turn as pageable, pinned, registered or managed memory (the
  rest on the device), plus one call with the kinds mixed: the output bits equal the all-device call, which the rest of
  the suite holds to the oracle.  Pageable outputs of 1 B, 256 KiB +- 1, 1 MiB +- 1 and 64 MiB +- 1 land on the edges
  of the pinned ring that stages them (and past its 64 MiB limit).
* Call sequences without synchronisation that reuse and grow the per-thread scratch slots, switch streams and nest
  entries: each output equals the same call made alone.
"""
import ctypes as ct
import glob
import os

import numpy as np
import pytest

from tests.conftest import ir_movie

pytestmark = pytest.mark.gpu

torch = pytest.importorskip("torch")

from librir_b200 import _lib, movie, signal_processing as sp, tools, video_io as vio  # noqa: E402

SENTINEL = 0xA5
N, H, W = 4, 16, 32
META = 3
LS = 64  # padded plane line size of the split / merge cases


@pytest.fixture(scope="module")
def lib():
    torch.cuda.set_device(0)
    lib = _lib.load()
    lib.rirb_set_stream(None)
    return lib


def cudart():
    """The CUDA runtime torch loaded (cudaMallocManaged is not in torch.cuda.cudart())."""
    for name in ["libcudart.so.12"] + sorted(glob.glob(os.path.join(os.path.dirname(torch.__file__), "..", "nvidia", "cuda_runtime",
                                                                    "lib", "libcudart.so*"))) + ["/usr/local/cuda/lib64/libcudart.so"]:
        try:
            rt = ct.CDLL(name)
            rt.cudaMallocManaged.argtypes = [ct.POINTER(ct.c_void_p), ct.c_size_t, ct.c_uint]
            rt.cudaFree.argtypes = [ct.c_void_p]
            return rt
        except OSError:
            continue
    pytest.fail("no CUDA runtime library to allocate managed memory with")


# ---------------------------------------------------------------------------------------------
# buffers of every kind
# ---------------------------------------------------------------------------------------------
KINDS = ("pageable", "pinned", "registered", "managed", "device")


class Buf:
    """`data` (a numpy array) copied into a buffer of one memory kind; `.ptr`, `.read()` -> its bytes now."""

    def __init__(self, kind, data, pool):
        raw = np.ascontiguousarray(data).reshape(-1).view(np.uint8)
        self.kind, self.nbytes = kind, raw.size
        if kind in ("pageable", "registered"):
            self.host = raw.copy()
            self.ptr = self.host.ctypes.data
            if kind == "registered":
                assert int(torch.cuda.cudart().cudaHostRegister(self.ptr, self.nbytes, 0)) == 0
                pool.append(lambda p=self.ptr: torch.cuda.cudart().cudaHostUnregister(p))
        elif kind == "pinned":
            self.t = torch.from_numpy(raw.copy()).pin_memory()
            self.ptr = self.t.data_ptr()
        elif kind == "device":
            self.t = torch.from_numpy(raw.copy()).cuda()
            self.ptr = self.t.data_ptr()
        else:
            rt = cudart()
            p = ct.c_void_p()
            assert rt.cudaMallocManaged(ct.byref(p), max(self.nbytes, 1), 1) == 0
            self.ptr = p.value
            ct.memmove(self.ptr, raw.ctypes.data, self.nbytes)
            pool.append(lambda p=self.ptr, rt=rt: rt.cudaFree(p))

    def read(self):
        torch.cuda.synchronize()
        if self.kind in ("pageable", "registered"):
            return self.host.copy()
        if self.kind == "managed":
            return np.frombuffer(ct.string_at(self.ptr, self.nbytes), np.uint8).copy()
        return self.t.cpu().numpy().copy()


@pytest.fixture
def pool():
    """Clean-ups of registered and managed buffers, run after the case whatever happened in it."""
    fns = []
    yield fns
    torch.cuda.synchronize()
    for f in reversed(fns):
        f()


# ---------------------------------------------------------------------------------------------
# the entries: operands (role, initial contents) and the call
# ---------------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def data(lib):
    mov = ir_movie(N, H, W, seed=77)
    lo, hi = vio.precode_movie(mov, 2, True, 0)
    bp_full = sp.bad_pixels_create(mov[0])
    bpl = vio.LoaderBadPixels(mov[0])
    it = (np.arange(H * W) % 251).astype(np.uint8).reshape(H, W)
    planes = [np.ascontiguousarray(np.random.default_rng(k).integers(0, 256, (H, LS), dtype=np.uint8)) for k in range(3)]
    sx = np.array([0.5, -1.25, 2.0, 0.75][:N], np.float64)
    sy = np.array([0.25, 1.5, -0.5, 0.0][:N], np.float64)
    each = H * W * 2
    zsrc = mov.reshape(-1).view(np.uint8)
    d_src = torch.from_numpy(zsrc.copy()).cuda()
    d_dst = torch.zeros(N * (each + 64), dtype=torch.uint8, device="cuda")
    d_sizes = torch.zeros(N, dtype=torch.int64, device="cuda")
    assert lib.rirb_zstd_encode_batch(d_src.data_ptr(), N, each, 0, d_dst.data_ptr(), each + 64, d_sizes.data_ptr()) == 0
    sizes = d_sizes.cpu().numpy()
    frames = d_dst.cpu().numpy().reshape(N, each + 64)
    zframes = np.concatenate([frames[i, : sizes[i]] for i in range(N)])
    zoff = np.concatenate([[0], np.cumsum(sizes)[:-1]]).astype(np.int64)
    yield dict(mov=mov, lo=lo, hi=hi, bp_full=bp_full, bpl=bpl, bp_rows=bpl.handle, it=it, planes=planes, sx=sx, sy=sy, each=each, zsrc=zsrc,
               zframes=zframes, zoff=zoff, zsizes=sizes.astype(np.uint32))
    sp.bad_pixels_destroy(bp_full)


BG = np.zeros(1, np.uint16)


def _lossy(lib, p):
    h = lib.rirb_lossy_open(W, H, H, 6, 2, 5.0, 32, 0, 1)
    try:
        return lib.rirb_lossy_add_images(h, p["frames"], N, p["out"], p["errors"])
    finally:
        lib.rirb_lossy_close(h)


def entries(d):
    """name -> ([(operand, role, initial array)], call(lib, pointers)); role: in / out / io (read and written)."""
    mov, f32 = d["mov"], d["mov"].astype(np.float32)
    z16, z8, zf = np.zeros_like(mov), np.zeros(mov.shape, np.uint8), np.zeros(mov.shape, np.float32)
    sx, sy = d["sx"], d["sy"]
    fx, fy = sx.astype(np.float32), sy.astype(np.float32)
    pl = d["planes"]
    each = d["each"]
    return {
        "translate": ([("src", "in", mov), ("dst", "out", z16), ("dx", "in", fx), ("dy", "in", fy)],
                      lambda lib, p: lib.rirb_translate_batch(ord("H"), p["src"], p["dst"], W, H, N, p["dx"], p["dy"], N,
                                                              BG.ctypes.data, b"nearest")),
        "gaussian_u16": ([("src", "in", mov), ("dst", "out", zf)],
                         lambda lib, p: lib.rirb_gaussian_filter_u16_batch(p["src"], p["dst"], W, H, N, 1.0)),
        "gaussian_f32": ([("src", "in", f32), ("dst", "out", zf)],
                         lambda lib, p: lib.rirb_gaussian_filter_batch(p["src"], p["dst"], W, H, N, 1.5)),
        "bp_correct": ([("in", "in", mov), ("out", "out", z16)],
                       lambda lib, p: lib.rirb_bad_pixels_correct_batch(d["bp_full"], p["in"], p["out"], N)),
        "bp_correct_gaussian": ([("in", "in", mov), ("corrected", "out", z16), ("smoothed", "out", zf)],
                                lambda lib, p: lib.rirb_bad_pixels_correct_gaussian_batch(d["bp_full"], p["in"], p["corrected"],
                                                                                          p["smoothed"], N, 1.0)),
        "remove_bad_pixels": ([("frames", "io", mov)],
                              lambda lib, p: lib.rirb_loader_remove_bad_pixels(d["bp_rows"], p["frames"], N, H * W)),
        "remove_motion": ([("in", "in", mov), ("out", "out", z16), ("shift_x", "in", sx), ("shift_y", "in", sy)],
                          lambda lib, p: lib.rirb_loader_remove_motion(p["in"], p["out"], W, H - META, N, H * W, p["shift_x"],
                                                                       p["shift_y"])),
        "read_movie": ([("lo", "in", d["lo"]), ("hi", "in", d["hi"]), ("out", "out", z16), ("shift_x", "in", sx), ("shift_y", "in", sy)],
                       lambda lib, p: lib.rirb_loader_read_movie(d["bp_rows"], p["lo"], p["hi"], N, W, H, 100, 0, p["shift_x"],
                                                                 p["shift_y"], META, p["out"])),
        "finish_frames": ([("frames", "io", mov), ("shift_x", "in", sx), ("shift_y", "in", sy)],
                          lambda lib, p: lib.rirb_loader_finish_frames(d["bp_rows"], p["frames"], N, W, H, 100, 0, p["shift_x"],
                                                                       p["shift_y"], META)),
        "split_yuv444": ([("img", "in", mov[0]), ("it", "in", d["it"]), ("y_plane", "out", pl[0]), ("u_plane", "out", pl[1]),
                          ("v_plane", "out", pl[2])],
                         lambda lib, p: lib.rirb_split_yuv444(p["img"], p["it"], W, H, p["y_plane"], p["u_plane"], p["v_plane"], LS, LS,
                                                              LS)),
        "merge_yuv444": ([("y_plane", "in", pl[0]), ("u_plane", "in", pl[1]), ("v_plane", "in", pl[2]), ("img", "out", z16[0]),
                          ("it", "out", z8[0])],
                         lambda lib, p: lib.rirb_merge_yuv444(p["y_plane"], p["u_plane"], p["v_plane"], LS, LS, LS, W, H, p["img"],
                                                              p["it"])),
        "split_yuv420": ([("img", "in", mov[0]), ("it", "in", d["it"]), ("y_plane", "out", np.concatenate([pl[0], pl[1]])),
                          ("u_plane", "out", pl[2])],
                         lambda lib, p: lib.rirb_split_yuv420(p["img"], p["it"], W, H, p["y_plane"], LS, p["u_plane"], LS)),
        "merge_yuv420": ([("y_plane", "in", np.concatenate([pl[0], pl[1]])), ("u_plane", "in", pl[2]), ("img", "out", z16[0]),
                          ("it", "out", z8[0])],
                         lambda lib, p: lib.rirb_merge_yuv420(p["y_plane"], LS, p["u_plane"], LS, W, H, p["img"], p["it"])),
        "precode": ([("movie", "in", mov), ("lo", "out", z8), ("hi", "out", z8)],
                    lambda lib, p: lib.rirb_precode_movie(p["movie"], N, W, H, 2, 1, 0, p["lo"], p["hi"])),
        "precode_stats": ([("movie", "in", mov), ("lo", "out", z8), ("hi", "out", z8), ("minmax", "out", np.zeros(2, np.uint32)),
                           ("hist", "out", np.zeros(65536, np.uint64))],
                          lambda lib, p: lib.rirb_precode_movie_stats(p["movie"], N, W, H, 2, 1, 0, p["lo"], p["hi"], p["minmax"], p["hist"],
                                                                      0)),
        "decode": ([("lo", "in", d["lo"]), ("hi", "in", d["hi"]), ("movie", "out", z16)],
                   lambda lib, p: lib.rirb_decode_movie(p["lo"], p["hi"], N, W, H, 2, 1, 0, p["movie"])),
        "lossy": ([("frames", "in", mov), ("out", "out", z16), ("errors", "out", np.zeros((N, 2), np.int32))],
                  lambda lib, p: _lossy(lib, p)),
        "movie_stats": ([("pixels", "in", mov), ("minmax", "out", np.zeros(2, np.uint32)), ("hist", "out", np.zeros(65536, np.uint64))],
                        lambda lib, p: lib.rirb_movie_stats(p["pixels"], mov.size, p["minmax"], p["hist"], 0)),
        "zstd_encode": ([("src", "in", d["zsrc"]), ("dst", "out", np.zeros((N, each + 64), np.uint8)), ("sizes", "out", np.zeros(N, np.int64))],
                        lambda lib, p: lib.rirb_zstd_encode_batch(p["src"], N, each, 0, p["dst"], each + 64, p["sizes"])),
        "zstd_decode": ([("src", "in", d["zframes"]), ("offsets", "in", d["zoff"]), ("sizes", "in", d["zsizes"]),
                         ("dst", "out", np.zeros((N, each), np.uint8)), ("status", "out", np.zeros(N, np.int64))],
                        lambda lib, p: lib.rirb_zstd_decode_batch(p["src"], p["offsets"], p["sizes"], N, p["dst"], each, each, p["status"])),
        "process_movie_host": ([("frames", "in", mov), ("dx", "in", fx), ("dy", "in", fy), ("lo", "out", z8), ("hi", "out", z8),
                                ("smoothed", "out", zf)],
                               lambda lib, p: lib.rirb_process_movie_host(d["bp_full"], p["frames"], N, W, H, 1.0, p["dx"], p["dy"],
                                                                          b"nearest", 0, 2, 1, 0, p["lo"], p["hi"], p["smoothed"])),
    }


ENTRY_OPERANDS = {  # kept in step with entries(): parametrisation happens before the module fixtures exist
    "translate": ("src", "dst", "dx", "dy"), "gaussian_u16": ("src", "dst"), "gaussian_f32": ("src", "dst"),
    "bp_correct": ("in", "out"), "bp_correct_gaussian": ("in", "corrected", "smoothed"), "remove_bad_pixels": ("frames",),
    "remove_motion": ("in", "out", "shift_x", "shift_y"), "read_movie": ("lo", "hi", "out", "shift_x", "shift_y"),
    "finish_frames": ("frames", "shift_x", "shift_y"), "split_yuv444": ("img", "it", "y_plane", "u_plane", "v_plane"),
    "merge_yuv444": ("y_plane", "u_plane", "v_plane", "img", "it"), "split_yuv420": ("img", "it", "y_plane", "u_plane"),
    "merge_yuv420": ("y_plane", "u_plane", "img", "it"), "precode": ("movie", "lo", "hi"),
    "precode_stats": ("movie", "lo", "hi", "minmax", "hist"), "decode": ("lo", "hi", "movie"), "lossy": ("frames", "out", "errors"),
    "movie_stats": ("pixels", "minmax", "hist"), "zstd_encode": ("src", "dst", "sizes"),
    "zstd_decode": ("src", "offsets", "sizes", "dst", "status"), "process_movie_host": ("frames", "dx", "dy", "lo", "hi", "smoothed"),
}
DEVICE_ONLY = ("zstd_encode", "zstd_decode")  # kernels dereference every operand: pageable memory is refused


def run(lib, spec, kinds, pool):
    """Call the entry with operand i in memory kind kinds[i]; -> (status, {written operand: bytes after the call})."""
    ops, call = spec
    bufs = {name: Buf(k, init, pool) for (name, _, init), k in zip(ops, kinds)}
    rc = call(lib, {n: b.ptr for n, b in bufs.items()})
    lib.rirb_synchronize()
    return rc, {name: bufs[name].read() for name, role, _ in ops if role != "in"}


def test_entry_table_matches_the_operand_list(data):
    assert {k: tuple(n for n, _, _ in v[0]) for k, v in entries(data).items()} == ENTRY_OPERANDS


KIND_CASES = [(e, op, k) for e, ops in ENTRY_OPERANDS.items() for op in ops for k in KINDS[:-1]] + [
    (e, "mixed", "mixed") for e in ENTRY_OPERANDS]


@pytest.mark.parametrize("entry,operand,kind", KIND_CASES, ids=[f"{e}-{o}-{k}" for e, o, k in KIND_CASES])
def test_every_kind_of_memory_on_every_operand(lib, data, pool, entry, operand, kind):
    spec = entries(data)[entry]
    names = ENTRY_OPERANDS[entry]
    rc0, want = run(lib, spec, ["device"] * len(names), pool)
    assert rc0 == 0, _lib.last_error()
    if kind == "mixed":
        kinds = [KINDS[(i + 1) % len(KINDS)] for i in range(len(names))]
        if entry in DEVICE_ONLY:
            kinds = [k if k != "pageable" else "managed" for k in kinds]
    else:
        kinds = [kind if n == operand else "device" for n in names]
    before = _lib.launch_count()
    rc, got = run(lib, spec, kinds, pool)
    if entry in DEVICE_ONLY and "pageable" in kinds:
        assert rc == -1 and "pageable" in _lib.last_error() and _lib.launch_count() == before
        return
    assert rc == 0, _lib.last_error()
    for name in want:
        assert np.array_equal(got[name], want[name]), f"{entry}: {name} differs with {dict(zip(names, kinds))}"


RING_EDGES = [1, (256 << 10) - 1, 256 << 10, (256 << 10) + 1, (1 << 20) - 1, 1 << 20, (1 << 20) + 1, (64 << 20) - 1, 64 << 20,
              (64 << 20) + 1]


@pytest.mark.parametrize("nbytes", RING_EDGES)
def test_pageable_outputs_on_the_staging_ring_edges(lib, nbytes):
    """One uint8 row of `nbytes` pixels shifted by one pixel: every byte of the pageable output, written through the ring
    chunk by chunk (or by the driver above 64 MiB), equals the device output."""
    src = np.random.default_rng(nbytes).integers(0, 256, nbytes, dtype=np.uint8)
    out = np.full(nbytes, SENTINEL ^ 0xFF, np.uint8)
    one, zero = np.ones(1, np.float32), np.zeros(1, np.float32)
    bg = np.zeros(1, np.uint8)
    assert lib.rirb_translate_batch(ord("B"), src.ctypes.data, out.ctypes.data, nbytes, 1, 1, one.ctypes.data, zero.ctypes.data, 1,
                                    bg.ctypes.data, b"nearest") == 0, _lib.last_error()
    d_out = torch.zeros(nbytes, dtype=torch.uint8, device="cuda")
    assert lib.rirb_translate_batch(ord("B"), src.ctypes.data, d_out.data_ptr(), nbytes, 1, 1, one.ctypes.data, zero.ctypes.data, 1,
                                    bg.ctypes.data, b"nearest") == 0
    assert np.array_equal(d_out.cpu().numpy(), out)


# ---------------------------------------------------------------------------------------------
# overlap at the C ABI
# ---------------------------------------------------------------------------------------------
OVERLAP_PAIRS = {
    "translate": [("src", "dst"), ("dx", "dst")], "gaussian_u16": [("src", "dst")], "gaussian_f32": [("src", "dst")],
    "bp_correct": [("in", "out")], "bp_correct_gaussian": [("in", "corrected"), ("in", "smoothed"), ("corrected", "smoothed")],
    "remove_motion": [("in", "out")], "read_movie": [("lo", "out"), ("hi", "out")],
    "split_yuv444": [("img", "u_plane"), ("it", "y_plane"), ("u_plane", "v_plane")], "merge_yuv444": [("u_plane", "img"), ("img", "it")],
    "split_yuv420": [("img", "y_plane"), ("y_plane", "u_plane")], "merge_yuv420": [("y_plane", "img"), ("img", "it")],
    "precode": [("movie", "lo"), ("lo", "hi")], "precode_stats": [("movie", "hi"), ("lo", "hi"), ("minmax", "hist")],
    "decode": [("lo", "movie"), ("hi", "movie")], "lossy": [("frames", "out"), ("out", "errors")],
    "movie_stats": [("pixels", "hist"), ("minmax", "hist")], "zstd_encode": [("src", "dst"), ("dst", "sizes")],
    "zstd_decode": [("offsets", "dst"), ("dst", "status")],
}
OVERLAP_CASES = [(e, a, b, by) for e, pairs in OVERLAP_PAIRS.items() for a, b in pairs for by in ("element", "row", "frame")]


def overlap_bytes(arr, by):
    if by == "element" or arr.ndim < 2:
        return arr.itemsize
    if by == "row":
        return arr.shape[-1] * arr.itemsize
    return arr.shape[-2] * arr.shape[-1] * arr.itemsize


@pytest.mark.parametrize("entry,a,b,by", OVERLAP_CASES, ids=[f"{e}-{a}-{b}-{by}" for e, a, b, by in OVERLAP_CASES])
def test_device_operands_that_overlap_are_refused(lib, data, entry, a, b, by):
    ops, call = entries(data)[entry]
    init = {n: np.ascontiguousarray(x).reshape(-1).view(np.uint8) for n, _, x in ops}
    arrs = {n: np.asarray(x) for n, _, x in ops}
    ov = min(overlap_bytes(arrs[b], by), init[a].size, init[b].size)
    backing = torch.full((init[a].size + init[b].size - ov + 64,), SENTINEL, dtype=torch.uint8, device="cuda")
    backing[: init[a].size].copy_(torch.from_numpy(init[a].copy()))
    at = {a: 0, b: init[a].size - ov}
    others = {n: torch.from_numpy(init[n].copy()).cuda() for n in init if n not in at}
    ptrs = {n: backing.data_ptr() + off for n, off in at.items()} | {n: t.data_ptr() for n, t in others.items()}
    torch.cuda.synchronize()
    snapshot = backing.cpu().numpy().copy()
    before = _lib.launch_count()
    rc = call(lib, ptrs)
    torch.cuda.synchronize()
    after = backing.cpu().numpy()
    assert np.array_equal(after, snapshot), f"{entry}: {int((after != snapshot).sum())} bytes of the overlapping operands changed"
    assert rc == -1 and "overlap" in _lib.last_error(), (rc, _lib.last_error())
    assert _lib.launch_count() == before


def test_process_movie_host_refuses_overlapping_host_operands(lib, data):
    """Its copies run on three streams at once: an output over an input races with a later sub-chunk's upload."""
    mov = data["mov"]
    buf = np.zeros(mov.nbytes + mov.size, np.uint8)
    buf[: mov.nbytes] = mov.reshape(-1).view(np.uint8)
    dx = np.zeros(N, np.float32)
    before = _lib.launch_count()
    rc = lib.rirb_process_movie_host(data["bp_full"], buf.ctypes.data, N, W, H, 1.0, dx.ctypes.data, dx.ctypes.data, b"nearest", 0, 2,
                                     1, 0, buf.ctypes.data + mov.nbytes - W, buf.ctypes.data + mov.nbytes, None)
    assert rc == -1 and "overlap" in _lib.last_error() and _lib.launch_count() == before


@pytest.mark.parametrize("by", ["element", "row", "frame"])
def test_overlapping_host_operands_give_the_out_of_place_answer(lib, data, by):
    """Host operands are staged into separate device buffers, so a shared byte is read before it is written."""
    mov = data["mov"]
    ov = overlap_bytes(mov, by)
    want = sp.translate_batch(mov, 0.5, -0.75, "nearest")
    buf = np.zeros(2 * mov.nbytes - ov, np.uint8)
    buf[: mov.nbytes] = mov.reshape(-1).view(np.uint8)
    dx, dy, bg = np.full(1, 0.5, np.float32), np.full(1, -0.75, np.float32), np.zeros(1, np.uint16)
    rc = lib.rirb_translate_batch(ord("H"), buf.ctypes.data, buf.ctypes.data + mov.nbytes - ov, W, H, N, dx.ctypes.data, dy.ctypes.data,
                                  1, bg.ctypes.data, b"nearest")
    assert rc == 0, _lib.last_error()
    got = buf[mov.nbytes - ov:].view(np.uint16).reshape(mov.shape)
    assert np.array_equal(got, want)


def test_documented_in_place_entries_take_equal_device_pointers(lib, data):
    mov = data["mov"]
    sx, sy = data["sx"], data["sy"]
    out_of_place = vio.remove_motion(mov, sx, sy, META)
    d = torch.from_numpy(mov.view(np.int16).copy()).cuda().view(torch.uint16)
    vio.remove_motion(d, sx, sy, META, out=d)
    assert np.array_equal(d.cpu().view(torch.int16).numpy().view(np.uint16), out_of_place)
    host = mov.copy()
    assert lib.rirb_bad_pixels_correct_batch(data["bp_full"], host.ctypes.data, host.ctypes.data, N) == 0
    d = torch.from_numpy(mov.view(np.int16).copy()).cuda().view(torch.uint16)
    sp.bad_pixels_correct_batch(data["bp_full"], d, out=d)
    assert np.array_equal(d.cpu().view(torch.int16).numpy().view(np.uint16), host)


# ---------------------------------------------------------------------------------------------
# wrong torch CUDA outputs at the facade: a guard behind every short view
# ---------------------------------------------------------------------------------------------
TDT = {np.dtype(np.uint8): torch.uint8, np.dtype(np.uint16): torch.uint16, np.dtype(np.float32): torch.float32}


class Guarded:
    """A view of `shape` at the start of a 0xA5 buffer that holds `full` elements of `dtype`."""

    def __init__(self, shape, full, dtype):
        esz = np.dtype(dtype).itemsize
        self.n = int(np.prod(shape)) * esz
        self.buf = torch.full((int(np.prod(full)) * esz + 64,), SENTINEL, dtype=torch.uint8, device="cuda")
        self.t = self.buf[: self.n].view(TDT[np.dtype(dtype)]).view(*shape)

    def guard_intact(self):
        torch.cuda.synchronize()
        return bool((self.buf[self.n:] == SENTINEL).all().item())


def dev(a):
    return torch.from_numpy(a.view(np.int16) if a.dtype == np.uint16 else a).cuda().view(TDT[a.dtype])


SHORT = {"frame": lambda s: (s[0] - 1,) + s[1:], "row": lambda s: s[:-2] + (s[-2] - 1, s[-1]), "col": lambda s: s[:-1] + (s[-1] - 1,)}


def facade_calls(d, tmp_path):
    mov = d["mov"]
    path = str(tmp_path / "m.z")
    with tools.ZFileWriter(path, W, H, method=1) as wr:
        wr.add_images(mov, list(range(N)))
    bpl = d["bpl"]
    return {  # entry -> (output operand, its dtype, call(out))
        "translate_batch-out": (np.uint16, lambda o: sp.translate_batch(dev(mov), 0.5, 0.25, "nearest", out=o)),
        "gaussian_filter_batch-out": (np.float32, lambda o: sp.gaussian_filter_batch(dev(mov), 1.0, out=o)),
        "bad_pixels_correct_batch-out": (np.uint16, lambda o: sp.bad_pixels_correct_batch(d["bp_full"], dev(mov), out=o)),
        "bad_pixels_correct_gaussian_batch-out": (np.uint16, lambda o: sp.bad_pixels_correct_gaussian_batch(d["bp_full"], dev(mov), out=o)),
        "bad_pixels_correct_gaussian_batch-smoothed": (
            np.float32, lambda o: sp.bad_pixels_correct_gaussian_batch(d["bp_full"], dev(mov), smoothed=o)),
        "precode_movie-lo": (np.uint8, lambda o: vio.precode_movie(dev(mov), 2, True, 0, out=(o, dev(np.zeros(mov.shape, np.uint8))))),
        "precode_movie-hi": (np.uint8, lambda o: vio.precode_movie(dev(mov), 2, True, 0, out=(dev(np.zeros(mov.shape, np.uint8)), o))),
        "decode_movie-out": (np.uint16, lambda o: vio.decode_movie(dev(d["lo"]), dev(d["hi"]), 2, True, 0, out=o)),
        "remove_motion-out": (np.uint16, lambda o: vio.remove_motion(dev(mov), d["sx"], d["sy"], META, out=o)),
        "read_movie-out": (np.uint16, lambda o: vio.read_movie(dev(d["lo"]), dev(d["hi"]), bpl, 100, 0, d["sx"], d["sy"], META, out=o)),
        "LossyPreconditioner.add_images-out": (np.uint16, lambda o: vio.LossyPreconditioner(W, H).add_images(dev(mov), out=o)),
        "ZFileReader.read_images-out": (np.uint16, lambda o: tools.ZFileReader(path).read_images(0, N, out=o)),
    }


FACADE_CASES = [(e, s) for e in ("translate_batch-out", "gaussian_filter_batch-out", "bad_pixels_correct_batch-out",
                                 "bad_pixels_correct_gaussian_batch-out", "bad_pixels_correct_gaussian_batch-smoothed", "precode_movie-lo",
                                 "precode_movie-hi", "decode_movie-out", "remove_motion-out", "read_movie-out",
                                 "LossyPreconditioner.add_images-out", "ZFileReader.read_images-out") for s in SHORT]


@pytest.mark.parametrize("entry,short", FACADE_CASES, ids=[f"{e}-short_{s}" for e, s in FACADE_CASES])
def test_short_device_output_is_refused_and_the_guard_survives(lib, data, tmp_path, entry, short):
    dtype, call = facade_calls(data, tmp_path)[entry]
    g = Guarded(SHORT[short]((N, H, W)), (N, H, W), dtype)
    before = _lib.launch_count()
    try:
        call(g.t)
        err = None
    except RuntimeError as e:
        err = str(e)
    assert g.guard_intact(), f"{entry}: the call wrote past a view {short} short"
    operand = entry.split("-")[1]
    assert err is not None and operand in err, err
    assert _lib.launch_count() == before


# ---------------------------------------------------------------------------------------------
# strided numpy inputs that the facade copies: the same bits as the contiguous call
# ---------------------------------------------------------------------------------------------
def strided_calls(d):
    mov, lo, hi = d["mov"], d["lo"], d["hi"]
    wide = np.zeros((2 * N, H, 2 * W), np.uint16)
    wide[::2, :, ::2] = mov
    lw, hw = np.zeros((2 * N, H, 2 * W), np.uint8), np.zeros((2 * N, H, 2 * W), np.uint8)
    lw[::2, :, ::2], hw[::2, :, ::2] = lo, hi
    bpl = d["bpl"]
    s, sl, sh = wide[::2, :, ::2], lw[::2, :, ::2], hw[::2, :, ::2]
    return {
        "translate_batch": lambda m: sp.translate_batch(m(s), 0.5, 0.25, "nearest"),
        "gaussian_filter_batch": lambda m: sp.gaussian_filter_batch(m(s), 1.0),
        "bad_pixels_correct_batch": lambda m: sp.bad_pixels_correct_batch(d["bp_full"], m(s)),
        "bad_pixels_correct_gaussian_batch": lambda m: np.concatenate(
            [x.view(np.uint8).reshape(-1) for x in sp.bad_pixels_correct_gaussian_batch(d["bp_full"], m(s))]),
        "precode_movie": lambda m: np.stack(vio.precode_movie(m(s), 2, True, 0)),
        "decode_movie": lambda m: vio.decode_movie(m(sl), m(sh), 2, True, 0),
        "read_movie": lambda m: vio.read_movie(m(sl), m(sh), bpl, 100, 0, d["sx"], d["sy"], META),
        "remove_motion": lambda m: vio.remove_motion(m(s), d["sx"], d["sy"], META),
        "LossyPreconditioner.add_images": lambda m: vio.LossyPreconditioner(W, H, removeBadPixels=True).add_images(m(s))[0],
        "process_movie_host": lambda m: np.stack(movie.process_movie_host(type("BP", (), {"handle": d["bp_full"]})(), m(s), d["sx"],
                                                                          d["sy"], gop=2)),
    }


@pytest.mark.parametrize("entry", ["translate_batch", "gaussian_filter_batch", "bad_pixels_correct_batch",
                                   "bad_pixels_correct_gaussian_batch", "precode_movie", "decode_movie", "read_movie", "remove_motion",
                                   "LossyPreconditioner.add_images", "process_movie_host"])
def test_strided_numpy_input_gives_the_contiguous_answer(lib, data, entry):
    call = strided_calls(data)[entry]
    assert np.array_equal(call(lambda a: a), call(np.ascontiguousarray))


# ---------------------------------------------------------------------------------------------
# scratch slots under load
# ---------------------------------------------------------------------------------------------
def test_host_staging_grows_a_slot_that_an_unsynchronised_call_still_reads(lib, data):
    """Call 1 stages its host input in slot 0 and writes a device output, so it returns before its kernel ran; call 2
    stages a four times larger host input into slot 0, which must grow under it."""
    small = ir_movie(8, 64, 128, seed=3)
    big = ir_movie(32, 64, 128, seed=4)
    want_small = sp.translate_batch(small, 0.5, 0.25, "nearest")
    want_big = sp.translate_batch(big, -0.5, 1.25, "nearest")
    for _ in range(3):
        d_out = torch.empty((8, 64, 128), dtype=torch.uint16, device="cuda")
        dx, dy, bg = np.full(1, 0.5, np.float32), np.full(1, 0.25, np.float32), np.zeros(1, np.uint16)
        lib.rirb_set_stream(ct.c_void_p(torch.cuda.current_stream().cuda_stream))
        assert lib.rirb_translate_batch(ord("H"), small.ctypes.data, d_out.data_ptr(), 128, 64, 8, dx.ctypes.data, dy.ctypes.data, 1,
                                        bg.ctypes.data, b"nearest") == 0
        got_big = sp.translate_batch(big, -0.5, 1.25, "nearest")
        torch.cuda.synchronize()
        assert np.array_equal(d_out.cpu().view(torch.int16).numpy().view(np.uint16), want_small)
        assert np.array_equal(got_big, want_big)
        lib.rirb_release_thread_resources()  # the next round grows slot 0 from nothing again


def test_a_fresh_stream_waits_for_work_still_using_the_slots(lib, data):
    mov = ir_movie(16, 64, 128, seed=5)
    want = sp.gaussian_filter_batch(mov, 1.0)
    want2 = sp.gaussian_filter_batch(mov[::-1].copy(), 1.0)
    d_out = torch.empty((16, 64, 128), dtype=torch.float32, device="cuda")
    assert lib.rirb_gaussian_filter_u16_batch(mov.ctypes.data, d_out.data_ptr(), 128, 64, 16, 1.0) == 0  # slot 0, no sync
    s = torch.cuda.Stream()
    lib.rirb_set_stream(ct.c_void_p(s.cuda_stream))
    got2 = np.empty_like(want2)
    rev = mov[::-1].copy()
    assert lib.rirb_gaussian_filter_u16_batch(rev.ctypes.data, got2.ctypes.data, 128, 64, 16, 1.0) == 0  # slot 0 again
    lib.rirb_set_stream(None)
    torch.cuda.synchronize()
    assert np.array_equal(d_out.cpu().numpy(), want)
    assert np.array_equal(got2, want2)


def test_nested_entries_give_what_they_give_alone(lib, data):
    """read_movie with motion stages into slots 0-5 and translates; finish_frames calls remove_motion, which stages its
    shifts; bad_pixels_create uses slots 6-7 between them.  Host operands throughout, no synchronisation in between."""
    mov = data["mov"]
    lo, hi, sx, sy = data["lo"], data["hi"], data["sx"], data["sy"]
    bpl = vio.LoaderBadPixels(mov[0])
    alone_read = vio.read_movie(lo, hi, bpl, 100, 0, sx, sy, META)
    alone_finish = vio.finish_frames(mov.copy(), bpl, 100, 0, sx, sy, META)
    alone_bp = sp.bad_pixels_list(sp.bad_pixels_create(mov[1]))
    d_lo, d_hi = dev(lo), dev(hi)
    _lib.use_torch_stream()
    outs = []
    for _ in range(2):
        out = torch.empty((N, H, W), dtype=torch.uint16, device="cuda")
        vio.read_movie(d_lo, d_hi, bpl, 100, 0, sx, sy, META, out=out)
        fin = vio.finish_frames(mov.copy(), bpl, 100, 0, sx, sy, META)
        h = sp.bad_pixels_create(mov[1])
        outs.append((out, fin, sp.bad_pixels_list(h)))
        sp.bad_pixels_destroy(h)
    torch.cuda.synchronize()
    for out, fin, bpls in outs:
        assert np.array_equal(out.cpu().view(torch.int16).numpy().view(np.uint16), alone_read)
        assert np.array_equal(fin, alone_finish)
        assert np.array_equal(bpls[0], alone_bp[0]) and bpls[1] == alone_bp[1]
