"""Every facade entry checks its array operands before the library sees a pointer.

The C ABI takes bare pointers and trusts them for the whole extent the call implies: frames x height x width elements of
the type the entry reads or writes.  A numpy view with gaps, an output one frame / row / column short, the wrong dtype or
``hi`` planes of another shape than ``lo`` would be read or written as if they were that dense buffer -- past the end of
an allocation, or into the wrong elements with no error.  The checks live in ``signal_processing._operand``; each case
here hands one entry one wrong operand and expects a ``RuntimeError`` that names the operand, raised before anything is
launched.  No case needs a device: the refusal happens in Python.  Inputs that an entry copies when they are strided
(instead of refusing them) are compared with the contiguous call in ``tests/test_gpu_operand_contract.py``.
"""
import numpy as np
import pytest

from librir_b200 import _lib, movie, signal_processing as sp, tools, video_io as vio

N, H, W = 3, 8, 16
HANDLE = 7919  # a bad-pixel handle number no test creates: its frame size is registered by the `bp_handle` fixture


@pytest.fixture
def bp_handle(monkeypatch):
    monkeypatch.setattr(sp, "_BP_SHAPES", {**getattr(sp, "_BP_SHAPES", {}), HANDLE: (H, W)}, raising=False)
    return HANDLE


def wrong(a, kind):
    """`a` (a correct operand) made wrong in one way."""
    if kind == "strided_frames":  # a[::2]: same shape, every other frame of a larger stack
        return np.zeros((2 * a.shape[0],) + a.shape[1:], a.dtype)[::2]
    if kind == "strided_cols":  # a[:, :, ::2]
        return np.zeros(a.shape[:-1] + (2 * a.shape[-1],), a.dtype)[..., ::2]
    if kind == "dtype":
        return np.zeros(a.shape, np.float32 if a.dtype != np.float32 else np.uint16)
    if kind == "short_frame":
        return np.zeros((a.shape[0] - 1,) + a.shape[1:], a.dtype)
    if kind == "short_row":
        return np.zeros(a.shape[:-2] + (a.shape[-2] - 1, a.shape[-1]), a.dtype)
    if kind == "short_col":
        return np.zeros(a.shape[:-1] + (a.shape[-1] - 1,), a.dtype)
    raise ValueError(kind)


OUT_KINDS = ("strided_frames", "strided_cols", "dtype", "short_frame", "short_row", "short_col")
INPLACE_KINDS = ("strided_frames", "strided_cols", "dtype")
SHAPE_KINDS = ("short_frame", "short_row", "short_col")


def u16(shape=(N, H, W)):
    return np.full(shape, 8000, np.uint16)


def u8(shape=(N, H, W)):
    return np.zeros(shape, np.uint8)


def f32(shape=(N, H, W)):
    return np.zeros(shape, np.float32)


class _LoaderBP(vio.LoaderBadPixels):
    def __init__(self):  # the frame size of a real detection, without the detection (which needs a device)
        self.height, self.width, self.rows, self.handle = H, W, H - 3, 0

    def __del__(self):
        pass


class _Lossy(vio.LossyPreconditioner):
    def __init__(self):
        self.width, self.height, self.lossy_height, self.handle = W, H, H, 0

    def __del__(self):
        pass


class _Reader(tools.ZFileReader):
    def __init__(self):
        self.width, self.height, self.images, self.threads, self.handle = W, H, N, 0, 0

    def __del__(self):
        pass


# entry -> (operands of a correct call, call(ops), [(operand, kinds)])
ENTRIES = {
    "translate_batch": (
        lambda: dict(frames=u16(), out=u16()),
        lambda o: sp.translate_batch(o["frames"], 0.5, 0.25, "nearest", out=o["out"]),
        [("out", OUT_KINDS)]),
    "gaussian_filter_batch": (
        lambda: dict(frames=f32(), out=f32()),
        lambda o: sp.gaussian_filter_batch(o["frames"], 1.0, out=o["out"]),
        [("out", OUT_KINDS)]),
    "bad_pixels_correct_batch": (
        lambda: dict(frames=u16(), out=u16()),
        lambda o: sp.bad_pixels_correct_batch(HANDLE, o["frames"], out=o["out"]),
        [("frames", ("dtype", "short_row", "short_col")), ("out", OUT_KINDS)]),
    "bad_pixels_correct_gaussian_batch": (
        lambda: dict(frames=u16(), out=u16(), smoothed=f32()),
        lambda o: sp.bad_pixels_correct_gaussian_batch(HANDLE, o["frames"], 1.0, out=o["out"], smoothed=o["smoothed"]),
        [("frames", ("dtype", "short_row", "short_col")), ("out", OUT_KINDS), ("smoothed", OUT_KINDS)]),
    "precode_movie": (
        lambda: dict(movie=u16(), lo=u8(), hi=u8()),
        lambda o: vio.precode_movie(o["movie"], 4, True, 0, out=(o["lo"], o["hi"])),
        [("movie", ("dtype",)), ("lo", OUT_KINDS), ("hi", OUT_KINDS)]),
    "decode_movie": (
        lambda: dict(lo=u8(), hi=u8(), out=u16()),
        lambda o: vio.decode_movie(o["lo"], o["hi"], 4, True, 0, out=o["out"]),
        [("lo", ("dtype",)), ("hi", ("dtype",) + SHAPE_KINDS), ("out", OUT_KINDS)]),
    "remove_motion": (
        lambda: dict(frames=u16(), out=u16()),
        lambda o: vio.remove_motion(o["frames"], [0.5] * N, [0.25] * N, out=o["out"]),
        [("frames", ("dtype",)), ("out", OUT_KINDS)]),
    "read_movie": (
        lambda: dict(lo=u8(), hi=u8(), out=u16()),
        lambda o: vio.read_movie(o["lo"], o["hi"], None, 100, 0, out=o["out"]),
        [("lo", ("dtype",)), ("hi", ("dtype",) + SHAPE_KINDS), ("out", OUT_KINDS)]),
    "finish_frames": (
        lambda: dict(frames=u16()),
        lambda o: vio.finish_frames(o["frames"], None, 100),
        [("frames", INPLACE_KINDS)]),
    "LoaderBadPixels.remove": (
        lambda: dict(frames=u16()),
        lambda o: _LoaderBP().remove(o["frames"]),
        [("frames", INPLACE_KINDS)]),
    "LossyPreconditioner.add_images": (
        lambda: dict(frames=u16(), out=u16()),
        lambda o: _Lossy().add_images(o["frames"], out=o["out"]),
        [("frames", ("dtype",)), ("out", OUT_KINDS)]),
    "ZFileReader.read_images": (
        lambda: dict(out=u16()),
        lambda o: _Reader().read_images(0, N, out=o["out"]),
        [("out", OUT_KINDS)]),
    "process_movie_host": (
        lambda: dict(frames=u16(), lo=u8(), hi=u8(), smoothed=f32()),
        lambda o: movie.process_movie_host(type("BP", (), {"handle": HANDLE})(), o["frames"], np.zeros(N, np.float32),
                                           np.zeros(N, np.float32), gop=4, lo=o["lo"], hi=o["hi"], smoothed=o["smoothed"]),
        [("frames", ("dtype",)), ("lo", OUT_KINDS), ("hi", OUT_KINDS), ("smoothed", OUT_KINDS)]),
}

CASES = [(entry, op, kind) for entry, (_, _, ops) in ENTRIES.items() for op, kinds in ops for kind in kinds]


def refused(call, name):
    before = _lib.launch_count()
    with pytest.raises(RuntimeError, match=rf"\b{name}\b"):
        call()
    assert _lib.launch_count() == before


@pytest.mark.parametrize("entry,operand,kind", CASES, ids=[f"{e}-{o}-{k}" for e, o, k in CASES])
def test_wrong_operand_is_refused_by_name(bp_handle, entry, operand, kind):
    make, call, _ = ENTRIES[entry]
    ops = make()
    ops[operand] = wrong(ops[operand], kind)
    refused(lambda: call(ops), operand)


@pytest.mark.parametrize("shifts", ["float64", "short", "dy_short"])
def test_translate_batch_refuses_device_shift_arrays_it_would_misread(shifts):
    """Torch shift arrays go to the library as they are: float32, one per frame (or one for all), dx and dy alike."""
    torch = pytest.importorskip("torch")
    frames, out = u16(), u16()
    dx, dy = torch.zeros(N, dtype=torch.float32), torch.zeros(N, dtype=torch.float32)
    if shifts == "float64":
        dx = dx.double()
    elif shifts == "short":
        dx, dy = dx[:-1], dy[:-1]
    else:
        dy = dy[:-1]
    refused(lambda: sp.translate_batch(frames, dx, dy, "nearest", out=out), "dx" if shifts != "dy_short" else "dy")


@pytest.mark.parametrize("entry", ["translate_batch", "gaussian_filter_batch", "bad_pixels_correct_batch", "precode_movie",
                                   "decode_movie", "read_movie", "remove_motion", "LossyPreconditioner.add_images"])
def test_read_only_numpy_output_is_refused(bp_handle, entry):
    make, call, _ = ENTRIES[entry]
    ops = make()
    name = "lo" if entry == "precode_movie" else "out"
    ops[name].flags.writeable = False
    refused(lambda: call(ops), name)


@pytest.mark.parametrize("entry", ["bad_pixels_correct_batch", "remove_motion"])
def test_strided_in_place_frames_are_refused(bp_handle, entry):
    """``out is frames`` asks for the result in ``frames`` itself; a copy of a strided view would drop it."""
    frames = wrong(u16(), "strided_frames")
    if entry == "bad_pixels_correct_batch":
        refused(lambda: sp.bad_pixels_correct_batch(HANDLE, frames, out=frames), "frames")
    else:
        refused(lambda: vio.remove_motion(frames, [0.0] * N, [0.0] * N, out=frames), "frames")


def test_precode_movie_out_must_be_a_pair():
    with pytest.raises(RuntimeError, match="pair"):
        vio.precode_movie(u16(), out=(u8(),))


def test_zfile_writer_refuses_a_device_stack_of_another_dtype(tmp_path):
    """Numpy stacks are converted to uint16; a tensor goes to the library as it is, so its dtype must be uint16."""
    torch = pytest.importorskip("torch")
    w = tools.ZFileWriter.__new__(tools.ZFileWriter)
    w.width, w.height, w.threads, w.handle = W, H, 0, 0
    refused(lambda: w.add_images(torch.zeros((N, H, W), dtype=torch.float32), list(range(N))), "frames")


def test_the_pointer_helper_refuses_strided_numpy():
    """The last line behind every entry: ``_ptr`` never hands the library the base address of a view with gaps."""
    with pytest.raises(RuntimeError, match="contiguous"):
        sp._ptr(wrong(u16(), "strided_cols"))
    sp._ptr(u16())
