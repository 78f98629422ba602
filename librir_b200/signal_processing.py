"""Host-side mirror of ``librir.signal_processing`` for the hot path.

Same names, arguments, defaults and error behaviour as the reference's ctypes wrappers
(src/python/librir/signal_processing/rir_signal_processing.py: translate :23-82,
gaussian_filter :85-113, find_median_pixel :116-147, bad_pixels_* :273-316) and its
``BadPixels`` class (BadPixels.py:16-29) -- but every call lands in the CUDA library.

The ``*_batch`` functions are additive: they take a stack of frames ``[n, h, w]`` as a numpy
array (staged through the GPU) or as a torch CUDA tensor (zero copies, runs on torch's current
stream) and process it in one launch.
"""
from __future__ import annotations

import ctypes as ct

import numpy as np

from . import _lib

_DTYPES = {
    np.dtype(np.bool_): "?",
    np.dtype(np.int8): "b",
    np.dtype(np.uint8): "B",
    np.dtype(np.int16): "h",
    np.dtype(np.uint16): "H",
    np.dtype(np.int32): "i",
    np.dtype(np.uint32): "I",
    np.dtype(np.int64): "l",
    np.dtype(np.uint64): "L",
    np.dtype(np.float32): "f",
    np.dtype(np.float64): "d",
}


def toCharP(s):
    """librir/low_level/misc.py toCharP: str -> bytes."""
    return s.encode("ascii") if isinstance(s, str) else bytes(s)


# ----------------------------------------------------------------------------------------
# buffer helpers: numpy (host) or torch CUDA tensor (device)
# ----------------------------------------------------------------------------------------
def _is_torch(x) -> bool:
    return type(x).__module__.startswith("torch")


_TORCH_NP_DTYPES = {}  # filled on first use: every operand check of a torch tensor looks its dtype up here


def _torch_np_dtype(t):
    if not _TORCH_NP_DTYPES:
        import torch

        _TORCH_NP_DTYPES.update({
            torch.bool: np.dtype(np.bool_), torch.int8: np.dtype(np.int8), torch.uint8: np.dtype(np.uint8),
            torch.int16: np.dtype(np.int16), torch.uint16: np.dtype(np.uint16), torch.int32: np.dtype(np.int32),
            torch.uint32: np.dtype(np.uint32), torch.int64: np.dtype(np.int64), torch.uint64: np.dtype(np.uint64),
            torch.float32: np.dtype(np.float32), torch.float64: np.dtype(np.float64),
        })
    return _TORCH_NP_DTYPES[t.dtype]


def _ptr(x):
    if _is_torch(x):
        if not x.is_contiguous():
            raise RuntimeError("librir_b200: tensors must be contiguous")
        return ct.c_void_p(x.data_ptr())
    if not x.flags.c_contiguous:  # the library reads and writes dense buffers from the first element's address
        raise RuntimeError("librir_b200: arrays must be contiguous")
    return x.ctypes.data_as(ct.c_void_p)


def _dtype_of(x):
    return _torch_np_dtype(x) if _is_torch(x) else x.dtype


def _operand(x, what, name, shape=None, dtype=None, copy=False):
    """Check an array operand of ``what`` before its pointer goes to the library, which trusts the pointer for the whole
    extent the call implies: ``dtype`` and ``shape`` (None: any) must match exactly, and the buffer must be dense.  A
    strided numpy input is copied when ``copy`` (operands the library only reads); otherwise -- outputs, in-place
    operands, torch tensors -- it is refused, as is a read-only numpy output.  ``dtype`` may be a tuple of the dtypes
    accepted.  Returns the operand to hand to ``_ptr``."""
    try:
        dt = _dtype_of(x)
    except KeyError:  # a torch dtype the library has no code for
        dt = None
    allowed = [np.dtype(d) for d in (dtype if isinstance(dtype, tuple) else (dtype,))] if dtype is not None else None
    if allowed is not None and dt not in allowed:
        raise RuntimeError(f"{what}: {name} must be {' or '.join(d.name for d in allowed)}, not {x.dtype}")
    if shape is not None and tuple(x.shape) != tuple(shape):
        raise RuntimeError(f"{what}: {name} has shape {tuple(x.shape)}, expected {tuple(shape)}")
    if _is_torch(x):
        if not x.is_contiguous():
            raise RuntimeError(f"{what}: {name} must be a contiguous tensor")
        return x
    if not x.flags.c_contiguous:
        if not copy:
            raise RuntimeError(f"{what}: {name} is a strided view; the library writes it as a dense array")
        x = np.ascontiguousarray(x)
    elif not copy and not x.flags.writeable:
        raise RuntimeError(f"{what}: {name} is read-only")
    return x


def _empty_like(x, dtype=None):
    if _is_torch(x):
        import torch

        if dtype is None:
            return torch.empty_like(x)
        tdt = {np.dtype(np.float32): torch.float32, np.dtype(np.uint16): torch.uint16, np.dtype(np.uint8): torch.uint8}[
            np.dtype(dtype)]
        return torch.empty(x.shape, dtype=tdt, device=x.device)
    return np.empty(x.shape, dtype=dtype or x.dtype)


def _prepare_device_call(x):
    if _is_torch(x):
        if not x.is_cuda:
            raise RuntimeError("librir_b200: torch tensors must live on a CUDA device (use numpy for host data)")
        _lib.use_torch_stream()


# ----------------------------------------------------------------------------------------
# translate
# ----------------------------------------------------------------------------------------
def translate(image, dx, dy, strategy=str(), background=None):
    """Sub-pixel shift of one 2-D image by ``(dx, dy)`` with bilinear weights (rir_signal_processing.py:23-82).

    ``strategy`` decides what the pixels without a source get: ``""`` / ``"noborder"`` keep the input's value,
    ``"constant"`` (alias of ``"background"``) writes ``background``, ``"nearest"`` repeats the closest valid
    row / column, ``"wrap"`` continues from the opposite edge.  Result: same shape and dtype as ``image``.
    """
    lib = _lib.load()
    if len(image.shape) != 2:
        raise RuntimeError("translate: wrong input image dimension")
    if strategy == "background" and background is None:
        raise RuntimeError("translate: wrong background value")

    strategy = toCharP(strategy)
    if strategy == b"constant":
        strategy = b"background"
    img = np.ascontiguousarray(image)
    # "noborder" pixels keep the source value; the other strategies write every pixel
    res = np.copy(img, "C") if strategy in (b"", b"noborder") else np.empty_like(img)
    _back = np.zeros((1), dtype=img.dtype)
    if background is not None:
        _back[0] = background
    _tr = np.zeros((2), dtype=np.float32)
    _tr[0] = dx
    _tr[1] = dy
    _dtype = _DTYPES.get(image.dtype, None)
    if _dtype is None:
        raise RuntimeError("An error occured while calling 'translate'")
    r = lib.translate(ord(_dtype), _ptr(img), _ptr(res), img.shape[1], img.shape[0], _tr[0], _tr[1], _ptr(_back), strategy)
    _lib.check(r, "translate")
    return res


def translate_batch(frames, dx, dy, strategy=str(), background=None, out=None):
    """``translate`` on a stack ``[n, h, w]``; ``dx``/``dy`` scalars or per-frame sequences.  ``out``: same shape and dtype
    as ``frames``.  A strided numpy ``frames`` is copied first; a strided ``out`` is refused."""
    lib = _lib.load()
    if len(frames.shape) != 3:
        raise RuntimeError("translate_batch: wrong input dimension")
    if strategy == "background" and background is None:
        raise RuntimeError("translate: wrong background value")
    strategy = toCharP(strategy)
    if strategy == b"constant":
        strategy = b"background"
    _prepare_device_call(frames)
    frames = _operand(frames, "translate_batch", "frames", copy=True)
    n, h, w = frames.shape
    dt = _dtype_of(frames)
    code = _DTYPES.get(dt)
    if code is None:
        raise RuntimeError("An error occured while calling 'translate'")
    if out is None:
        out = frames.clone() if _is_torch(frames) else np.copy(frames, "C")
    out = _operand(out, "translate_batch", "out", frames.shape, dt)
    if _is_torch(dx):
        ns = dx.numel()
        sx = _operand(dx, "translate_batch", "dx", (ns,) if ns != 1 else None, np.float32)
        sy = _operand(dy, "translate_batch", "dy", tuple(dx.shape), np.float32)
        if ns not in (1, n):
            raise RuntimeError(f"translate_batch: dx has {ns} shifts for {n} frames")
    else:
        sx = np.ascontiguousarray(np.atleast_1d(dx), dtype=np.float32)
        sy = np.ascontiguousarray(np.atleast_1d(dy), dtype=np.float32)
        ns = sx.size
    _back = np.zeros((1), dtype=dt)
    if background is not None:
        _back[0] = background
    r = lib.rirb_translate_batch(ord(code), _ptr(frames), _ptr(out), w, h, n, _ptr(sx), _ptr(sy), ns, _ptr(_back), strategy)
    _lib.check(r, "translate")
    return out


# ----------------------------------------------------------------------------------------
# gaussian
# ----------------------------------------------------------------------------------------
def gaussian_filter(image, sigma=1.0):
    """Gaussian smoothing of one 2-D image, radius ``max(1, int(2 * sigma))``, taps outside the image dropped and the
    rest renormalised (rir_signal_processing.py:85-113).  The output is float32 whatever the input dtype."""
    lib = _lib.load()
    if len(image.shape) != 2:
        raise RuntimeError("gaussian_filter: wrong input image dimension")
    res = np.empty(image.shape, dtype=np.float32)
    if image.dtype == np.uint16:
        # the uint16 -> float32 conversion of the reference wrapper (rir_signal_processing.py:100) happens
        # in the kernel: half the upload, no host pass (the conversion is exact either way)
        img = np.ascontiguousarray(image)
        r = lib.rirb_gaussian_filter_u16_batch(_ptr(img), _ptr(res), img.shape[1], img.shape[0], 1, sigma)
    else:
        img = np.ascontiguousarray(image, dtype=np.float32)
        r = lib.gaussian_filter(_ptr(img), _ptr(res), img.shape[1], img.shape[0], sigma)
    _lib.check(r, "gaussian_filter")
    return res


def gaussian_filter_batch(frames, sigma=1.0, out=None):
    """Gaussian filter of a stack ``[n, h, w]`` (float32, or uint16 converted on the fly) into float32 ``out`` of the same
    shape.  A strided numpy ``frames`` is copied first; a strided ``out`` is refused."""
    lib = _lib.load()
    if len(frames.shape) != 3:
        raise RuntimeError("gaussian_filter_batch: wrong input dimension")
    _prepare_device_call(frames)
    frames = _operand(frames, "gaussian_filter_batch", "frames", copy=True)
    n, h, w = frames.shape
    dt = _dtype_of(frames)
    if out is None:
        out = _empty_like(frames, np.float32)
    out = _operand(out, "gaussian_filter_batch", "out", frames.shape, np.float32)
    if dt == np.uint16:
        r = lib.rirb_gaussian_filter_u16_batch(_ptr(frames), _ptr(out), w, h, n, sigma)
    elif dt == np.float32:
        r = lib.rirb_gaussian_filter_batch(_ptr(frames), _ptr(out), w, h, n, sigma)
    else:
        raise RuntimeError("gaussian_filter_batch: frames must be uint16 or float32")
    _lib.check(r, "gaussian_filter")
    return out


# ----------------------------------------------------------------------------------------
# statistics
# ----------------------------------------------------------------------------------------
def find_median_pixel(image, percent=0.5, mask=None):
    """Quantile of a uint16 image through its histogram: the smallest level whose cumulated count reaches
    ``percent * size`` (optionally over the pixels where ``mask`` is non-zero); rir_signal_processing.py:116-147."""
    lib = _lib.load()
    if len(image.shape) != 2:
        raise RuntimeError("find_median_pixel: wrong input image dimension")
    image = np.ascontiguousarray(image.astype(dtype=np.uint16, copy=False))
    if mask is not None:
        mask = np.ascontiguousarray(mask.astype(dtype=np.uint8, copy=False))
        res = lib.find_median_pixel_mask(_ptr(image), _ptr(mask), image.size, float(percent))
    else:
        res = lib.find_median_pixel(_ptr(image), image.size, float(percent))
    return _lib.check(res, "find_median_pixel")


# ----------------------------------------------------------------------------------------
# connected components
# ----------------------------------------------------------------------------------------
# columns of the statistics rows of ``label_batch``; the centroid is ``stats[..., SUM_X] / stats[..., AREA]``
AREA, X_MIN, Y_MIN, X_MAX, Y_MAX, SUM_X, SUM_Y, SUM_VALUE, MAX_VALUE, ARGMAX = range(10)


def label_batch(frames, threshold, connectivity=8, max_components=256, labels=None):
    """Connected components of ``frames > threshold`` for a uint16 stack ``[n, h, w]``, with per-component statistics.

    ``threshold``: a scalar or one value per frame (sequence, numpy array or tensor of uint16 range).  ``connectivity``:
    4 or 8.  Returns ``(labels, counts, stats)``: int32 ``labels [n, h, w]`` (0 background, 1..K numbered in raster order
    of each component's first pixel, as ``scipy.ndimage.label``), int32 ``counts [n]`` (the true K of each frame) and
    int64 ``stats [n, max_components, 10]`` whose row ``k - 1`` describes label ``k`` (columns ``AREA`` .. ``ARGMAX``;
    rows past ``min(K, max_components)`` are zero).  numpy in gives numpy out; a torch CUDA tensor gives tensors on its
    device.  ``labels``: an int32 output of the same shape, or None."""
    lib = _lib.load()
    what = "label_batch"
    if len(frames.shape) != 3:
        raise RuntimeError(f"{what}: wrong input dimension")
    if connectivity not in (4, 8):
        raise RuntimeError(f"{what}: connectivity must be 4 or 8, not {connectivity}")
    if int(max_components) != max_components or max_components < 0:
        raise RuntimeError(f"{what}: max_components must be a non-negative integer")
    max_components = int(max_components)
    _prepare_device_call(frames)
    frames = _operand(frames, what, "frames", dtype=np.uint16, copy=True)
    n, h, w = frames.shape
    thr, nt = _label_thresholds(threshold, what, n)
    if _is_torch(frames):
        import torch

        if labels is None:
            labels = torch.empty((n, h, w), dtype=torch.int32, device=frames.device)
        counts = torch.empty(n, dtype=torch.int32, device=frames.device)
        stats = torch.zeros((n, max_components, 10), dtype=torch.int64, device=frames.device)
    else:
        if labels is None:
            labels = np.empty((n, h, w), np.int32)
        counts = np.empty(n, np.int32)
        stats = np.zeros((n, max_components, 10), np.int64)
    labels = _operand(labels, what, "labels", (n, h, w), np.int32)
    r = lib.rirb_label_batch(_ptr(frames), w, h, n, _ptr(thr), nt, connectivity, _ptr(labels), _ptr(counts), _ptr(stats),
                             max_components)
    _lib.check(r, what)
    return labels, counts, stats


def _label_thresholds(threshold, what, n):
    """``threshold`` of a labelling call: one uint16 value or one per frame, as a dense host array or a device tensor."""
    if _is_torch(threshold):
        thr = _operand(threshold.reshape(-1), what, "threshold", dtype=np.uint16)
        nt = thr.numel()
    else:
        t = np.asarray(threshold).reshape(-1)
        if t.size and (not np.all(np.isfinite(t)) or np.any(t != np.floor(t)) or t.min() < 0 or t.max() > 65535):
            raise RuntimeError(f"{what}: thresholds must be integers in [0, 65535]")
        thr = np.ascontiguousarray(t, dtype=np.uint16)
        nt = thr.size
    if nt not in (1, n):
        raise RuntimeError(f"{what}: {nt} thresholds for {n} frames")
    return thr, nt


# columns of the statistics rows of ``label_movie``; the centroid is ``stats[:, EV_SUM_X] / stats[:, EV_VOLUME]`` (likewise
# t and y) and the duration ``stats[:, EV_T_LAST] - stats[:, EV_T_FIRST] + 1``
(EV_VOLUME, EV_T_FIRST, EV_T_LAST, EV_X_MIN, EV_Y_MIN, EV_X_MAX, EV_Y_MAX, EV_SUM_T, EV_SUM_X, EV_SUM_Y, EV_SUM_VALUE,
 EV_MAX_VALUE, EV_ARGMAX) = range(13)


def label_movie(frames, threshold, connectivity=26, max_events=256, labels=None):
    """Events of a uint16 movie ``[n, h, w]``: the connected components of ``frames > threshold`` in space and time, with
    per-event statistics.

    ``threshold``: a scalar or one value per frame, as for ``label_batch``.  ``connectivity``: 6, 18 or 26 over the axes
    ``(t, y, x)`` (``scipy.ndimage.generate_binary_structure(3, 1 | 2 | 3)``).  Returns ``(labels, count, stats)``: int32
    ``labels [n, h, w]`` (0 background, 1..K numbered in raster order of each event's first voxel, as
    ``scipy.ndimage.label`` on the volume), ``count`` (K, a Python int) and int64 ``stats [max_events, 13]`` whose row
    ``k - 1`` describes event ``k`` (columns ``EV_VOLUME`` .. ``EV_ARGMAX``; ``EV_ARGMAX`` is ``t * h * w + y * w + x``;
    rows past ``min(K, max_events)`` are zero).  numpy in gives numpy out; a torch CUDA tensor gives tensors on its
    device.  ``labels``: an int32 output of the same shape, or None.  The whole movie is one call: two events that merge
    in a later frame are one event."""
    lib = _lib.load()
    what = "label_movie"
    if len(frames.shape) != 3:
        raise RuntimeError(f"{what}: wrong input dimension")
    if connectivity not in (6, 18, 26):
        raise RuntimeError(f"{what}: connectivity must be 6, 18 or 26, not {connectivity}")
    if int(max_events) != max_events or max_events < 0:
        raise RuntimeError(f"{what}: max_events must be a non-negative integer")
    max_events = int(max_events)
    _prepare_device_call(frames)
    frames = _operand(frames, what, "frames", dtype=np.uint16, copy=True)
    n, h, w = frames.shape
    thr, nt = _label_thresholds(threshold, what, n)
    count = np.zeros(1, np.int32)  # the entry waits for its stream, so a host count is ready when it returns
    if _is_torch(frames):
        import torch

        if labels is None:
            labels = torch.empty((n, h, w), dtype=torch.int32, device=frames.device)
        stats = torch.zeros((max_events, 13), dtype=torch.int64, device=frames.device)
    else:
        if labels is None:
            labels = np.empty((n, h, w), np.int32)
        stats = np.zeros((max_events, 13), np.int64)
    labels = _operand(labels, what, "labels", (n, h, w), np.int32)
    r = lib.rirb_label_movie(_ptr(frames), w, h, n, _ptr(thr), nt, connectivity, _ptr(labels), _ptr(count), _ptr(stats),
                             max_events)
    _lib.check(r, what)
    return labels, int(count[0]), stats


# ----------------------------------------------------------------------------------------
# bad pixels
# ----------------------------------------------------------------------------------------
def bad_pixels_create(first_image):
    """Run the bad-pixel detection on ``first_image`` and keep the flagged set (and the clamp level) behind a new
    handle, which is what the call returns (rir_signal_processing.py:273-289)."""
    lib = _lib.load()
    if _is_torch(first_image):
        _prepare_device_call(first_image)
        img = first_image
    else:
        img = np.array(first_image, dtype=np.uint16, order="C")
    img = _operand(img, "bad_pixels_create", "first_image", dtype=np.uint16, copy=True)
    if len(img.shape) != 2:
        raise RuntimeError("bad_pixels_create: wrong input image dimension")
    ret = lib.bad_pixels_create(_ptr(img), img.shape[1], img.shape[0])
    if ret <= 0:
        raise RuntimeError(f"'bad_pixels_create': {_lib.last_error()}")
    _BP_SHAPES[ret] = tuple(img.shape)
    return ret


_BP_SHAPES = {}  # handle -> (h, w) of the image it was created on: the frame size the batch calls read and write


def _bp_frames(handle, frames, what, copy=True):
    """``frames`` of a batch call on a bad-pixel handle: uint16 ``[n, h, w]`` with the handle's ``(h, w)``."""
    hw = _BP_SHAPES.get(handle)
    if len(frames.shape) != 3:
        raise RuntimeError(f"{what}: wrong input dimension")
    return _operand(frames, what, "frames", (frames.shape[0],) + hw if hw else None, np.uint16, copy=copy)


def bad_pixels_correct_gaussian_batch(handle, frames, sigma=1.0, out=None, smoothed=None):
    """``bad_pixels_correct_batch`` followed by ``gaussian_filter_batch`` of the corrected frames, in one pass over the
    movie: returns ``(corrected uint16 [n,h,w], smoothed float32 [n,h,w])``.  A strided numpy ``frames`` is copied
    first; a strided ``out`` or ``smoothed`` is refused."""
    lib = _lib.load()
    _prepare_device_call(frames)
    what = "bad_pixels_correct_gaussian_batch"
    frames = _bp_frames(handle, frames, what)
    if out is None:
        out = _empty_like(frames)
    if smoothed is None:
        smoothed = _empty_like(frames, np.float32)
    out = _operand(out, what, "out", frames.shape, np.uint16)
    smoothed = _operand(smoothed, what, "smoothed", frames.shape, np.float32)
    res = lib.rirb_bad_pixels_correct_gaussian_batch(handle, _ptr(frames), _ptr(out), _ptr(smoothed), frames.shape[0], float(sigma))
    _lib.check(res, "bad_pixels_correct_gaussian")
    return out, smoothed


def bad_pixels_destroy(handle):
    """Release a handle obtained from ``bad_pixels_create``."""
    _lib.load().bad_pixels_destroy(handle)
    _BP_SHAPES.pop(handle, None)


def bad_pixels_correct(handle, img):
    """Median-replace the handle's flagged pixels in ``img`` and clamp the rest; returns a new uint16 image."""
    lib = _lib.load()
    img = np.ascontiguousarray(img, dtype=np.uint16)
    out = np.empty(img.shape, dtype=np.uint16)
    res = lib.bad_pixels_correct(handle, _ptr(img), _ptr(out))
    if res < 0:
        raise RuntimeError("'bad_pixels_correct': unknown error")
    return out


def bad_pixels_correct_batch(handle, frames, out=None):
    """Correct a stack ``[n, h, w]`` of uint16 frames in one launch (``out is frames``: in place).  A strided numpy
    ``frames`` is copied first; a strided ``out`` is refused."""
    lib = _lib.load()
    _prepare_device_call(frames)
    inplace = out is frames
    frames = _bp_frames(handle, frames, "bad_pixels_correct_batch", copy=not inplace)
    if out is None:
        out = _empty_like(frames)
    out = frames if inplace else _operand(out, "bad_pixels_correct_batch", "out", frames.shape, np.uint16)
    res = lib.rirb_bad_pixels_correct_batch(handle, _ptr(frames), _ptr(out), frames.shape[0])
    _lib.check(res, "bad_pixels_correct")
    return out


def bad_pixels_list(handle):
    """Raster-ordered ``(x, y)`` list and clamp level held by a handle (introspection)."""
    lib = _lib.load()
    k = _lib.check(lib.rirb_bad_pixels_count(handle), "bad_pixels_count")
    xy = np.zeros((max(k, 1), 2), dtype=np.int32)
    clamp = ct.c_int(0)
    _lib.check(lib.rirb_bad_pixels_get(handle, _ptr(xy), k, ct.byref(clamp)), "bad_pixels_get")
    return xy[:k], clamp.value


class BadPixels:
    """Owner of a bad-pixel handle: detection at construction, ``correct`` per image, release on deletion
    (BadPixels.py:16-29)."""

    def __init__(self, first_image):
        self.handle = bad_pixels_create(first_image)

    def __del__(self):
        try:
            bad_pixels_destroy(self.handle)
        except Exception:
            pass

    def correct(self, img):
        return bad_pixels_correct(self.handle, img)

    def correct_batch(self, frames, out=None):
        return bad_pixels_correct_batch(self.handle, frames, out)

    def correct_gaussian_batch(self, frames, sigma=1.0, out=None, smoothed=None):
        return bad_pixels_correct_gaussian_batch(self.handle, frames, sigma, out, smoothed)


__all__ = [
    "translate",
    "translate_batch",
    "gaussian_filter",
    "gaussian_filter_batch",
    "find_median_pixel",
    "label_batch",
    "label_movie",
    "bad_pixels_create",
    "bad_pixels_correct",
    "bad_pixels_correct_batch",
    "bad_pixels_correct_gaussian_batch",
    "bad_pixels_destroy",
    "bad_pixels_list",
    "BadPixels",
]
