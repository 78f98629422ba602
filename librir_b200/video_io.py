"""Host-side mirror of the slices of ``librir.video_io`` that sit on the hot path.

* the lossless writer's pre-coder: what ``H264Capture::AddFrame`` does to a frame before handing
  it to the codec (h264.cpp:1022-1131: key-frame decision :1050-1064, byte-plane split
  :1066-1103) and its inverse ``VideoGrabber::toArray`` (h264.cpp:3016-3051), plus this repo's
  temporal-delta option (DESIGN.md, parity unpinned);
* the file loader's per-frame hooks: ``IRFileLoader::removeBadPixels`` (IRFileLoader.cpp:722-802),
  ``removeMotionGeneric`` (:617-627) and the ``.regfile`` reader ``loadTranslationFile``
  (:822-847) / writer ``MaskedRegistratorECC.to_reg_file`` (masked_registration_ecc.py:214-215).

The bitstream stage (ffmpeg / x264 / zstd) stays on the host and outside this package.
"""
from __future__ import annotations

import numpy as np

from . import _lib
from .signal_processing import _empty_like, _is_torch, _operand, _prepare_device_call, _ptr, bad_pixels_create, bad_pixels_destroy

DEFAULT_GOP = 50  # H264_Saver default, h264.cpp:1052-1061 / setParameter "GOP"


def linesize(width: int, align: int = 32) -> int:
    """Row stride av_frame_get_buffer(frame, 32) gives an 8-bit plane (h264.cpp:1041)."""
    return (width + align - 1) // align * align


def key_frames(nframes: int, gop: int = DEFAULT_GOP) -> np.ndarray:
    """AddFrame's key-frame decision for a writer starting at frame 0 (h264.cpp:1050-1061)."""
    key = np.zeros(nframes, dtype=np.uint8)
    _lib.check(_lib.load().rirb_key_frames(nframes, gop, _ptr(key)), "key_frames")
    return key


# ----------------------------------------------------------------------------------------
# per-frame AVFrame layouts
# ----------------------------------------------------------------------------------------
def split_yuv444(image, it=None, ls=None):
    """YUV444P branch of AddFrame: returns planes (Y, U, V), each ``[h, linesize]``;
    U = low bytes, V = high bytes, Y = ``it`` (integration-time image) or 0."""
    lib = _lib.load()
    img = np.ascontiguousarray(image, dtype=np.uint16)
    if img.ndim != 2:
        raise RuntimeError("split_yuv444: wrong input image dimension")
    h, w = img.shape
    ls = ls or linesize(w)
    planes = [np.zeros((h, ls), dtype=np.uint8) for _ in range(3)]
    itp = _ptr(np.ascontiguousarray(it, dtype=np.uint8)) if it is not None else None
    r = lib.rirb_split_yuv444(_ptr(img), itp, w, h, _ptr(planes[0]), _ptr(planes[1]), _ptr(planes[2]), ls, ls, ls)
    _lib.check(r, "split_yuv444")
    return planes


def merge_yuv444(y, u, v, width):
    """toArray, YUV444P branch: returns (image uint16 [h,w], it uint8 [h,w])."""
    lib = _lib.load()
    y, u, v = (np.ascontiguousarray(p, dtype=np.uint8) for p in (y, u, v))
    h, ls = u.shape
    img = np.zeros((h, width), dtype=np.uint16)
    it = np.zeros((h, width), dtype=np.uint8)
    r = lib.rirb_merge_yuv444(_ptr(y), _ptr(u), _ptr(v), y.shape[1], ls, v.shape[1], width, h, _ptr(img), _ptr(it))
    _lib.check(r, "merge_yuv444")
    return img, it


def split_yuv420(image, it=None, ls=None):
    """YUV420P branch of AddFrame: luma plane ``[2h, linesize]`` (rows [0,h) low bytes, rows
    [h,2h) high bytes) and, when ``it`` is given, the U plane holding it."""
    lib = _lib.load()
    img = np.ascontiguousarray(image, dtype=np.uint16)
    if img.ndim != 2:
        raise RuntimeError("split_yuv420: wrong input image dimension")
    h, w = img.shape
    ls = ls or linesize(w)
    y = np.zeros((2 * h, ls), dtype=np.uint8)  # the writer memsets the whole buffer first (h264.cpp:1088)
    u = np.zeros((h, ls), dtype=np.uint8) if it is not None else None
    itp = _ptr(np.ascontiguousarray(it, dtype=np.uint8)) if it is not None else None
    r = lib.rirb_split_yuv420(_ptr(img), itp, w, h, _ptr(y), ls, _ptr(u) if u is not None else None, ls)
    _lib.check(r, "split_yuv420")
    return (y, u) if it is not None else y


def merge_yuv420(y, width, u=None):
    lib = _lib.load()
    y = np.ascontiguousarray(y, dtype=np.uint8)
    h = y.shape[0] // 2
    img = np.zeros((h, width), dtype=np.uint16)
    if u is None:
        r = lib.rirb_merge_yuv420(_ptr(y), y.shape[1], None, 0, width, h, _ptr(img), None)
        _lib.check(r, "merge_yuv420")
        return img
    u = np.ascontiguousarray(u, dtype=np.uint8)
    it = np.zeros((h, width), dtype=np.uint8)
    r = lib.rirb_merge_yuv420(_ptr(y), y.shape[1], _ptr(u), u.shape[1], width, h, _ptr(img), _ptr(it))
    _lib.check(r, "merge_yuv420")
    return img, it


# ----------------------------------------------------------------------------------------
# whole movies (dense planes)
# ----------------------------------------------------------------------------------------
def precode_movie(movie, gop=DEFAULT_GOP, delta=False, first_frame=0, out=None, stats=None):
    """Byte-plane split (+ optional temporal delta) of ``movie[t, h, w]`` (numpy or torch CUDA
    uint16).  Returns ``(lo, hi)`` uint8 ``[t, h, w]``.  ``stats``: a :class:`librir_b200.movie.MovieStats`
    to fold the same frames into (min / max / histogram) in the same pass over them.  ``out``: a ``(lo, hi)`` pair of
    uint8 arrays of ``movie``'s shape.  A strided numpy ``movie`` is copied first; strided planes are refused."""
    lib = _lib.load()
    if len(movie.shape) != 3:
        raise RuntimeError("precode_movie: wrong input dimension")
    _prepare_device_call(movie)
    movie = _operand(movie, "precode_movie", "movie", dtype=np.uint16, copy=True)
    t, h, w = movie.shape
    if out is not None and len(out) != 2:
        raise RuntimeError("precode_movie: out must be a (lo, hi) pair")
    lo, hi = out if out is not None else (_empty_like(movie, np.uint8), _empty_like(movie, np.uint8))
    lo = _operand(lo, "precode_movie", "lo", movie.shape, np.uint8)
    hi = _operand(hi, "precode_movie", "hi", movie.shape, np.uint8)
    if stats is not None:
        import ctypes as ct

        if stats._fresh:
            stats._sums[65536] = 0
        r = lib.rirb_precode_movie_stats(_ptr(movie), t, w, h, gop, int(bool(delta)), first_frame, _ptr(lo), _ptr(hi),
                                         ct.c_void_p(stats.minmax.data_ptr()), ct.c_void_p(stats.hist.data_ptr()),
                                         0 if stats._fresh else 1)
        _lib.check(r, "precode_movie_stats")
        stats._fresh = False
        stats._sums[65536] += t * h * w
        return lo, hi
    r = lib.rirb_precode_movie(_ptr(movie), t, w, h, gop, int(bool(delta)), first_frame, _ptr(lo), _ptr(hi))
    _lib.check(r, "precode_movie")
    return lo, hi


def decode_movie(lo, hi, gop=DEFAULT_GOP, delta=False, first_frame=0, out=None):
    """Inverse of :func:`precode_movie`: uint8 planes ``lo`` / ``hi`` ``[t, h, w]`` -> uint16 ``out`` of the same shape.
    Strided numpy planes are copied first; a strided ``out`` is refused."""
    lib = _lib.load()
    _prepare_device_call(lo)
    if len(lo.shape) != 3:
        raise RuntimeError("decode_movie: wrong input dimension")
    lo = _operand(lo, "decode_movie", "lo", dtype=np.uint8, copy=True)
    hi = _operand(hi, "decode_movie", "hi", lo.shape, np.uint8, copy=True)
    t, h, w = lo.shape
    mov = out if out is not None else _empty_like(lo, np.uint16)
    mov = _operand(mov, "decode_movie", "out", lo.shape, np.uint16)
    r = lib.rirb_decode_movie(_ptr(lo), _ptr(hi), t, w, h, gop, int(bool(delta)), first_frame, _ptr(mov))
    _lib.check(r, "decode_movie")
    return mov


class LosslessPrecoder:
    """Frame-at-a-time front of the lossless writer, mirroring ``H264_Saver::addImageLossLess``
    -> ``H264Capture::AddFrame`` up to the point where the frame is handed to the codec.

    ``add_image`` returns what the codec would be given for that frame: ``(key, Y, U, V)`` for
    the default YUV444P layout (or ``(key, Y)`` / ``(key, Y, U)`` for YUV420P)."""

    def __init__(self, width, height, gop=DEFAULT_GOP, pix_fmt="yuv444p"):
        if pix_fmt not in ("yuv444p", "yuv420p"):
            raise RuntimeError("LosslessPrecoder: unknown pixel format")
        self.width, self.height, self.gop, self.pix_fmt = width, height, gop, pix_fmt
        self.frame_counter = 0
        self.last_key_frame = 0

    def add_image(self, img, it=None, key=False):
        img = np.ascontiguousarray(img, dtype=np.uint16)
        if img.shape != (self.height, self.width):
            raise RuntimeError("add_image: wrong image size")
        # key-frame rule, h264.cpp:1052-1061 (the IT overload compares with '>', :1165)
        if self.frame_counter == 0:
            key = True
        elif (self.frame_counter - self.last_key_frame > self.gop) if it is not None else (
                self.frame_counter - self.last_key_frame >= self.gop):
            key = True
        if key:
            self.last_key_frame = self.frame_counter
        self.frame_counter += 1
        if self.pix_fmt == "yuv444p":
            y, u, v = split_yuv444(img, it)
            return key, y, u, v
        res = split_yuv420(img, it)
        return (key,) + (res if isinstance(res, tuple) else (res,))


# ----------------------------------------------------------------------------------------
# loader hooks
# ----------------------------------------------------------------------------------------
class LoaderBadPixels:
    """``IRFileLoader::setBadPixelsEnabled`` + ``removeBadPixels``: detection on the first frame
    without its last 3 (metadata) rows, in-place correction of rows ``[0, h-3)``."""

    def __init__(self, first_image, meta_rows=3):
        first = np.ascontiguousarray(first_image, dtype=np.uint16)
        self.height, self.width = first.shape
        self.rows = self.height - meta_rows
        self.handle = bad_pixels_create(first[: self.rows])

    def __del__(self):
        try:
            bad_pixels_destroy(self.handle)
        except Exception:
            pass

    def remove(self, frames):
        """In place on uint16 ``frames[n, h, w]`` (or one ``[h, w]`` frame); returns ``frames``.  Strided views are refused."""
        lib = _lib.load()
        _prepare_device_call(frames)
        n = 1 if len(frames.shape) == 2 else frames.shape[0]
        if tuple(frames.shape[-2:]) != (self.height, self.width):
            raise RuntimeError("remove_bad_pixels: wrong image size")
        _operand(frames, "remove_bad_pixels", "frames", dtype=np.uint16)
        r = lib.rirb_loader_remove_bad_pixels(self.handle, _ptr(frames), n, self.height * self.width)
        _lib.check(r, "remove_bad_pixels")
        return frames


def remove_motion(frames, shifts_x, shifts_y, meta_rows=3, out=None):
    """``removeMotionGeneric`` on a stack: frame t is translated by ``(-shifts_x[t], -shifts_y[t])``
    on rows ``[0, h-meta_rows)``; the metadata rows pass through.  uint16 ``frames``; ``out``: same shape and dtype
    (``out is frames``: in place).  A strided numpy ``frames`` is copied first (unless in place); a strided ``out`` is
    refused."""
    lib = _lib.load()
    _prepare_device_call(frames)
    inplace = out is frames
    frames = _operand(frames, "remove_motion", "frames", dtype=np.uint16, copy=not inplace)
    single = len(frames.shape) == 2
    n = 1 if single else frames.shape[0]
    h, w = frames.shape[-2:]
    sx = np.ascontiguousarray(np.atleast_1d(shifts_x), dtype=np.float64)
    sy = np.ascontiguousarray(np.atleast_1d(shifts_y), dtype=np.float64)
    if sx.size != n or sy.size != n:
        raise RuntimeError("remove_motion: one shift per frame expected")
    if out is None:
        out = _empty_like(frames)
    out = frames if inplace else _operand(out, "remove_motion", "out", frames.shape, np.uint16)
    r = lib.rirb_loader_remove_motion(_ptr(frames), _ptr(out), w, h - meta_rows, n, h * w, _ptr(sx), _ptr(sy))
    _lib.check(r, "remove_motion")
    return out


def finish_frames(frames, bad_pixels=None, min_T=0, min_T_height=0, shifts_x=None, shifts_y=None, meta_rows=3):
    """The same chain as :func:`read_movie` for frames that are uint16 already (decoded from the zstd movie file):
    ``+= min_T`` -> ``removeBadPixels`` -> ``removeMotion``, IN PLACE on ``frames`` ``[n, h, w]`` (numpy or torch CUDA).
    What ``load_image`` of ``libvideo_io_b200.so`` runs after the decode.  Strided views are refused."""
    lib = _lib.load()
    _prepare_device_call(frames)
    _operand(frames, "finish_frames", "frames", dtype=np.uint16)
    single = len(frames.shape) == 2
    n = 1 if single else frames.shape[0]
    h, w = frames.shape[-2:]
    sx = sy = None
    if shifts_x is not None or shifts_y is not None:
        sx = np.ascontiguousarray(np.atleast_1d(shifts_x), dtype=np.float64)
        sy = np.ascontiguousarray(np.atleast_1d(shifts_y), dtype=np.float64)
        if sx.size != n or sy.size != n:
            raise RuntimeError("finish_frames: one shift per frame expected")
    r = lib.rirb_loader_finish_frames(bad_pixels.handle if bad_pixels is not None else 0, _ptr(frames), n, w, h, int(min_T), int(min_T_height),
                                      _ptr(sx) if sx is not None else None, _ptr(sy) if sy is not None else None, int(meta_rows))
    _lib.check(r, "loader_finish_frames")
    return frames


def read_movie(lo, hi, bad_pixels=None, min_T=0, min_T_height=0, shifts_x=None, shifts_y=None, meta_rows=3, out=None):
    """``IRFileLoader::readImage``'s post-decode chain (IRFileLoader.cpp:1168-1247, calibration 0) on a
    run of decoded frames: byte planes ``lo``/``hi`` ``[n, h, w]`` (what ``VideoGrabber::toArray`` merges,
    h264.cpp:3016-3051) -> ``+= min_T`` on the first ``min_T_height`` rows -> ``removeBadPixels`` on rows
    ``[0, h-meta_rows)`` (``bad_pixels``: a :class:`LoaderBadPixels` or None) -> ``removeMotion`` by the
    per-frame shifts of the ``.regfile`` (None: off).  Returns uint16 ``[n, h, w]`` (``out``: of ``lo``'s shape).
    Strided numpy planes are copied first; a strided ``out`` is refused."""
    lib = _lib.load()
    _prepare_device_call(lo)
    single = len(lo.shape) == 2
    n = 1 if single else lo.shape[0]
    h, w = lo.shape[-2:]
    lo = _operand(lo, "read_movie", "lo", dtype=np.uint8, copy=True)
    hi = _operand(hi, "read_movie", "hi", lo.shape, np.uint8, copy=True)
    handle = 0
    if bad_pixels is not None:
        if (bad_pixels.height, bad_pixels.width) != (h, w) or bad_pixels.rows != h - meta_rows:
            raise RuntimeError("read_movie: wrong image size for this bad-pixel state")
        handle = bad_pixels.handle
    sx = sy = None
    if shifts_x is not None or shifts_y is not None:
        sx = np.ascontiguousarray(np.atleast_1d(shifts_x), dtype=np.float64)
        sy = np.ascontiguousarray(np.atleast_1d(shifts_y), dtype=np.float64)
        if sx.size != n or sy.size != n:
            raise RuntimeError("read_movie: one shift per frame expected")
    if out is None:
        out = _empty_like(lo, np.uint16)
    out = _operand(out, "read_movie", "out", lo.shape, np.uint16)
    r = lib.rirb_loader_read_movie(handle, _ptr(lo), _ptr(hi), n, w, h, int(min_T), int(min_T_height),
                                   _ptr(sx) if sx is not None else None, _ptr(sy) if sy is not None else None, int(meta_rows),
                                   _ptr(out))
    _lib.check(r, "read_movie")
    return out


class LossyPreconditioner:
    """``H264_Saver``'s lossy "bounded-error" pre-conditioner (``addImageLossyNoCamera``, h264.cpp:2253-2424):
    frames in temperature, IN TIME ORDER -> the frames the lossless encoder then receives, pixels that stay
    within the per-frame error bounds being frozen to a reference / running-average value.  Parameters are the
    saver's string parameters (h264.cpp:1709-1781) with their defaults (PrivateData(), :1663-1665).
    ``variant="add_loss"`` selects ``H264_Saver::addLoss`` (h264.cpp:2426-2607, what ``h264_add_loss`` runs) instead;
    ``memcpyQuirk=False`` replaces the compiled reference's overlapping memcpy of its spread window by a memmove."""

    def __init__(self, width, height, lossy_height=None, lowValueError=6, highValueError=2, stdFactor=5.0, runningAverage=32,
                 subtractMin=False, removeBadPixels=False, variant="add_image_lossy", memcpyQuirk=True):
        lib = _lib.load()
        self.width, self.height = int(width), int(height)
        self.lossy_height = self.height if lossy_height is None else int(lossy_height)
        self.handle = lib.rirb_lossy_open(self.width, self.height, self.lossy_height, int(lowValueError), int(highValueError),
                                          float(stdFactor), int(runningAverage), int(bool(subtractMin)), int(bool(removeBadPixels)))
        if self.handle <= 0:
            raise RuntimeError(f"An error occured while calling 'lossy_open': {_lib.last_error()}")
        self.variant = str(variant)
        _lib.check(lib.rirb_lossy_set_parameter(self.handle, b"variant", self.variant.encode()), "lossy_set_parameter")
        _lib.check(lib.rirb_lossy_set_parameter(self.handle, b"memcpyQuirk", b"1" if memcpyQuirk else b"0"), "lossy_set_parameter")

    def __del__(self):
        try:
            _lib.load().rirb_lossy_close(self.handle)
        except Exception:
            pass

    def add_images(self, frames, out=None):
        """``frames``: uint16 ``[n, h, w]`` (or one ``[h, w]`` frame), numpy or torch CUDA.  Returns
        ``(out, errors)`` with ``errors[t] = (BackgroundError, ForegroundError)`` of frame t.  ``out``: uint16 of
        ``frames``' shape.  A strided numpy ``frames`` is copied first; a strided ``out`` is refused."""
        lib = _lib.load()
        _prepare_device_call(frames)
        frames = _operand(frames, "lossy add_images", "frames", dtype=np.uint16, copy=True)
        single = len(frames.shape) == 2
        n = 1 if single else frames.shape[0]
        if tuple(frames.shape[-2:]) != (self.height, self.width):
            raise RuntimeError("lossy add_images: wrong image size")
        if out is None:
            out = _empty_like(frames)
        out = _operand(out, "lossy add_images", "out", frames.shape, np.uint16)
        errors = np.zeros((n, 2), dtype=np.int32)
        r = lib.rirb_lossy_add_images(self.handle, _ptr(frames), n, _ptr(out), _ptr(errors))
        _lib.check(r, "lossy_add_images")
        return out, errors


def load_translation_file(filename, nframes=None):
    """``IRFileLoader::loadTranslationFile`` (IRFileLoader.cpp:822-847): tab-separated file, one
    header line, 4 columns; shifts are columns 1 and 2.  Returns ``(x, y)`` float64 arrays."""
    with open(filename) as f:
        f.readline()
        rows = [ln.split() for ln in f if ln.strip()]
    try:
        ar = np.array(rows, dtype=np.float32)  # the reference parses floats (Array2D<float>)
    except ValueError as e:
        raise RuntimeError(f"error while loading motion correction file: {e}")
    if ar.ndim != 2 or ar.shape[1] != 4:
        raise RuntimeError("error while loading motion correction file: 4 columns expected")
    if nframes is not None and ar.shape[0] != nframes:
        raise RuntimeError("wrong number of images in motion correction file")
    return ar[:, 1].astype(np.float64), ar[:, 2].astype(np.float64)


def save_translation_file(filename, x, y, confidence=None):
    """``MaskedRegistratorECC.to_reg_file`` layout (a pandas ``to_csv(sep="\\t")`` of the three
    columns below with the frame index in front)."""
    x = np.asarray(x, dtype=np.float64)
    y = np.asarray(y, dtype=np.float64)
    c = np.ones_like(x) if confidence is None else np.asarray(confidence, dtype=np.float64)
    with open(filename, "w") as f:
        f.write("\tx-axis translations\ty-axis translations\tConfidence level\n")
        for i in range(len(x)):
            f.write(f"{i}\t{float(x[i])!r}\t{float(y[i])!r}\t{float(c[i])!r}\n")


__all__ = [
    "DEFAULT_GOP", "linesize", "key_frames", "split_yuv444", "merge_yuv444", "split_yuv420", "merge_yuv420",
    "precode_movie", "decode_movie", "LosslessPrecoder", "LoaderBadPixels", "remove_motion", "read_movie", "finish_frames", "LossyPreconditioner",
    "load_translation_file",
    "save_translation_file",
]
