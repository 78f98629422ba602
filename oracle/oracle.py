"""ctypes front-end of the CPU oracle (oracle.c) and of the compiled reference (oracle/_ref).

TEST INFRASTRUCTURE ONLY -- see the header of oracle.c.  Two back-ends with one interface:

* ``port``  : liboracle.so, the C restatement built from oracle/oracle.c (always available).
* ``ref``   : oracle/_ref/libs/libsignal_processing.so, the reference's own sources compiled
              by oracle/build_ref.sh (available where it was built; it travels to the GPU box).

Function names follow the reference's Python API (librir/signal_processing/
rir_signal_processing.py) so that the parity tests read like the reference's own tests.
"""
from __future__ import annotations

import ctypes as ct
import os
import subprocess

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
_PORT_PATH = os.path.join(_HERE, "liboracle.so")
_REF_DIR = os.path.join(_HERE, "_ref", "libs")
_REF_PATH = os.path.join(_REF_DIR, "libsignal_processing.so")
_REF_OMP_PATH = os.path.join(_REF_DIR, "libsignal_processing_omp.so")

_DTYPE_CODES = {
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


def build(force: bool = False) -> None:
    """Compile liboracle.so (and oracle/_ref when /root/reference is present)."""
    src = os.path.join(_HERE, "oracle.c")
    if force or not os.path.exists(_PORT_PATH) or os.path.getmtime(_PORT_PATH) < os.path.getmtime(src):
        subprocess.check_call(["make", "-C", _HERE, "-B", "liboracle.so"], stdout=subprocess.DEVNULL)
    if os.path.isdir(os.environ.get("LIBRIR_REFERENCE", "/root/reference")):
        subprocess.check_call(["bash", os.path.join(_HERE, "build_ref.sh")], stdout=subprocess.DEVNULL)


_port = None
_ref = None
_ref_omp = None


def port_lib() -> ct.CDLL:
    global _port
    if _port is None:
        build()
        _port = ct.CDLL(_PORT_PATH)
        _port.orc_get_background.restype = ct.c_uint
    return _port


def have_ref() -> bool:
    return os.path.exists(_REF_PATH)


def ref_lib(omp: bool = False) -> ct.CDLL:
    """The compiled reference (stock flags; ``omp=True``: same sources with -fopenmp)."""
    global _ref, _ref_omp
    if omp:
        if _ref_omp is None:
            ct.CDLL(os.path.join(_REF_DIR, "libtools.so"), mode=ct.RTLD_GLOBAL)
            _ref_omp = ct.CDLL(_REF_OMP_PATH)
        return _ref_omp
    if _ref is None:
        ct.CDLL(os.path.join(_REF_DIR, "libtools.so"), mode=ct.RTLD_GLOBAL)
        _ref = ct.CDLL(_REF_PATH)
    return _ref


def _p(a: np.ndarray):
    return a.ctypes.data_as(ct.c_void_p)


def _c(a, dtype=None) -> np.ndarray:
    return np.ascontiguousarray(a, dtype=dtype)


# ----------------------------------------------------------------------------------------
# interface shared by both back-ends
# ----------------------------------------------------------------------------------------
class _Base:
    kind = "?"

    # -- translate -----------------------------------------------------------------------
    def translate(self, image, dx, dy, strategy="", background=None):
        """Semantics of librir.signal_processing.translate (rir_signal_processing.py:23-82)."""
        if image.ndim != 2:
            raise RuntimeError("translate: wrong input image dimension")
        if strategy == "background" and background is None:
            raise RuntimeError("translate: wrong background value")
        if strategy == "constant":
            strategy = "background"
        img = np.copy(image, "C")
        res = np.copy(image, "C")
        back = np.zeros(1, dtype=img.dtype)
        if background is not None:
            back[0] = background
        code = _DTYPE_CODES.get(img.dtype)
        if code is None:
            raise RuntimeError("An error occured while calling 'translate'")
        r = self._translate(ord(code), img, res, img.shape[1], img.shape[0], np.float32(dx), np.float32(dy), back,
                            strategy.encode())
        if r < 0:
            raise RuntimeError("An error occured while calling 'translate'")
        return res

    # -- gaussian ------------------------------------------------------------------------
    def gaussian_filter(self, image, sigma=1.0):
        if image.ndim != 2:
            raise RuntimeError("gaussian_filter: wrong input image dimension")
        img = np.array(image, dtype=np.float32, order="C")
        res = np.zeros(image.shape, dtype=np.float32)
        self._gaussian(img, res, img.shape[1], img.shape[0], float(sigma))
        return res


class Port(_Base):
    """The C restatement (oracle.c)."""

    kind = "port"

    def __init__(self):
        self.lib = port_lib()

    def _translate(self, code, img, res, w, h, dx, dy, back, strategy):
        f = self.lib.orc_translate
        f.argtypes = [ct.c_int, ct.c_void_p, ct.c_void_p, ct.c_int, ct.c_int, ct.c_float, ct.c_float, ct.c_void_p,
                      ct.c_char_p]
        return f(code, _p(img), _p(res), w, h, dx, dy, _p(back), strategy)

    def _gaussian(self, img, res, w, h, sigma):
        f = self.lib.orc_gaussian_filter
        f.argtypes = [ct.c_void_p, ct.c_void_p, ct.c_int, ct.c_int, ct.c_float]
        return f(_p(img), _p(res), w, h, sigma)

    def gaussian_kernel(self, sigma):
        self.lib.orc_gaussian_radius.argtypes = [ct.c_float]
        r = self.lib.orc_gaussian_radius(float(sigma))
        k = np.zeros((2 * r + 1, 2 * r + 1), dtype=np.float32)
        self.lib.orc_gaussian_kernel.argtypes = [ct.c_float, ct.c_int, ct.c_void_p]
        self.lib.orc_gaussian_kernel(float(sigma), r, _p(k))
        return k

    # bad pixels ------------------------------------------------------------------------
    def bad_pixels_detect(self, first, std_factor=5.0):
        """Returns (xy[K,2] int32 raster-ordered, global_threshold, clamp_value)."""
        img = _c(first, np.uint16)
        h, w = img.shape
        f = self.lib.orc_bad_pixels_detect
        f.argtypes = [ct.c_void_p, ct.c_int, ct.c_int, ct.c_double, ct.c_void_p, ct.c_int, ct.c_void_p]
        thr = ct.c_int(0)
        cap = img.size
        xy = np.zeros((cap, 2), dtype=np.int32)
        k = f(_p(img), w, h, float(std_factor), _p(xy), cap, ct.byref(thr))
        self.lib.orc_bad_pixels_clamp_value.argtypes = [ct.c_void_p, ct.c_int, ct.c_int]
        clamp = self.lib.orc_bad_pixels_clamp_value(_p(img), w, h)
        return xy[:k].copy(), thr.value, clamp

    def bad_pixels_correct_with(self, xy, clamp, image):
        img = _c(image, np.uint16)
        out = np.zeros_like(img)
        h, w = img.shape
        xy = _c(xy, np.int32)
        f = self.lib.orc_bad_pixels_correct
        f.argtypes = [ct.c_void_p, ct.c_void_p, ct.c_int, ct.c_int, ct.c_void_p, ct.c_int, ct.c_int]
        f(_p(img), _p(out), w, h, _p(xy), len(xy), int(clamp))
        return out

    def bad_pixels_correct_inplace(self, xy, clamp, image):
        """BadPixels::correct with in == out (sequential: later pixels see earlier corrections)."""
        img = np.array(image, dtype=np.uint16, order="C")
        h, w = img.shape
        xy = _c(xy, np.int32)
        f = self.lib.orc_bad_pixels_correct
        f.argtypes = [ct.c_void_p, ct.c_void_p, ct.c_int, ct.c_int, ct.c_void_p, ct.c_int, ct.c_int]
        f(_p(img), _p(img), w, h, _p(xy), len(xy), int(clamp))
        return img

    def bad_pixels_create(self, first):
        xy, _thr, clamp = self.bad_pixels_detect(first)
        return (xy, clamp)

    def bad_pixels_correct(self, handle, image):
        return self.bad_pixels_correct_with(handle[0], handle[1], image)

    def bad_pixels_destroy(self, handle):
        pass

    def loader_remove_bad_pixels(self, image, xy):
        """IRFileLoader::removeBadPixels on rows [0,h) of ``image`` (caller crops h-3)."""
        img = np.array(image, dtype=np.uint16, order="C")
        h, w = img.shape
        xy = _c(xy, np.int32)
        f = self.lib.orc_loader_remove_bad_pixels
        f.argtypes = [ct.c_void_p, ct.c_int, ct.c_int, ct.c_void_p, ct.c_int]
        f(_p(img), w, h, _p(xy), len(xy))
        return img

    def loader_remove_motion(self, image, shift_x, shift_y):
        img = np.array(image, dtype=np.uint16, order="C")
        h, w = img.shape
        f = self.lib.orc_loader_remove_motion
        f.argtypes = [ct.c_void_p, ct.c_int, ct.c_int, ct.c_double, ct.c_double]
        f(_p(img), w, h, float(shift_x), float(shift_y))
        return img

    def lossy_open(self, w, h, stop_h, low_error=6, high_error=2, std_factor=5.0, running_average=32, subtract_min=False,
                   bp_enabled=False, variant=0, memcpy_quirk=True, exact_squares=False, saturating_round=False):
        """H264_Saver::addImageLossyNoCamera state (h264.cpp:2253-2424; variant=1: addLoss, :2426-2607); returns an
        opaque state for lossy_add.  memcpy_quirk: reproduce the compiled reference's overlapping memcpy (oracle.c).
        exact_squares / saturating_round: arithmetic the reference does NOT have (exact squares in stdDev; a saturating
        conversion with NaN -> 0 in the bound update), for tests that show its own arithmetic matters."""
        f = self.lib.orc_lossy_open
        f.restype = ct.c_void_p
        f.argtypes = [ct.c_int, ct.c_int, ct.c_int, ct.c_int, ct.c_int, ct.c_double, ct.c_int, ct.c_int, ct.c_int]
        st = ct.c_void_p(f(w, h, stop_h, low_error, high_error, std_factor, running_average, int(subtract_min), int(bp_enabled)))
        g = self.lib.orc_lossy_configure
        g.restype = None
        g.argtypes = [ct.c_void_p, ct.c_int, ct.c_int]
        g(st, int(variant), int(memcpy_quirk))
        g = self.lib.orc_lossy_counterfactual
        g.restype = None
        g.argtypes = [ct.c_void_p, ct.c_int, ct.c_int]
        g(st, int(exact_squares), int(saturating_round))
        return st

    def lossy_std_dev(self, prev, img, img_dl=None, back=0):
        """stdDev (h264.cpp:1993-2036) on flat arrays: (background, foreground) spreads; img_dl=None: un-split."""
        prev, img = _c(prev, np.uint16).ravel(), _c(img, np.uint16).ravel()
        dl = None if img_dl is None else _c(img_dl, np.uint16).ravel()
        out = np.zeros(2, dtype=np.float64)
        f = self.lib.orc_lossy_std_dev
        f.restype = None
        f.argtypes = [ct.c_void_p, ct.c_void_p, ct.c_int, ct.c_void_p, ct.c_uint, ct.c_void_p]
        f(_p(prev), _p(img), img.size, None if dl is None else _p(dl), int(back), _p(out))
        return float(out[0]), float(out[1])

    def lossy_bounds(self, variant, sd0, sd1, mean0, mean1, std_factor, low_error, high_error):
        """One frame's bound update (h264.cpp:2367-2376 / :2559-2567): returns (lowError, highError)."""
        e = np.array([low_error, high_error], dtype=np.int32)
        f = self.lib.orc_lossy_bounds
        f.restype = None
        f.argtypes = [ct.c_int, ct.c_double, ct.c_double, ct.c_double, ct.c_double, ct.c_double, ct.c_void_p]
        f(int(variant), sd0, sd1, mean0, mean1, std_factor, _p(e))
        return int(e[0]), int(e[1])

    def lossy_add(self, state, image):
        """One frame through the pre-conditioner: returns (frame handed to the lossless encoder, (lowError, highError))."""
        img = _c(image, np.uint16)
        out = np.empty_like(img)
        err = np.zeros(2, dtype=np.int32)
        f = self.lib.orc_lossy_add_image
        f.restype = None
        f.argtypes = [ct.c_void_p, ct.c_void_p, ct.c_void_p, ct.c_void_p]
        f(state, _p(img), _p(out), _p(err))
        return out, (int(err[0]), int(err[1]))

    def lossy_get_min(self, state):
        """MIN_T of a subtractMin state (what rirb_lossy_get_min reports)."""
        f = self.lib.orc_lossy_get_min
        f.restype = ct.c_int
        f.argtypes = [ct.c_void_p]
        return int(f(state))

    def lossy_close(self, state):
        f = self.lib.orc_lossy_close
        f.restype = None
        f.argtypes = [ct.c_void_p]
        f(state)

    def loader_read_image(self, lo, hi, xy=None, min_T=0, min_T_height=0, shift=None, meta_rows=3):
        """IRFileLoader::readImage after the decoder, calibration == 0 (IRFileLoader.cpp:1168-1247):
        toArray's merge (h264.cpp:3016-3051) -> += min_T on the first min_T_height rows (:1174-1179)
        -> removeBadPixels(pixels, w, h-3) (:1241) -> removeMotion(pixels, w, h-3, pos) (:1243)."""
        lo = np.asarray(lo, dtype=np.uint8)
        hi = np.asarray(hi, dtype=np.uint8)
        img = (lo.astype(np.uint16) | (hi.astype(np.uint16) << 8)).astype(np.uint16)
        h, w = img.shape
        if min_T and min_T_height:
            rows = min(h, int(min_T_height))
            img[:rows] = (img[:rows].astype(np.int64) + int(min_T)).astype(np.uint16)  # unsigned short += int: wraps
        hb = h - meta_rows
        if xy is not None and len(xy):
            img[:hb] = self.loader_remove_bad_pixels(img[:hb], xy)
        if shift is not None:
            img[:hb] = self.loader_remove_motion(img[:hb], shift[0], shift[1])
        return img

    # stats -----------------------------------------------------------------------------
    def find_median_pixel(self, image, percent=0.5, mask=None):
        img = _c(image, np.uint16)
        if mask is None:
            f = self.lib.orc_find_median_pixel
            f.argtypes = [ct.c_void_p, ct.c_int, ct.c_float]
            return f(_p(img), img.size, float(percent))
        m = _c(mask, np.uint8)
        f = self.lib.orc_find_median_pixel_mask
        f.argtypes = [ct.c_void_p, ct.c_void_p, ct.c_int, ct.c_float]
        return f(_p(img), _p(m), img.size, float(percent))

    def get_background(self, image):
        img = _c(image, np.uint16)
        f = self.lib.orc_get_background
        f.argtypes = [ct.c_void_p, ct.c_int]
        return int(f(_p(img), img.size))

    def movie_stats(self, movie):
        mov = _c(movie, np.uint16)
        hist = np.zeros(65536, dtype=np.uint64)
        lo, hi = ct.c_uint(0), ct.c_uint(0)
        f = self.lib.orc_movie_stats
        f.argtypes = [ct.c_void_p, ct.c_size_t, ct.c_void_p, ct.c_void_p, ct.c_void_p]
        f(_p(mov), mov.size, ct.byref(lo), ct.byref(hi), _p(hist))
        return lo.value, hi.value, hist

    def quantile_from_hist(self, hist, percent):
        hist = _c(hist, np.uint64)
        f = self.lib.orc_quantile_from_hist
        f.argtypes = [ct.c_void_p, ct.c_ulonglong, ct.c_float]
        return f(_p(hist), int(hist.sum()), float(percent))

    # pre-coder -------------------------------------------------------------------------
    def split_444(self, image, it=None, linesize=None):
        """H264Capture::AddFrame, YUV444P branch: returns (Y, U, V) planes [h][linesize]."""
        img = _c(image, np.uint16)
        h, w = img.shape
        ls = linesize or ((w + 31) // 32) * 32
        planes = [np.full((h, ls), 0xAA, dtype=np.uint8) for _ in range(3)]
        itp = _p(_c(it, np.uint8)) if it is not None else None
        f = self.lib.orc_split_444
        f.argtypes = [ct.c_void_p, ct.c_void_p, ct.c_int, ct.c_int, ct.c_void_p, ct.c_void_p, ct.c_void_p, ct.c_int,
                      ct.c_int, ct.c_int]
        f(_p(img), itp, w, h, _p(planes[0]), _p(planes[1]), _p(planes[2]), ls, ls, ls)
        return planes

    def merge_444(self, y, u, v, w):
        h, ls = u.shape
        img = np.zeros((h, w), dtype=np.uint16)
        it = np.zeros((h, w), dtype=np.uint8)
        f = self.lib.orc_merge_444
        f.argtypes = [ct.c_void_p, ct.c_void_p, ct.c_void_p, ct.c_int, ct.c_int, ct.c_int, ct.c_int, ct.c_int,
                      ct.c_void_p, ct.c_void_p]
        f(_p(_c(y)), _p(_c(u)), _p(_c(v)), ls, ls, ls, w, h, _p(img), _p(it))
        return img, it

    def split_420(self, image, linesize=None):
        img = _c(image, np.uint16)
        h, w = img.shape
        ls = linesize or ((w + 31) // 32) * 32
        y = np.full((2 * h, ls), 0xAA, dtype=np.uint8)
        f = self.lib.orc_split_420
        f.argtypes = [ct.c_void_p, ct.c_int, ct.c_int, ct.c_void_p, ct.c_int]
        f(_p(img), w, h, _p(y), ls)
        return y

    def merge_420(self, y, w):
        h2, ls = y.shape
        h = h2 // 2
        img = np.zeros((h, w), dtype=np.uint16)
        f = self.lib.orc_merge_420
        f.argtypes = [ct.c_void_p, ct.c_int, ct.c_int, ct.c_int, ct.c_void_p]
        f(_p(_c(y)), ls, w, h, _p(img))
        return img

    def key_frames(self, nframes, gop=50):
        k = np.zeros(nframes, dtype=np.uint8)
        f = self.lib.orc_key_frames
        f.argtypes = [ct.c_int, ct.c_int, ct.c_void_p]
        f(nframes, gop, _p(k))
        return k

    def precode_movie(self, movie, gop=50, delta=False):
        mov = _c(movie, np.uint16)
        t, h, w = mov.shape
        lo = np.zeros((t, h, w), dtype=np.uint8)
        hi = np.zeros((t, h, w), dtype=np.uint8)
        f = self.lib.orc_precode_movie
        f.argtypes = [ct.c_void_p, ct.c_int, ct.c_int, ct.c_int, ct.c_int, ct.c_int, ct.c_void_p, ct.c_void_p]
        f(_p(mov), t, w, h, gop, int(delta), _p(lo), _p(hi))
        return lo, hi

    def decode_movie(self, lo, hi, gop=50, delta=False):
        lo = _c(lo, np.uint8)
        hi = _c(hi, np.uint8)
        t, h, w = lo.shape
        mov = np.zeros((t, h, w), dtype=np.uint16)
        f = self.lib.orc_decode_movie
        f.argtypes = [ct.c_void_p, ct.c_void_p, ct.c_int, ct.c_int, ct.c_int, ct.c_int, ct.c_int, ct.c_void_p]
        f(_p(lo), _p(hi), t, w, h, gop, int(delta), _p(mov))
        return mov


class Ref(_Base):
    """The reference's own compiled C facade (signal_processing.h:29-94)."""

    kind = "reference"

    def __init__(self, omp: bool = False):
        self.lib = ref_lib(omp)
        self.omp = omp

    def _translate(self, code, img, res, w, h, dx, dy, back, strategy):
        f = self.lib.translate
        f.argtypes = [ct.c_int, ct.c_void_p, ct.c_void_p, ct.c_int, ct.c_int, ct.c_float, ct.c_float, ct.c_void_p,
                      ct.c_char_p]
        return f(code, _p(img), _p(res), w, h, dx, dy, _p(back), strategy)

    def _gaussian(self, img, res, w, h, sigma):
        f = self.lib.gaussian_filter
        f.argtypes = [ct.c_void_p, ct.c_void_p, ct.c_int, ct.c_int, ct.c_float]
        return f(_p(img), _p(res), w, h, sigma)

    def bad_pixels_create(self, first):
        img = np.array(first, dtype=np.uint16, order="C")
        f = self.lib.bad_pixels_create
        f.argtypes = [ct.c_void_p, ct.c_int, ct.c_int]
        return f(_p(img), img.shape[1], img.shape[0])

    def bad_pixels_correct(self, handle, image):
        img = np.array(image, dtype=np.uint16, order="C")
        out = np.zeros(img.shape, dtype=np.uint16)
        f = self.lib.bad_pixels_correct
        f.argtypes = [ct.c_int, ct.c_void_p, ct.c_void_p]
        if f(handle, _p(img), _p(out)) < 0:
            raise RuntimeError("'bad_pixels_correct': unknown error")
        return out

    def bad_pixels_destroy(self, handle):
        self.lib.bad_pixels_destroy.argtypes = [ct.c_int]
        self.lib.bad_pixels_destroy(handle)

    def find_median_pixel(self, image, percent=0.5, mask=None):
        img = _c(image, np.uint16)
        if mask is None:
            f = self.lib.find_median_pixel
            f.argtypes = [ct.c_void_p, ct.c_int, ct.c_float]
            return f(_p(img), img.size, float(percent))
        m = _c(mask, np.uint8)
        f = self.lib.find_median_pixel_mask
        f.argtypes = [ct.c_void_p, ct.c_void_p, ct.c_int, ct.c_float]
        return f(_p(img), _p(m), img.size, float(percent))


    # header-only templates reached through oracle/ref_shim.cpp ---------------------------
    def _shim(self):
        if not hasattr(self, "_shim_lib"):
            self._shim_lib = ct.CDLL(os.path.join(_REF_DIR, "libref_shim.so"))
        return self._shim_lib

    def bad_pixels_list(self, first, std_factor=5.0):
        img = _c(first, np.uint16)
        h, w = img.shape
        xy = np.zeros((img.size, 2), dtype=np.int32)
        f = self._shim().ref_bad_pixels_list
        f.argtypes = [ct.c_void_p, ct.c_int, ct.c_int, ct.c_double, ct.c_void_p, ct.c_int]
        k = f(_p(img), w, h, float(std_factor), _p(xy), img.size)
        return xy[:k].copy()

    def loader_remove_motion(self, image, shift_x, shift_y):
        img = np.array(image, dtype=np.uint16, order="C")
        h, w = img.shape
        f = self._shim().ref_remove_motion
        f.argtypes = [ct.c_void_p, ct.c_int, ct.c_int, ct.c_double, ct.c_double]
        f(_p(img), w, h, float(shift_x), float(shift_y))
        return img


def best():
    """The strongest oracle available: the compiled reference if present, else the port."""
    return Ref() if have_ref() else Port()
