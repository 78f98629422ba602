"""Host-side mirror of ``librir.tools`` for the file formats either side of the path (SURVEY.md 8f-3).

* ``attrs_*`` functions and the ``FileAttributes`` class: same names, arguments, return types and
  error behaviour as librir/tools/rir_tools.py:76-420 and librir/tools/FileAttributes.py:32-161,
  over ``rirb_attrs_*`` (rir::FileAttributes, FileAttributes.cpp).
* ``ZFileWriter`` / ``ZFileReader``: the zstd movie file of ZFile.cpp (the reference only reaches it
  from C++ -- ``IRFileLoader`` reads it, IRFileLoader.cpp:331-370); runs of frames are compressed by a
  pool of host threads, and frame buffers may be torch CUDA tensors.
"""
from __future__ import annotations

import atexit
import ctypes as ct
import os
from typing import Dict

import numpy as np

from . import _lib
from .signal_processing import _operand, _ptr


def _bytes_of(x, enc) -> bytes:
    if isinstance(x, bytes):
        return x
    if isinstance(x, str):
        return x.encode(enc)
    return str(x).encode(enc)


def _to_string(b: bytes) -> str:
    """librir/low_level/misc.py:56-61 toString: ascii, else utf8, NULs dropped."""
    try:
        return b.decode("ascii").replace("\x00", "")
    except UnicodeDecodeError:
        return b.decode("utf8").replace("\x00", "")


def attrs_open_file(filename):
    """Open attribute file and returns a handle to it"""
    return _lib.load().rirb_attrs_open_file(str(filename).encode("ascii"))


def attrs_open_buffer(buf: bytes):
    """Open attributes from an in-memory file. Attributes are read-only."""
    res = _lib.load().rirb_attrs_open_from_memory(ct.cast(ct.c_char_p(buf), ct.c_void_p), len(buf))
    if res == 0:
        raise RuntimeError("cannot read attributes from memory")
    return res


def attrs_close(handle):
    _lib.load().rirb_attrs_close(int(handle))


def attrs_discard(handle):
    _lib.load().rirb_attrs_discard(int(handle))


def attrs_flush(handle):
    if _lib.load().rirb_attrs_flush(int(handle)) < 0:
        raise RuntimeError("An error occured while calling 'attrs_flush'")


def attrs_image_count(handle):
    tmp = _lib.load().rirb_attrs_image_count(int(handle))
    if tmp < 0:
        raise RuntimeError("An error occured while calling 'attrs_image_count'")
    return tmp


def attrs_global_attribute_count(handle):
    tmp = _lib.load().rirb_attrs_global_attribute_count(int(handle))
    if tmp < 0:
        raise RuntimeError("An error occured while calling 'attrs_global_attribute_count'")
    return tmp


def attrs_frame_attribute_count(handle, pos):
    tmp = _lib.load().rirb_attrs_frame_attribute_count(int(handle), int(pos))
    if tmp < 0:
        raise RuntimeError("An error occured while calling 'attrs_frame_attribute_count'")
    return tmp


def _get_blob(fn, what, *ids) -> bytes:
    n = ct.c_int(200)
    buf = ct.create_string_buffer(200)
    tmp = fn(*ids, buf, ct.byref(n))
    if tmp == -2:  # too small: the call wrote the needed size
        buf = ct.create_string_buffer(max(1, n.value))
        tmp = fn(*ids, buf, ct.byref(n))
    if tmp < 0:
        raise RuntimeError(f"An error occured while calling '{what}'")
    return buf.raw[: n.value]


def attrs_global_attribute_name(handle, index) -> str:
    return _to_string(_get_blob(_lib.load().rirb_attrs_global_attribute_name, "attrs_global_attribute_name", int(handle), int(index)))


def attrs_global_attribute_value(handle, index) -> bytes:
    return _get_blob(_lib.load().rirb_attrs_global_attribute_value, "attrs_global_attribute_value", int(handle), int(index))


def attrs_frame_attribute_name(handle, frame, index) -> str:
    return _to_string(_get_blob(_lib.load().rirb_attrs_frame_attribute_name, "attrs_frame_attribute_name", int(handle), int(frame), int(index)))


def attrs_frame_attribute_value(handle, frame, index) -> bytes:
    return _get_blob(_lib.load().rirb_attrs_frame_attribute_value, "attrs_frame_attribute_value", int(handle), int(frame), int(index))


def attrs_frame_timestamp(handle, frame):
    t = ct.c_longlong(0)
    if _lib.load().rirb_attrs_frame_timestamp(int(handle), int(frame), ct.byref(t)) < 0:
        raise RuntimeError("An error occured while calling 'attrs_frame_timestamp'")
    return np.int64(t.value)


def attrs_timestamps(handle):
    times = np.zeros((attrs_image_count(handle)), dtype=np.int64)
    if _lib.load().rirb_attrs_timestamps(int(handle), times.ctypes.data_as(ct.c_void_p)) < 0:
        raise RuntimeError("An error occured while calling 'attrs_timestamps'")
    return times


def attrs_set_times(handle, times):
    if not isinstance(times, np.ndarray) or (times.dtype != np.int64):
        times = np.array(list(times), dtype=np.int64)
    times = np.ascontiguousarray(times)
    if _lib.load().rirb_attrs_set_times(int(handle), times.ctypes.data_as(ct.c_void_p), int(times.shape[0])) < 0:
        raise RuntimeError("An error occured while calling 'attrs_set_times'")


def attrs_set_time(handle, frame, time):
    if _lib.load().rirb_attrs_set_time(int(handle), int(frame), int(time)) < 0:
        raise RuntimeError("An error occured while calling 'attrs_set_time'")


def _pack(attributes, enc):
    keys, values, klens, vlens = bytes(), bytes(), [], []
    for k, v in attributes.items():
        ks, vs = _bytes_of(k, enc), _bytes_of(v, enc)
        klens.append(len(ks))
        vlens.append(len(vs))
        keys += ks
        values += vs
    kl = np.array(klens, dtype=np.int32)
    vl = np.array(vlens, dtype=np.int32)
    return keys, kl, values, vl


def attrs_set_frame_attributes(handle, frame, attributes):
    if type(attributes) is not dict:
        raise RuntimeError("attrs_set_frame_attributes: wrong attributes type (should be dict)")
    keys, kl, values, vl = _pack(attributes, "ascii")  # rir_tools.py:340-351 encodes frame attributes as ascii
    tmp = _lib.load().rirb_attrs_set_frame_attributes(int(handle), int(frame), ct.cast(ct.c_char_p(keys), ct.c_void_p),
                                                      kl.ctypes.data_as(ct.c_void_p), ct.cast(ct.c_char_p(values), ct.c_void_p),
                                                      vl.ctypes.data_as(ct.c_void_p), len(attributes))
    if tmp < 0:
        raise RuntimeError("An error occured while calling 'attrs_set_frame_attributes'")


def attrs_set_global_attributes(handle, attributes):
    if type(attributes) is not dict:
        raise RuntimeError("attrs_set_global_attributes: wrong attributes type (should be dict)")
    keys, kl, values, vl = _pack(attributes, "utf8")  # rir_tools.py:392-403 encodes global attributes as utf8
    tmp = _lib.load().rirb_attrs_set_global_attributes(int(handle), ct.cast(ct.c_char_p(keys), ct.c_void_p),
                                                       kl.ctypes.data_as(ct.c_void_p), ct.cast(ct.c_char_p(values), ct.c_void_p),
                                                       vl.ctypes.data_as(ct.c_void_p), len(attributes))
    if tmp < 0:
        raise RuntimeError("An error occured while calling 'attrs_set_global_attributes'")


class FileAttributes(object):
    """
    Small class handling file attributes based on librir attributes format
    (librir/tools/FileAttributes.py:32-161: same interface).

    Newly defined attributes are only written to the file when the FileAttributes object is closed
    or the flush() function is called.
    """

    _attributes: Dict[str, bytes]

    @classmethod
    def from_buffer(cls, buffer: bytes):
        return cls(attrs_open_buffer(buffer))

    @classmethod
    def from_filename(cls, filename: os.PathLike):
        return cls(attrs_open_file(filename))

    def __init__(self, handle):
        self.handle = handle
        self._timestamps = attrs_timestamps(self.handle)
        self._attributes = {}
        for i in range(attrs_global_attribute_count(self.handle)):
            self._attributes[attrs_global_attribute_name(self.handle, i)] = attrs_global_attribute_value(self.handle, i)
        atexit.register(self.close)

    def close(self):
        """Write attributes and close the file. The FileAttributes object cannot be used anymore."""
        if self.handle:
            self.attributes = self._attributes
            self.timestamps = self._timestamps
            attrs_close(self.handle)
            self.handle = 0

    def flush(self):
        if self.handle:
            attrs_flush(self.handle)

    def discard(self):
        """Close the file (the reference's attrs_discard writes what was already handed to the handle, tools.cpp:124-131)."""
        if not self.handle:
            return
        attrs_discard(self.handle)
        self.handle = 0

    def __enter__(self):
        return self

    def __exit__(self, exc_type, exc_val, exc_tb):
        return self.close()

    def is_open(self):
        return self.handle > 0

    def frame_count(self):
        return self._timestamps.shape[0]

    @property
    def timestamps(self):
        """Get/set the timestamps within the file"""
        return self._timestamps

    @timestamps.setter
    def timestamps(self, times):
        attrs_set_times(self.handle, times)
        if not isinstance(times, np.ndarray) or times.dtype != np.int64:
            times = np.array(list(times), dtype=np.int64)
        self._timestamps = times

    @property
    def attributes(self) -> Dict[str, bytes]:
        """Get/set the global file attributes"""
        return self._attributes

    @attributes.setter
    def attributes(self, attributes):
        attrs_set_global_attributes(self.handle, attributes)
        self._attributes = attributes

    def frame_attributes(self, frame_index):
        """Returns the frame attributes for given frame index"""
        return {
            attrs_frame_attribute_name(self.handle, frame_index, i): attrs_frame_attribute_value(self.handle, frame_index, i)
            for i in range(attrs_frame_attribute_count(self.handle, frame_index))
        }

    def set_frame_attributes(self, frame_index, attributes):
        """Set the frame attributes for given frame index"""
        attrs_set_frame_attributes(self.handle, frame_index, attributes)


# ----------------------------------------------------------------------------------------
# zstd movie file (ZFile.cpp)
# ----------------------------------------------------------------------------------------
def _is_torch(x) -> bool:
    return type(x).__module__.startswith("torch")


class ZFileWriter:
    """``z_open_file_write`` / ``z_write_image`` / ``z_close_file`` (ZFile.cpp:255-296, 483-542, 410-452)."""

    def __init__(self, filename, width, height, rate=50, method=1, clevel=2, threads=0, gop=50, coder="host"):
        """``method`` 1 = zstd of the raw image (the reference's files), 2 = byte planes + zstd, 3 = temporal delta with
        key frames every ``gop`` images + byte planes + zstd (video_io.h:298-305); 2 and 3 pre-code on the GPU.
        ``coder`` "host" = zstd on host threads at ``clevel``; "gpu" = the device coder (Huffman-literal zstd frames that any
        zstd decoder reads; ``clevel`` does not apply; needs a CUDA device); "gpu-lz" = the device coder with LZ matches in
        the blocks where they make the frame smaller (the high-byte planes of methods 2/3 above all)."""
        if coder not in ("host", "gpu", "gpu-lz"):
            raise ValueError(f"coder must be 'host', 'gpu' or 'gpu-lz', not {coder!r}")
        lib = _lib.load()
        self.handle = lib.rirb_z_open_file_write_gop(str(filename).encode(), int(width), int(height), int(rate), int(method),
                                                     int(clevel), int(gop))
        if self.handle <= 0:
            raise RuntimeError(f"cannot open '{filename}' for writing: {_lib.last_error()}")
        if coder != "host" and (lib.rirb_z_set_coder(self.handle, 1) != 0 or lib.rirb_z_set_lz(self.handle, int(coder == "gpu-lz")) != 0):
            err = _lib.last_error()
            lib.rirb_z_close_file(self.handle)
            self.handle = 0
            raise RuntimeError(f"cannot use the device coder for '{filename}': {err}")
        self.width, self.height, self.threads = int(width), int(height), int(threads)

    def add_image(self, img, timestamp):
        self.add_images(np.asarray(img)[None] if not _is_torch(img) else img[None], [timestamp])

    def add_images(self, frames, timestamps):
        """frames ``[n, h, w]`` uint16 (numpy, or a torch CUDA tensor: one download), timestamps ``[n]`` in ns."""
        ts = np.ascontiguousarray(timestamps, dtype=np.int64)
        if _is_torch(frames):
            _operand(frames, "ZFileWriter.add_images", "frames", dtype=(np.uint16, np.int16))
            ptr, shape = ct.c_void_p(frames.data_ptr()), tuple(frames.shape)
            if frames.is_cuda:
                _lib.use_torch_stream()
        else:
            frames = np.ascontiguousarray(frames, dtype=np.uint16)
            ptr, shape = frames.ctypes.data_as(ct.c_void_p), frames.shape
        if len(shape) != 3 or shape[1] != self.height or shape[2] != self.width or shape[0] != ts.shape[0]:
            raise RuntimeError("ZFileWriter.add_images: wrong frame stack or timestamp count")
        _lib.check(_lib.load().rirb_z_write_images(self.handle, ptr, shape[0], ts.ctypes.data_as(ct.c_void_p), self.threads), "z_write_images")

    def close(self) -> int:
        """Patch the sample count, append the attribute trailer; returns the bytes of headers + records."""
        if not self.handle:
            return 0
        n = _lib.load().rirb_z_close_file(self.handle)
        self.handle = 0
        return int(n)

    def __enter__(self):
        return self

    def __exit__(self, *exc):
        self.close()


class ZFileReader:
    """``z_open_file_read`` / ``z_read_image`` / ``z_get_timestamps`` (ZFile.cpp:124-253, 544-641)."""

    def __init__(self, filename, threads=0):
        lib = _lib.load()
        self.handle = lib.rirb_z_open_file_read(str(filename).encode())
        if self.handle <= 0:
            raise RuntimeError(f"cannot open '{filename}': {_lib.last_error()}")
        w, h = ct.c_int(0), ct.c_int(0)
        lib.rirb_z_image_size(self.handle, ct.byref(w), ct.byref(h))
        self.width, self.height, self.threads = w.value, h.value, int(threads)
        self.images = lib.rirb_z_image_count(self.handle)
        self.timestamps = np.zeros(self.images, dtype=np.int64)
        if self.images:
            lib.rirb_z_get_timestamps(self.handle, self.timestamps.ctypes.data_as(ct.c_void_p))

    def __len__(self):
        return self.images

    def read_image(self, pos):
        return self.read_images(pos, 1)[0]

    def read_images(self, pos=0, count=None, out=None):
        """Frames ``[pos, pos + count)`` -> uint16 ``[count, h, w]`` (``out``: numpy array or torch CUDA tensor of that
        shape, uint16 or int16 -- the same bits; strided views are refused)."""
        if count is None:
            count = self.images - pos
        if out is None:
            out = np.empty((count, self.height, self.width), dtype=np.uint16)
        _operand(out, "ZFileReader.read_images", "out", (count, self.height, self.width), (np.uint16, np.int16))
        if _is_torch(out) and out.is_cuda:
            _lib.use_torch_stream()
        ptr = _ptr(out)
        _lib.check(_lib.load().rirb_z_read_images(self.handle, int(pos), int(count), ptr, None, self.threads), "z_read_images")
        return out

    def close(self):
        if self.handle:
            _lib.load().rirb_z_close_file(self.handle)
            self.handle = 0

    def __enter__(self):
        return self

    def __exit__(self, *exc):
        self.close()


__all__ = [n for n in dir() if n.startswith("attrs_")] + ["FileAttributes", "ZFileWriter", "ZFileReader"]
