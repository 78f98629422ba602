"""ctypes loader for libsignal_processing_b200.so (the C ABI of include/librir_b200.h).

Mirrors librir/low_level/misc.py:98-136 (loadDlls: glob the package's libs/ directory and
``ctypes.cdll.LoadLibrary`` what matches).  The library is built in-tree by
``librir_b200/csrc/Makefile`` (see ``__graft_entry__.build``).  There is no fallback of any
kind: if the library is missing, import fails; if no CUDA device is usable, every compute
entry returns -1 and the wrappers raise ``RuntimeError`` with the library's message.
"""
from __future__ import annotations

import ctypes as ct
import glob
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_DIR = os.path.join(_HERE, "libs")


def lib_path() -> str:
    found = sorted(glob.glob(os.path.join(LIB_DIR, "*signal_processing*.so")))
    if not found:
        raise ImportError(
            "librir_b200: libs/libsignal_processing_b200.so is not built "
            "(run `python -c 'import __graft_entry__ as g; g.build()'` or `make -C librir_b200/csrc`)"
        )
    return found[0]


_vp, _i, _ll, _f, _sz = ct.c_void_p, ct.c_int, ct.c_longlong, ct.c_float, ct.c_size_t

# name -> (restype, argtypes); the single source of truth the symbol test checks against
# include/librir_b200.h
SIGNATURES = {
    # Part 1: the reference's interface
    "translate": (_i, [_i, _vp, _vp, _i, _i, _f, _f, _vp, ct.c_char_p]),
    "gaussian_filter": (_i, [_vp, _vp, _i, _i, _f]),
    "find_median_pixel": (_i, [_vp, _i, _f]),
    "find_median_pixel_mask": (_i, [_vp, _vp, _i, _f]),
    "bad_pixels_create": (_i, [_vp, _i, _i]),
    "bad_pixels_correct": (_i, [_i, _vp, _vp]),
    "bad_pixels_destroy": (None, [_i]),
    "extract_times": (_i, [_vp, _i, _vp, _i, _vp, _vp]),
    "resample_time_serie": (_i, [_vp, _vp, _i, _vp, _i, _i, ct.c_double, _vp, _vp]),
    "label_image": (_i, [_i, _vp, _vp, _i, _i, _vp, _vp, _vp]),
    "keep_largest_area": (_i, [_i, _vp, _vp, _i, _i, _vp, _i]),
    "hash_bytes": (_sz, [_vp, _sz]),
    # Part 2: additive
    "rirb_device_count": (_i, []),
    "rirb_set_device": (_i, [_i]),
    "rirb_set_stream": (_i, [_vp]),
    "rirb_synchronize": (_i, []),
    "rirb_last_error": (ct.c_char_p, []),
    "rirb_kernel_launch_count": (_ll, []),
    "rirb_version": (ct.c_char_p, []),
    "rirb_set_parameter": (_i, [ct.c_char_p, ct.c_char_p]),
    "rirb_translate_batch": (_i, [_i, _vp, _vp, _i, _i, _ll, _vp, _vp, _ll, _vp, ct.c_char_p]),
    "rirb_gaussian_filter_batch": (_i, [_vp, _vp, _i, _i, _ll, _f]),
    "rirb_gaussian_filter_u16_batch": (_i, [_vp, _vp, _i, _i, _ll, _f]),
    "rirb_bad_pixels_correct_batch": (_i, [_i, _vp, _vp, _ll]),
    "rirb_bad_pixels_correct_gaussian_batch": (_i, [_i, _vp, _vp, _vp, _ll, _f]),
    "rirb_bad_pixels_count": (_i, [_i]),
    "rirb_bad_pixels_get": (_i, [_i, _vp, _i, _vp]),
    "rirb_loader_remove_bad_pixels": (_i, [_i, _vp, _ll, _sz]),
    "rirb_loader_remove_motion": (_i, [_vp, _vp, _i, _i, _ll, _sz, _vp, _vp]),
    "rirb_loader_read_movie": (_i, [_i, _vp, _vp, _ll, _i, _i, _i, _i, _vp, _vp, _i, _vp]),
    "rirb_loader_finish_frames": (_i, [_i, _vp, _ll, _i, _i, _i, _i, _vp, _vp, _i]),
    "rirb_split_yuv444": (_i, [_vp, _vp, _i, _i, _vp, _vp, _vp, _i, _i, _i]),
    "rirb_merge_yuv444": (_i, [_vp, _vp, _vp, _i, _i, _i, _i, _i, _vp, _vp]),
    "rirb_split_yuv420": (_i, [_vp, _vp, _i, _i, _vp, _i, _vp, _i]),
    "rirb_merge_yuv420": (_i, [_vp, _i, _vp, _i, _i, _i, _vp, _vp]),
    "rirb_precode_movie": (_i, [_vp, _ll, _i, _i, _i, _i, _ll, _vp, _vp]),
    "rirb_precode_movie_stats": (_i, [_vp, _ll, _i, _i, _i, _i, _ll, _vp, _vp, _vp, _vp, _i]),
    "rirb_decode_movie": (_i, [_vp, _vp, _ll, _i, _i, _i, _i, _ll, _vp]),
    "rirb_key_frames": (_i, [_ll, _i, _vp]),
    "rirb_lossy_open": (_i, [_i, _i, _i, _i, _i, ct.c_double, _i, _i, _i]),
    "rirb_lossy_add_images": (_i, [_i, _vp, _ll, _vp, _vp]),
    "rirb_lossy_close": (None, [_i]),
    "rirb_lossy_get_min": (_i, [_i, _vp]),
    "rirb_release_thread_resources": (None, []),
    "rirb_lossy_set_parameter": (_i, [_i, ct.c_char_p, ct.c_char_p]),
    "rirb_process_movie_host": (_i, [_i, _vp, _ll, _i, _i, _f, _vp, _vp, ct.c_char_p, ct.c_uint, _i, _i, _ll, _vp, _vp, _vp]),
    "rirb_movie_stats": (_i, [_vp, _sz, _vp, _vp, _i]),
    "rirb_hist_quantile": (_i, [_vp, _ll, _f]),
    "rirb_get_background": (_i, [_vp, _i]),
    # Part 3: file formats (host code)
    "rirb_attrs_open_file": (_i, [ct.c_char_p]),
    "rirb_attrs_open_from_memory": (_i, [_vp, _ll]),
    "rirb_attrs_close": (None, [_i]),
    "rirb_attrs_discard": (None, [_i]),
    "rirb_attrs_abandon": (None, [_i]),
    "rirb_attrs_flush": (_i, [_i]),
    "rirb_attrs_image_count": (_i, [_i]),
    "rirb_attrs_global_attribute_count": (_i, [_i]),
    "rirb_attrs_global_attribute_name": (_i, [_i, _i, _vp, _vp]),
    "rirb_attrs_global_attribute_value": (_i, [_i, _i, _vp, _vp]),
    "rirb_attrs_frame_attribute_count": (_i, [_i, _i]),
    "rirb_attrs_frame_attribute_name": (_i, [_i, _i, _i, _vp, _vp]),
    "rirb_attrs_frame_attribute_value": (_i, [_i, _i, _i, _vp, _vp]),
    "rirb_attrs_frame_timestamp": (_i, [_i, _i, _vp]),
    "rirb_attrs_timestamps": (_i, [_i, _vp]),
    "rirb_attrs_set_times": (_i, [_i, _vp, _i]),
    "rirb_attrs_set_time": (_i, [_i, _i, _ll]),
    "rirb_attrs_set_frame_attributes": (_i, [_i, _i, _vp, _vp, _vp, _vp, _i]),
    "rirb_attrs_set_global_attributes": (_i, [_i, _vp, _vp, _vp, _vp, _i]),
    "rirb_z_open_file_write": (_i, [ct.c_char_p, _i, _i, _i, _i, _i]),
    "rirb_z_open_file_write_gop": (_i, [ct.c_char_p, _i, _i, _i, _i, _i, _i]),
    "rirb_z_write_image": (_i, [_i, _vp, _ll]),
    "rirb_z_write_images": (_i, [_i, _vp, _ll, _vp, _i]),
    "rirb_z_close_file": (_ll, [_i]),
    "rirb_z_open_file_read": (_i, [ct.c_char_p]),
    "rirb_z_image_count": (_i, [_i]),
    "rirb_z_method": (_i, [_i]),
    "rirb_z_image_size": (_i, [_i, _vp, _vp]),
    "rirb_z_get_timestamps": (_i, [_i, _vp]),
    "rirb_z_read_image": (_i, [_i, _i, _vp, _vp]),
    "rirb_z_read_images": (_i, [_i, _i, _i, _vp, _vp, _i]),
    "rirb_z_set_coder": (_i, [_i, _i]),
    "rirb_z_set_lz": (_i, [_i, _i]),
    "rirb_zstd_encode_batch": (_i, [_vp, _ll, _ll, _ll, _vp, _ll, _vp]),
    "rirb_zstd_encode_batch_lz": (_i, [_vp, _ll, _ll, _ll, _vp, _ll, _vp]),
    "rirb_zstd_decode_batch": (_i, [_vp, _vp, _vp, _ll, _vp, _ll, _ll, _vp]),
    # Part 4: registration front end
    "rirb_ecc_open": (_i, [_i, _i]),
    "rirb_ecc_close": (None, [_i]),
    "rirb_ecc_set_mask": (_i, [_i, _i, _vp]),
    "rirb_ecc_set_image": (_i, [_i, _i, _vp, _i]),
    "rirb_ecc_reset_reference": (_i, [_i, _f, _f]),
    "rirb_ecc_quantile": (_i, [_i, _i, _f, _i]),
    "rirb_ecc_compute": (_i, [_i, _f, _i, _i, ct.c_double, _vp, _vp, _vp]),
    "rirb_ecc_track_config": (_i, [_i, _f, ct.c_double, _i]),
    "rirb_ecc_track_set_median": (_i, [_i, ct.c_double]),
    "rirb_ecc_track": (_i, [_i, _i, _vp, _ll, _i, _i, _i, _i, _i, _i, _vp, _vp, _vp, _vp, _vp]),
    "rirb_ecc_track_state": (_i, [_i, _vp, _vp, _vp, _vp]),
}

_lib = None


def load() -> ct.CDLL:
    """Load the library once and attach restype/argtypes to every declared entry."""
    global _lib
    if _lib is None:
        lib = ct.cdll.LoadLibrary(lib_path())
        for name, (res, args) in SIGNATURES.items():
            fn = getattr(lib, name)  # AttributeError if the .so lacks a declared symbol
            fn.restype = res
            fn.argtypes = args
        _lib = lib
    return _lib


def set_parameter(key: str, value) -> None:
    """``rirb_set_parameter``: process-wide kernel-variant switches ("translate_tma", "gauss_tma", "loader_fused", "ecc_fused", "lossy_run")."""
    check(load().rirb_set_parameter(key.encode(), str(int(value)).encode()), "set_parameter")


def last_error() -> str:
    return load().rirb_last_error().decode(errors="replace")


def check(status: int, what: str) -> int:
    """Python side of the reference's convention: negative status -> RuntimeError."""
    if status < 0:
        raise RuntimeError(f"An error occured while calling '{what}': {last_error()}")
    return status


def device_available() -> bool:
    return load().rirb_device_count() > 0


def use_torch_stream() -> None:
    """Point the calling thread's library stream at torch's current CUDA stream."""
    import torch

    load().rirb_set_stream(ct.c_void_p(torch.cuda.current_stream().cuda_stream))


def launch_count() -> int:
    return int(load().rirb_kernel_launch_count())
