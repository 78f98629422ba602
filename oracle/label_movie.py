"""oracle/label_movie.py -- TEST INFRASTRUCTURE ONLY (never imported by librir_b200).

The contract of ``rirb_label_movie`` restated on the CPU: events are ``scipy.ndimage.label`` on the 3-D mask of the
``[n, h, w]`` movie with ``generate_binary_structure(3, 1 | 2 | 3)`` for connectivity 6 | 18 | 26 (numbered in
``(t, y, x)`` raster order of each event's first voxel); statistics are numpy int64 reductions, in the style of
``oracle/label.py``'s ``stats_frame``.  Columns: volume, t_first, t_last, x_min, y_min, x_max, y_max, sum t, sum x, sum y,
sum value, max value, argmax (``t * h * w + y * w + x`` of the first voxel in raster order holding the maximum; not
``scipy.ndimage.maximum_position``, whose tie rule is not raster-first).  Rows past ``min(K, max_events)`` are zero, as
``librir_b200.signal_processing.label_movie`` returns them.
"""
from __future__ import annotations

import numpy as np
from scipy import ndimage

MOVIE_COLUMNS = 13


def structure3(connectivity: int):
    if connectivity not in (6, 18, 26):
        raise ValueError("connectivity must be 6, 18 or 26")
    return ndimage.generate_binary_structure(3, {6: 1, 18: 2, 26: 3}[connectivity])


def stats_movie(frames, lab, k):
    """int64 [k, 13] statistics of event labels ``lab`` (1..k, shape [n, h, w]) over the values of ``frames``."""
    out = np.zeros((k, MOVIE_COLUMNS), np.int64)
    if k == 0:
        return out
    n, h, w = lab.shape
    flat = lab.reshape(-1)
    idx = np.flatnonzero(flat)  # (t, y, x) raster order
    ell = flat[idx].astype(np.int64) - 1
    ts, rest = np.divmod(idx.astype(np.int64), h * w)
    ys, xs = np.divmod(rest, w)
    v = np.asarray(frames).reshape(-1)[idx].astype(np.int64)
    big, none = np.iinfo(np.int64).max, -1
    np.add.at(out[:, 0], ell, 1)
    for col, coord, fill, op in ((1, ts, big, np.minimum), (2, ts, none, np.maximum), (3, xs, big, np.minimum),
                                 (4, ys, big, np.minimum), (5, xs, none, np.maximum), (6, ys, none, np.maximum)):
        out[:, col] = fill
        op.at(out[:, col], ell, coord)
    np.add.at(out[:, 7], ell, ts)
    np.add.at(out[:, 8], ell, xs)
    np.add.at(out[:, 9], ell, ys)
    np.add.at(out[:, 10], ell, v)
    np.maximum.at(out[:, 11], ell, v)
    first = np.full(k, big, np.int64)
    at_max = v == out[ell, 11]
    np.minimum.at(first, ell[at_max], idx[at_max].astype(np.int64))
    out[:, 12] = first
    return out


def label_movie(frames, thresholds, connectivity=26, max_events=256):
    """(labels int32 [n,h,w], count int, stats int64 [max_events, 13]) of a uint16 movie ``[n, h, w]``."""
    frames = np.asarray(frames)
    n = frames.shape[0]
    thr = np.broadcast_to(np.asarray(thresholds).reshape(-1), (n,)).astype(np.int64)
    mask = frames > thr[:, None, None]
    lab, k = ndimage.label(mask, structure=structure3(connectivity))
    lab = lab.astype(np.int32)
    stats = np.zeros((max_events, MOVIE_COLUMNS), np.int64)
    if max_events and k:
        m = min(int(k), max_events)
        stats[:m] = stats_movie(frames, lab, int(k))[:m]
    return lab, int(k), stats
