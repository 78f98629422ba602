"""oracle/label.py -- TEST INFRASTRUCTURE ONLY (never imported by librir_b200).

The contract of ``rirb_label_batch`` restated on the CPU: labels and counts from ``scipy.ndimage.label`` with the 4- or
8-neighbour structure (raster order of each component's first pixel), statistics as numpy int64 reductions.  Columns:
area, x_min, y_min, x_max, y_max, sum x, sum y, sum value, max value, argmax (y * w + x of the first pixel in raster order
holding the maximum; not ``scipy.ndimage.maximum_position``, whose tie rule is not raster-first).  Rows past
``min(K, max_components)`` are zero, as ``librir_b200.signal_processing.label_batch`` returns them.
"""
from __future__ import annotations

import numpy as np
from scipy import ndimage

COLUMNS = 10


def structure(connectivity: int):
    if connectivity not in (4, 8):
        raise ValueError("connectivity must be 4 or 8")
    return ndimage.generate_binary_structure(2, 1 if connectivity == 4 else 2)


def label_frame(frame, threshold, connectivity):
    """int32 labels and the component count of one frame."""
    lab, k = ndimage.label(np.asarray(frame) > threshold, structure=structure(connectivity))
    return lab.astype(np.int32), int(k)


def stats_frame(frame, lab, k):
    """int64 [k, 10] statistics of labels ``lab`` (1..k) over the values of ``frame``."""
    out = np.zeros((k, COLUMNS), np.int64)
    if k == 0:
        return out
    h, w = lab.shape
    flat = lab.reshape(-1)
    idx = np.flatnonzero(flat)  # raster order
    ell = flat[idx].astype(np.int64) - 1
    ys, xs = np.divmod(idx.astype(np.int64), w)
    v = np.asarray(frame).reshape(-1)[idx].astype(np.int64)
    np.add.at(out[:, 0], ell, 1)
    out[:, 1] = np.iinfo(np.int64).max
    out[:, 2] = np.iinfo(np.int64).max
    out[:, 3] = -1
    out[:, 4] = -1
    np.minimum.at(out[:, 1], ell, xs)
    np.minimum.at(out[:, 2], ell, ys)
    np.maximum.at(out[:, 3], ell, xs)
    np.maximum.at(out[:, 4], ell, ys)
    np.add.at(out[:, 5], ell, xs)
    np.add.at(out[:, 6], ell, ys)
    np.add.at(out[:, 7], ell, v)
    np.maximum.at(out[:, 8], ell, v)
    first = np.full(k, np.iinfo(np.int64).max, np.int64)
    at_max = v == out[ell, 8]
    np.minimum.at(first, ell[at_max], idx[at_max].astype(np.int64))
    out[:, 9] = first
    return out


def label_batch(frames, thresholds, connectivity=8, max_components=256):
    """(labels int32 [n,h,w], counts int32 [n], stats int64 [n, max_components, 10]) of a uint16 stack."""
    frames = np.asarray(frames)
    n = frames.shape[0]
    thr = np.broadcast_to(np.asarray(thresholds).reshape(-1), (n,))
    labels = np.zeros(frames.shape, np.int32)
    counts = np.zeros(n, np.int32)
    stats = np.zeros((n, max_components, COLUMNS), np.int64)
    for t in range(n):
        labels[t], counts[t] = label_frame(frames[t], int(thr[t]), connectivity)
        if max_components and counts[t]:
            s = stats_frame(frames[t], labels[t], int(counts[t]))
            m = min(int(counts[t]), max_components)
            stats[t, :m] = s[:m]
    return labels, counts, stats
