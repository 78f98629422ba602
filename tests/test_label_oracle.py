"""The connected-component oracle (oracle/label.py) on the CPU: equal to an independent pure-Python flood fill on random
small masks at both connectivities, equal to OpenCV's connectedComponentsWithStats up to the numbering, and the C entry
fails loudly without a device."""
from collections import deque

import numpy as np
import pytest

from librir_b200 import _lib, signal_processing as sp
from oracle import label as OL

NEIGHBOURS = {4: [(-1, 0), (1, 0), (0, -1), (0, 1)], 8: [(dy, dx) for dy in (-1, 0, 1) for dx in (-1, 0, 1) if dy or dx]}


def flood_fill(frame, threshold, connectivity):
    """Labels numbered in raster order of each component's first pixel, and the statistics rows, by breadth-first search."""
    h, w = frame.shape
    mask = frame > threshold
    lab = np.zeros((h, w), np.int32)
    rows = []
    for y0 in range(h):
        for x0 in range(w):
            if not mask[y0, x0] or lab[y0, x0]:
                continue
            k = len(rows) + 1
            lab[y0, x0] = k
            todo, px = deque([(y0, x0)]), []
            while todo:
                y, x = todo.popleft()
                px.append((y, x))
                for dy, dx in NEIGHBOURS[connectivity]:
                    ny, nx = y + dy, x + dx
                    if 0 <= ny < h and 0 <= nx < w and mask[ny, nx] and not lab[ny, nx]:
                        lab[ny, nx] = k
                        todo.append((ny, nx))
            px.sort()
            vals = [int(frame[y, x]) for y, x in px]
            top = max(vals)
            arg = next(y * w + x for (y, x), v in zip(px, vals) if v == top)
            rows.append([len(px), min(x for _, x in px), min(y for y, _ in px), max(x for _, x in px), max(y for y, _ in px),
                         sum(x for _, x in px), sum(y for y, _ in px), sum(vals), top, arg])
    return lab, len(rows), np.array(rows, np.int64).reshape(-1, 10)


def random_cases(n):
    rng = np.random.default_rng(2024)
    for i in range(n):
        h, w = (int(v) for v in rng.integers(1, 14, 2))
        density = rng.choice([0.2, 0.41, 0.5, 0.59, 0.8])
        mask = rng.random((h, w)) < density
        vals = rng.integers(0, 6, (h, w)).astype(np.uint16)  # few levels: ties for the maximum are common
        yield i, np.where(mask, 100 + vals, vals).astype(np.uint16)


@pytest.mark.parametrize("connectivity", [4, 8])
def test_oracle_equals_flood_fill_on_random_masks(connectivity):
    for i, frame in random_cases(200):
        want_lab, want_k, want_stats = flood_fill(frame, 50, connectivity)
        lab, k = OL.label_frame(frame, 50, connectivity)
        assert k == want_k, i
        np.testing.assert_array_equal(lab, want_lab, err_msg=str(i))
        np.testing.assert_array_equal(OL.stats_frame(frame, lab, k), want_stats, err_msg=str(i))
        # the batch form: capacity below K keeps the first rows, the rest stay zero
        cap = max(1, k // 2)
        _, counts, stats = OL.label_batch(frame[None], 50, connectivity, cap)
        assert counts[0] == k
        np.testing.assert_array_equal(stats[0, : min(k, cap)], want_stats[:cap])


@pytest.mark.parametrize("connectivity", [4, 8])
def test_oracle_partitions_match_opencv(connectivity):
    cv2 = pytest.importorskip("cv2")
    rng = np.random.default_rng(7)
    for i in range(60):
        h, w = (int(v) for v in rng.integers(1, 60, 2))
        frame = (rng.random((h, w)) < rng.choice([0.3, 0.5, 0.59, 0.7])).astype(np.uint16) * 1000
        lab, k = OL.label_frame(frame, 0, connectivity)
        stats = OL.stats_frame(frame, lab, k)
        n, cvlab, cvstats, cvcent = cv2.connectedComponentsWithStats((frame > 0).astype(np.uint8), connectivity=connectivity,
                                                                     ltype=cv2.CV_32S)
        assert n - 1 == k, i
        # the permutation of labels: cv2 label -> oracle label, one to one
        fg = lab > 0
        pairs = np.unique(np.stack([cvlab[fg], lab[fg]], 1), axis=0)
        assert len(pairs) == k and len(np.unique(pairs[:, 0])) == k and len(np.unique(pairs[:, 1])) == k, i
        assert not np.any(cvlab[~fg]), i
        perm = np.zeros(k + 1, np.int64)
        perm[pairs[:, 0]] = pairs[:, 1]
        ours = stats[perm[1:] - 1]
        np.testing.assert_array_equal(ours[:, sp.AREA], cvstats[1:, cv2.CC_STAT_AREA])
        np.testing.assert_array_equal(ours[:, sp.X_MIN], cvstats[1:, cv2.CC_STAT_LEFT])
        np.testing.assert_array_equal(ours[:, sp.Y_MIN], cvstats[1:, cv2.CC_STAT_TOP])
        np.testing.assert_array_equal(ours[:, sp.X_MAX] - ours[:, sp.X_MIN] + 1, cvstats[1:, cv2.CC_STAT_WIDTH])
        np.testing.assert_array_equal(ours[:, sp.Y_MAX] - ours[:, sp.Y_MIN] + 1, cvstats[1:, cv2.CC_STAT_HEIGHT])
        np.testing.assert_allclose(ours[:, sp.SUM_X] / ours[:, sp.AREA], cvcent[1:, 0], rtol=0, atol=1e-9)
        np.testing.assert_allclose(ours[:, sp.SUM_Y] / ours[:, sp.AREA], cvcent[1:, 1], rtol=0, atol=1e-9)


def test_oracle_centroid_is_scipy_center_of_mass():
    from scipy import ndimage

    rng = np.random.default_rng(3)
    frame = (rng.random((40, 50)) < 0.55).astype(np.uint16) * 7
    lab, k = OL.label_frame(frame, 0, 8)
    stats = OL.stats_frame(frame, lab, k)
    com = np.array(ndimage.center_of_mass(np.ones_like(lab), lab, np.arange(1, k + 1)))
    assert np.array_equal(stats[:, sp.SUM_Y] / stats[:, sp.AREA], com[:, 0])
    assert np.array_equal(stats[:, sp.SUM_X] / stats[:, sp.AREA], com[:, 1])


def test_facade_checks_its_arguments():
    frames = np.zeros((2, 4, 5), np.uint16)
    for call in (
        lambda: sp.label_batch(frames[0], 1),  # not a stack
        lambda: sp.label_batch(frames, 1, connectivity=6),
        lambda: sp.label_batch(frames, [1, 2, 3]),  # neither one nor one per frame
        lambda: sp.label_batch(frames, 70000),
        lambda: sp.label_batch(frames, 1.5),
        lambda: sp.label_batch(frames, 1, max_components=-1),
        lambda: sp.label_batch(frames.astype(np.int32), 1),
        lambda: sp.label_batch(frames, 1, labels=np.zeros((2, 4, 5), np.int64)),
    ):
        with pytest.raises(RuntimeError):
            call()
    lib = _lib.load()
    lab = np.zeros(frames.shape, np.int32)
    cnt = np.zeros(2, np.int32)
    thr = np.zeros(1, np.uint16)
    assert lib.rirb_label_batch(frames.ctypes.data, 5, 4, 2, thr.ctypes.data, 1, 6, lab.ctypes.data, cnt.ctypes.data, None, 0) == -1
    assert "connectivity" in _lib.last_error()
    assert lib.rirb_label_batch(frames.ctypes.data, 5, 4, 2, thr.ctypes.data, 3, 8, lab.ctypes.data, cnt.ctypes.data, None, 0) == -1
    assert lib.rirb_label_batch(frames.ctypes.data, 65536, 32768, 2, thr.ctypes.data, 1, 8, lab.ctypes.data, cnt.ctypes.data, None, 0) == -1
    assert "bad arguments" in _lib.last_error()
    assert lib.rirb_label_batch(frames.ctypes.data, 5, 4, 0, thr.ctypes.data, 0, 8, lab.ctypes.data, cnt.ctypes.data, None, 0) == 0


@pytest.mark.skipif(_lib.device_available(), reason="checks behaviour WITHOUT a CUDA device")
def test_label_batch_without_a_device_fails_loudly():
    frames = np.ones((2, 4, 5), np.uint16)
    with pytest.raises(RuntimeError) as e:
        sp.label_batch(frames, 0)
    assert "no CPU fallback" in str(e.value)
    lib = _lib.load()
    lab = np.zeros(frames.shape, np.int32)
    cnt = np.zeros(2, np.int32)
    thr = np.zeros(1, np.uint16)
    assert lib.rirb_label_batch(frames.ctypes.data, 5, 4, 2, thr.ctypes.data, 1, 8, lab.ctypes.data, cnt.ctypes.data, None, 0) == -1
    assert "no CPU fallback" in _lib.last_error()
