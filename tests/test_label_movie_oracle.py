"""The event oracle (oracle/label_movie.py) on the CPU: equal to an independent pure-Python 3-D flood fill on small
random volumes at 6-, 18- and 26-connectivity, equal to the per-frame oracle on single frames, right on planted volumes
whose event count depends on the connectivity, and the C entry refuses bad arguments without a device."""
from collections import deque

import numpy as np
import pytest

from librir_b200 import _lib, signal_processing as sp
from oracle import label as OL
from oracle import label_movie as OM


def stencil(connectivity):
    """(dt, dy, dx) offsets of generate_binary_structure(3, r), written out by hand: r = number of non-zero axes allowed."""
    r = {6: 1, 18: 2, 26: 3}[connectivity]
    return [(dt, dy, dx) for dt in (-1, 0, 1) for dy in (-1, 0, 1) for dx in (-1, 0, 1)
            if (dt, dy, dx) != (0, 0, 0) and abs(dt) + abs(dy) + abs(dx) <= r]


def flood_fill(frames, threshold, connectivity):
    """Labels numbered in (t, y, x) raster order of each event's first voxel, and the 13-column rows, by breadth-first
    search."""
    n, h, w = frames.shape
    mask = frames > threshold
    lab = np.zeros((n, h, w), np.int32)
    rows = []
    nbrs = stencil(connectivity)
    for t0 in range(n):
        for y0 in range(h):
            for x0 in range(w):
                if not mask[t0, y0, x0] or lab[t0, y0, x0]:
                    continue
                k = len(rows) + 1
                lab[t0, y0, x0] = k
                todo, vox = deque([(t0, y0, x0)]), []
                while todo:
                    t, y, x = todo.popleft()
                    vox.append((t, y, x))
                    for dt, dy, dx in nbrs:
                        nt, ny, nx = t + dt, y + dy, x + dx
                        if 0 <= nt < n and 0 <= ny < h and 0 <= nx < w and mask[nt, ny, nx] and not lab[nt, ny, nx]:
                            lab[nt, ny, nx] = k
                            todo.append((nt, ny, nx))
                vox.sort()
                vals = [int(frames[v]) for v in vox]
                top = max(vals)
                arg = next(t * h * w + y * w + x for (t, y, x), v in zip(vox, vals) if v == top)
                ts = [v[0] for v in vox]
                ys = [v[1] for v in vox]
                xs = [v[2] for v in vox]
                rows.append([len(vox), min(ts), max(ts), min(xs), min(ys), max(xs), max(ys), sum(ts), sum(xs), sum(ys), sum(vals),
                             top, arg])
    return lab, len(rows), np.array(rows, np.int64).reshape(-1, 13)


def random_volumes(count, seed):
    rng = np.random.default_rng(seed)
    for i in range(count):
        n, h, w = (int(v) for v in rng.integers(1, 9, 3))
        density = rng.choice([0.1, 0.2, 0.31, 0.5, 0.7])
        mask = rng.random((n, h, w)) < density
        vals = rng.integers(0, 5, (n, h, w))  # few levels: ties for the maximum are common
        yield i, np.where(mask, 100 + vals, vals).astype(np.uint16)


@pytest.mark.parametrize("connectivity", [6, 18, 26])
def test_oracle_equals_flood_fill_on_random_volumes(connectivity):
    for i, frames in random_volumes(120, 100 + connectivity):
        want_lab, want_k, want_stats = flood_fill(frames, 50, connectivity)
        lab, k, stats = OM.label_movie(frames, 50, connectivity, max_events=want_k + 3)
        assert k == want_k, i
        np.testing.assert_array_equal(lab, want_lab, err_msg=str(i))
        np.testing.assert_array_equal(stats[:k], want_stats, err_msg=str(i))
        assert not stats[k:].any(), i
        # capacity below K keeps the first rows
        cap = max(1, k // 2)
        _, _, part = OM.label_movie(frames, 50, connectivity, max_events=cap)
        np.testing.assert_array_equal(part[:min(k, cap)], want_stats[:cap], err_msg=str(i))


@pytest.mark.parametrize("connectivity,plane", [(6, 4), (18, 8), (26, 8)])
def test_single_frames_equal_the_per_frame_oracle(connectivity, plane):
    rng = np.random.default_rng(connectivity)
    for i in range(40):
        h, w = (int(v) for v in rng.integers(1, 30, 2))
        frame = np.where(rng.random((h, w)) < rng.choice([0.3, 0.5, 0.6]), 100 + rng.integers(0, 4, (h, w)), 0).astype(np.uint16)
        lab, k, st = OM.label_movie(frame[None], 50, connectivity, 512)
        lab2, counts, st2 = OL.label_batch(frame[None], 50, plane, 512)
        assert k == counts[0], i
        np.testing.assert_array_equal(lab, lab2, err_msg=str(i))
        m = min(k, 512)
        pairs = [(sp.EV_VOLUME, sp.AREA), (sp.EV_X_MIN, sp.X_MIN), (sp.EV_Y_MIN, sp.Y_MIN), (sp.EV_X_MAX, sp.X_MAX),
                 (sp.EV_Y_MAX, sp.Y_MAX), (sp.EV_SUM_X, sp.SUM_X), (sp.EV_SUM_Y, sp.SUM_Y), (sp.EV_SUM_VALUE, sp.SUM_VALUE),
                 (sp.EV_MAX_VALUE, sp.MAX_VALUE), (sp.EV_ARGMAX, sp.ARGMAX)]
        for a, b in pairs:
            np.testing.assert_array_equal(st[:m, a], st2[0, :m, b], err_msg=f"{i} {a}")
        assert not st[:m, sp.EV_T_FIRST].any() and not st[:m, sp.EV_T_LAST].any() and not st[:m, sp.EV_SUM_T].any()


def planted(step, n=6, size=12):
    """One lit pixel per frame, moved by ``step`` (dy, dx) from frame to frame."""
    frames = np.zeros((n, size, size), np.uint16)
    for t in range(n):
        frames[t, 1 + step[0] * t, 1 + step[1] * t] = 1000 + t
    return frames


def test_planted_volumes():
    diag = planted((1, 1))  # corner-to-corner through time: only the 3 x 3 block reaches it
    assert OM.label_movie(diag, 0, 26)[1] == 1
    assert OM.label_movie(diag, 0, 18)[1] == 6
    assert OM.label_movie(diag, 0, 6)[1] == 6
    side = planted((0, 1))  # an edge neighbour in the next frame
    assert OM.label_movie(side, 0, 26)[1] == 1
    assert OM.label_movie(side, 0, 18)[1] == 1
    assert OM.label_movie(side, 0, 6)[1] == 6
    blink = np.zeros((9, 4, 5), np.uint16)
    blink[::2, 2, 3] = 500  # on in every other frame: nothing joins the "on" frames
    for conn in (6, 18, 26):
        lab, k, st = OM.label_movie(blink, 0, conn)
        assert k == 5
        np.testing.assert_array_equal(st[:5, sp.EV_T_FIRST], [0, 2, 4, 6, 8])
        np.testing.assert_array_equal(st[:5, sp.EV_ARGMAX], [t * 20 + 13 for t in (0, 2, 4, 6, 8)])
        assert lab[4, 2, 3] == 3
    # the whole-event statistics of the diagonal
    _, k, st = OM.label_movie(diag, 0, 26)
    np.testing.assert_array_equal(st[0], [6, 0, 5, 1, 1, 6, 6, 15, 21, 21, sum(range(1000, 1006)), 1005, 5 * 144 + 6 * 12 + 6])


def test_facade_checks_its_arguments():
    frames = np.zeros((2, 4, 5), np.uint16)
    for call in (
        lambda: sp.label_movie(frames[0], 1),  # not a stack
        lambda: sp.label_movie(frames, 1, connectivity=8),
        lambda: sp.label_movie(frames, [1, 2, 3]),  # neither one nor one per frame
        lambda: sp.label_movie(frames, 70000),
        lambda: sp.label_movie(frames, 1.5),
        lambda: sp.label_movie(frames, 1, max_events=-1),
        lambda: sp.label_movie(frames.astype(np.int32), 1),
        lambda: sp.label_movie(frames, 1, labels=np.zeros((2, 4, 5), np.int64)),
        lambda: sp.label_movie(frames, 1, labels=np.zeros((2, 4, 10), np.int32)[:, :, ::2]),  # a strided output
    ):
        with pytest.raises(RuntimeError):
            call()


def test_c_entry_refuses_bad_arguments_without_a_device():
    lib = _lib.load()
    frames = np.zeros((2, 4, 5), np.uint16)
    lab = np.zeros(frames.shape, np.int32)
    cnt = np.full(1, -3, np.int32)
    stats = np.zeros((4, 13), np.int64)
    thr = np.zeros(2, np.uint16)

    def call(nframes=2, nthr=1, conn=26, cap=4, w=5, h=4, st=stats.ctypes.data):
        return lib.rirb_label_movie(frames.ctypes.data, w, h, nframes, thr.ctypes.data, nthr, conn, lab.ctypes.data,
                                    cnt.ctypes.data, st, cap)

    for conn in (4, 8, 0):
        assert call(conn=conn) == -1
        assert "connectivity" in _lib.last_error() and str(conn) in _lib.last_error()
    assert call(nthr=3) == -1 and "bad arguments" in _lib.last_error()
    assert call(cap=-1) == -1 and "bad arguments" in _lib.last_error()
    assert call(cap=-1, st=None) == -1 and "bad arguments" in _lib.last_error()
    assert call(w=65536, h=32768) == -1 and "bad arguments" in _lib.last_error()
    assert call(nframes=-1) == -1 and "bad arguments" in _lib.last_error()
    assert call(nframes=2 ** 40, nthr=1, w=1 << 15, h=1 << 15) == -1 and "2^48" in _lib.last_error()
    assert (cnt == -3).all() and not lab.any() and not stats.any()  # nothing written by a refused call
    assert call(nframes=0, nthr=0) == 0 and cnt[0] == 0  # no frames, no events


@pytest.mark.skipif(_lib.device_available(), reason="checks behaviour WITHOUT a CUDA device")
def test_label_movie_without_a_device_fails_loudly():
    frames = np.ones((2, 4, 5), np.uint16)
    with pytest.raises(RuntimeError) as e:
        sp.label_movie(frames, 0)
    assert "no CPU fallback" in str(e.value)
    lib = _lib.load()
    lab = np.zeros(frames.shape, np.int32)
    cnt = np.zeros(1, np.int32)
    thr = np.zeros(1, np.uint16)
    assert lib.rirb_label_movie(frames.ctypes.data, 5, 4, 2, thr.ctypes.data, 1, 26, lab.ctypes.data, cnt.ctypes.data, None, 0) == -1
    assert "no CPU fallback" in _lib.last_error()
