"""rirb_label_batch on the device, bit for bit against oracle/label.py (scipy.ndimage.label + int64 reductions): labels,
counts and statistics at connectivity 4 and 8, on edge shapes around the 32 x 32 tile, patterns that stress the border
merges (spirals, combs, U-shapes, noise around the percolation densities), the IR movie, thresholds, capacity, batches of
more than 65,535 frames, determinism and the operand contract."""

import numpy as np
import pytest

from oracle import label as OL
from tests.conftest import ir_movie

pytestmark = pytest.mark.gpu

torch = pytest.importorskip("torch")

from librir_b200 import _lib, signal_processing as sp  # noqa: E402

TILE = 32
THR = 500


# ---- patterns: boolean masks of shape (h, w) -----------------------------------------------------------------------
def spiral(h, w):
    """One width-1 path winding inwards through every ring (rings 2 px apart, each opened next to its corner)."""
    m = np.zeros((h, w), bool)
    k = 0
    while 2 * k <= h - 1 - 2 * k and 2 * k <= w - 1 - 2 * k:
        t, l, b, r = 2 * k, 2 * k, h - 1 - 2 * k, w - 1 - 2 * k
        m[t, l:r + 1] = m[b, l:r + 1] = True
        m[t:b + 1, l] = m[t:b + 1, r] = True
        if t + 1 < b:
            m[t + 1, l] = False
            if t + 2 <= b and l + 1 <= r:
                m[t + 2, l + 1] = True
        k += 1
    return m


def comb(h, w):
    """Teeth on every other column that meet only on the last row."""
    m = np.zeros((h, w), bool)
    m[:, ::2] = True
    m[-1, :] = True
    return m


def u_shapes(h, w):
    """Pairs of bars 4 px apart joined only on the last row."""
    m = np.zeros((h, w), bool)
    x = np.arange(w)
    m[:, (x % 6 == 0) | (x % 6 == 4)] = True
    m[-1, x % 6 <= 4] = True
    return m


def patterns(h, w, seed):
    rng = np.random.default_rng(seed)
    y, x = np.mgrid[0:h, 0:w]
    out = {
        "empty": np.zeros((h, w), bool),
        "full": np.ones((h, w), bool),
        "checker": (x + y) % 2 == 0,
        "hstripes": y % 2 == 0,
        "vstripes": x % 2 == 0,
        "diagonal": (x - y) % 3 == 0,  # 8- but not 4-connected
        "spiral": spiral(h, w),
        "comb": comb(h, w),
        "comb_up": comb(h, w)[::-1],
        "u_shapes": u_shapes(h, w),
    }
    for d in (0.3, 0.41, 0.5, 0.59, 0.7):
        out[f"noise{d}"] = rng.random((h, w)) < d
    return out


def to_frames(masks, seed):
    """uint16 frames: foreground THR+1 .. THR+8 (ties for the maximum), background 0 .. THR."""
    rng = np.random.default_rng(seed)
    fr = []
    for m in masks:
        fr.append(np.where(m, THR + 1 + rng.integers(0, 8, m.shape), rng.integers(0, THR + 1, m.shape)).astype(np.uint16))
    return np.stack(fr)


def check(frames, thr, conn, cap=64, device=True):
    want = OL.label_batch(frames, thr, conn, cap)
    src = torch.from_numpy(frames.view(np.int16)).cuda().view(torch.uint16) if device else frames
    got = sp.label_batch(src, thr, conn, cap)
    got = [g.cpu().numpy() if device else g for g in got]
    for name, a, b in zip(("labels", "counts", "stats"), got, want):
        if not np.array_equal(a, b):
            bad = np.argwhere(a != b)
            pytest.fail(f"{name} differ at {len(bad)} places, first {bad[:3].tolist()}: got {a[tuple(bad[0])]}, want {b[tuple(bad[0])]}")
    return got


SHAPES = [(1, 1), (1, 300), (300, 1), (7, 5), (TILE - 1, TILE - 1), (TILE, TILE), (TILE + 1, TILE + 1), (TILE - 1, TILE + 1),
          (TILE + 1, TILE - 1), (2 * TILE + 1, 3 * TILE - 1), (509, 641), (512, 640), (1024, 1024), (2048, 2048)]


@pytest.fixture(scope="module", autouse=True)
def device():
    if not torch.cuda.is_available():
        pytest.skip("needs a CUDA device")
    torch.cuda.set_device(0)


@pytest.mark.parametrize("conn", [4, 8])
@pytest.mark.parametrize("shape", SHAPES, ids=[f"{h}x{w}" for h, w in SHAPES])
def test_patterns_equal_the_oracle(shape, conn):
    h, w = shape
    pats = patterns(h, w, seed=h * 7919 + w)
    frames = to_frames(list(pats.values()), seed=w)
    check(frames, THR, conn)


@pytest.mark.parametrize("conn", [4, 8])
def test_ir_movie_thresholded_at_several_levels(conn):
    mov = ir_movie(8, 512, 640)
    for level in (8500, 9500, 9900, 10500, 15000):
        check(mov, level, conn, cap=256)
    # per-frame thresholds in one call, numpy host operands too
    check(mov, np.array([8500, 9500, 9900, 10500, 15000, 9000, 9700, 0], np.uint16), conn, cap=256, device=False)


def test_thresholds_per_frame_scalar_and_extremes():
    h, w = 70, 90
    frames = to_frames(list(patterns(h, w, 5).values()), 6)
    n = len(frames)
    per = np.arange(n, dtype=np.uint16) * 37 + 400
    check(frames, per, 8)
    check(frames, per[3], 4)
    labels, counts, stats = sp.label_batch(frames, 65535, 8)  # nothing is above 65535
    assert not labels.any() and not counts.any() and not stats.any()
    zeros = np.zeros((3, h, w), np.uint16)
    labels, counts, stats = sp.label_batch(zeros, 0, 4)  # 0 > 0 is false
    assert not labels.any() and not counts.any() and not stats.any()
    d = torch.from_numpy(per.view(np.int16)).cuda().view(torch.uint16)  # device thresholds
    got = sp.label_batch(torch.from_numpy(frames.view(np.int16)).cuda().view(torch.uint16), d, 8)
    want = OL.label_batch(frames, per, 8, 256)
    for a, b in zip(got, want):
        np.testing.assert_array_equal(a.cpu().numpy(), b)


def test_capacity_below_the_count_and_sentinel_rows():
    lib = _lib.load()
    h, w = 64, 96
    rng = np.random.default_rng(11)
    masks = [rng.random((h, w)) < 0.4, np.zeros((h, w), bool)]
    masks[1][5:9, 5:9] = masks[1][20:30, 40:45] = True  # two components, fewer than the capacity
    frames = to_frames(masks, 12)
    cap = 5
    want_l, want_c, want_s = OL.label_batch(frames, THR, 8, cap)
    assert want_c[0] > cap and want_c[1] == 2
    for kind in ("host", "device"):
        stats = np.full((2, cap, 10), -7, np.int64)
        labels = np.zeros(frames.shape, np.int32)
        counts = np.zeros(2, np.int32)
        thr = np.array([THR], np.uint16)
        if kind == "host":
            rc = lib.rirb_label_batch(frames.ctypes.data, w, h, 2, thr.ctypes.data, 1, 8, labels.ctypes.data, counts.ctypes.data,
                                      stats.ctypes.data, cap)
            got_s = stats
        else:
            ds = torch.from_numpy(stats).cuda()
            rc = lib.rirb_label_batch(frames.ctypes.data, w, h, 2, thr.ctypes.data, 1, 8, labels.ctypes.data, counts.ctypes.data,
                                      ds.data_ptr(), cap)
            torch.cuda.synchronize()
            got_s = ds.cpu().numpy()
        assert rc == 0, _lib.last_error()
        np.testing.assert_array_equal(counts, want_c)
        np.testing.assert_array_equal(labels, want_l)
        np.testing.assert_array_equal(got_s[0], want_s[0])
        np.testing.assert_array_equal(got_s[1, :2], want_s[1, :2])
        assert np.all(got_s[1, 2:] == -7), "rows past K_t were written"


def test_more_than_65535_frames_in_one_call():
    rng = np.random.default_rng(21)
    n = 70_001
    frames = np.where(rng.random((n, 3, 5)) < 0.5, THR + 1 + rng.integers(0, 4, (n, 3, 5)), 0).astype(np.uint16)
    per = rng.integers(THR - 1, THR + 4, n).astype(np.uint16)
    check(frames, per, 4, cap=8)


def test_two_runs_give_identical_bits():
    frames = to_frames([np.random.default_rng(s).random((512, 640)) < 0.59 for s in range(6)], 31)
    d = torch.from_numpy(frames.view(np.int16)).cuda().view(torch.uint16)
    a = sp.label_batch(d, THR, 8, 4096)
    b = sp.label_batch(d, THR, 8, 4096)
    for x, y in zip(a, b):
        assert torch.equal(x, y)


# ---- operand contract ---------------------------------------------------------------------------------------------
from tests.test_gpu_operand_contract import KINDS, Buf  # noqa: E402


@pytest.fixture
def pool():
    fns = []
    yield fns
    torch.cuda.synchronize()
    for f in reversed(fns):
        f()


N, H, W, CAP = 3, 40, 70, 16


def contract_operands():
    frames = to_frames([np.random.default_rng(s).random((H, W)) < 0.5 for s in range(N)], 41)
    return dict(frames=frames, thresholds=np.array([THR, THR - 3, THR + 2], np.uint16), labels=np.zeros((N, H, W), np.int32),
                counts=np.zeros(N, np.int32), stats=np.full((N, CAP, 10), -5, np.int64))


def run_contract(lib, kinds, pool):
    ops = contract_operands()
    bufs = {k: Buf(kinds.get(k, "device"), v, pool) for k, v in ops.items()}
    rc = lib.rirb_label_batch(bufs["frames"].ptr, W, H, N, bufs["thresholds"].ptr, N, 8, bufs["labels"].ptr, bufs["counts"].ptr,
                              bufs["stats"].ptr, CAP)
    assert rc == 0, _lib.last_error()
    return {k: bufs[k].read() for k in ("labels", "counts", "stats")}


@pytest.mark.parametrize("kind", KINDS[:-1])
@pytest.mark.parametrize("operand", ["frames", "thresholds", "labels", "counts", "stats"])
def test_every_kind_of_memory_gives_the_device_bits(operand, kind, pool):
    lib = _lib.load()
    lib.rirb_set_stream(None)
    want = run_contract(lib, {}, pool)
    got = run_contract(lib, {operand: kind}, pool)
    for k in want:
        assert np.array_equal(got[k], want[k]), (operand, kind, k)
    ops = contract_operands()
    wl, wc, ws = OL.label_batch(ops["frames"], ops["thresholds"], 8, CAP)
    assert np.array_equal(want["labels"].view(np.int32).reshape(wl.shape), wl)
    assert np.array_equal(want["counts"].view(np.int32), wc)
    s = want["stats"].view(np.int64).reshape(N, CAP, 10)
    for t in range(N):
        m = min(int(wc[t]), CAP)
        assert np.array_equal(s[t, :m], ws[t, :m]) and np.all(s[t, m:] == -5)


@pytest.mark.parametrize("pair", [("labels", "counts"), ("labels", "stats"), ("counts", "stats"), ("frames", "labels"),
                                  ("thresholds", "counts")])
def test_overlapping_device_operands_are_refused_without_a_launch(pair):
    lib = _lib.load()
    lib.rirb_set_stream(None)
    npx = N * H * W
    # one device buffer holds every operand; the second of the pair is moved onto the first
    sizes = dict(frames=npx * 2, thresholds=N * 2, labels=npx * 4, counts=N * 4, stats=N * CAP * 80)
    offs, at = {}, 0
    for k, s in sizes.items():
        offs[k] = at
        at += (s + 255) // 256 * 256
    buf = torch.full((at,), 0xA5, dtype=torch.uint8, device="cuda")
    offs[pair[1]] = offs[pair[0]] + 2  # every operand is longer than 2 bytes
    base = buf.data_ptr()
    before = _lib.launch_count()
    rc = lib.rirb_label_batch(base + offs["frames"], W, H, N, base + offs["thresholds"], N, 8, base + offs["labels"],
                              base + offs["counts"], base + offs["stats"], CAP)
    torch.cuda.synchronize()
    assert rc == -1 and "overlap" in _lib.last_error()
    assert _lib.launch_count() == before
    assert bool((buf == 0xA5).all()), "a refused call wrote to the buffer"


def test_misaligned_frame_views_are_accepted():
    frames = to_frames([np.random.default_rng(s).random((37, 53)) < 0.55 for s in range(4)], 51)
    raw = torch.zeros(frames.size + 1, dtype=torch.int16, device="cuda")
    raw[1:] = torch.from_numpy(frames.reshape(-1).view(np.int16)).cuda()
    view = raw[1:].view(torch.uint16).reshape(frames.shape)  # 2 bytes past a 256-byte boundary
    lab = torch.zeros(frames.size + 1, dtype=torch.int32, device="cuda")[1:].reshape(frames.shape)
    got = sp.label_batch(view, THR, 8, 32, labels=lab)
    want = OL.label_batch(frames, THR, 8, 32)
    for a, b in zip(got, want):
        np.testing.assert_array_equal(a.cpu().numpy(), b)
