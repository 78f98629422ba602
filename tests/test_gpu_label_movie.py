"""rirb_label_movie on the device, bit for bit against oracle/label_movie.py (scipy.ndimage.label on the (t, y, x) volume + int64
reductions): labels, count and statistics at connectivity 6, 18 and 26, on edge shapes around the 32 x 32 tile, movies
of the 2-D adversarial patterns, temporal adversaries (late merges, late-born events, deep union chains, helices, 3-D
percolation noise), the IR movie, capacity, more than 65,535 frames, determinism and the operand contract."""

import numpy as np
import pytest

from oracle import label_movie as OM
from tests.conftest import ir_movie

pytestmark = pytest.mark.gpu

torch = pytest.importorskip("torch")

from librir_b200 import _lib, signal_processing as sp  # noqa: E402

TILE = 32
THR = 500
CONNS = [6, 18, 26]


# ---- 2-D patterns (boolean masks of shape (h, w)) ------------------------------------------------------------------
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
    out = [spiral(h, w), comb(h, w), comb(h, w)[::-1], u_shapes(h, w), y % 2 == 0, x % 2 == 0, (x + y) % 2 == 0,
           (x - y) % 3 == 0]
    out += [rng.random((h, w)) < d for d in (0.3, 0.41, 0.59)]
    return out


def to_frames(masks, seed):
    """uint16 frames: foreground THR+1 .. THR+8 (ties for the maximum), background 0 .. THR."""
    masks = np.asarray(masks)
    rng = np.random.default_rng(seed)
    return np.where(masks, THR + 1 + rng.integers(0, 8, masks.shape), rng.integers(0, THR + 1, masks.shape)).astype(np.uint16)


def dev(a):
    return torch.from_numpy(np.ascontiguousarray(a).view(np.int16)).cuda().view(torch.uint16)


def check(frames, thr, conn, cap=64, device=True):
    want_l, want_k, want_s = OM.label_movie(frames, thr, conn, cap)
    got_l, got_k, got_s = sp.label_movie(dev(frames) if device else frames, thr, conn, cap)
    if device:
        got_l, got_s = got_l.cpu().numpy(), got_s.cpu().numpy()
    assert got_k == want_k, f"count {got_k}, want {want_k}"
    for name, a, b in (("labels", got_l, want_l), ("stats", got_s, want_s)):
        if not np.array_equal(a, b):
            bad = np.argwhere(a != b)
            pytest.fail(f"{name} differ at {len(bad)} places, first {bad[:3].tolist()}: got {a[tuple(bad[0])]}, want {b[tuple(bad[0])]}")
    return got_l, got_k, got_s


@pytest.fixture(scope="module", autouse=True)
def device():
    if not torch.cuda.is_available():
        pytest.skip("needs a CUDA device")
    torch.cuda.set_device(0)


# ---- shapes ---------------------------------------------------------------------------------------------------------
SHAPES = [(1, 1, 1), (1, 7, 5), (2, 33, 31), (3, 1, 300), (5, 300, 1), (12, TILE - 1, TILE - 1), (12, TILE, TILE),
          (12, TILE + 1, TILE + 1), (12, TILE - 1, TILE + 1), (22, 2 * TILE + 1, 3 * TILE - 1), (40, 509, 641), (40, 512, 640)]


@pytest.mark.parametrize("conn", CONNS)
@pytest.mark.parametrize("shape", SHAPES, ids=[f"{n}x{h}x{w}" for n, h, w in SHAPES])
def test_pattern_movies_equal_the_oracle(shape, conn):
    n, h, w = shape
    pats = patterns(h, w, seed=h * 7919 + w)
    # each pattern held for two frames, then the next one: links to itself and to a different pattern
    masks = [pats[(t // 2) % len(pats)] for t in range(n)]
    check(to_frames(masks, seed=n + w), THR, conn)


# ---- temporal adversaries -------------------------------------------------------------------------------------------
@pytest.mark.parametrize("conn", CONNS)
def test_blobs_born_apart_merge_late(conn):
    n, h, w = 60, 40, 70
    m = np.zeros((n, h, w), bool)
    m[:, 10:20, 5:15] = True  # the left blob, from frame 0
    m[:, 25:35, 50:60] = True  # the right blob, from frame 0
    m[50:, 14:30, 5:60] = True  # frame 50 on: a bridge
    _, k, st = check(to_frames(m, 1), THR, conn)
    assert k == 1 and st[0, sp.EV_T_FIRST] == 0 and st[0, sp.EV_T_LAST] == n - 1


@pytest.mark.parametrize("conn", CONNS)
def test_late_born_event_high_in_raster_order_merges_into_an_earlier_one(conn):
    n, h, w = 12, 64, 64
    m = np.zeros((n, h, w), bool)
    m[0:, 50:60, 50:60] = True  # born in frame 0, low in the frame
    m[3:, 2:8, 2:8] = True  # born in frame 3, first in raster order of its frame
    m[6:, 4:52, 6:52] = True  # frame 6 on: joins the two
    m[1, 0, 0] = True  # an isolated voxel, born between them
    lab, k, st = check(to_frames(m, 2), THR, conn)
    assert k == 2 and lab[3, 2, 2] == 1 and lab[1, 0, 0] == 2


@pytest.mark.parametrize("conn", CONNS)
def test_comb_through_time(conn):
    """One component per frame at its own x, joined only through the last frame: deep union chains."""
    n, h, w = 200, 6, 400
    m = np.zeros((n, h, w), bool)
    for t in range(n - 1):
        m[t:, 2, 2 * t] = True  # a tooth born in frame t at x = 2t, lasting to the end
    m[n - 1, 2, :] = True
    _, k, _ = check(to_frames(m, 3), THR, conn, cap=8)
    assert k == 1


@pytest.mark.parametrize("conn", CONNS)
def test_helix_connected_only_through_frames(conn):
    n, h, w = 120, 48, 48
    m = np.zeros((n, h, w), bool)
    for t in range(n):
        a = 2 * np.pi * t / 40
        y, x = int(round(24 + 10 * np.sin(a))), int(round(24 + 10 * np.cos(a)))
        m[t, y - 1:y + 2, x - 1:x + 2] = True  # a 3 x 3 dot: the next frame's dot overlaps it at every connectivity
        y2, x2 = int(round(24 - 10 * np.sin(a))), int(round(24 - 10 * np.cos(a)))
        m[t, y2 - 1:y2 + 2, x2 - 1:x2 + 2] = True  # the second strand
    _, k, _ = check(to_frames(m, 4), THR, conn)
    assert k == 2


@pytest.mark.parametrize("conn,density", [(6, 0.31), (18, 0.14), (26, 0.10), (6, 0.5), (26, 0.2)])
def test_noise_at_the_percolation_density(conn, density):
    rng = np.random.default_rng(conn)
    m = rng.random((30, 200, 300)) < density
    check(to_frames(m, 5), THR, conn, cap=4096)


@pytest.mark.parametrize("conn", CONNS)
def test_full_and_empty_volumes(conn):
    full = np.ones((25, 70, 90), bool)
    _, k, st = check(to_frames(full, 6), THR, conn)
    assert k == 1 and st[0, sp.EV_VOLUME] == full.size
    _, k, st = check(to_frames(~full, 7), THR, conn)
    assert k == 0 and not st.any()


# ---- the IR movie ---------------------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def ir():
    return ir_movie(200, 512, 640, drift=0.05)


@pytest.mark.parametrize("conn", CONNS)
def test_ir_movie_at_several_thresholds(ir, conn):
    n = len(ir)
    for level in (9500, 9900, 15000):
        _, k, st = check(ir, level, conn, cap=512)
        if level == 15000:  # only the stuck-hot pixels: each one is an event over the whole movie
            assert k > 100 and np.all(st[:k, sp.EV_VOLUME] == n) and np.all(st[:k, sp.EV_T_LAST] == n - 1)
    # above the background, the drifting spot is one event over every frame
    _, k, st = check(ir, 10100, conn, cap=512)
    spot = st[:k][st[:k, sp.EV_VOLUME] > n]
    assert len(spot) == 1 and spot[0, sp.EV_T_FIRST] == 0 and spot[0, sp.EV_T_LAST] == n - 1


@pytest.mark.parametrize("conn", [6, 26])
def test_ir_movie_with_per_frame_thresholds(ir, conn):
    per = (10300 + 7 * (np.arange(len(ir)) % 50)).astype(np.uint16)
    check(ir, per, conn, cap=512)  # device frames, host thresholds
    check(ir[:60], per[:60], conn, cap=512, device=False)  # host frames and thresholds
    want = OM.label_movie(ir, per, conn, 512)
    got = sp.label_movie(dev(ir), dev(per), conn, 512)  # device thresholds
    assert got[1] == want[1]
    np.testing.assert_array_equal(got[0].cpu().numpy(), want[0])
    np.testing.assert_array_equal(got[2].cpu().numpy(), want[2])


# ---- capacity -------------------------------------------------------------------------------------------------------
def test_capacity_and_sentinel_rows():
    lib = _lib.load()
    rng = np.random.default_rng(11)
    n, h, w = 6, 40, 60
    frames = to_frames(rng.random((n, h, w)) < 0.2, 12)
    _, K, full = OM.label_movie(frames, THR, 26, 10_000)
    assert K > 20
    for cap in (0, 7, K, K + 9):
        check(frames, THR, 26, cap=cap)
    thr = np.array([THR], np.uint16)
    for kind in ("host", "device"):
        for cap in (7, K + 9):
            stats = np.full((cap, 13), -7, np.int64)
            labels = np.zeros(frames.shape, np.int32)
            count = np.zeros(1, np.int32)
            ds = torch.from_numpy(stats).cuda() if kind == "device" else None
            rc = lib.rirb_label_movie(frames.ctypes.data, w, h, n, thr.ctypes.data, 1, 26, labels.ctypes.data, count.ctypes.data,
                                      ds.data_ptr() if ds is not None else stats.ctypes.data, cap)
            assert rc == 0, _lib.last_error()
            got = ds.cpu().numpy() if ds is not None else stats
            m = min(K, cap)
            assert count[0] == K
            np.testing.assert_array_equal(got[:m], full[:m])
            assert np.all(got[m:] == -7), "rows past K were written"
    # stats = NULL through the C entry
    labels = np.zeros(frames.shape, np.int32)
    count = np.zeros(1, np.int32)
    assert lib.rirb_label_movie(frames.ctypes.data, w, h, n, thr.ctypes.data, 1, 26, labels.ctypes.data, count.ctypes.data, None,
                                16) == 0, _lib.last_error()
    assert count[0] == K
    np.testing.assert_array_equal(labels, OM.label_movie(frames, THR, 26, 0)[0])


# ---- limits ---------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("conn", CONNS)
def test_more_than_65535_frames(conn):
    rng = np.random.default_rng(21 + conn)
    n = 70_001
    m = rng.random((n, 3, 5)) < 0.3
    m[:, 1, 2] = True  # on in every frame: one event spans them all
    frames = to_frames(m, 22)
    lab, _, _ = check(frames, THR, conn, cap=16)
    assert lab[0, 1, 2] > 0 and np.all(lab[:, 1, 2] == lab[0, 1, 2])


def test_single_pixel_chain_over_all_frames():
    n = 70_001
    m = np.zeros((n, 2, 3), bool)
    m[:, 1, 1] = True
    for conn in CONNS:
        lab, k, st = check(to_frames(m, 23), THR, conn, cap=2)
        assert k == 1 and st[0, sp.EV_VOLUME] == n and st[0, sp.EV_SUM_T] == n * (n - 1) // 2


# ---- consistency ----------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("conn,plane", [(6, 4), (18, 8), (26, 8)])
def test_one_frame_gives_the_labels_of_label_batch(conn, plane):
    frames = to_frames([np.random.default_rng(31).random((300, 400)) < 0.55], 32)
    a, k, _ = sp.label_movie(dev(frames), THR, conn, 16)
    b, counts, _ = sp.label_batch(dev(frames), THR, plane, 16)
    assert torch.equal(a, b) and k == int(counts[0])


def test_two_runs_give_identical_bits():
    frames = to_frames(np.random.default_rng(41).random((20, 512, 640)) < 0.2, 42)
    d = dev(frames)
    a = sp.label_movie(d, THR, 26, 4096)
    b = sp.label_movie(d, THR, 26, 4096)
    assert a[1] == b[1] and torch.equal(a[0], b[0]) and torch.equal(a[2], b[2])


# ---- operand contract -----------------------------------------------------------------------------------------------
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
    frames = to_frames(np.random.default_rng(51).random((N, H, W)) < 0.3, 52)
    return dict(frames=frames, thresholds=np.array([THR, THR - 3, THR + 2], np.uint16), labels=np.zeros((N, H, W), np.int32),
                count=np.full(1, -1, np.int32), stats=np.full((CAP, 13), -5, np.int64))


def run_contract(lib, kinds, pool):
    ops = contract_operands()
    bufs = {k: Buf(kinds.get(k, "device"), v, pool) for k, v in ops.items()}
    rc = lib.rirb_label_movie(bufs["frames"].ptr, W, H, N, bufs["thresholds"].ptr, N, 18, bufs["labels"].ptr, bufs["count"].ptr,
                              bufs["stats"].ptr, CAP)
    assert rc == 0, _lib.last_error()
    return {k: bufs[k].read() for k in ("labels", "count", "stats")}


@pytest.mark.parametrize("kind", KINDS[:-1])
@pytest.mark.parametrize("operand", ["frames", "thresholds", "labels", "count", "stats"])
def test_every_kind_of_memory_gives_the_device_bits(operand, kind, pool):
    lib = _lib.load()
    lib.rirb_set_stream(None)
    want = run_contract(lib, {}, pool)
    got = run_contract(lib, {operand: kind}, pool)
    for k in want:
        assert np.array_equal(got[k], want[k]), (operand, kind, k)
    ops = contract_operands()
    wl, wk, ws = OM.label_movie(ops["frames"], ops["thresholds"], 18, CAP)
    assert np.array_equal(want["labels"].view(np.int32).reshape(wl.shape), wl)
    assert want["count"].view(np.int32)[0] == wk
    s = want["stats"].view(np.int64).reshape(CAP, 13)
    m = min(wk, CAP)
    assert np.array_equal(s[:m], ws[:m]) and np.all(s[m:] == -5)


@pytest.mark.parametrize("pair", [("labels", "count"), ("labels", "stats"), ("count", "stats"), ("frames", "labels"),
                                  ("thresholds", "count"), ("frames", "stats")])
def test_overlapping_device_operands_are_refused_without_a_launch(pair):
    lib = _lib.load()
    lib.rirb_set_stream(None)
    npx = N * H * W
    sizes = dict(frames=npx * 2, thresholds=N * 2, labels=npx * 4, count=4, stats=CAP * 13 * 8)
    offs, at = {}, 0
    for k, s in sizes.items():
        offs[k] = at
        at += (s + 255) // 256 * 256
    buf = torch.full((at,), 0xA5, dtype=torch.uint8, device="cuda")
    offs[pair[1]] = offs[pair[0]] + 2  # every operand is longer than 2 bytes
    base = buf.data_ptr()
    before = _lib.launch_count()
    rc = lib.rirb_label_movie(base + offs["frames"], W, H, N, base + offs["thresholds"], N, 26, base + offs["labels"],
                              base + offs["count"], base + offs["stats"], CAP)
    torch.cuda.synchronize()
    assert rc == -1 and "overlap" in _lib.last_error()
    assert _lib.launch_count() == before
    assert bool((buf == 0xA5).all()), "a refused call wrote to the buffer"


def test_misaligned_frame_views_are_accepted():
    frames = to_frames(np.random.default_rng(61).random((4, 37, 53)) < 0.3, 62)
    raw = torch.zeros(frames.size + 1, dtype=torch.int16, device="cuda")
    raw[1:] = torch.from_numpy(frames.reshape(-1).view(np.int16)).cuda()
    view = raw[1:].view(torch.uint16).reshape(frames.shape)  # 2 bytes past a 256-byte boundary
    lab = torch.zeros(frames.size + 1, dtype=torch.int32, device="cuda")[1:].reshape(frames.shape)
    got = sp.label_movie(view, THR, 26, 32, labels=lab)
    want = OM.label_movie(frames, THR, 26, 32)
    assert got[1] == want[1]
    np.testing.assert_array_equal(got[0].cpu().numpy(), want[0])
    np.testing.assert_array_equal(got[2].cpu().numpy(), want[2])


def test_strided_numpy_input_is_copied_and_strided_outputs_are_refused():
    big = to_frames(np.random.default_rng(71).random((4, 30, 80)) < 0.3, 72)
    view = big[:, :, ::2]  # strided input
    lab, k, st = sp.label_movie(view, THR, 18, 64)
    want = OM.label_movie(np.ascontiguousarray(view), THR, 18, 64)
    assert k == want[1]
    np.testing.assert_array_equal(lab, want[0])
    np.testing.assert_array_equal(st, want[2])
    out = np.zeros((4, 30, 80), np.int32)[:, :, ::2]
    with pytest.raises(RuntimeError, match="strided"):
        sp.label_movie(view, THR, 18, 64, labels=out)
    tout = torch.zeros((4, 30, 80), dtype=torch.int32, device="cuda")[:, :, ::2]
    with pytest.raises(RuntimeError):
        sp.label_movie(dev(view), THR, 18, 64, labels=tout)
