"""Randomised tests of the device zstd kernels.  The decoder (rirb_zstd_decode_batch) runs the random valid, mutated and
truncated frames of tests/test_zdecoder_fuzz.py in mixed batches (frames at every offset mod 16 of the source, the
last ones ending within 16 bytes of its end, capacities one byte short, 8 MiB records at window log 23) and must give
the status and bytes of the host build of the same per-frame code, and libzstd's content for every valid frame: the
warp version (32 lanes, the aligned 16-byte loads) computes the same function as the sequential one.  Coder 1
(rirb_zstd_encode_batch) and coder 2 (rirb_zstd_encode_batch_lz) run payloads aimed at their rules (symbol ranges,
weight descriptions, count ties, the length limit, literal counts, block and segment edges, match lengths, long
literal runs, sort chunks) and must write oracle/zcoder.py's and oracle/zlz.py's frames byte for byte, which libzstd
and the device decoder give back.  ``RIRB_FUZZ_SEED=<n> RIRB_FUZZ_SCALE=<k>`` runs k times as many cases from other
seeds."""
import numpy as np
import pytest

from tests import test_zdecoder_fuzz as F
from tests import vio_cases as C
from tests import zlz_cases as L

pytestmark = pytest.mark.gpu

torch = pytest.importorskip("torch")
if not torch.cuda.is_available():  # pragma: no cover
    pytest.skip("needs a CUDA device", allow_module_level=True)

from librir_b200 import _lib  # noqa: E402
from librir_b200 import entropy as E  # noqa: E402
from oracle import zcoder as Z1  # noqa: E402
from oracle import zlz as Z2  # noqa: E402
from tests.test_gpu_zcoder import device_encode  # noqa: E402
from tests.test_gpu_zlz import device_encode_lz  # noqa: E402

SEED, SCALE = F.SEED, F.SCALE
GUARD = 0xA5


@pytest.fixture(scope="module")
def host_decode(tmp_path_factory):
    return F.build_host_decoder(tmp_path_factory.mktemp("zdhost"))


def decode_batch(frames, cap, rng, stride=None):
    """rirb_zstd_decode_batch with frame i at an offset = i mod 16 (plus 0 or 16) of the source and 0-15 bytes after
    the last frame -> (statuses, [n + 2, stride] output whose first and last rows are guard rows)."""
    n = len(frames)
    stride = stride or cap + 64
    blob, offs = bytearray(), []
    for i, f in enumerate(frames):
        blob += b"\xee" * ((i - len(blob)) % 16 + 16 * int(rng.integers(0, 2)))
        offs.append(len(blob))
        blob += f
    blob += b"\xee" * int(rng.integers(0, 16))
    src = torch.from_numpy(np.frombuffer(bytes(blob) or b"\xee", np.uint8).copy()).cuda()
    off = torch.from_numpy(np.array(offs, np.int64)).cuda()
    size = torch.from_numpy(np.array([len(f) for f in frames], np.uint32).view(np.int32)).cuda()
    dst = torch.full((n + 2, stride), GUARD, dtype=torch.uint8, device="cuda")
    status = torch.full((n,), 7777, dtype=torch.int64, device="cuda")
    _lib.use_torch_stream()
    assert _lib.load().rirb_zstd_decode_batch(src.data_ptr(), off.data_ptr(), size.data_ptr(), n, dst[1:].data_ptr(), stride,
                                              cap, status.data_ptr()) == 0, _lib.last_error()
    torch.cuda.synchronize()
    out = dst.cpu().numpy()
    assert (out[0] == GUARD).all() and (out[-1] == GUARD).all()
    return status.cpu().numpy(), out


def check_against_host(frames, cap, rng, host_decode, payloads=None):
    """Every frame: the device's status and bytes are the host harness's, and nothing lands behind the capacity.  For a
    frame with a known payload (None: a mutated frame) both give the payload, or -1 / -2 when it does not fit / has a
    checksum."""
    st, out = decode_batch(frames, cap, rng)
    for i, f in enumerate(frames):
        hs, hb = host_decode(f, cap)
        assert st[i] == hs, (i, st[i], hs)
        assert out[1 + i, :max(hs, 0)].tobytes() == hb, i
        assert (out[1 + i, cap:] == GUARD).all(), i
        if payloads is not None and payloads[i] is not None:
            data, p = payloads[i]
            want = F.expected_status(data, p) if len(data) <= cap else (-2 if p.get(F.P_CHECKSUM) else -1)
            assert hs == want, (i, len(data), cap, hs, p)
            if hs >= 0:
                assert hb == data, i
    return st


def test_decoder_batches(host_decode):
    """Mixed batches of valid and mutated frames up to 400 KB; every third batch with a capacity one byte short of the
    longest payload."""
    rng = np.random.default_rng(701 + SEED)
    for b in range(3 * SCALE):
        frames, pays = [], []
        for i in range(40):
            frame, data, p = F.valid_frame(rng, 40 * b + i, max_len=400_000)
            if rng.random() < 0.4:
                frames.append(F.mutate(rng, frame))
                pays.append(None)
            else:
                frames.append(frame)
                pays.append((data, p))
        longest = max(len(x[0]) for x in pays if x is not None)
        cap = max(0, longest - 1) if b % 3 == 2 else longest + int(rng.integers(0, 64))
        st = check_against_host(frames, cap, rng, host_decode, pays)
        assert (st >= 0).any()


def test_decoder_large_records(host_decode):
    """2048 x 2048 x 2-byte method-1 records (8 MiB, offsets past 2^20) at window log 23, with and without the content
    size, one of them mutated, next to a small frame."""
    rng = np.random.default_rng(702 + SEED)
    mov = C.movie(2, 2048, 2048, seed=int(rng.integers(0, 1000)))
    frames, pays = [], []
    for k in range(2):
        data = mov[k].reshape(-1).view(np.uint8)
        p = {F.P_LEVEL: int(rng.integers(-3, 6)), F.P_WINDOW_LOG: 23, F.P_CONTENT_SIZE: k}
        frames.append(F.compress(data, p))
        pays.append((data.tobytes(), p))
    frames.append(F.mutate(rng, frames[int(rng.integers(0, 2))]))
    pays.append(None)
    frame, data, p = F.valid_frame(rng, 0, max_len=20_000)
    frames.append(frame)
    pays.append((data, p))
    check_against_host(frames, 2048 * 2048 * 2 + int(rng.integers(0, 16)), rng, host_decode, pays)


# ---- coder 1 ------------------------------------------------------------------------------------------------------------
def from_counts(rng, counts):
    """A shuffled payload in which byte value s appears counts[s] times."""
    x = np.repeat(np.arange(len(counts), dtype=np.uint8), counts)
    rng.shuffle(x)
    return x


def coder1_payload(rng):
    """A payload aimed at one of coder 1's rules (DESIGN §7 r3): the largest symbol at 127 / 128 / 129 (nibble against
    FSE weights), many distinct weights (long weight descriptions), one weight value, many equal counts (the tie-breaks
    of the sort and the merge), Fibonacci-like counts (the length limit), or a length from the literal-count and block
    edges."""
    kind = int(rng.integers(0, 7))
    if kind == 0:
        top = int(rng.choice([127, 128, 129]))
        counts = np.minimum(rng.geometric(rng.uniform(0.02, 0.3), top + 1), 400) * int(rng.integers(1, 4))
        counts[top] = max(1, counts[top])
        return from_counts(rng, counts)
    if kind == 1:
        return from_counts(rng, rng.integers(0, 2 ** int(rng.integers(1, 11)), 256) + 1)
    if kind == 2:
        k = 2 ** int(rng.integers(1, 9))
        return from_counts(rng, np.full(k, int(rng.integers(1, 400))))
    if kind == 3:
        levels = rng.integers(1, 300, int(rng.integers(1, 4)))
        return from_counts(rng, levels[rng.integers(0, len(levels), int(rng.integers(2, 257)))])
    if kind == 4:
        f = [1, 1]
        while len(f) < int(rng.integers(18, 27)):
            f.append(f[-1] + f[-2])
        counts = np.array(f, np.int64)
        counts = np.maximum(1, counts + rng.integers(-2, 3, len(counts)) * (counts > 3))
        return from_counts(rng, rng.permutation(counts))
    n = int(rng.choice([1, 2, 3, 4, 5, 6, 1023, 1024, 131071, 131072, 131073, 262143, 262144, 262145,
                        int(rng.integers(0, 300_000))]))
    if kind == 5:
        return np.minimum(rng.geometric(rng.uniform(0.01, 0.5), n), 255).astype(np.uint8)
    return rng.integers(0, int(rng.integers(1, 257)), n).astype(np.uint8)


def random_segment(rng, n):
    return 0 if n == 0 or rng.random() < 0.6 else int(rng.integers(1, n + 1))


def check_coder(frames, payloads, segment, restate, host_decode, rng):
    """Frames are the restatement's byte for byte; libzstd, the device decoder and the host harness give the payloads."""
    for i, (f, p) in enumerate(zip(frames, payloads)):
        assert f == restate(p, segment), (i, len(p), segment)
        assert E.zstd_decompress(f) == p.tobytes(), i
    pays = [(p.tobytes(), {}) for p in payloads]
    check_against_host(frames, payloads.shape[1], rng, host_decode, pays)


def test_coder1_random_payloads(host_decode):
    rng = np.random.default_rng(703 + SEED)
    for case in range(60 * SCALE):
        data = coder1_payload(rng)
        seg = random_segment(rng, len(data))
        frames = device_encode(data[None], seg)
        check_coder(frames, data[None], seg, Z1.encode_frame, host_decode, rng)


def test_coder1_batches(host_decode):
    """Batches of 2-12 payloads of one length from different generators."""
    rng = np.random.default_rng(704 + SEED)
    for case in range(10 * SCALE):
        first = coder1_payload(rng)
        n = max(1, min(len(first), 100_000))
        batch = np.stack([first[:n] if len(first) >= n else np.resize(first, n)] +
                         [np.resize(coder1_payload(rng), n) for _ in range(int(rng.integers(1, 12)))])
        seg = random_segment(rng, n)
        check_coder(device_encode(batch, seg), batch, seg, Z1.encode_frame, host_decode, rng)


# ---- coder 2 ------------------------------------------------------------------------------------------------------------
def coder2_payload(rng):
    """(payload, segment) aimed at coder 2: periodic data, runs, matches of exactly 7 / 8 / 9 bytes, matches that end
    at a block or segment end, literal runs around 65,535 / 65,536 / 100,000 before a match."""
    kind = int(rng.integers(0, 6))
    r = rng.integers(0, 256, 140_000).astype(np.uint8)
    if kind == 0:
        n = int(rng.integers(1, 150_000))
        x = np.resize(r[:int(rng.integers(1, 3000))], n)
        noise = rng.random(n) < rng.choice([0, 0.002, 0.02])
        x[noise] = rng.integers(0, 256, int(noise.sum()))
        return x, random_segment(rng, n)
    if kind == 1:
        x = L.runs(int(rng.integers(1, 150_000)), int(rng.integers(0, 1 << 30)), lo=int(rng.integers(1, 10)))
        return x, random_segment(rng, len(x))
    if kind == 2:
        m = int(rng.choice([7, 8, 9]))
        parts = [r[:2000]]
        for s in rng.integers(0, 2000 - m, int(rng.integers(1, 400))):
            parts += [r[2000 + int(rng.integers(0, 130_000)):][:int(rng.integers(1, 40))], r[s:s + m]]
        return np.concatenate(parts), 0
    if kind == 3:  # every segment (and block) ends inside a match
        seg = int(rng.choice([int(rng.integers(100, 5000)), 131072]))
        x = np.resize(r[:int(rng.integers(1, 90))], seg * int(rng.integers(1, 4)))
        return x, seg if rng.random() < 0.5 else 0
    if kind == 4:
        ll = min(int(rng.choice([65534, 65535, 65536, 65537, 100_000, int(rng.integers(60_000, 131_000))])), 131_000)
        m = int(rng.integers(3, 131_072 - ll + 1)) if ll < 131_069 else 3
        return np.concatenate([r[:ll], r[:min(m, ll)]]), 0
    n = int(rng.integers(0, 20_000))
    return np.minimum(rng.geometric(0.1, n), 255).astype(np.uint8), random_segment(rng, n)


def test_coder2_random_payloads(host_decode):
    rng = np.random.default_rng(705 + SEED)
    for case in range(60 * SCALE):
        data, seg = coder2_payload(rng)
        frames = device_encode_lz(data[None], seg)
        check_coder(frames, data[None], seg, Z2.encode_frame_lz, host_decode, rng)


def test_coder2_many_blocks_in_one_call(host_decode):
    """More than 512 blocks in one call (small segments), so the candidate sort runs in several chunks."""
    rng = np.random.default_rng(706 + SEED)
    for case in range(2 * SCALE):
        n, seg = int(rng.integers(2000, 6000)), int(rng.integers(60, 300))
        count = -(-600 // Z1.n_blocks(n, seg)) + int(rng.integers(0, 8))
        batch = np.stack([np.resize(coder2_payload(rng)[0], n) if n else np.zeros(0, np.uint8) for _ in range(count)])
        assert count * Z1.n_blocks(n, seg) > 512
        check_coder(device_encode_lz(batch, seg), batch, seg, Z2.encode_frame_lz, host_decode, rng)
