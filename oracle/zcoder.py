"""Restatement in numpy of the device zstd coder (librir_b200/csrc/zcoder.cu), byte for byte.

The coder writes one zstd frame (RFC 8878) per payload using a small subset of the format:
  frame header   magic, Frame_Header_Descriptor 0xA0 (Single_Segment_Flag, 4-byte Frame_Content_Size), no checksum
  blocks         at most 128 KiB, never across a segment boundary; per block the first that applies of
                 RLE (all bytes equal), compressed (Huffman literals + zero sequences, if smaller than raw), raw
  literals       Huffman code lengths <= 11 bits, weights in direct 4-bit form when the largest symbol is <= 128,
                 else FSE-compressed (accuracy log 6); one stream up to 1023 literals, four streams with a jump table above

Tie-breaks (DESIGN.md section 7 f-3 states them too; the kernel does the same):
  1. symbols present are sorted by (count, symbol) ascending;
  2. Huffman merges take the smaller weight of the front of the leaf queue and the front of the node queue, the leaf when
     the weights are equal;
  3. depths above 11 are cut with the JPEG (ITU T.81 K.3) adjustment of the per-length counts, then lengths are handed out
     longest first along the order of rule 1;
  4. canonical codes: longest length first, symbols of one length in ascending order, codes counting up from 0;
  5. FSE weights: each weight value present gets max(1, count * 64 // n) slots; while the sum is above 64 the value with the
     most slots (smallest value on a tie) gives one up, while below the value with the highest count (smallest value on a
     tie) takes one; the two last weights are the states' initial symbols, each in the first table cell holding it.
The checks against an independent decoder are in tests/test_zcoder.py (the system libzstd).
"""
from __future__ import annotations

import numpy as np

BLOCK = 128 * 1024
MAX_BITS = 11
FSE_LOG = 6
MAGIC = b"\x28\xb5\x2f\xfd"


def frame_bound(nbytes: int, segment: int = 0) -> int:
    """Largest frame the coder can write for a payload of `nbytes`: raw blocks plus headers."""
    return 9 + 3 * max(1, n_blocks(nbytes, segment)) + nbytes


def blocks_of(nbytes: int, segment: int = 0):
    """(offset, length) of the blocks of a payload cut into segments of `segment` bytes (0: one segment)."""
    seg = nbytes if segment <= 0 else segment
    out = []
    for s0 in range(0, nbytes, max(seg, 1)):
        s1 = min(nbytes, s0 + seg)
        out += [(b, min(BLOCK, s1 - b)) for b in range(s0, s1, BLOCK)]
    return out


def n_blocks(nbytes: int, segment: int = 0) -> int:
    return len(blocks_of(nbytes, segment))


def code_lengths(counts: np.ndarray) -> np.ndarray:
    """Length-limited Huffman code lengths (rules 1-3) for a histogram with >= 2 symbols present."""
    syms = [s for s in range(256) if counts[s] > 0]
    order = sorted(syms, key=lambda s: (int(counts[s]), s))
    n = len(order)
    leaf_w = [int(counts[s]) for s in order]
    node_w, kids = [], []  # internal nodes in creation order; children: ("l", i) or ("n", j)
    li = ni = 0
    for _ in range(n - 1):
        pick = []
        for _k in range(2):
            if li < n and (ni >= len(node_w) or leaf_w[li] <= node_w[ni]):
                pick.append(("l", li, leaf_w[li]))
                li += 1
            else:
                pick.append(("n", ni, node_w[ni]))
                ni += 1
        node_w.append(pick[0][2] + pick[1][2])
        kids.append((pick[0][:2], pick[1][:2]))
    ndepth = [0] * (n - 1)
    depth = [0] * n
    for j in range(n - 2, -1, -1):
        for kind, i in kids[j]:
            if kind == "l":
                depth[i] = ndepth[j] + 1
            else:
                ndepth[i] = ndepth[j] + 1
    maxd = max(depth)
    bl = [0] * (max(maxd, MAX_BITS) + 2)
    for d in depth:
        bl[d] += 1
    for i in range(maxd, MAX_BITS, -1):
        while bl[i] > 0:
            j = i - 2
            while bl[j] == 0:
                j -= 1
            bl[i] -= 2
            bl[i - 1] += 1
            bl[j + 1] += 2
            bl[j] -= 1
    lens = np.zeros(256, np.int64)
    k = 0
    for ln in range(min(maxd, MAX_BITS), 0, -1):
        for _ in range(bl[ln]):
            lens[order[k]] = ln
            k += 1
    return lens


def canonical_codes(lens: np.ndarray) -> np.ndarray:
    """Rule 4 (RFC 8878 4.2.1.3: lowest weight first, natural order within a weight)."""
    maxb = int(lens.max())
    start = [0] * (maxb + 2)
    val = 0
    for ln in range(maxb, 0, -1):
        start[ln] = val
        val = (val + int((lens == ln).sum())) >> 1
    codes = np.zeros(256, np.int64)
    for s in range(256):
        if lens[s]:
            codes[s] = start[lens[s]]
            start[lens[s]] += 1
    return codes


class _Bits:
    """Forward little-endian bit writer."""

    def __init__(self):
        self.v = 0
        self.n = 0

    def put(self, value: int, nbits: int):
        self.v |= (value & ((1 << nbits) - 1)) << self.n
        self.n += nbits

    def close(self) -> bytes:  # end mark, then zero padding to a byte
        self.put(1, 1)
        return self.v.to_bytes((self.n + 7) // 8, "little")


def fse_normalize(w: np.ndarray) -> list:
    """Rule 5: slots out of 64 for each weight value 0..max(w)."""
    top = int(w.max())
    cnt = [int((w == v).sum()) for v in range(top + 1)]
    n = len(w)
    norm = [max(1, c * 64 // n) if c else 0 for c in cnt]
    while sum(norm) > 64:
        v = max(range(top + 1), key=lambda v: (norm[v], -v))
        norm[v] -= 1
    while sum(norm) < 64:
        v = max(range(top + 1), key=lambda v: (cnt[v], -v))
        norm[v] += 1
    return norm


def fse_ncount(norm: list) -> bytes:
    """FSE table description (RFC 8878 4.1.1), accuracy log 6, no 'less than 1' probabilities."""
    b = _Bits()
    b.put(FSE_LOG - 5, 4)
    remaining = (1 << FSE_LOG) + 1
    threshold = 1 << FSE_LOG
    nbits = FSE_LOG + 1
    s = 0
    prev0 = False
    top = len(norm)
    while s < top and remaining > 1:
        if prev0:
            start = s
            while norm[s] == 0:
                s += 1
            while s >= start + 3:
                start += 3
                b.put(3, 2)
            b.put(s - start, 2)
        count = norm[s]
        s += 1
        mx = (2 * threshold - 1) - remaining
        remaining -= count
        v = count + 1
        if v >= threshold:
            v += mx
        b.put(v, nbits - 1 if v < mx else nbits)
        prev0 = v == 1
        while remaining < threshold:
            nbits -= 1
            threshold >>= 1
    assert remaining == 1
    return b.v.to_bytes((b.n + 7) // 8, "little")


def fse_table(norm: list):
    """Decoding table (RFC 8878 4.1.1): symbol, nbBits, baseline per state."""
    size = 1 << FSE_LOG
    sym = [0] * size
    step = (size >> 1) + (size >> 3) + 3
    pos = 0
    for s, c in enumerate(norm):
        for _ in range(c):
            sym[pos] = s
            pos = (pos + step) & (size - 1)
    assert pos == 0
    nxt = list(norm)
    nb = [0] * size
    base = [0] * size
    for u in range(size):
        x = nxt[sym[u]]
        nxt[sym[u]] += 1
        nb[u] = FSE_LOG - (x.bit_length() - 1)
        base[u] = (x << nb[u]) - size
    return sym, nb, base


def fse_weights(w: np.ndarray):
    """FSE-compressed weights (RFC 8878 4.2.1.2), or None when they cannot be written (one weight value, >= 128 bytes)."""
    if len(set(w.tolist())) < 2:
        return None
    norm = fse_normalize(w)
    head = fse_ncount(norm)
    sym, nb, base = fse_table(norm)
    n = len(w)

    def first_state(x):
        return sym.index(x)

    def encode(x, v):  # the state holding x whose transition reaches v, and the bits that select v
        for u in range(64):
            if sym[u] == x and base[u] <= v < base[u] + (1 << nb[u]):
                return u, v - base[u], nb[u]
        raise AssertionError

    # state of each of the two interleaved chains; decoding reads bits in the reverse of the order written here
    state = [None, None]
    state[(n - 1) & 1] = first_state(int(w[n - 1]))
    state[(n - 2) & 1] = first_state(int(w[n - 2]))
    b = _Bits()
    for k in range(n - 3, -1, -1):
        u, val, bits = encode(int(w[k]), state[k & 1])
        b.put(val, bits)
        state[k & 1] = u
    b.put(state[1], FSE_LOG)
    b.put(state[0], FSE_LOG)
    body = head + b.close()
    return body if len(body) < 128 else None


def tree_description(lens: np.ndarray):
    """Huffman_Tree_Description bytes, or None when the weights cannot be written."""
    maxb = int(lens.max())
    last = int(np.nonzero(lens)[0].max())
    w = np.where(lens[:last] > 0, maxb + 1 - lens[:last], 0).astype(np.int64)
    if last <= 128:
        pad = np.concatenate([w, [0]]) if last & 1 else w
        return bytes([127 + last]) + bytes((pad[0::2] << 4 | pad[1::2]).astype(np.uint8).tolist())
    body = fse_weights(w)
    return None if body is None else bytes([len(body)]) + body


def huff_stream(lit: np.ndarray, lens: np.ndarray, codes: np.ndarray) -> bytes:
    """One Huffman stream: the last literal first, so that a decoder reading backward meets the first one first."""
    r = lit[::-1].astype(np.int64)
    ln = lens[r]
    cd = codes[r]
    pos = np.concatenate([[0], np.cumsum(ln)[:-1]])
    total = int(ln.sum())
    bits = np.zeros(total + 1, np.uint8)
    for k in range(MAX_BITS):
        m = ln > k
        bits[pos[m] + k] = (cd[m] >> k) & 1
    bits[total] = 1
    return np.packbits(bits, bitorder="little").tobytes()


def _block_header(last: bool, btype: int, size: int) -> bytes:
    return (int(last) | btype << 1 | size << 3).to_bytes(3, "little")


def encode_block(data: np.ndarray, last: bool) -> bytes:
    n = len(data)
    counts = np.bincount(data, minlength=256)
    if n > 0 and (counts > 0).sum() == 1:
        return _block_header(last, 1, n) + bytes([int(data[0])])
    raw = _block_header(last, 0, n) + data.tobytes()
    if n == 0:
        return raw
    lens = code_lengths(counts)
    tree = tree_description(lens)
    if tree is None:
        return raw
    codes = canonical_codes(lens)
    if n <= 1023:
        streams = huff_stream(data, lens, codes)
        csize = len(tree) + len(streams)
        if csize >= n:
            return raw
        lh = (2 | 0 << 2 | n << 4 | csize << 14).to_bytes(3, "little")
    else:
        seg = (n + 3) // 4
        parts = [huff_stream(data[i * seg:min(n, (i + 1) * seg)], lens, codes) for i in range(4)]
        if max(len(p) for p in parts[:3]) > 0xFFFF:
            return raw
        jump = b"".join(len(p).to_bytes(2, "little") for p in parts[:3])
        streams = jump + b"".join(parts)
        csize = len(tree) + len(streams)
        if csize >= n:
            return raw
        if max(n, csize) <= 16383:
            lh = (2 | 2 << 2 | n << 4 | csize << 18).to_bytes(4, "little")
        else:
            lh = (2 | 3 << 2 | n << 4 | csize << 22).to_bytes(5, "little")
    body = lh + tree + streams + b"\x00"
    if len(body) >= n:
        return raw
    return _block_header(last, 2, len(body)) + body


def encode_frame(payload, segment: int = 0) -> bytes:
    """One zstd frame for `payload` (bytes-like or uint8 array), blocks cut at multiples of `segment` bytes (0: none)."""
    data = np.frombuffer(bytes(payload), np.uint8) if not isinstance(payload, np.ndarray) else np.ascontiguousarray(payload).reshape(-1).view(np.uint8)
    n = len(data)
    out = [MAGIC, bytes([0xA0]), n.to_bytes(4, "little")]
    blocks = blocks_of(n, segment) or [(0, 0)]
    for i, (a, ln) in enumerate(blocks):
        out.append(encode_block(data[a:a + ln], i == len(blocks) - 1))
    return b"".join(out)
