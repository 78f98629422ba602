"""Restatement in numpy of coder 2, the device zstd coder with LZ matches (librir_b200/csrc/zcoder.cu, the zl_* kernels and
rirb_zstd_encode_batch_lz), byte for byte.  Coder 2 is coder 1 (oracle/zcoder.py) plus an LZ form per block; the rules
follow, and DESIGN.md section 7 f-3 states them too.  The checks against an independent decoder are in tests/test_zlz.py
(the system libzstd)."""
from __future__ import annotations

import numpy as np

from oracle.zcoder import MAGIC, _Bits, _block_header, blocks_of, encode_block

#   candidates  per block x[0..n): for p <= n-8, cand(p) = the largest q < p with x[q:q+8] == x[p:p+8], else none (a stable
#               sort of (8-byte key, position) within the block); matches never reach outside the block
#   parse       greedy: from p = 0 while p <= n-8, a candidate gives the sequence (LL = p - lit, ML = common prefix of x[p:]
#               and x[cand(p):] (overlap semantics: runs get offset 1), offset = p - cand(p)), then p += ML, lit = p;
#               no candidate: p += 1.  The bytes from lit to the end of the block are trailing literals.
#   sequences   Offset_Value = offset + 3 always (no repeat codes, no state across blocks); LL, ML and OF each in mode RLE
#               when all their codes in the block are equal, else Predefined; FSE bitstream of RFC 8878 3.1.1.3.2; the
#               initial state of each table is the first cell holding the last sequence's code
#   literals    Huffman under coder 1's rules when coder 1 would compress the literal bytes, else RLE when they are one
#               value, else raw
#   block       coder 1's RLE block if it applies; else the smaller of coder 1's form and the LZ form (the LZ form needs at
#               least one sequence; coder 1 wins a tie).  Coder 1's form is raw when neither beats the raw block.
# A frame where no block takes the LZ form is byte-identical to coder 1's.

MIN_MATCH = 8
LL_DEF = [4, 3, 2, 2, 2, 2, 2, 2, 2, 2, 2, 2, 2, 1, 1, 1, 2, 2, 2, 2, 2, 2, 2, 2, 2, 3, 2, 1, 1, 1, 1, 1, -1, -1, -1, -1]
ML_DEF = [1, 4, 3, 2, 2, 2, 2, 2, 2] + [1] * 37 + [-1] * 7
OF_DEF = [1, 1, 1, 1, 1, 1, 2, 2, 2] + [1] * 15 + [-1] * 5
LL_BASE = list(range(16)) + [16, 18, 20, 22, 24, 28, 32, 40, 48, 64] + [1 << k for k in range(7, 17)]
LL_BITS = [0] * 16 + [1, 1, 1, 1, 2, 2, 3, 3, 4, 6] + list(range(7, 17))
ML_BASE = list(range(3, 35)) + [35, 37, 39, 41, 43, 47, 51, 59, 67, 83, 99] + [(1 << k) + 3 for k in range(7, 17)]
ML_BITS = [0] * 32 + [1, 1, 1, 1, 2, 2, 3, 3, 4, 4, 5] + list(range(7, 17))


def candidates(x: np.ndarray) -> np.ndarray:
    """cand(p) for p = 0 .. n-8 (-1: none)."""
    m = len(x) - MIN_MATCH + 1
    if m <= 0:
        return np.zeros(0, np.int64)
    keys = np.zeros(m, np.uint64)
    for k in range(MIN_MATCH):
        keys |= x[k:k + m].astype(np.uint64) << np.uint64(8 * k)
    order = np.argsort(keys, kind="stable")
    sk = keys[order]
    cand = np.full(m, -1, np.int64)
    same = np.flatnonzero(sk[1:] == sk[:-1])
    cand[order[same + 1]] = order[same]
    return cand


def match_length(x: np.ndarray, p: int, q: int) -> int:
    """Common prefix of x[p:] and x[q:] (q < p)."""
    n, L, step = len(x), 0, 64
    while p + L < n:
        k = min(step, n - p - L)
        ne = np.flatnonzero(x[p + L:p + L + k] != x[q + L:q + L + k])
        if len(ne):
            return L + int(ne[0])
        L += k
        step *= 2
    return L


def parse(x: np.ndarray):
    """The greedy parse of one block: [(LL, ML, offset)], the literal bytes (uint8)."""
    cand = candidates(x)
    has = np.flatnonzero(cand >= 0)
    seqs, lits = [], []
    p = lit = 0
    while True:
        i = np.searchsorted(has, p)
        if i == len(has):
            break
        p = int(has[i])
        q = int(cand[p])
        L = match_length(x, p, q)
        seqs.append((p - lit, L, p - q))
        lits.append(x[lit:p])
        p += L
        lit = p
    lits.append(x[lit:])
    return seqs, np.concatenate(lits).astype(np.uint8)


def replay(seqs, literals: np.ndarray) -> np.ndarray:
    """What a decoder rebuilds from a block's sequences and literals (the check of the parse)."""
    out, li = [], 0
    for ll, ml, off in seqs:
        out.extend(literals[li:li + ll].tolist())
        li += ll
        for _ in range(ml):
            out.append(out[-off])
    out.extend(literals[li:].tolist())
    return np.array(out, np.uint8)


def _literal_header(kind: int, n: int) -> bytes:
    """Raw (0) or RLE (1) Literals_Section_Header (RFC 8878 3.1.1.3.1.1)."""
    if n <= 31:
        return bytes([kind | n << 3])
    if n <= 4095:
        return (kind | 1 << 2 | n << 4).to_bytes(2, "little")
    return (kind | 3 << 2 | n << 4).to_bytes(3, "little")


def literals_section(lit: np.ndarray) -> bytes:
    n = len(lit)
    c1 = encode_block(lit, False)
    if n > 0 and (c1[0] >> 1) & 3 == 2:
        return c1[3:-1]  # coder 1's compressed body without its Number_of_Sequences byte
    if n > 0 and (lit == lit[0]).all():
        return _literal_header(1, n) + bytes([int(lit[0])])
    return _literal_header(0, n) + lit.tobytes()


def _code(base: list, v: int) -> int:
    return int(np.searchsorted(np.array(base), v, side="right")) - 1


def fse_table_log(norm: list, log: int):
    """Decoding table (RFC 8878 4.1.1) with 'less than 1' (-1) probabilities: symbol, nbBits, baseline per state."""
    size = 1 << log
    sym = [0] * size
    high = size - 1
    nxt = []
    for s, c in enumerate(norm):
        if c == -1:
            sym[high] = s
            high -= 1
        nxt.append(1 if c == -1 else c)
    step = (size >> 1) + (size >> 3) + 3
    pos = 0
    for s, c in enumerate(norm):
        for _ in range(max(c, 0)):
            sym[pos] = s
            pos = (pos + step) & (size - 1)
            while pos > high:
                pos = (pos + step) & (size - 1)
    assert pos == 0
    nb = [0] * size
    base = [0] * size
    for u in range(size):
        x = nxt[sym[u]]
        nxt[sym[u]] += 1
        nb[u] = log - (x.bit_length() - 1)
        base[u] = (x << nb[u]) - size
    return sym, nb, base


_PREDEF = [(LL_DEF, 6), (OF_DEF, 5), (ML_DEF, 6)]


def sequences_section(seqs) -> bytes:
    n = len(seqs)
    llc = [_code(LL_BASE, ll) for ll, _, _ in seqs]
    mlc = [_code(ML_BASE, ml) for _, ml, _ in seqs]
    ofv = [off + 3 for _, _, off in seqs]
    ofc = [v.bit_length() - 1 for v in ofv]
    codes = [llc, ofc, mlc]  # table order LL, OF, ML
    rle = [len(set(c)) == 1 for c in codes]
    head = bytes([n]) if n < 128 else bytes([(n >> 8) + 128, n & 0xFF])
    head += bytes([rle[0] << 6 | rle[1] << 4 | rle[2] << 2])
    head += bytes(c[0] for c, r in zip(codes, rle) if r)
    tabs = [fse_table_log(norm, log) for norm, log in _PREDEF]
    state = [0, 0, 0]
    b = _Bits()

    def extra(i):
        b.put(seqs[i][0] - LL_BASE[llc[i]], LL_BITS[llc[i]])
        b.put(seqs[i][1] - ML_BASE[mlc[i]], ML_BITS[mlc[i]])
        b.put(ofv[i] - (1 << ofc[i]), ofc[i])

    for t in range(3):
        if not rle[t]:
            state[t] = tabs[t][0].index(codes[t][n - 1])
    extra(n - 1)
    for i in range(n - 2, -1, -1):
        for t in (1, 2, 0):  # OF, ML, LL
            if rle[t]:
                continue
            sym, nb, base = tabs[t]
            v = state[t]
            u = next(u for u in range(len(sym)) if sym[u] == codes[t][i] and base[u] <= v < base[u] + (1 << nb[u]))
            b.put(v - base[u], nb[u])
            state[t] = u
        extra(i)
    for t, log in ((2, 6), (1, 5), (0, 6)):  # ML, OF, LL
        if not rle[t]:
            b.put(state[t], log)
    return head + b.close()


def encode_block_lz(data: np.ndarray, last: bool) -> bytes:
    c1 = encode_block(data, last)
    if (c1[0] >> 1) & 3 == 1:
        return c1
    seqs, lits = parse(data)
    if not seqs:
        return c1
    body = literals_section(lits) + sequences_section(seqs)
    return _block_header(last, 2, len(body)) + body if 3 + len(body) < len(c1) else c1


def encode_frame_lz(payload, segment: int = 0) -> bytes:
    """Coder 2's frame for `payload`: coder 1's frame header and block cuts, each block by encode_block_lz."""
    data = np.frombuffer(bytes(payload), np.uint8) if not isinstance(payload, np.ndarray) else np.ascontiguousarray(payload).reshape(-1).view(np.uint8)
    n = len(data)
    out = [MAGIC, bytes([0xA0]), n.to_bytes(4, "little")]
    blocks = blocks_of(n, segment) or [(0, 0)]
    for i, (a, ln) in enumerate(blocks):
        out.append(encode_block_lz(data[a:a + ln], i == len(blocks) - 1))
    return b"".join(out)
