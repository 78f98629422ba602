// librir_b200/csrc/zdecoder.cu -- the device zstd decoder: standalone zstd frames (RFC 8878) in HBM -> their content in HBM.
//
// Coverage: every single frame without a dictionary -- both header forms, content sizes of 0/1/2/4/8 bytes, raw / RLE /
// compressed blocks, raw / RLE / Huffman / treeless literals in 1 or 4 streams, Huffman weights as nibbles or FSE-coded,
// code lengths up to 11 bits, all three sequence-count forms and the predefined / RLE / FSE / repeat table modes of LL, OF
// and ML, repeat offsets, overlapping matches and matches into earlier blocks of the frame.  A frame with a dictionary
// ID or a content checksum, a skippable frame and bytes after the last block are refused (status -2): the host decodes
// those.  Every byte is untrusted: no read leaves [offset, offset + size) of its frame, no write leaves its dst slot, and
// what RFC 8878 and libzstd check is checked (status -1 for that frame only).
//
// Three launches per batch:
//   zd_scan_kernel      one thread per frame: frame header, every block header, literals and sequence-count headers;
//                       whether the frame has sequences at all
//   zd_literals_kernel  ZD_LIT_CTAS warps per frame, each takes every ZD_LIT_CTAS-th Huffman literals section of its
//                       frame: table from the section (or, treeless, from the last one before it that has a table),
//                       then one lane per stream.  Output to the frame's literal scratch, or straight into dst for a
//                       frame without sequences (every frame of the device coder)
//   zd_frames_kernel    one warp per frame, blocks in order: lane 0 builds the FSE tables and decodes sequences in runs
//                       of 32, the warp copies literals and matches (match byte k = out[start - off + k % off], so an
//                       overlapping match needs no serial pass)
// The per-frame bodies are __host__ __device__ so that the same code can be exercised without a device.
#include "../../include/librir_b200.h"
#include "common.cuh"
#include "kernels.h"

namespace rirb {

namespace {

#ifdef __CUDA_ARCH__
#define ZD_WIDTH 32
#else
#define ZD_WIDTH 1
#endif

__host__ __device__ inline int zd_lane()
{
#ifdef __CUDA_ARCH__
    return threadIdx.x & 31;
#else
    return 0;
#endif
}
__host__ __device__ inline void zd_sync()
{
#ifdef __CUDA_ARCH__
    __syncwarp();
#endif
}
__host__ __device__ inline int zd_highbit(unsigned long long v)  // v > 0
{
#ifdef __CUDA_ARCH__
    return 63 - __clzll((long long)v);
#else
    return 63 - __builtin_clzll(v);
#endif
}

constexpr unsigned ZD_BLOCK_MAX = 128 * 1024;
constexpr int ZD_HUF_LOG = 11;
constexpr int ZD_LIT_CTAS = 8;  // warps per frame in zd_literals_kernel (a 640x512 record is 5 blocks)
constexpr int ZD_SEQ_RUN = 32;  // sequences decoded by lane 0 before the warp executes them

// predefined distributions and code tables (RFC 8878 3.1.1.3.2.2 and 3.1.1.3.2.1.1)
#define ZD_LL_DEF 4, 3, 2, 2, 2, 2, 2, 2, 2, 2, 2, 2, 2, 1, 1, 1, 2, 2, 2, 2, 2, 2, 2, 2, 2, 3, 2, 1, 1, 1, 1, 1, -1, -1, -1, -1
#define ZD_ML_DEF                                                                                                              \
    1, 4, 3, 2, 2, 2, 2, 2, 2, 1, 1, 1, 1, 1, 1, 1, 1, 1, 1, 1, 1, 1, 1, 1, 1, 1, 1, 1, 1, 1, 1, 1, 1, 1, 1, 1, 1, 1, 1, 1, 1, \
        1, 1, 1, 1, 1, -1, -1, -1, -1, -1, -1, -1
#define ZD_OF_DEF 1, 1, 1, 1, 1, 1, 2, 2, 2, 1, 1, 1, 1, 1, 1, 1, 1, 1, 1, 1, 1, 1, 1, 1, -1, -1, -1, -1, -1
#define ZD_LL_BASE                                                                                                             \
    0, 1, 2, 3, 4, 5, 6, 7, 8, 9, 10, 11, 12, 13, 14, 15, 16, 18, 20, 22, 24, 28, 32, 40, 48, 64, 0x80, 0x100, 0x200, 0x400,    \
        0x800, 0x1000, 0x2000, 0x4000, 0x8000, 0x10000
#define ZD_LL_BITS 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 1, 1, 1, 1, 2, 2, 3, 3, 4, 6, 7, 8, 9, 10, 11, 12, 13, 14, 15, 16
#define ZD_ML_BASE                                                                                                             \
    3, 4, 5, 6, 7, 8, 9, 10, 11, 12, 13, 14, 15, 16, 17, 18, 19, 20, 21, 22, 23, 24, 25, 26, 27, 28, 29, 30, 31, 32, 33, 34, 35, \
        37, 39, 41, 43, 47, 51, 59, 67, 83, 99, 0x83, 0x103, 0x203, 0x403, 0x803, 0x1003, 0x2003, 0x4003, 0x8003, 0x10003
#define ZD_ML_BITS                                                                                                             \
    0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 1, 1, 1, 1, 2, 2, 3, 3, 4, 4, \
        5, 7, 8, 9, 10, 11, 12, 13, 14, 15, 16

__constant__ short d_def[3][53] = {{ZD_LL_DEF}, {ZD_OF_DEF}, {ZD_ML_DEF}};
__constant__ unsigned d_ll_base[36] = {ZD_LL_BASE};
__constant__ unsigned char d_ll_bits[36] = {ZD_LL_BITS};
__constant__ unsigned d_ml_base[53] = {ZD_ML_BASE};
__constant__ unsigned char d_ml_bits[53] = {ZD_ML_BITS};
#ifndef __CUDA_ARCH__
const short h_def[3][53] = {{ZD_LL_DEF}, {ZD_OF_DEF}, {ZD_ML_DEF}};
const unsigned h_ll_base[36] = {ZD_LL_BASE};
const unsigned char h_ll_bits[36] = {ZD_LL_BITS};
const unsigned h_ml_base[53] = {ZD_ML_BASE};
const unsigned char h_ml_bits[53] = {ZD_ML_BITS};
#endif
#ifdef __CUDA_ARCH__
#define ZD_TAB(name) d_##name
#else
#define ZD_TAB(name) h_##name
#endif

// the table kinds, in the order of the Symbol_Compression_Modes fields: LL, OF, ML
__host__ __device__ constexpr int zd_max_sym(int kind) { return kind == 0 ? 35 : kind == 1 ? 31 : 52; }
__host__ __device__ constexpr int zd_max_log(int kind) { return kind == 1 ? 8 : 9; }
__host__ __device__ constexpr int zd_def_log(int kind) { return kind == 1 ? 5 : 6; }
__host__ __device__ constexpr int zd_def_nsym(int kind) { return kind == 0 ? 36 : kind == 1 ? 29 : 53; }

// ---- bounded reads ---------------------------------------------------------------------------------------------------
// 8 bytes at b[i..i+8) little-endian, bytes outside [0, len) read as 0 and never touched
__host__ __device__ inline unsigned long long zd_load8(const u8* b, long long len, long long i)
{
#ifdef __CUDA_ARCH__
    const uintptr_t a = reinterpret_cast<uintptr_t>(b + i) & ~(uintptr_t)7;
    if (i >= 0 && (const u8*)a >= b && (const u8*)a + 16 <= b + len) {
        const unsigned long long lo = *(const unsigned long long*)a, hi = *(const unsigned long long*)(a + 8);
        const int sh = (int)((reinterpret_cast<uintptr_t>(b + i) & 7) * 8);
        return sh ? (lo >> sh) | (hi << (64 - sh)) : lo;
    }
#endif
    unsigned long long v = 0;
    for (int k = 0; k < 8; ++k)
        if (i + k >= 0 && i + k < len) v |= (unsigned long long)b[i + k] << (8 * k);
    return v;
}

// Backward bitstream (Huffman streams, FSE weights, sequences): bits [0, pos) are unread; reads past the start give
// zeros and make pos negative (an overflow the callers reject).
struct ZdBits {
    const u8* b;
    long long len, pos, cb;  // container = bytes [cb, cb + 8)
    unsigned long long c;
};
__host__ __device__ inline bool zd_bits_init(ZdBits& s, const u8* b, long long len)
{
    s.b = b;
    s.len = len;
    if (len <= 0 || b[len - 1] == 0) return false;  // the last byte holds the end mark
    s.pos = 8 * (len - 1) + zd_highbit(b[len - 1]);
    s.cb = -1000;
    s.c = 0;
    return true;
}
__host__ __device__ inline unsigned zd_peek(ZdBits& s, int n)  // n <= 32
{
    if (n == 0) return 0;
    const long long lo = s.pos - n;  // may be negative: the container then holds zeros below the start
    if (lo < s.cb * 8 || s.pos > s.cb * 8 + 64) {
        s.cb = ((s.pos + 7) >> 3) - 8;
        s.c = zd_load8(s.b, s.len, s.cb);
    }
    return (unsigned)((s.c >> (lo - s.cb * 8)) & ((1ull << n) - 1));
}
__host__ __device__ inline unsigned zd_read(ZdBits& s, int n)
{
    const unsigned v = zd_peek(s, n);
    s.pos -= n;
    return v;
}

// ---- FSE tables -------------------------------------------------------------------------------------------------------
struct ZdFse {
    unsigned short base;
    unsigned char sym, nb;
};

// normalised counts (RFC 8878 4.1.1) at f[pos..end) -> norm[0..*nsym), *log; returns bytes used or -1
__host__ __device__ inline long long zd_read_ncount(const u8* f, long long pos, long long end, int max_log, int max_sym, short* norm,
                                                    int* nsym, int* log)
{
    const long long len = end - pos;
    if (len <= 0) return -1;
    long long bit = 0;
    auto bits = [&](int n) -> unsigned {
        const unsigned long long w = zd_load8(f + pos, len, bit >> 3);
        return (unsigned)((w >> (bit & 7)) & ((1ull << n) - 1));
    };
    const int al = (int)bits(4) + 5;
    bit += 4;
    if (al > max_log) return -1;
    int remaining = 1 << al, s = 0;
    while (remaining > 0 && s <= max_sym) {
        const int nb = zd_highbit((unsigned)remaining + 1) + 1;
        unsigned val = bits(nb);
        const unsigned lower_mask = (1u << (nb - 1)) - 1;
        const unsigned threshold = (1u << nb) - 1 - ((unsigned)remaining + 1);
        if ((val & lower_mask) < threshold) {
            val &= lower_mask;
            bit += nb - 1;
        } else {
            if (val > lower_mask) val -= threshold;
            bit += nb;
        }
        const int p = (int)val - 1;
        remaining -= p < 0 ? -p : p;
        norm[s++] = (short)p;
        if (p == 0) {
            for (;;) {
                const int rep = (int)bits(2);
                bit += 2;
                for (int k = 0; k < rep; ++k) {
                    if (s > max_sym) return -1;
                    norm[s++] = 0;
                }
                if (rep != 3) break;
            }
        }
        if (bit > 8 * len) return -1;
    }
    if (remaining != 0 || bit > 8 * len) return -1;
    *nsym = s;
    *log = al;
    return (bit + 7) >> 3;
}

// decoding table of 1 << log cells; state_desc: 256 scratch words; false if the counts do not fill the table
__host__ __device__ inline bool zd_fse_build(ZdFse* t, const short* norm, int nsym, int log, unsigned short* state_desc)
{
    const int size = 1 << log;
    int high = size;
    for (int s = 0; s < nsym; ++s)
        if (norm[s] == -1) {
            if (high <= 0) return false;
            t[--high].sym = (unsigned char)s;
            state_desc[s] = 1;
        }
    const int step = (size >> 1) + (size >> 3) + 3, mask = size - 1;
    int pos = 0;
    for (int s = 0; s < nsym; ++s) {
        if (norm[s] <= 0) continue;
        state_desc[s] = (unsigned short)norm[s];
        for (int i = 0; i < norm[s]; ++i) {
            t[pos].sym = (unsigned char)s;
            do {
                pos = (pos + step) & mask;
            } while (pos >= high);
        }
    }
    if (pos != 0) return false;
    for (int i = 0; i < size; ++i) {
        const unsigned next = state_desc[t[i].sym]++;
        const int nb = log - zd_highbit(next);
        t[i].nb = (unsigned char)nb;
        t[i].base = (unsigned short)((next << nb) - size);
    }
    return true;
}

// ---- literals -----------------------------------------------------------------------------------------------------------
struct ZdLit {
    int type, streams;
    unsigned hsize, regen, csize;  // header bytes, regenerated bytes, bytes after the header
};
// literals section header at f[pos..end)
__host__ __device__ inline bool zd_lit_header(const u8* f, long long pos, long long end, ZdLit& L)
{
    if (pos >= end) return false;
    const unsigned b0 = f[pos];
    L.type = b0 & 3;
    const int sf = (b0 >> 2) & 3;
    auto byte = [&](int k) -> unsigned { return pos + k < end ? f[pos + k] : 0u; };
    if (L.type < 2) {
        L.streams = 1;
        if ((sf & 1) == 0) {
            L.hsize = 1;
            L.regen = b0 >> 3;
        } else if (sf == 1) {
            L.hsize = 2;
            L.regen = (b0 >> 4) + (byte(1) << 4);
        } else {
            L.hsize = 3;
            L.regen = (b0 >> 4) + (byte(1) << 4) + (byte(2) << 12);
        }
        L.csize = L.type == 0 ? L.regen : 1;
    } else {
        L.streams = sf == 0 ? 1 : 4;
        const unsigned long long h = (unsigned long long)b0 | (byte(1) << 8) | (byte(2) << 16) | ((unsigned long long)byte(3) << 24) |
                                     ((unsigned long long)byte(4) << 32);
        if (sf < 2) {
            L.hsize = 3;
            L.regen = (unsigned)(h >> 4) & 0x3FF;
            L.csize = (unsigned)(h >> 14) & 0x3FF;
        } else if (sf == 2) {
            L.hsize = 4;
            L.regen = (unsigned)(h >> 4) & 0x3FFF;
            L.csize = (unsigned)(h >> 18) & 0x3FFF;
        } else {
            L.hsize = 5;
            L.regen = (unsigned)(h >> 4) & 0x3FFFF;
            L.csize = (unsigned)(h >> 22) & 0x3FFFF;
        }
        if (L.streams == 4 && L.regen < 6) return false;
    }
    return pos + L.hsize + L.csize <= end;
}

// Huffman table description at f[pos..end) -> weights w[0..nsym); returns its bytes or -1
__host__ __device__ inline long long zd_huf_weights(const u8* f, long long pos, long long end, u8* w, int* nsym, short* norm, ZdFse* ft,
                                                    unsigned short* sd)
{
    if (pos >= end) return -1;
    const unsigned hb = f[pos];
    int nw = 0;
    long long used;
    if (hb >= 128) {
        nw = (int)hb - 127;
        used = 1 + (nw + 1) / 2;
        if (pos + used > end) return -1;
        for (int i = 0; i < nw; ++i) {
            const unsigned b = f[pos + 1 + i / 2];
            w[i] = (u8)((i & 1) ? (b & 15) : (b >> 4));
        }
    } else {
        if (hb == 0 || pos + 1 + hb > end) return -1;
        used = 1 + hb;
        int ns = 0, log = 0;
        const long long nc = zd_read_ncount(f, pos + 1, pos + 1 + hb, 6, 255, norm, &ns, &log);
        if (nc < 0 || nc >= hb || !zd_fse_build(ft, norm, ns, log, sd)) return -1;
        ZdBits s;
        if (!zd_bits_init(s, f + pos + 1 + nc, hb - nc)) return -1;
        unsigned s1 = zd_read(s, log), s2 = zd_read(s, log);
        if (s.pos < 0) return -1;
        // two interleaved states; the stream ends when a read goes past its start (same limits as libzstd: at most
        // 255 weights, the last one from the other state)
        for (;;) {
            if (nw > 253) return -1;
            w[nw++] = ft[s1].sym;
            s1 = ft[s1].base + zd_read(s, ft[s1].nb);
            if (s.pos < 0) {
                w[nw++] = ft[s2].sym;
                break;
            }
            if (nw > 253) return -1;
            w[nw++] = ft[s2].sym;
            s2 = ft[s2].base + zd_read(s, ft[s2].nb);
            if (s.pos < 0) {
                w[nw++] = ft[s1].sym;
                break;
            }
        }
    }
    // the last weight is implied: the total has to reach the next power of two
    unsigned total = 0;
    for (int i = 0; i < nw; ++i) {
        if (w[i] > ZD_HUF_LOG) return -1;
        if (w[i]) total += 1u << (w[i] - 1);
    }
    if (total == 0) return -1;
    const int log = zd_highbit(total) + 1;
    if (log > ZD_HUF_LOG) return -1;
    const unsigned rest = (1u << log) - total;
    if (rest & (rest - 1)) return -1;
    w[nw] = (u8)(zd_highbit(rest) + 1);
    int ones = 0;
    for (int i = 0; i <= nw; ++i) ones += w[i] == 1;
    if (ones < 2 || (ones & 1)) return -1;
    *nsym = nw + 1;
    return used;
}

// Shared work space of one Huffman literals section
struct ZdHufSmem {
    unsigned short table[1 << ZD_HUF_LOG];  // symbol | bits << 8
    unsigned short start[256];
    u8 w[256];
    short norm[256];
    unsigned short sd[256];
    ZdFse ft[64];
    int log, nsym, ok;
};

// one stream of count symbols from f[s0..s1) into out
__host__ __device__ inline bool zd_huf_stream(const u8* b, long long len, const unsigned short* table, int log, u8* out, unsigned count)
{
    ZdBits s;
    if (!zd_bits_init(s, b, len)) return false;
    for (unsigned k = 0; k < count; ++k) {
        const unsigned e = table[zd_peek(s, log)];
        s.pos -= e >> 8;
        out[k] = (u8)e;
        if (s.pos < 0) return false;
    }
    return s.pos == 0;
}

// Decodes the Huffman literals section at f[lit..) (whose table is described at f[tree..)) into out, by the calling warp
// (or one host thread).  Returns false for a malformed section.  All lanes return the same value.
__host__ __device__ inline bool zd_huf_section(const u8* f, long long fsize, long long lit, long long tree, u8* out, ZdHufSmem& sm)
{
    const int lane = zd_lane();
    ZdLit L, T;
    const bool okL = zd_lit_header(f, lit, fsize, L) && zd_lit_header(f, tree, fsize, T) && T.type == 2;
    long long tsize = 0;
    if (lane == 0) {
        sm.ok = 0;
        if (okL) {
            tsize = zd_huf_weights(f, tree + T.hsize, tree + T.hsize + T.csize, sm.w, &sm.nsym, sm.norm, sm.ft, sm.sd);
            if (tsize >= 0) {
                unsigned total = 0;
                for (int i = 0; i < sm.nsym; ++i)
                    if (sm.w[i]) total += 1u << (sm.w[i] - 1);
                sm.log = zd_highbit(total);
                unsigned rank[ZD_HUF_LOG + 2] = {0};
                for (int i = 0; i < sm.nsym; ++i)
                    if (sm.w[i]) rank[sm.w[i]] += 1u << (sm.w[i] - 1);
                unsigned next[ZD_HUF_LOG + 2], acc = 0;
                for (int wv = 1; wv <= ZD_HUF_LOG + 1; ++wv) {
                    next[wv] = acc;
                    acc += rank[wv];
                }
                for (int i = 0; i < sm.nsym; ++i)
                    if (sm.w[i]) {
                        sm.start[i] = (unsigned short)next[sm.w[i]];
                        next[sm.w[i]] += 1u << (sm.w[i] - 1);
                    }
                sm.ok = 1;
            }
        }
    }
    zd_sync();
    if (!sm.ok) return false;
    for (int i = lane; i < sm.nsym; i += ZD_WIDTH) {
        const int wv = sm.w[i];
        if (!wv) continue;
        const unsigned short e = (unsigned short)(i | ((sm.log + 1 - wv) << 8));
        for (unsigned k = 0; k < (1u << (wv - 1)); ++k) sm.table[sm.start[i] + k] = e;
    }
    zd_sync();
    // the streams: after the table description (compressed literals) or right after the header (treeless)
    const u8* st = f + lit + L.hsize;
    long long slen = L.csize;
    if (L.type == 2) {
        // the tree of this very section: tsize was computed by lane 0 only; recompute cheaply from the header byte
        const unsigned hb = f[lit + L.hsize];
        const long long ts = hb >= 128 ? 1 + ((long long)hb - 127 + 1) / 2 : 1 + (long long)hb;
        st += ts;
        slen -= ts;
        if (slen <= 0) return false;
    }
    bool ok = true;
    if (L.streams == 1) {
        if (lane == 0) ok = zd_huf_stream(st, slen, sm.table, sm.log, out, L.regen);
    } else {
        if (slen < 6) return false;
        const long long l1 = st[0] | (st[1] << 8), l2 = st[2] | (st[3] << 8), l3 = st[4] | (st[5] << 8);
        const long long l4 = slen - 6 - l1 - l2 - l3;
        const unsigned seg = (L.regen + 3) / 4;
        if (l4 < 0 || 3 * seg > L.regen) return false;
        if (lane < 4) {
            const long long off[4] = {6, 6 + l1, 6 + l1 + l2, 6 + l1 + l2 + l3};
            const long long len[4] = {l1, l2, l3, l4};
            for (int k = lane; k < 4; k += ZD_WIDTH)
                ok = ok && zd_huf_stream(st + off[k], len[k], sm.table, sm.log, out + (size_t)k * seg, k < 3 ? seg : L.regen - 3 * seg);
        }
    }
#ifdef __CUDA_ARCH__
    ok = __all_sync(0xFFFFFFFFu, ok);
#endif
    return ok;
}

// ---- frames ------------------------------------------------------------------------------------------------------------
struct ZdFrame {
    long long data;  // offset of the first block header
    long long fcs;   // content size, -1 when the header has none
    unsigned bmax;   // Block_Maximum_Size
    int has_seq;     // some block has sequences
    int err;         // 0, -1 (malformed), -2 (refused)
};

// zd_scan_kernel's body: the frame header and every block header of one frame
__host__ __device__ inline void zd_scan_frame(const u8* f, long long size, long long cap, ZdFrame& fr)
{
    fr.err = -1;
    fr.has_seq = 0;
    if (size < 4) return;
    const unsigned magic = f[0] | (f[1] << 8) | (f[2] << 16) | ((unsigned)f[3] << 24);
    if ((magic & 0xFFFFFFF0u) == 0x184D2A50u) {
        fr.err = -2;
        return;
    }
    if (magic != 0xFD2FB528u || size < 5) return;
    const unsigned fhd = f[4];
    const int fcs_flag = fhd >> 6, single = (fhd >> 5) & 1, checksum = (fhd >> 2) & 1, dict = fhd & 3;
    if (fhd & 8) return;  // reserved bit
    long long pos = 5;
    unsigned long long window = 0;
    if (!single) {
        if (pos >= size) return;
        const unsigned wd = f[pos++];
        const int wlog = 10 + (wd >> 3);
        if (wlog > 31) return;
        window = (1ull << wlog) + ((1ull << wlog) >> 3) * (wd & 7);
    }
    pos += dict == 0 ? 0 : dict == 1 ? 1 : dict == 2 ? 2 : 4;
    const int fcs_bytes = fcs_flag == 0 ? (single ? 1 : 0) : fcs_flag == 1 ? 2 : fcs_flag == 2 ? 4 : 8;
    if (pos + fcs_bytes > size) return;
    if (dict || checksum) {
        fr.err = -2;
        return;
    }
    long long fcs = -1;
    if (fcs_bytes) {
        unsigned long long v = 0;
        for (int k = 0; k < fcs_bytes; ++k) v |= (unsigned long long)f[pos + k] << (8 * k);
        if (fcs_bytes == 2) v += 256;
        if (v > (unsigned long long)cap) return;
        fcs = (long long)v;
    }
    pos += fcs_bytes;
    if (single) window = (unsigned long long)fcs;
    fr.fcs = fcs;
    fr.data = pos;
    fr.bmax = (unsigned)(window < ZD_BLOCK_MAX ? window : ZD_BLOCK_MAX);
    long long out = 0, lits = 0;
    bool tree = false;
    for (;;) {
        if (pos + 3 > size) return;
        const unsigned h = f[pos] | (f[pos + 1] << 8) | (f[pos + 2] << 16);
        pos += 3;
        const int last = h & 1, type = (h >> 1) & 3;
        const unsigned bsize = h >> 3;
        if (type == 3 || bsize > fr.bmax) return;
        if (type == 1) {
            if (pos + 1 > size) return;
            out += bsize;
            pos += 1;
        } else {
            if (pos + bsize > size) return;
            if (type == 0) {
                out += bsize;
            } else {
                const long long end = pos + bsize;
                ZdLit L;
                if (!zd_lit_header(f, pos, end, L) || L.regen > fr.bmax) return;
                if (L.type == 2) tree = true;
                if (L.type == 3 && !tree) return;
                if ((L.type >= 2 && L.regen == 0)) return;
                lits += L.regen;
                out += L.regen;
                if (lits > cap) return;
                const long long q = pos + L.hsize + L.csize;
                if (q >= end) return;
                const unsigned b0 = f[q];
                if (b0 == 0) {
                    if (q + 1 != end) return;
                } else {
                    fr.has_seq = 1;
                }
            }
            pos += bsize;
        }
        if (last) break;
    }
    if (!fr.has_seq && (out > cap || (fcs >= 0 && out != fcs))) return;
    fr.err = pos == size ? 0 : -2;
}

// zd_literals_kernel's body: the Huffman literals sections k = part, part + parts, ... of one frame
__host__ __device__ inline void zd_literals_frame(const u8* f, long long size, ZdFrame& fr, u8* dst, u8* lit_scratch, int part,
                                                  int parts, ZdHufSmem& sm)
{
    long long pos = fr.data, out = 0, lits = 0, tree = -1;
    int k = 0;
    for (;;) {
        const unsigned h = f[pos] | (f[pos + 1] << 8) | (f[pos + 2] << 16);
        pos += 3;
        const int last = h & 1, type = (h >> 1) & 3;
        const unsigned bsize = h >> 3;
        if (type == 1) {
            out += bsize;
            pos += 1;
        } else {
            if (type == 0) {
                out += bsize;
            } else {
                ZdLit L;
                zd_lit_header(f, pos, pos + bsize, L);  // checked by the scan
                if (L.type == 2) tree = pos;
                if (L.type >= 2) {
                    if (k % parts == part) {
                        u8* to = fr.has_seq ? lit_scratch + lits : dst + out;
                        if (!zd_huf_section(f, size, pos, tree, to, sm)) {
                            if (zd_lane() == 0) fr.err = -1;
                            return;
                        }
                    }
                    ++k;
                    lits += L.regen;
                }
                out += L.regen;
            }
            pos += bsize;
        }
        if (last) break;
    }
}

// Shared work space of one frame's sequences
struct ZdSeqSmem {
    ZdFse t[3][512];
    short norm[256];
    unsigned short sd[256];
    int log[3];
    int have[3];  // a table of that kind has been set in this frame (for the repeat mode)
    unsigned ll[ZD_SEQ_RUN], ml[ZD_SEQ_RUN], off[ZD_SEQ_RUN];
    long long q;  // where the block's sequence bitstream starts
    int bad;
};

// one of the three tables of a block from mode `mode` at f[pos..end); returns bytes used or -1
__host__ __device__ inline long long zd_seq_table(const u8* f, long long pos, long long end, int kind, int mode, ZdSeqSmem& sm)
{
    ZdFse* t = sm.t[kind];
    if (mode == 0) {
        for (int s = 0; s < zd_def_nsym(kind); ++s) sm.norm[s] = ZD_TAB(def)[kind][s];
        if (!zd_fse_build(t, sm.norm, zd_def_nsym(kind), zd_def_log(kind), sm.sd)) return -1;
        sm.log[kind] = zd_def_log(kind);
        sm.have[kind] = 1;
        return 0;
    }
    if (mode == 1) {
        if (pos >= end || f[pos] > zd_max_sym(kind)) return -1;
        t[0].sym = f[pos];
        t[0].nb = 0;
        t[0].base = 0;
        sm.log[kind] = 0;
        sm.have[kind] = 1;
        return 1;
    }
    if (mode == 2) {
        int nsym = 0, log = 0;
        const long long used = zd_read_ncount(f, pos, end, zd_max_log(kind), zd_max_sym(kind), sm.norm, &nsym, &log);
        if (used < 0 || !zd_fse_build(t, sm.norm, nsym, log, sm.sd)) return -1;
        sm.log[kind] = log;
        sm.have[kind] = 1;
        return used;
    }
    return sm.have[kind] ? 0 : -1;
}

// warp copy of n literal bytes (from src, or the byte rle when src is null) to dst
__host__ __device__ inline void zd_put(u8* dst, const u8* src, int rle, long long n)
{
    for (long long k = zd_lane(); k < n; k += ZD_WIDTH) dst[k] = src ? src[k] : (u8)rle;
}

// zd_frames_kernel's body: one frame, blocks in order.  Returns the status.
__host__ __device__ inline long long zd_decode_frame(const u8* f, long long size, const ZdFrame& fr, u8* dst, long long cap,
                                                     const u8* lit_scratch, ZdSeqSmem& sm)
{
    if (fr.err) return fr.err;
    const int lane = zd_lane();
    long long pos = fr.data, out = 0, lits = 0;
    unsigned rep[3] = {1, 4, 8};
    if (lane == 0) sm.have[0] = sm.have[1] = sm.have[2] = 0;
    for (;;) {
        const unsigned h = f[pos] | (f[pos + 1] << 8) | (f[pos + 2] << 16);
        pos += 3;
        const int last = h & 1, type = (h >> 1) & 3;
        const unsigned bsize = h >> 3;
        if (type == 1) {
            if (out + bsize > cap) return -1;
            zd_put(dst + out, nullptr, f[pos], bsize);
            out += bsize;
            pos += 1;
        } else if (type == 0) {
            if (out + bsize > cap) return -1;
            zd_put(dst + out, f + pos, 0, bsize);
            out += bsize;
            pos += bsize;
        } else {
            const long long end = pos + bsize;
            ZdLit L;
            zd_lit_header(f, pos, end, L);
            const u8* lsrc = nullptr;  // literal bytes (null: RLE)
            int lrle = 0;
            if (L.type == 0)
                lsrc = f + pos + L.hsize;
            else if (L.type == 1)
                lrle = f[pos + L.hsize];
            else
                lsrc = lit_scratch + lits;
            if (L.type >= 2) lits += L.regen;
            long long q = pos + L.hsize + L.csize;
            const long long block_start = out;
            long long lcur = 0;  // literals of the block consumed
            if (!fr.has_seq) {
                if (L.type < 2) zd_put(dst + out, lsrc, lrle, L.regen);  // Huffman literals are in place already
                out += L.regen;
            } else {
                // Sequences_Section_Header
                long long nseq = f[q];
                if (nseq < 128) {
                    q += 1;
                } else if (nseq < 255) {
                    if (q + 2 > end) return -1;
                    nseq = ((nseq - 128) << 8) + f[q + 1];
                    q += 2;
                } else {
                    if (q + 3 > end) return -1;
                    nseq = f[q + 1] + ((long long)f[q + 2] << 8) + 0x7F00;
                    q += 3;
                }
                if (nseq == 0) {
                    if (q != end) return -1;
                } else {
                    if (q >= end) return -1;
                    const unsigned modes = f[q++];
                    if (modes & 3) return -1;
                    if (lane == 0) {
                        sm.bad = 0;
                        for (int kind = 0; kind < 3 && !sm.bad; ++kind) {
                            const long long used = zd_seq_table(f, q, end, kind, (modes >> (6 - 2 * kind)) & 3, sm);
                            if (used < 0)
                                sm.bad = 1;
                            else
                                q += used;
                        }
                        sm.q = q;
                    }
                    zd_sync();
                    if (sm.bad) return -1;
                    q = sm.q;
                    zd_sync();
                    // lane 0 decodes runs of sequences; the warp executes them
                    ZdBits bs;
                    unsigned st[3] = {0, 0, 0};
                    if (lane == 0) {
                        sm.bad = !zd_bits_init(bs, f + q, end - q);
                        if (!sm.bad) {
                            st[0] = zd_read(bs, sm.log[0]);
                            st[1] = zd_read(bs, sm.log[1]);
                            st[2] = zd_read(bs, sm.log[2]);
                        }
                    }
                    long long used_lits = 0, op = out;  // lane 0's view of the literals consumed and the output reached
                    for (long long s0 = 0; s0 < nseq; s0 += ZD_SEQ_RUN) {
                        const int run = (int)(nseq - s0 < ZD_SEQ_RUN ? nseq - s0 : ZD_SEQ_RUN);
                        if (lane == 0 && !sm.bad) {
                            for (int j = 0; j < run; ++j) {
                                const ZdFse& el = sm.t[0][st[0]];
                                const ZdFse& eo = sm.t[1][st[1]];
                                const ZdFse& em = sm.t[2][st[2]];
                                const int llc = el.sym, ofc = eo.sym, mlc = em.sym;
                                unsigned ofv = (1u << ofc) + zd_read(bs, ofc);
                                const unsigned mlv = ZD_TAB(ml_base)[mlc] + zd_read(bs, ZD_TAB(ml_bits)[mlc]);
                                const unsigned llv = ZD_TAB(ll_base)[llc] + zd_read(bs, ZD_TAB(ll_bits)[llc]);
                                if (s0 + j + 1 < nseq) {
                                    st[0] = el.base + zd_read(bs, el.nb);
                                    st[2] = em.base + zd_read(bs, em.nb);
                                    st[1] = eo.base + zd_read(bs, eo.nb);
                                }
                                unsigned offset;
                                if (ofv > 3) {
                                    offset = ofv - 3;
                                    rep[2] = rep[1];
                                    rep[1] = rep[0];
                                    rep[0] = offset;
                                } else {
                                    const int idx = (int)ofv - 1 + (llv == 0);
                                    if (idx == 0) {
                                        offset = rep[0];
                                    } else {
                                        offset = idx == 3 ? rep[0] - 1 : rep[idx];
                                        if (idx != 1) rep[2] = rep[1];
                                        rep[1] = rep[0];
                                        rep[0] = offset;
                                    }
                                }
                                used_lits += llv;
                                op += llv;
                                if (bs.pos < 0 || offset == 0 || used_lits > L.regen || offset > op || op + mlv > cap ||
                                    op + mlv - block_start > fr.bmax) {
                                    sm.bad = 1;
                                    break;
                                }
                                op += mlv;
                                sm.ll[j] = llv;
                                sm.ml[j] = mlv;
                                sm.off[j] = offset;
                            }
                        }
                        zd_sync();
                        if (sm.bad) return -1;
                        for (int j = 0; j < run; ++j) {
                            const long long ll = sm.ll[j], ml = sm.ml[j], off = sm.off[j];
                            zd_put(dst + out, lsrc ? lsrc + lcur : nullptr, lrle, ll);
                            lcur += ll;
                            out += ll;
                            zd_sync();  // a match may read the literals just written
                            u8* o = dst + out;
                            if (off >= ml)
                                for (long long k = lane; k < ml; k += ZD_WIDTH) o[k] = o[k - off];
                            else  // overlapping: every byte repeats one of the off bytes before the match
                                for (long long k = lane; k < ml; k += ZD_WIDTH) o[k] = o[k % off - off];
                            out += ml;
                            zd_sync();
                        }
                    }
                    if (lane == 0 && bs.pos != 0) sm.bad = 1;  // the bitstream must be consumed exactly
                    zd_sync();
                    if (sm.bad) return -1;
                    zd_sync();
                }
                // the literals after the last sequence
                const long long rest = (long long)L.regen - lcur;
                if (out + rest > cap) return -1;
                zd_put(dst + out, lsrc ? lsrc + lcur : nullptr, lrle, rest);
                out += rest;
                zd_sync();
            }
            pos = end;
            if (out - block_start > (long long)fr.bmax) return -1;
        }
        if (last) break;
    }
    if (out > cap || (fr.fcs >= 0 && out != fr.fcs)) return -1;
    return out;
}

__global__ void __launch_bounds__(128) zd_scan_kernel(const u8* __restrict__ src, const long long* __restrict__ offsets,
                                                      const unsigned* __restrict__ sizes, long long n, long long cap, ZdFrame* frames)
{
    const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    ZdFrame fr;
    zd_scan_frame(src + offsets[i], sizes[i], cap, fr);
    frames[i] = fr;
}

__global__ void __launch_bounds__(32) zd_literals_kernel(const u8* __restrict__ src, const long long* __restrict__ offsets,
                                                         const unsigned* __restrict__ sizes, ZdFrame* frames, u8* dst,
                                                         long long dst_stride, u8* lit_scratch, long long cap)
{
    __shared__ ZdHufSmem sm;
    const long long i = blockIdx.x;
    if (frames[i].err) return;
    zd_literals_frame(src + offsets[i], sizes[i], frames[i], dst + i * dst_stride, lit_scratch + i * cap, blockIdx.y, gridDim.y, sm);
}

__global__ void __launch_bounds__(32) zd_frames_kernel(const u8* __restrict__ src, const long long* __restrict__ offsets,
                                                       const unsigned* __restrict__ sizes, const ZdFrame* __restrict__ frames,
                                                       u8* dst, long long dst_stride, long long cap, const u8* lit_scratch,
                                                       long long lit_stride, long long* status)
{
    __shared__ ZdSeqSmem sm;
    const long long i = blockIdx.x;
    const ZdFrame fr = frames[i];
    const long long r = zd_decode_frame(src + offsets[i], sizes[i], fr, dst + i * dst_stride, cap, lit_scratch + i * lit_stride, sm);
    if (threadIdx.x == 0) status[i] = r;
}

}  // namespace

size_t zdecoder_scratch_bytes(long long n, long long cap)
{
    return (size_t)n * (((size_t)cap + 255) / 256 * 256) + (size_t)n * sizeof(ZdFrame) + 256;
}

int zdecoder_frame_plain(const u8* f, long long size, long long cap)
{
    ZdFrame fr;
    zd_scan_frame(f, size, cap, fr);
    return fr.err == 0 && !fr.has_seq;
}

int launch_zstd_decode(const u8* src, const long long* offsets, const unsigned* sizes, long long n, u8* dst, long long dst_stride,
                       long long cap, long long* status, void* scratch, cudaStream_t st)
{
    if (n <= 0) return 0;
    if (n > 0x7FFFFFFFll) {
        set_error("zstd_decode: too many frames in one batch (%lld)", n);
        return -1;
    }
    const long long lit_stride = (cap + 255) / 256 * 256;
    u8* lits = (u8*)scratch;
    ZdFrame* frames = (ZdFrame*)(lits + (size_t)n * lit_stride);
    RIRB_LAUNCH(zd_scan_kernel, (unsigned)((n + 127) / 128), 128, 0, st, src, offsets, sizes, n, cap, frames);
    RIRB_LAUNCH(zd_literals_kernel, dim3((unsigned)n, ZD_LIT_CTAS), 32, 0, st, src, offsets, sizes, frames, dst, dst_stride, lits, lit_stride);
    RIRB_LAUNCH(zd_frames_kernel, (unsigned)n, 32, 0, st, src, offsets, sizes, frames, dst, dst_stride, cap, lits, lit_stride, status);
    return 0;
}

}  // namespace rirb

using namespace rirb;

extern "C" int rirb_zstd_decode_batch(const unsigned char* src, const long long* offsets, const unsigned* sizes, long long n,
                                      unsigned char* dst, long long dst_stride, long long dst_capacity, long long* status)
{
    if (n < 0 || (n > 0 && (!src || !offsets || !sizes || !dst || !status)) || dst_capacity < 0 || dst_stride < dst_capacity) {
        set_error("zstd_decode_batch: bad arguments (device pointers, n >= 0, 0 <= dst_capacity <= dst_stride)");
        return -1;
    }
    if (rirb_device_count() <= 0) {
        set_error("zstd_decode_batch: no CUDA device (the decoder is a CUDA kernel; no CPU fallback)");
        return -1;
    }
    if (n == 0) return 0;
    // the extent of src is in the device-resident offsets / sizes, so src is not part of the overlap check
    if (refuse_pageable("zstd_decode_batch", {{"src", src, 0}, {"offsets", offsets, 0}, {"sizes", sizes, 0}, {"dst", dst, 0}, {"status", status, 0}}) ||
        refuse_overlap("zstd_decode_batch", {{"offsets", offsets, sizeof(long long) * (size_t)n}, {"sizes", sizes, sizeof(unsigned) * (size_t)n}},
                       {{"dst", dst, (size_t)n * (size_t)dst_stride}, {"status", status, sizeof(long long) * (size_t)n}}))
        return -1;
    cudaStream_t st = current_stream();
    void* scratch = nullptr;
    RIRB_CUDA_OK(cudaMallocAsync(&scratch, zdecoder_scratch_bytes(n, dst_capacity), st));
    const int rc = launch_zstd_decode(src, offsets, sizes, n, dst, dst_stride, dst_capacity, status, scratch, st);
    RIRB_CUDA_OK(cudaFreeAsync(scratch, st));
    return rc;
}
