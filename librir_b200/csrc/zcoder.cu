// librir_b200/csrc/zcoder.cu -- the device zstd coder: payloads in HBM -> standalone zstd frames (RFC 8878).
//
// The subset written (oracle/zcoder.py restates it byte for byte; DESIGN.md 7 f-3 states the tie-breaks):
//   frame    magic, Frame_Header_Descriptor 0xA0 (Single_Segment_Flag, 4-byte Frame_Content_Size), no checksum
//   blocks   <= 128 KiB, cut at segment boundaries (so each byte plane gets its own tables); per block the first that
//            applies of RLE (one byte value), compressed (Huffman literals + the sequence count 0, if smaller than the raw
//            block), raw
//   literals code lengths <= 11 bits; weights as 4-bit nibbles when the largest symbol is <= 128, else FSE-compressed
//            (accuracy log 6, header byte < 128; a block whose weights do not fit that is raw); one stream up to 1023
//            literals, four streams and a jump table above
//
// Three launches per batch:
//   zc_block_kernel   one CTA per zstd block: histogram (per-warp tables in shared memory), code construction and the
//                     table description (thread 0: <= 256 symbols), per-thread bit counts -> bit offsets (streams are
//                     written back to front, so a chunk's offset is the sum over the chunks AFTER it), bit packing into
//                     the block's fixed-size scratch slot (full words plain-stored, the two shared end words OR-ed)
//   zc_layout_kernel  frame sizes and where every block lands (fixed stride, or records packed back to back)
//   zc_copy_kernel    gathers header, streams (or the raw input bytes) of every block into place
#include "../../include/librir_b200.h"
#include "common.cuh"
#include "kernels.h"

namespace rirb {

namespace {

constexpr int ZC_THREADS = 256;
constexpr int ZC_BLOCK = 128 * 1024;
constexpr int ZC_MAX_BITS = 11;
constexpr int ZC_FSE_LOG = 6;
constexpr int ZC_HEAD = 256;                          // slot bytes reserved for block header + literals header + tree + jump
constexpr size_t ZC_SLOT = ZC_HEAD + ZC_BLOCK + 64;   // one block's compressed form (only used when it is smaller than raw)
constexpr int ZC_FRAME_HEAD = 9;                      // magic + descriptor + 4-byte content size

enum { ZB_RAW = 0, ZB_RLE = 1, ZB_COMP = 2 };

struct ZMeta {
    unsigned out_len;   // bytes of the block in the frame, its 3-byte header included
    unsigned head_len;  // bytes at the start of the slot that open the block
    unsigned kind;
    unsigned nstreams;
    unsigned s_off[4], s_len[4];  // Huffman streams inside the slot
};

struct ZGeom {
    long long bytes_each, seg, bps, bpp;  // payload bytes, segment bytes, blocks per full segment, blocks per payload
};

__host__ __device__ inline void block_span(const ZGeom& g, long long k, long long& off, int& len)
{
    if (g.bytes_each == 0) {
        off = 0;
        len = 0;
        return;
    }
    const long long s = k / g.bps, j = k % g.bps;
    const long long s0 = s * g.seg;
    const long long slen = (g.bytes_each - s0 < g.seg ? g.bytes_each - s0 : g.seg);
    off = s0 + j * ZC_BLOCK;
    const long long rest = slen - j * ZC_BLOCK;
    len = (int)(rest < ZC_BLOCK ? rest : ZC_BLOCK);
}

// forward little-endian bit writer over a zeroed byte buffer (thread 0 only)
struct BitW {
    unsigned char* b;
    int cap;
    int n = 0;
    __device__ __forceinline__ void put(unsigned v, int nb)
    {
        for (int i = 0; i < nb; ++i, ++n)
            if ((v >> i) & 1u && (n >> 3) < cap) b[n >> 3] |= (unsigned char)(1u << (n & 7));
    }
    __device__ int bytes() const { return (n + 7) >> 3; }
};

struct ZShared {
    unsigned hist[ZC_THREADS / 32][256];
    unsigned cnt[256];
    short sorted[256];
    unsigned char len[256];
    unsigned short code[256];
    unsigned tbits[ZC_THREADS];
    // code construction (thread 0)
    unsigned node_w[256];
    short kid[256][2];  // < 256: leaf index in `sorted`, else 256 + node
    unsigned char ndepth[256], depth[256];
    unsigned short bl[264];
    unsigned char tree[264];  // Huffman_Tree_Description (FSE form may be built longer before it is refused)
    unsigned char head[ZC_HEAD];
    int tree_len, kind, head_len, nstreams, seg;
    unsigned stotal[4], sbytes[4], soff[4];
    // FSE weight tables and canonical code starts (thread 0; shared memory rather than the stack)
    int fcnt[16], fnorm[16], fnxt[16];
    unsigned char fsym[64], fnb[64], fbase[64];
    unsigned cstart[16];
};

// Rules 1-3 of oracle/zcoder.py: Huffman over (count, symbol)-sorted leaves, leaf first on equal weights, JPEG K.3 cut to 11
// bits, lengths handed out longest first along the sorted order.  Then rule 4, canonical codes.
__device__ __forceinline__ void build_code(ZShared& s, int nsym)
{
    int li = 0, ni = 0, nn = 0;
    for (int m = 0; m < nsym - 1; ++m) {
        unsigned w = 0;
        for (int k = 0; k < 2; ++k) {
            const bool leaf = li < nsym && (ni >= nn || s.cnt[s.sorted[li]] <= s.node_w[ni]);
            if (leaf) {
                w += s.cnt[s.sorted[li]];
                s.kid[nn][k] = (short)li++;
            } else {
                w += s.node_w[ni];
                s.kid[nn][k] = (short)(256 + ni++);
            }
        }
        s.node_w[nn++] = w;
    }
    s.ndepth[nn - 1] = 0;
    int maxd = 0;
    for (int j = nn - 1; j >= 0; --j)
        for (int k = 0; k < 2; ++k) {
            const int c = s.kid[j][k];
            const int d = s.ndepth[j] + 1;
            if (c < 256) {
                s.depth[c] = (unsigned char)d;
                maxd = d > maxd ? d : maxd;
            } else {
                s.ndepth[c - 256] = (unsigned char)d;
            }
        }
    for (int i = 0; i < 264; ++i) s.bl[i] = 0;
    for (int i = 0; i < nsym; ++i) s.bl[s.depth[i]]++;
    for (int i = maxd; i > ZC_MAX_BITS; --i)
        while (s.bl[i] > 0) {
            int j = i - 2;
            while (s.bl[j] == 0) --j;
            s.bl[i] -= 2;
            s.bl[i - 1] += 1;
            s.bl[j + 1] += 2;
            s.bl[j] -= 1;
        }
    for (int i = 0; i < 256; ++i) s.len[i] = 0;
    int k = 0;
    const int top = maxd < ZC_MAX_BITS ? maxd : ZC_MAX_BITS;
    for (int ln = top; ln >= 1; --ln)
        for (int c = 0; c < s.bl[ln]; ++c) s.len[s.sorted[k++]] = (unsigned char)ln;
    unsigned* start = s.cstart;
    unsigned val = 0;
    for (int ln = top; ln >= 1; --ln) {
        start[ln] = val;
        val = (val + s.bl[ln]) >> 1;
    }
    for (int x = 0; x < 256; ++x)
        if (s.len[x]) s.code[x] = (unsigned short)start[s.len[x]]++;
}

// Rule 5 and RFC 8878 4.1.1 / 4.2.1.2: the weights w[0..n) as an FSE stream behind its table description.  Returns the bytes
// written to `out` (header byte excluded), or 0 when they cannot be written in this form.
__device__ __forceinline__ int fse_weights(ZShared& s, const unsigned char* w, int n, unsigned char* out, int cap)
{
    int top = 0, distinct = 0;
    int *cnt = s.fcnt, *norm = s.fnorm, *nxt = s.fnxt;
    unsigned char *sym = s.fsym, *nb = s.fnb, *base = s.fbase;
    for (int v = 0; v < 16; ++v) cnt[v] = norm[v] = 0;
    for (int i = 0; i < n; ++i) {
        distinct += cnt[w[i]] == 0;
        cnt[w[i]]++;
        top = w[i] > top ? w[i] : top;
    }
    if (distinct < 2) return 0;
    int sum = 0;
    for (int v = 0; v <= top; ++v) {
        norm[v] = cnt[v] ? (cnt[v] * 64 / n > 1 ? cnt[v] * 64 / n : 1) : 0;
        sum += norm[v];
    }
    while (sum > 64) {
        int b = 0;
        for (int v = 1; v <= top; ++v)
            if (norm[v] > norm[b]) b = v;
        norm[b]--;
        sum--;
    }
    while (sum < 64) {
        int b = 0;
        for (int v = 1; v <= top; ++v)
            if (cnt[v] > cnt[b]) b = v;
        norm[b]++;
        sum++;
    }
    for (int i = 0; i < cap; ++i) out[i] = 0;
    BitW bw{out, cap};
    // table description
    bw.put(ZC_FSE_LOG - 5, 4);
    int remaining = (1 << ZC_FSE_LOG) + 1, threshold = 1 << ZC_FSE_LOG, nbits = ZC_FSE_LOG + 1, sy = 0;
    bool prev0 = false;
    while (sy <= top && remaining > 1) {
        if (prev0) {
            int st = sy;
            while (norm[sy] == 0) ++sy;
            while (sy >= st + 3) {
                st += 3;
                bw.put(3, 2);
            }
            bw.put((unsigned)(sy - st), 2);
        }
        const int c = norm[sy++];
        const int mx = (2 * threshold - 1) - remaining;
        remaining -= c;
        int v = c + 1;
        if (v >= threshold) v += mx;
        bw.put((unsigned)v, v < mx ? nbits - 1 : nbits);
        prev0 = v == 1;
        while (remaining < threshold) {
            --nbits;
            threshold >>= 1;
        }
    }
    const int hbytes = bw.bytes();
    // decoding table
    {
        const int step = (64 >> 1) + (64 >> 3) + 3;
        int pos = 0;
        for (int x = 0; x <= top; ++x)
            for (int i = 0; i < norm[x]; ++i) {
                sym[pos] = (unsigned char)x;
                pos = (pos + step) & 63;
            }
        for (int x = 0; x < 16; ++x) nxt[x] = norm[x];
        for (int u = 0; u < 64; ++u) {
            const int xx = nxt[sym[u]]++;
            const int hb = 31 - __clz(xx);
            nb[u] = (unsigned char)(ZC_FSE_LOG - hb);
            base[u] = (unsigned char)((xx << nb[u]) - 64);
        }
    }
    // two interleaved chains (even / odd weights); the decoder reads the bits in the reverse of the order written
    BitW bs{out + hbytes, cap - hbytes};
    int st_even = 0, st_odd = 0;  // the chains of the even and of the odd weights
    for (int t = 0; t < 2; ++t) {
        const int k = n - 1 - t;
        int u = 0;
        while (sym[u] != w[k]) ++u;
        if (k & 1) st_odd = u;
        else st_even = u;
    }
    for (int k = n - 3; k >= 0; --k) {
        const int v = (k & 1) ? st_odd : st_even;
        int u = 0;
        while (!(sym[u] == w[k] && base[u] <= v && v < base[u] + (1 << nb[u]))) ++u;
        bs.put((unsigned)(v - base[u]), nb[u]);
        if (k & 1) st_odd = u;
        else st_even = u;
    }
    bs.put((unsigned)st_odd, ZC_FSE_LOG);
    bs.put((unsigned)st_even, ZC_FSE_LOG);
    bs.put(1, 1);
    const int total = hbytes + bs.bytes();
    return total < 128 && total <= cap ? total : 0;
}

// Huffman_Tree_Description into s.tree; false when the weights cannot be written
__device__ __forceinline__ bool tree_description(ZShared& s)
{
    int maxb = 0, last = 0;
    for (int x = 0; x < 256; ++x)
        if (s.len[x]) {
            maxb = s.len[x] > maxb ? s.len[x] : maxb;
            last = x;
        }
    unsigned char* w = s.ndepth;  // free by now: the weights of symbols 0 .. last-1
    for (int x = 0; x < last; ++x) w[x] = s.len[x] ? (unsigned char)(maxb + 1 - s.len[x]) : 0;
    if (last <= 128) {
        s.tree[0] = (unsigned char)(127 + last);
        for (int i = 0; i < (last + 1) / 2; ++i)
            s.tree[1 + i] = (unsigned char)((w[2 * i] << 4) | (2 * i + 1 < last ? w[2 * i + 1] : 0));
        s.tree_len = 1 + (last + 1) / 2;
        return true;
    }
    const int b = fse_weights(s, w, last, s.tree + 1, (int)sizeof(s.tree) - 1);
    if (!b) return false;
    s.tree[0] = (unsigned char)b;
    s.tree_len = 1 + b;
    return true;
}

__device__ inline void put_le(unsigned char* p, unsigned long long v, int n)
{
    for (int i = 0; i < n; ++i) p[i] = (unsigned char)(v >> (8 * i));
}

__global__ void __launch_bounds__(ZC_THREADS) zc_block_kernel(const u8* __restrict__ src, ZGeom g, u8* __restrict__ slots,
                                                             ZMeta* __restrict__ meta)
{
    __shared__ ZShared s;
    const int tid = threadIdx.x;
    const long long b = blockIdx.x;
    const long long k = b % g.bpp;
    long long off;
    int n;
    block_span(g, k, off, n);
    const u8* in = src + (b / g.bpp) * g.bytes_each + off;
    const bool last = k == g.bpp - 1;
    u8* slot = slots + (size_t)b * ZC_SLOT;

    for (int i = tid; i < (ZC_THREADS / 32) * 256; i += ZC_THREADS) (&s.hist[0][0])[i] = 0;
    __syncthreads();
    for (int i = tid; i < n; i += ZC_THREADS) atomicAdd(&s.hist[tid >> 5][in[i]], 1u);
    __syncthreads();
    unsigned c = 0;
    for (int w = 0; w < ZC_THREADS / 32; ++w) c += s.hist[w][tid];
    s.cnt[tid] = c;
    const int nsym = __syncthreads_count(c > 0);
    if (nsym >= 2) {
        int rank = 0;
        for (int x = 0; x < 256; ++x) {
            const unsigned cx = s.cnt[x];
            rank += cx > 0 && (cx < c || (cx == c && x < tid));
        }
        if (c) s.sorted[rank] = (short)tid;
    }
    __syncthreads();
    if (tid == 0) {
        s.kind = n == 0 ? ZB_RAW : nsym == 1 ? ZB_RLE : ZB_COMP;
        if (s.kind == ZB_COMP) {
            build_code(s, nsym);
            if (!tree_description(s)) s.kind = ZB_RAW;
        }
        s.nstreams = n <= 1023 ? 1 : 4;
        s.seg = (n + 3) / 4;
    }
    __syncthreads();
    const int kind0 = s.kind;
    // this thread's chunk of its stream
    const int ns = s.nstreams, tps = ZC_THREADS / ns, si = tid / tps, r = tid % tps;
    const int s0 = ns == 1 ? 0 : si * s.seg;
    const int s1 = ns == 1 ? n : min(n, (si + 1) * s.seg);
    const int chunk = (s1 - s0 + tps - 1) / tps;
    const int a = min(s1, s0 + r * chunk), e = min(s1, s0 + (r + 1) * chunk);
    if (kind0 == ZB_COMP) {
        unsigned bits = 0;
        for (int i = a; i < e; ++i) bits += s.len[in[i]];
        s.tbits[tid] = bits;
    }
    __syncthreads();
    if (tid == 0) {
        int kind = s.kind;
        if (kind == ZB_COMP) {
            unsigned streams = ns == 4 ? 6 : 0;
            bool fits = true;
            for (int q = 0; q < ns; ++q) {
                unsigned t = 0;
                for (int i = q * tps; i < (q + 1) * tps; ++i) t += s.tbits[i];
                s.stotal[q] = t;
                s.sbytes[q] = t / 8 + 1;
                streams += s.sbytes[q];
                if (q < 3 && s.sbytes[q] > 0xFFFF) fits = false;
            }
            const unsigned csize = (unsigned)s.tree_len + streams;
            const int lh = ns == 1 ? 3 : ((unsigned)n > csize ? (unsigned)n : csize) <= 16383 ? 4 : 5;
            const unsigned body = (unsigned)lh + csize + 1;
            if (!fits || body >= (unsigned)n) {
                kind = ZB_RAW;
            } else {
                put_le(s.head, 1u * last | ZB_COMP << 1 | body << 3, 3);
                unsigned long long h;
                if (lh == 3) h = 2ull | (unsigned long long)n << 4 | (unsigned long long)csize << 14;
                else if (lh == 4) h = 2ull | 2ull << 2 | (unsigned long long)n << 4 | (unsigned long long)csize << 18;
                else h = 2ull | 3ull << 2 | (unsigned long long)n << 4 | (unsigned long long)csize << 22;
                put_le(s.head + 3, h, lh);
                int p = 3 + lh;
                for (int i = 0; i < s.tree_len; ++i) s.head[p++] = s.tree[i];
                if (ns == 4)
                    for (int q = 0; q < 3; ++q, p += 2) put_le(s.head + p, s.sbytes[q], 2);
                s.head_len = p;
                unsigned o = ZC_HEAD;
                for (int q = 0; q < ns; ++q) {
                    s.soff[q] = o;
                    o += (s.sbytes[q] + 3) & ~3u;
                }
                meta[b].out_len = 3 + body;
            }
        }
        if (kind == ZB_RLE) {
            put_le(s.head, 1u * last | ZB_RLE << 1 | (unsigned)n << 3, 3);
            s.head[3] = in[0];
            s.head_len = 4;
            meta[b].out_len = 4;
        } else if (kind == ZB_RAW) {
            put_le(s.head, 1u * last | ZB_RAW << 1 | (unsigned)n << 3, 3);
            s.head_len = 3;
            meta[b].out_len = 3 + n;
        }
        s.kind = kind;
        meta[b].kind = kind;
        meta[b].head_len = s.head_len;
        meta[b].nstreams = kind == ZB_COMP ? ns : 0;
        for (int q = 0; q < 4; ++q) {
            meta[b].s_off[q] = kind == ZB_COMP && q < ns ? s.soff[q] : 0;
            meta[b].s_len[q] = kind == ZB_COMP && q < ns ? s.sbytes[q] : 0;
        }
    }
    __syncthreads();
    for (int i = tid; i < s.head_len; i += ZC_THREADS) slot[i] = s.head[i];
    if (s.kind != ZB_COMP) return;
    // zero the stream words, then pack: the chunk after this one (higher literal indices) holds the lower bit positions
    unsigned* words = (unsigned*)(slot + ZC_HEAD);
    const unsigned nwords = (s.soff[ns - 1] + ((s.sbytes[ns - 1] + 3) & ~3u) - ZC_HEAD) / 4;
    for (unsigned i = tid; i < nwords; i += ZC_THREADS) words[i] = 0;
    unsigned pos = 0;
    for (int i = r + 1; i < tps; ++i) pos += s.tbits[si * tps + i];
    __syncthreads();
    unsigned* sw = (unsigned*)(slot + s.soff[si]);
    unsigned wi = pos >> 5;
    int nacc = pos & 31;
    unsigned long long acc = 0;
    bool first = true;
    for (int i = e - 1; i >= a; --i) {
        const int x = in[i];
        acc |= (unsigned long long)s.code[x] << nacc;
        nacc += s.len[x];
        if (nacc >= 32) {
            if (first) atomicOr(sw + wi, (unsigned)acc);
            else sw[wi] = (unsigned)acc;
            first = false;
            ++wi;
            acc >>= 32;
            nacc -= 32;
        }
    }
    if (nacc > 0) atomicOr(sw + wi, (unsigned)acc);
    if (r == 0) atomicOr(sw + (s.stotal[si] >> 5), 1u << (s.stotal[si] & 31));  // end mark
}

// one thread per payload for the sizes; packed records need the running sum over payloads (one CTA, chunked scan)
__global__ void zc_layout_kernel(const ZMeta* __restrict__ meta, long long n, long long bpp, long long dst_stride, int rec_head,
                                 long long* __restrict__ sizes, long long* __restrict__ foff, long long* __restrict__ boff)
{
    __shared__ long long part[1024];
    const int tid = threadIdx.x;
    const long long per = (n + blockDim.x - 1) / blockDim.x;
    const long long i0 = tid * per, i1 = min(n, i0 + per);
    long long mine = 0;
    for (long long i = i0; i < i1; ++i) {
        long long f = ZC_FRAME_HEAD;
        for (long long k = 0; k < bpp; ++k) f += meta[i * bpp + k].out_len;
        if (sizes) sizes[i] = f;
        mine += rec_head + f;
    }
    part[tid] = mine;
    __syncthreads();
    if (tid == 0) {
        long long run = 0;
        for (int t = 0; t < (int)blockDim.x; ++t) {
            const long long v = part[t];
            part[t] = run;
            run += v;
        }
        if (dst_stride == 0) foff[n] = run;
    }
    __syncthreads();
    long long at = part[tid];
    for (long long i = i0; i < i1; ++i) {
        const long long fo = dst_stride > 0 ? i * dst_stride : at;
        foff[i] = fo;
        long long o = fo + rec_head + ZC_FRAME_HEAD;
        for (long long k = 0; k < bpp; ++k) {
            boff[i * bpp + k] = o;
            o += meta[i * bpp + k].out_len;
        }
        at = o;
    }
}

__global__ void __launch_bounds__(ZC_THREADS) zc_copy_kernel(const u8* __restrict__ src, ZGeom g, const u8* __restrict__ slots,
                                                            const ZMeta* __restrict__ meta, const long long* __restrict__ foff,
                                                            const long long* __restrict__ boff, int rec_head, u8* __restrict__ dst)
{
    const long long b = blockIdx.x;
    const long long k = b % g.bpp, i = b / g.bpp;
    const int tid = threadIdx.x;
    const ZMeta& m = meta[b];
    const u8* slot = slots + (size_t)b * ZC_SLOT;
    u8* out = dst + boff[b];
    if (k == 0 && tid < ZC_FRAME_HEAD) {
        const unsigned magic_fhd = 0xFD2FB528u;  // then the descriptor 0xA0 and the 4-byte content size
        dst[foff[i] + rec_head + tid] = tid < 4 ? (u8)(magic_fhd >> (8 * tid)) : tid == 4 ? (u8)0xA0 : (u8)((unsigned long long)g.bytes_each >> (8 * (tid - 5)));
    }
    for (unsigned j = tid; j < m.head_len; j += ZC_THREADS) out[j] = slot[j];
    out += m.head_len;
    if (m.kind == ZB_RAW) {
        long long off;
        int n;
        block_span(g, k, off, n);
        const u8* in = src + i * g.bytes_each + off;
        for (int j = tid; j < n; j += ZC_THREADS) out[j] = in[j];
    } else if (m.kind == ZB_COMP) {
        for (unsigned q = 0; q < m.nstreams; ++q) {
            const u8* p = slot + m.s_off[q];
            for (unsigned j = tid; j < m.s_len[q]; j += ZC_THREADS) out[j] = p[j];
            out += m.s_len[q];
        }
        if (tid == 0) out[0] = 0;  // Number_of_Sequences = 0
    }
}

}  // namespace

size_t zcoder_scratch_bytes(long long n, long long bytes_each, long long segment)
{
    const long long seg = segment > 0 && segment < bytes_each ? segment : (bytes_each > 0 ? bytes_each : 1);
    const long long bps = (seg + ZC_BLOCK - 1) / ZC_BLOCK;
    const long long nseg = bytes_each > 0 ? (bytes_each + seg - 1) / seg : 1;
    const long long last = bytes_each > 0 ? bytes_each - (nseg - 1) * seg : 0;
    const long long bpp = bytes_each > 0 ? (nseg - 1) * bps + (last + ZC_BLOCK - 1) / ZC_BLOCK : 1;
    const size_t nb = (size_t)(n * bpp);
    return nb * (ZC_SLOT + sizeof(ZMeta) + 8) + (size_t)(n + 1) * 8 + 256;
}

long long zcoder_frame_bound(long long bytes_each, long long segment)
{
    const long long seg = segment > 0 && segment < bytes_each ? segment : (bytes_each > 0 ? bytes_each : 1);
    const long long nseg = bytes_each > 0 ? (bytes_each + seg - 1) / seg : 1;
    const long long last = bytes_each > 0 ? bytes_each - (nseg - 1) * seg : 0;
    const long long bpp = bytes_each > 0 ? (nseg - 1) * ((seg + ZC_BLOCK - 1) / ZC_BLOCK) + (last + ZC_BLOCK - 1) / ZC_BLOCK : 1;
    return ZC_FRAME_HEAD + 3 * bpp + bytes_each;
}

int launch_zstd_encode(const u8* src, long long n, long long bytes_each, long long segment, u8* dst, long long dst_stride,
                       int rec_head, long long* sizes, long long** frame_offsets, void* scratch, cudaStream_t st)
{
    if (n <= 0) return 0;
    ZGeom g;
    g.bytes_each = bytes_each;
    g.seg = segment > 0 && segment < bytes_each ? segment : (bytes_each > 0 ? bytes_each : 1);
    g.bps = (g.seg + ZC_BLOCK - 1) / ZC_BLOCK;
    const long long nseg = bytes_each > 0 ? (bytes_each + g.seg - 1) / g.seg : 1;
    const long long last = bytes_each > 0 ? bytes_each - (nseg - 1) * g.seg : 0;
    g.bpp = bytes_each > 0 ? (nseg - 1) * g.bps + (last + ZC_BLOCK - 1) / ZC_BLOCK : 1;
    const long long nb = n * g.bpp;
    if (nb > 0x7FFFFFFFll) {
        set_error("zstd_encode: too many blocks in one batch (%lld)", nb);
        return -1;
    }
    u8* slots = (u8*)scratch;
    ZMeta* meta = (ZMeta*)(slots + (size_t)nb * ZC_SLOT);
    long long* boff = (long long*)(meta + nb);
    long long* foff = boff + nb;
    RIRB_LAUNCH(zc_block_kernel, (unsigned)nb, ZC_THREADS, 0, st, src, g, slots, meta);
    RIRB_LAUNCH(zc_layout_kernel, 1, 1024, 0, st, meta, n, g.bpp, dst_stride, rec_head, sizes, foff, boff);
    RIRB_LAUNCH(zc_copy_kernel, (unsigned)nb, ZC_THREADS, 0, st, src, g, slots, meta, foff, boff, rec_head, dst);
    if (frame_offsets) *frame_offsets = foff;
    return 0;
}

}  // namespace rirb

using namespace rirb;

extern "C" int rirb_zstd_encode_batch(const unsigned char* src, long long n, long long bytes_each, long long segment,
                                      unsigned char* dst, long long dst_stride, long long* sizes)
{
    if (!src || !dst || !sizes || n < 0 || bytes_each < 0 || bytes_each > 0xFFFFFFFFll || segment < 0 ||
        dst_stride < zcoder_frame_bound(bytes_each, segment)) {
        set_error("zstd_encode_batch: bad arguments (dst_stride must be at least %lld)", zcoder_frame_bound(bytes_each, segment));
        return -1;
    }
    if (n == 0) return 0;
    if (rirb_device_count() <= 0) {
        set_error("zstd_encode_batch: no CUDA device (the coder is a CUDA kernel; no CPU fallback)");
        return -1;
    }
    cudaStream_t st = current_stream();
    void* scratch = nullptr;
    RIRB_CUDA_OK(cudaMallocAsync(&scratch, zcoder_scratch_bytes(n, bytes_each, segment), st));
    const int rc = launch_zstd_encode(src, n, bytes_each, segment, dst, dst_stride, 0, sizes, nullptr, scratch, st);
    RIRB_CUDA_OK(cudaFreeAsync(scratch, st));
    return rc;
}
