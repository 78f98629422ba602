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
#include <cub/device/device_segmented_radix_sort.cuh>

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

enum { ZB_RAW = 0, ZB_RLE = 1, ZB_COMP = 2, ZB_LZ = 3 };  // ZB_LZ: coder 2's LZ form, the whole block in the slot's head

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

__device__ inline void put_le(unsigned char* p, unsigned long long v, int n)
{
    for (int i = 0; i < n; ++i) p[i] = (unsigned char)(v >> (8 * i));
}

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

// Raw (0) or RLE (1) Literals_Section_Header (RFC 8878 3.1.1.3.1.1); returns its bytes
__device__ inline int literal_header(unsigned char* p, unsigned kind, unsigned n)
{
    if (n <= 31) {
        p[0] = (unsigned char)(kind | n << 3);
        return 1;
    }
    const int h = n <= 4095 ? 2 : 3;
    put_le(p, kind | (h == 2 ? 1u : 3u) << 2 | n << 4, h);
    return h;
}

// One CTA codes the n bytes at `in` into its slot and meta entry.  LZ = false: a whole zstd block (coder 1).  LZ = true: the
// literals section of coder 2's LZ form -- the same Huffman code and the same "smaller than raw" test, but without the block
// header, and RLE / raw literal headers in place of RLE / raw blocks; meta.out_len is then the section's bytes.
template <bool LZ>
__device__ __forceinline__ void zc_block_body(const u8* __restrict__ in, int n, bool last, u8* __restrict__ slot, ZMeta* __restrict__ mb)
{
    __shared__ ZShared s;
    const int tid = threadIdx.x;

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
                const int h0 = LZ ? 0 : 3;
                if (!LZ) put_le(s.head, 1u * last | ZB_COMP << 1 | body << 3, 3);
                unsigned long long h;
                if (lh == 3) h = 2ull | (unsigned long long)n << 4 | (unsigned long long)csize << 14;
                else if (lh == 4) h = 2ull | 2ull << 2 | (unsigned long long)n << 4 | (unsigned long long)csize << 18;
                else h = 2ull | 3ull << 2 | (unsigned long long)n << 4 | (unsigned long long)csize << 22;
                put_le(s.head + h0, h, lh);
                int p = h0 + lh;
                for (int i = 0; i < s.tree_len; ++i) s.head[p++] = s.tree[i];
                if (ns == 4)
                    for (int q = 0; q < 3; ++q, p += 2) put_le(s.head + p, s.sbytes[q], 2);
                s.head_len = p;
                unsigned o = ZC_HEAD;
                for (int q = 0; q < ns; ++q) {
                    s.soff[q] = o;
                    o += (s.sbytes[q] + 3) & ~3u;
                }
                mb->out_len = LZ ? lh + csize : 3 + body;
            }
        }
        if (LZ && kind != ZB_COMP) {
            s.head_len = literal_header(s.head, kind == ZB_RLE ? 1 : 0, (unsigned)n);
            if (kind == ZB_RLE) s.head[s.head_len++] = in[0];
            mb->out_len = s.head_len + (kind == ZB_RAW ? n : 0);
        } else if (kind == ZB_RLE) {
            put_le(s.head, 1u * last | ZB_RLE << 1 | (unsigned)n << 3, 3);
            s.head[3] = in[0];
            s.head_len = 4;
            mb->out_len = 4;
        } else if (kind == ZB_RAW) {
            put_le(s.head, 1u * last | ZB_RAW << 1 | (unsigned)n << 3, 3);
            s.head_len = 3;
            mb->out_len = 3 + n;
        }
        s.kind = kind;
        mb->kind = kind;
        mb->head_len = s.head_len;
        mb->nstreams = kind == ZB_COMP ? ns : 0;
        for (int q = 0; q < 4; ++q) {
            mb->s_off[q] = kind == ZB_COMP && q < ns ? s.soff[q] : 0;
            mb->s_len[q] = kind == ZB_COMP && q < ns ? s.sbytes[q] : 0;
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

__global__ void __launch_bounds__(ZC_THREADS) zc_block_kernel(const u8* __restrict__ src, ZGeom g, u8* __restrict__ slots,
                                                             ZMeta* __restrict__ meta)
{
    const long long b = blockIdx.x;
    const long long k = b % g.bpp;
    long long off;
    int n;
    block_span(g, k, off, n);
    zc_block_body<false>(src + (b / g.bpp) * g.bytes_each + off, n, k == g.bpp - 1, slots + (size_t)b * ZC_SLOT, meta + b);
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


// ---- coder 2: coder 1 plus an LZ form per block (oracle/zlz.py restates it; DESIGN.md 7 f-3) ----
//   zl_keys_kernel    one CTA per block: the 8-byte key and the position of every p <= n-8, and the block's sort segment
//   (CUB)             stable segmented radix sort of (key, position), LZ_SORT_BLOCKS blocks at a time
//   zl_cand_kernel    one CTA per block: cand(p) = the position sorted just before p when its key is the same, else -1
//   zl_parse_kernel   one warp per block: the greedy parse (a ballot over 32 positions finds the next candidate, the match
//                     is extended 32 bytes per step), the sequences and the compacted literals into the block's scratch
//   zl_lit_kernel     the literals through coder 1's Huffman path (zc_block_body<true>)
//   zl_seq_kernel     one thread per block: the sequences section, the FSE bitstream written from the last sequence back
//   zl_choose_kernel  one CTA per block: when the LZ form is smaller than coder 1's form, the whole block into coder 1's slot
// then zc_layout_kernel and zc_copy_kernel as for coder 1.

constexpr int LZ_MIN = 8;                       // match length, and the bytes of a candidate key
constexpr int LZ_MAX_SEQ = ZC_BLOCK / LZ_MIN;   // every sequence covers at least LZ_MIN bytes of its block
constexpr long long LZ_SORT_BLOCKS = 512;       // blocks per candidate sort: 64 MB of input, 24 B of sort buffers a byte
constexpr int LZ_WARPS = 4;                     // warps (blocks) per CTA of zl_parse_kernel
constexpr int LZ_SEQ_THREADS = 64;              // threads (blocks) per CTA of zl_seq_kernel

struct ZSeq {
    unsigned ll, ml, off;
};

// predefined distributions (RFC 8878 3.1.1.3.2.2) in table order LL, OF, ML, and the LL / ML code baselines
__constant__ short zl_def[3][53] = {
    {4, 3, 2, 2, 2, 2, 2, 2, 2, 2, 2, 2, 2, 1, 1, 1, 2, 2, 2, 2, 2, 2, 2, 2, 2, 3, 2, 1, 1, 1, 1, 1, -1, -1, -1, -1},
    {1, 1, 1, 1, 1, 1, 2, 2, 2, 1, 1, 1, 1, 1, 1, 1, 1, 1, 1, 1, 1, 1, 1, 1, -1, -1, -1, -1, -1},
    {1, 4, 3, 2, 2, 2, 2, 2, 2, 1, 1, 1, 1, 1, 1, 1, 1, 1, 1, 1, 1, 1, 1, 1, 1, 1, 1, 1, 1, 1, 1, 1, 1, 1, 1, 1, 1, 1, 1, 1, 1,
     1, 1, 1, 1, 1, -1, -1, -1, -1, -1, -1, -1}};
__constant__ unsigned char zl_nsym[3] = {36, 29, 53}, zl_log[3] = {6, 5, 6};
__constant__ unsigned zl_ll_base[36] = {0,  1,  2,  3,  4,  5,  6,  7,  8,  9,  10, 11, 12, 13, 14, 15, 16, 18, 20, 22, 24, 28, 32, 40, 48, 64,
                                        0x80, 0x100, 0x200, 0x400, 0x800, 0x1000, 0x2000, 0x4000, 0x8000, 0x10000};
__constant__ unsigned char zl_ll_bits[36] = {0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 1, 1, 1, 1, 2, 2, 3, 3, 4, 6, 7, 8, 9, 10, 11, 12, 13, 14, 15, 16};
__constant__ unsigned zl_ml_base[53] = {3,  4,  5,  6,  7,  8,  9,  10, 11, 12, 13, 14, 15, 16, 17, 18, 19, 20, 21, 22, 23, 24, 25, 26, 27, 28, 29,
                                        30, 31, 32, 33, 34, 35, 37, 39, 41, 43, 47, 51, 59, 67, 83, 99, 0x83, 0x103, 0x203, 0x403, 0x803,
                                        0x1003, 0x2003, 0x4003, 0x8003, 0x10003};
__constant__ unsigned char zl_ml_bits[53] = {0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0,
                                             0, 0, 0, 0, 0, 1, 1, 1, 1, 2, 2, 3, 3, 4, 4, 5, 7, 8, 9, 10, 11, 12, 13, 14, 15, 16};

__global__ void zl_keys_kernel(const u8* __restrict__ src, ZGeom g, long long b0, unsigned long long* __restrict__ keys,
                               unsigned* __restrict__ pos, int* __restrict__ seg_begin, int* __restrict__ seg_end)
{
    const long long cb = blockIdx.x, b = b0 + cb;
    long long off;
    int n;
    block_span(g, b % g.bpp, off, n);
    const u8* in = src + (b / g.bpp) * g.bytes_each + off;
    const int m = n >= LZ_MIN ? n - LZ_MIN + 1 : 0;
    const int base = (int)cb * ZC_BLOCK;
    for (int p = threadIdx.x; p < m; p += blockDim.x) {
        unsigned long long k = 0;
        for (int j = 0; j < LZ_MIN; ++j) k |= (unsigned long long)in[p + j] << (8 * j);
        keys[base + p] = k;
        pos[base + p] = (unsigned)p;
    }
    if (threadIdx.x == 0) {
        seg_begin[cb] = base;
        seg_end[cb] = base + m;
    }
}

__global__ void zl_cand_kernel(const unsigned long long* __restrict__ keys, const unsigned* __restrict__ pos,
                               const int* __restrict__ seg_begin, const int* __restrict__ seg_end, int* __restrict__ cand)
{
    const int a = seg_begin[blockIdx.x], e = seg_end[blockIdx.x];
    for (int i = a + (int)threadIdx.x; i < e; i += blockDim.x)
        cand[a + pos[i]] = i > a && keys[i] == keys[i - 1] ? (int)pos[i - 1] : -1;
}

__global__ void __launch_bounds__(32 * LZ_WARPS) zl_parse_kernel(const u8* __restrict__ src, ZGeom g, long long b0, long long nbc,
                                                                 const int* __restrict__ cand, u8* __restrict__ lits,
                                                                 ZSeq* __restrict__ seqs, unsigned* __restrict__ nseq,
                                                                 unsigned* __restrict__ nlit)
{
    const long long cb = (long long)blockIdx.x * LZ_WARPS + threadIdx.x / 32;
    if (cb >= nbc) return;
    const int lane = threadIdx.x & 31;
    const long long b = b0 + cb;
    long long off;
    int n;
    block_span(g, b % g.bpp, off, n);
    const u8* in = src + (b / g.bpp) * g.bytes_each + off;
    const int* cd = cand + cb * ZC_BLOCK;
    u8* lo = lits + b * ZC_BLOCK;
    ZSeq* sq = seqs + b * LZ_MAX_SEQ;
    int p = 0, lit = 0, ns = 0, nl = 0;
    while (p <= n - LZ_MIN) {
        const int i = p + lane;
        const unsigned has = __ballot_sync(~0u, i <= n - LZ_MIN && cd[i] >= 0);
        if (!has) {
            p += 32;
            continue;
        }
        p += __ffs(has) - 1;
        const int q = cd[p];
        int len = 0;
        for (;;) {  // common prefix of in[p..n) and in[q..n), q < p: the bytes compared are the input's, so runs overlap
            const int j = p + len + lane;
            const unsigned ne = __ballot_sync(~0u, j >= n || in[j] != in[q + len + lane]);
            if (ne) {
                len += __ffs(ne) - 1;
                break;
            }
            len += 32;
        }
        for (int k = lane; k < p - lit; k += 32) lo[nl + k] = in[lit + k];
        if (lane == 0) sq[ns] = ZSeq{(unsigned)(p - lit), (unsigned)len, (unsigned)(p - q)};
        nl += p - lit;
        ++ns;
        p += len;
        lit = p;
    }
    for (int k = lane; k < n - lit; k += 32) lo[nl + k] = in[lit + k];
    if (lane == 0) {
        nseq[b] = (unsigned)ns;
        nlit[b] = (unsigned)(nl + n - lit);
    }
}

__global__ void __launch_bounds__(ZC_THREADS) zl_lit_kernel(const u8* __restrict__ lits, const unsigned* __restrict__ nlit,
                                                           u8* __restrict__ slots, ZMeta* __restrict__ meta)
{
    const long long b = blockIdx.x;
    zc_block_body<true>(lits + b * ZC_BLOCK, (int)nlit[b], false, slots + (size_t)b * ZC_SLOT, meta + b);
}

// FSE decoding table of a predefined distribution (RFC 8878 4.1.1, 'less than 1' probabilities at the top), and the states
// of every symbol in ascending order: first[s] .. first[s + 1] in list
struct ZFse {
    unsigned char sym[64], nb[64], first[54], list[64];
    unsigned short base[64];
    short nxt[53];
};

__device__ void fse_predefined(ZFse& t, int which)
{
    const short* norm = zl_def[which];
    const int nsym = zl_nsym[which], log = zl_log[which], size = 1 << log;
    int high = size - 1;
    for (int s = 0; s < nsym; ++s) {
        if (norm[s] == -1) t.sym[high--] = (unsigned char)s;
        t.nxt[s] = norm[s] == -1 ? 1 : norm[s];
    }
    const int step = (size >> 1) + (size >> 3) + 3;
    int pos = 0;
    for (int s = 0; s < nsym; ++s)
        for (int i = 0; i < norm[s]; ++i) {
            t.sym[pos] = (unsigned char)s;
            do pos = (pos + step) & (size - 1);
            while (pos > high);
        }
    for (int u = 0; u < size; ++u) {
        const int x = t.nxt[t.sym[u]]++;
        t.nb[u] = (unsigned char)(log - (31 - __clz(x)));
        t.base[u] = (unsigned short)((x << t.nb[u]) - size);
    }
    int k = 0;
    for (int s = 0; s < nsym; ++s) {
        t.first[s] = (unsigned char)k;
        for (int u = 0; u < size; ++u)
            if (t.sym[u] == s) t.list[k++] = (unsigned char)u;
    }
    t.first[nsym] = (unsigned char)k;
}

__device__ __forceinline__ unsigned ll_code(unsigned v)
{
    if (v < 16) return v;
    if (v >= 64) return (31 - __clz(v)) + 19;
    unsigned c = 24;
    while (zl_ll_base[c] > v) --c;
    return c;
}

__device__ __forceinline__ unsigned ml_code(unsigned ml)
{
    const unsigned v = ml - 3;
    if (v < 32) return v;
    if (v >= 128) return (31 - __clz(v)) + 36;
    unsigned c = 42;
    while (zl_ml_base[c] > ml) --c;
    return c;
}

// forward little-endian bit writer into out[0 .. cap); ok turns false when the bytes do not fit
struct SeqBits {
    u8* out;
    unsigned cap, n = 0;
    unsigned long long acc = 0;
    int nacc = 0;
    bool ok = true;
    __device__ __forceinline__ void byte(unsigned v)
    {
        if (n < cap) out[n] = (u8)v;
        else ok = false;
        ++n;
    }
    __device__ __forceinline__ void put(unsigned v, int nb)
    {
        acc |= (unsigned long long)(v & ((1u << nb) - 1u)) << nacc;  // nb <= 17
        nacc += nb;
        while (nacc >= 8) {
            byte((unsigned)acc & 0xFF);
            acc >>= 8;
            nacc -= 8;
        }
    }
};

__global__ void __launch_bounds__(LZ_SEQ_THREADS) zl_seq_kernel(const ZSeq* __restrict__ seqs, const unsigned* __restrict__ nseq,
                                                                long long nb, u8* __restrict__ out, unsigned* __restrict__ out_len)
{
    __shared__ ZFse t[3];  // LL, OF, ML
    if (threadIdx.x < 3) fse_predefined(t[threadIdx.x], threadIdx.x);
    __syncthreads();
    const long long b = (long long)blockIdx.x * LZ_SEQ_THREADS + threadIdx.x;
    if (b >= nb) return;
    const int n = (int)nseq[b];
    if (n == 0) {
        out_len[b] = 0;
        return;
    }
    const ZSeq* sq = seqs + b * LZ_MAX_SEQ;
    auto codes = [&](int i, unsigned c[3]) {
        c[0] = ll_code(sq[i].ll);
        c[1] = 31 - __clz(sq[i].off + 3);
        c[2] = ml_code(sq[i].ml);
    };
    unsigned c0[3], c[3];
    codes(0, c0);
    bool rle[3] = {true, true, true};
    for (int i = 1; i < n; ++i) {
        codes(i, c);
        for (int x = 0; x < 3; ++x) rle[x] = rle[x] && c[x] == c0[x];
    }
    SeqBits w{out + b * ZC_BLOCK, (unsigned)ZC_BLOCK};
    if (n < 128) {
        w.byte((unsigned)n);
    } else {
        w.byte((unsigned)(n >> 8) + 128);
        w.byte((unsigned)n & 0xFF);
    }
    w.byte((unsigned)rle[0] << 6 | (unsigned)rle[1] << 4 | (unsigned)rle[2] << 2);
    for (int x = 0; x < 3; ++x)
        if (rle[x]) w.byte(c0[x]);
    auto extra = [&](int i, const unsigned c[3]) {
        w.put(sq[i].ll - zl_ll_base[c[0]], zl_ll_bits[c[0]]);
        w.put(sq[i].ml - zl_ml_base[c[2]], zl_ml_bits[c[2]]);
        w.put(sq[i].off + 3 - (1u << c[1]), (int)c[1]);
    };
    unsigned state[3] = {0, 0, 0};
    codes(n - 1, c);
    for (int x = 0; x < 3; ++x)
        if (!rle[x]) state[x] = t[x].list[t[x].first[c[x]]];
    extra(n - 1, c);
    for (int i = n - 2; i >= 0; --i) {
        codes(i, c);
#pragma unroll
        for (int o = 0; o < 3; ++o) {  // OF, ML, LL
            const int x = o == 0 ? 1 : o == 1 ? 2 : 0;
            if (rle[x]) continue;
            const ZFse& f = t[x];
            const unsigned v = state[x];
            int k = f.first[c[x]];
            while (!(f.base[f.list[k]] <= v && v < f.base[f.list[k]] + (1u << f.nb[f.list[k]]))) ++k;
            const unsigned u = f.list[k];
            w.put(v - f.base[u], f.nb[u]);
            state[x] = u;
        }
        extra(i, c);
    }
    if (!rle[2]) w.put(state[2], 6);
    if (!rle[1]) w.put(state[1], 5);
    if (!rle[0]) w.put(state[0], 6);
    w.put(1, 1);
    if (w.nacc > 0) w.byte((unsigned)w.acc);
    out_len[b] = w.ok ? w.n : 0;
}

__global__ void __launch_bounds__(ZC_THREADS) zl_choose_kernel(ZGeom g, const u8* __restrict__ lits, const unsigned* __restrict__ nlit,
                                                              const u8* __restrict__ lslots, const ZMeta* __restrict__ lmeta,
                                                              const u8* __restrict__ sbuf, const unsigned* __restrict__ slen,
                                                              u8* __restrict__ slots, ZMeta* __restrict__ meta)
{
    const long long b = blockIdx.x;
    const int tid = threadIdx.x;
    const unsigned sl = slen[b];
    const unsigned kind1 = meta[b].kind, len1 = meta[b].out_len;
    if (sl == 0 || kind1 == ZB_RLE) return;
    const ZMeta& lm = lmeta[b];
    const unsigned body = lm.out_len + sl;
    if (3 + body >= len1) return;  // coder 1's form wins ties
    u8* o = slots + (size_t)b * ZC_SLOT;
    const u8* ls = lslots + (size_t)b * ZC_SLOT;
    if (tid == 0) {
        const unsigned last = b % g.bpp == g.bpp - 1;
        const unsigned h = last | ZB_COMP << 1 | body << 3;
        o[0] = (u8)h;
        o[1] = (u8)(h >> 8);
        o[2] = (u8)(h >> 16);
    }
    unsigned at = 3;
    for (unsigned j = tid; j < lm.head_len; j += ZC_THREADS) o[at + j] = ls[j];
    at += lm.head_len;
    if (lm.kind == ZB_COMP) {
        for (unsigned q = 0; q < lm.nstreams; ++q) {
            for (unsigned j = tid; j < lm.s_len[q]; j += ZC_THREADS) o[at + j] = ls[lm.s_off[q] + j];
            at += lm.s_len[q];
        }
    } else if (lm.kind == ZB_RAW) {
        const u8* lp = lits + b * ZC_BLOCK;
        for (unsigned j = tid; j < nlit[b]; j += ZC_THREADS) o[at + j] = lp[j];
        at += nlit[b];
    }
    const u8* sp = sbuf + b * ZC_BLOCK;
    for (unsigned j = tid; j < sl; j += ZC_THREADS) o[at + j] = sp[j];
    __syncthreads();  // every thread has read meta[b]
    if (tid == 0) {
        ZMeta m = {};
        m.out_len = m.head_len = 3 + body;
        m.kind = ZB_LZ;
        meta[b] = m;
    }
}

// the sort of one chunk of blocks: its buffers, and the CUB work space for a chunk of `blocks` blocks
size_t lz_sort_temp_bytes(long long blocks)
{
    size_t t = 0;
    cub::DoubleBuffer<unsigned long long> k(nullptr, nullptr);
    cub::DoubleBuffer<unsigned> v(nullptr, nullptr);
    cub::DeviceSegmentedRadixSort::SortPairs(nullptr, t, k, v, (int)(blocks * ZC_BLOCK), (int)blocks, (const int*)nullptr,
                                             (const int*)nullptr);
    return t;
}
}  // namespace

static bool zc_geometry(long long n, long long bytes_each, long long segment, ZGeom& g, long long& nb)
{
    g.bytes_each = bytes_each;
    g.seg = segment > 0 && segment < bytes_each ? segment : (bytes_each > 0 ? bytes_each : 1);
    g.bps = (g.seg + ZC_BLOCK - 1) / ZC_BLOCK;
    const long long nseg = bytes_each > 0 ? (bytes_each + g.seg - 1) / g.seg : 1;
    const long long last = bytes_each > 0 ? bytes_each - (nseg - 1) * g.seg : 0;
    g.bpp = bytes_each > 0 ? (nseg - 1) * g.bps + (last + ZC_BLOCK - 1) / ZC_BLOCK : 1;
    nb = n * g.bpp;
    return nb <= 0x7FFFFFFFll;
}

size_t zcoder_scratch_bytes(long long n, long long bytes_each, long long segment)
{
    ZGeom g;
    long long nb;
    zc_geometry(n, bytes_each, segment, g, nb);
    return (size_t)nb * (ZC_SLOT + sizeof(ZMeta) + 8) + (size_t)(n + 1) * 8 + 256;
}

// coder 2's part of the scratch, behind coder 1's: per block a literals slot + meta, the literal bytes, the sequences, the
// sequences section and three counts; then the buffers of one candidate sort
struct LzScratch {
    u8 *lslots, *lits, *sbuf;
    ZMeta* lmeta;
    ZSeq* seqs;
    unsigned *nseq, *nlit, *slen;
    unsigned long long* keys[2];
    unsigned* pos[2];
    int *seg_begin, *seg_end;
    void* temp;
    size_t temp_bytes;
    size_t total;
};

static LzScratch lz_scratch(char* base, long long n, long long bytes_each, long long segment)
{
    ZGeom g;
    long long nb;
    zc_geometry(n, bytes_each, segment, g, nb);
    const long long chunk = nb < LZ_SORT_BLOCKS ? nb : LZ_SORT_BLOCKS;
    size_t at = (zcoder_scratch_bytes(n, bytes_each, segment) + 255) & ~(size_t)255;
    auto take = [&](size_t bytes) {
        char* p = base ? base + at : nullptr;
        at += (bytes + 255) & ~(size_t)255;
        return p;
    };
    LzScratch z;
    z.lslots = (u8*)take((size_t)nb * ZC_SLOT);
    z.lmeta = (ZMeta*)take((size_t)nb * sizeof(ZMeta));
    z.lits = (u8*)take((size_t)nb * ZC_BLOCK);
    z.seqs = (ZSeq*)take((size_t)nb * LZ_MAX_SEQ * sizeof(ZSeq));
    z.sbuf = (u8*)take((size_t)nb * ZC_BLOCK);
    z.nseq = (unsigned*)take((size_t)nb * 4);
    z.nlit = (unsigned*)take((size_t)nb * 4);
    z.slen = (unsigned*)take((size_t)nb * 4);
    for (int i = 0; i < 2; ++i) z.keys[i] = (unsigned long long*)take((size_t)chunk * ZC_BLOCK * 8);
    for (int i = 0; i < 2; ++i) z.pos[i] = (unsigned*)take((size_t)chunk * ZC_BLOCK * 4);
    z.seg_begin = (int*)take((size_t)chunk * 4);
    z.seg_end = (int*)take((size_t)chunk * 4);
    z.temp_bytes = lz_sort_temp_bytes(chunk);
    z.temp = take(z.temp_bytes);
    z.total = at;
    return z;
}

size_t zcoder_lz_scratch_bytes(long long n, long long bytes_each, long long segment)
{
    return lz_scratch(nullptr, n, bytes_each, segment).total;
}

long long zcoder_frame_bound(long long bytes_each, long long segment)
{
    ZGeom g;
    long long nb;
    zc_geometry(1, bytes_each, segment, g, nb);
    return ZC_FRAME_HEAD + 3 * g.bpp + bytes_each;
}

static int zstd_encode(bool lz, const u8* src, long long n, long long bytes_each, long long segment, u8* dst, long long dst_stride,
                       int rec_head, long long* sizes, long long** frame_offsets, void* scratch, cudaStream_t st)
{
    if (n <= 0) return 0;
    ZGeom g;
    long long nb;
    if (!zc_geometry(n, bytes_each, segment, g, nb)) {
        set_error("zstd_encode: too many blocks in one batch (%lld)", nb);
        return -1;
    }
    u8* slots = (u8*)scratch;
    ZMeta* meta = (ZMeta*)(slots + (size_t)nb * ZC_SLOT);
    long long* boff = (long long*)(meta + nb);
    long long* foff = boff + nb;
    RIRB_LAUNCH(zc_block_kernel, (unsigned)nb, ZC_THREADS, 0, st, src, g, slots, meta);
    if (lz) {
        const LzScratch z = lz_scratch((char*)scratch, n, bytes_each, segment);
        for (long long b0 = 0; b0 < nb; b0 += LZ_SORT_BLOCKS) {
            const long long nbc = nb - b0 < LZ_SORT_BLOCKS ? nb - b0 : LZ_SORT_BLOCKS;
            RIRB_LAUNCH(zl_keys_kernel, (unsigned)nbc, ZC_THREADS, 0, st, src, g, b0, z.keys[0], z.pos[0], z.seg_begin, z.seg_end);
            cub::DoubleBuffer<unsigned long long> k(z.keys[0], z.keys[1]);
            cub::DoubleBuffer<unsigned> v(z.pos[0], z.pos[1]);
            size_t temp = z.temp_bytes;
            RIRB_CUDA_OK(cub::DeviceSegmentedRadixSort::SortPairs(z.temp, temp, k, v, (int)(nbc * ZC_BLOCK), (int)nbc, z.seg_begin,
                                                                  z.seg_end, 0, 64, st));
            int* cand = (int*)k.Alternate();  // the keys before the sort are not needed any more
            RIRB_LAUNCH(zl_cand_kernel, (unsigned)nbc, ZC_THREADS, 0, st, k.Current(), v.Current(), z.seg_begin, z.seg_end, cand);
            RIRB_LAUNCH(zl_parse_kernel, (unsigned)((nbc + LZ_WARPS - 1) / LZ_WARPS), 32 * LZ_WARPS, 0, st, src, g, b0, nbc, cand,
                        z.lits, z.seqs, z.nseq, z.nlit);
        }
        RIRB_LAUNCH(zl_lit_kernel, (unsigned)nb, ZC_THREADS, 0, st, z.lits, z.nlit, z.lslots, z.lmeta);
        RIRB_LAUNCH(zl_seq_kernel, (unsigned)((nb + LZ_SEQ_THREADS - 1) / LZ_SEQ_THREADS), LZ_SEQ_THREADS, 0, st, z.seqs, z.nseq, nb,
                    z.sbuf, z.slen);
        RIRB_LAUNCH(zl_choose_kernel, (unsigned)nb, ZC_THREADS, 0, st, g, z.lits, z.nlit, z.lslots, z.lmeta, z.sbuf, z.slen, slots, meta);
    }
    RIRB_LAUNCH(zc_layout_kernel, 1, 1024, 0, st, meta, n, g.bpp, dst_stride, rec_head, sizes, foff, boff);
    RIRB_LAUNCH(zc_copy_kernel, (unsigned)nb, ZC_THREADS, 0, st, src, g, slots, meta, foff, boff, rec_head, dst);
    if (frame_offsets) *frame_offsets = foff;
    return 0;
}

int launch_zstd_encode(const u8* src, long long n, long long bytes_each, long long segment, u8* dst, long long dst_stride,
                       int rec_head, long long* sizes, long long** frame_offsets, void* scratch, cudaStream_t st)
{
    return zstd_encode(false, src, n, bytes_each, segment, dst, dst_stride, rec_head, sizes, frame_offsets, scratch, st);
}

int launch_zstd_encode_lz(const u8* src, long long n, long long bytes_each, long long segment, u8* dst, long long dst_stride,
                          int rec_head, long long* sizes, long long** frame_offsets, void* scratch, cudaStream_t st)
{
    return zstd_encode(true, src, n, bytes_each, segment, dst, dst_stride, rec_head, sizes, frame_offsets, scratch, st);
}

}  // namespace rirb

using namespace rirb;

static int encode_batch(bool lz, const unsigned char* src, long long n, long long bytes_each, long long segment, unsigned char* dst,
                        long long dst_stride, long long* sizes)
{
    const char* name = lz ? "zstd_encode_batch_lz" : "zstd_encode_batch";
    if (!src || !dst || !sizes || n < 0 || bytes_each < 0 || bytes_each > 0xFFFFFFFFll || segment < 0 ||
        dst_stride < zcoder_frame_bound(bytes_each, segment)) {
        set_error("%s: bad arguments (dst_stride must be at least %lld)", name, zcoder_frame_bound(bytes_each, segment));
        return -1;
    }
    if (n == 0) return 0;
    if (rirb_device_count() <= 0) {
        set_error("%s: no CUDA device (the coder is a CUDA kernel; no CPU fallback)", name);
        return -1;
    }
    if (refuse_pageable(name, {{"src", src, 0}, {"dst", dst, 0}, {"sizes", sizes, 0}}) ||
        refuse_overlap(name, {{"src", src, (size_t)n * (size_t)bytes_each}},
                       {{"dst", dst, (size_t)n * (size_t)dst_stride}, {"sizes", sizes, sizeof(long long) * (size_t)n}}))
        return -1;
    cudaStream_t st = current_stream();
    void* scratch = nullptr;
    RIRB_CUDA_OK(cudaMallocAsync(&scratch, lz ? zcoder_lz_scratch_bytes(n, bytes_each, segment) : zcoder_scratch_bytes(n, bytes_each, segment), st));
    const int rc = (lz ? launch_zstd_encode_lz : launch_zstd_encode)(src, n, bytes_each, segment, dst, dst_stride, 0, sizes, nullptr, scratch, st);
    RIRB_CUDA_OK(cudaFreeAsync(scratch, st));
    return rc;
}

extern "C" int rirb_zstd_encode_batch(const unsigned char* src, long long n, long long bytes_each, long long segment,
                                      unsigned char* dst, long long dst_stride, long long* sizes)
{
    return encode_batch(false, src, n, bytes_each, segment, dst, dst_stride, sizes);
}

extern "C" int rirb_zstd_encode_batch_lz(const unsigned char* src, long long n, long long bytes_each, long long segment,
                                         unsigned char* dst, long long dst_stride, long long* sizes)
{
    return encode_batch(true, src, n, bytes_each, segment, dst, dst_stride, sizes);
}
