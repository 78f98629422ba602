// librir_b200/csrc/translate.cu -- sub-pixel translation (the resampling step of motion correction).
//
// Reference semantics: rir::translate<T,U> Filters.h:249-326 (+ TranslateBorder :238-244,
// detail::wrap/cast :231-235), C facade signal_processing.cpp:14-73, motion-correction variant
// removeMotionGeneric IRFileLoader.cpp:617-627.  Restated in SURVEY.md appendix A.4.
//
// Arithmetic: source coordinates in float32, blend in float64 with the reference's operation
// order and NO fused multiply-add (__dmul_rn/__dadd_rn), truncating store -- so integer outputs
// are bit-identical to the reference, not merely within +-1 LSB.
//
// Three kernels:
//   translate_generic_kernel<T,U>  every dtype / strategy, one thread per destination pixel.
//   translate_u16_tma_kernel       the uint16 hot path: the source window of a 128x128 destination
//                                  tile is fetched by ONE TMA box load at the per-frame position
//                                  (x0 + floor(-dx), y0 + floor(-dy)); a thread turns 8
//                                  pixels of a row with two 128-bit shared-memory reads, the
//                                  vertical blend in exact 64-bit integer arithmetic and 4 fp64
//                                  operations per pixel, no type conversions (see the comments there).
//   translate_u16_kernel           same arithmetic without shared memory, 4 pixels per thread:
//                                  widths that are not a multiple of 8 / unaligned buffers.
#include <stdlib.h>

#include "common.cuh"
#include "kernels.h"
#include "sort9.cuh"
#include "tma.cuh"

namespace rirb {

// ------------------------------------------------------------------------------------------------
// pixel traits: promotion to double in the blend, detail::cast<U>(double) on the way out
// ------------------------------------------------------------------------------------------------
template <typename T> struct Pix {
    __device__ static __forceinline__ double to_double(T v) { return (double)v; }
    __device__ static __forceinline__ T from_double(double v) { return (T)v; }  // cvt.rzi for integers, rn for float
};
struct BoolPix {  // storage type of numpy bool: one byte, 0/1
    u8 v;
};
template <> struct Pix<BoolPix> {
    __device__ static __forceinline__ double to_double(BoolPix b) { return b.v ? 1.0 : 0.0; }  // bool -> int -> double
    __device__ static __forceinline__ BoolPix from_double(double v) { return BoolPix{(u8)(v != 0.0)}; }
};

// (size_t)float as x86-64 evaluates it for negative inputs: truncate as signed 64-bit, reinterpret.
__device__ __forceinline__ unsigned long long f2size(float v) { return (unsigned long long)(long long)v; }
__device__ __forceinline__ unsigned long long wrap_idx(unsigned long long v, unsigned long long n) { return (v + n) % n; }

__device__ __forceinline__ double blend4(double p1, double p2, double p3, double p4, double u, double v)
{
    const double omv = __dsub_rn(1.0, v);
    const double omu = __dsub_rn(1.0, u);
    const double left = __dadd_rn(__dmul_rn(p1, omv), __dmul_rn(p2, v));
    const double right = __dadd_rn(__dmul_rn(p3, omv), __dmul_rn(p4, v));
    return __dadd_rn(__dmul_rn(left, omu), __dmul_rn(right, u));
}

// Source accessors: where translate_pixel reads src[row][col] from.
// The reference indexes the image flat, src[col + row * w], and its in-range branch can produce col = w + 1 or
// row = h + 1: when px (py) lies within half a float ulp below w (h), px + 1.0f rounds UP to the next integer, the
// `rt == w` clamp does not fire, and Filters.h:300-310 reads one pixel into the next row -- or, on the last row(s),
// past the end of the buffer (undefined there).  Every accessor keeps the flat meaning (so the defined cases match
// the reference bit for bit) and clamps the index to the frame's last pixel (so the undefined ones stay in bounds).
template <typename T> struct GlobalSrc {
    const T* __restrict__ p;
    int w;
    long long npx;  // w * h
    __device__ __forceinline__ T operator()(long long row, long long col) const
    {
        const long long i = row * w + col;
        return p[i < npx ? i : npx - 1];
    }
};

// One destination pixel, any strategy.  Returns false when dst must be left untouched.
template <typename T, typename U, typename SRC>
__device__ __forceinline__ bool translate_pixel(const SRC& src, int w, int h, int x, int y, float dx, float dy, int strategy,
                                                U background, U& result)
{
    const float px = (float)x - dx;
    const float py = (float)y - dy;
    const float fw = (float)w, fh = (float)h;
    long long l, rt, t, b;
    double u, v;
    if (px < 0 || px >= fw || py < 0 || py >= fh) {
        if (strategy == STRAT_NOBORDER) return false;
        if (strategy == STRAT_BACKGROUND) {
            result = background;
            return true;
        }
        if (strategy == STRAT_NEAREST) {
            long long sx = px < 0 ? 0 : (px >= fw ? w - 1 : (long long)px);
            long long sy = py < 0 ? 0 : (py >= fh ? h - 1 : (long long)py);
            // plain conversion T -> U (identity for the facade; u16 -> float in the motion variant)
            result = Pix<U>::from_double(Pix<T>::to_double(src(sy, sx)));
            return true;
        }
        l = (long long)wrap_idx(f2size(px), (unsigned long long)w);
        rt = (long long)wrap_idx(f2size(px + 1.0f), (unsigned long long)w);
        t = (long long)wrap_idx(f2size(py), (unsigned long long)h);
        b = (long long)wrap_idx(f2size(py + 1.0f), (unsigned long long)h);
        u = (double)fabsf(px - (float)(int)px);
        v = (double)fabsf(py - (float)(int)py);
    } else {
        l = (long long)px;
        rt = (long long)(px + 1.0f);
        if (rt == w) rt = l;
        t = (long long)py;
        b = (long long)(py + 1.0f);
        if (b == h) b = t;
        u = (double)(px - (float)l);
        v = (double)((float)b - py);
    }
    const double p1 = Pix<T>::to_double(src(b, l));
    const double p2 = Pix<T>::to_double(src(t, l));
    const double p3 = Pix<T>::to_double(src(b, rt));
    const double p4 = Pix<T>::to_double(src(t, rt));
    result = Pix<U>::from_double(blend4(p1, p2, p3, p4, u, v));
    return true;
}
template <typename T, typename U>
__device__ __forceinline__ bool translate_pixel(const T* __restrict__ src, int w, int h, int x, int y, float dx, float dy,
                                                int strategy, U background, U& result)
{
    return translate_pixel<T, U>(GlobalSrc<T>{src, w, (long long)w * h}, w, h, x, y, dx, dy, strategy, background, result);
}

template <typename T>
__global__ void __launch_bounds__(256)
translate_generic_kernel(const T* __restrict__ src, T* __restrict__ dst, int w, int h, long long nframes, size_t frame_stride,
                         const float* __restrict__ dxs, const float* __restrict__ dys, float dx0, float dy0, int strategy,
                         T background)
{
    const int x = blockIdx.x * blockDim.x + threadIdx.x;
    const int y = blockIdx.y * blockDim.y + threadIdx.y;
    if (x >= w || y >= h) return;
    for (long long f = blockIdx.z; f < nframes; f += gridDim.z) {
        const float dx = dxs ? dxs[f] : dx0;
        const float dy = dys ? dys[f] : dy0;
        T r;
        if (translate_pixel<T, T>(src + f * frame_stride, w, h, x, y, dx, dy, strategy, background, r))
            dst[f * frame_stride + (size_t)y * w + x] = r;
    }
}

template <typename T>
static int launch_generic(const void* src, void* dst, int w, int h, long long nframes, const float* dxs, const float* dys,
                          float dx0, float dy0, int strategy, const void* background_host, cudaStream_t st)
{
    T bg = *reinterpret_cast<const T*>(background_host);
    dim3 block(32, 8);
    dim3 grid((unsigned)ceil_div(w, 32), (unsigned)ceil_div(h, 8), (unsigned)min(nframes, 32768LL));
    RIRB_LAUNCH(translate_generic_kernel<T>, grid, block, 0, st, (const T*)src, (T*)dst, w, h, nframes, (size_t)w * h, dxs, dys,
                dx0, dy0, strategy, bg);
    return 0;
}

// ------------------------------------------------------------------------------------------------
// uint16 hot path
// ------------------------------------------------------------------------------------------------
// Exact-integer vertical blend.  For a destination row, py = (float)y - dy, and in the in-range
// case v = (float)b - py, 1-v are the reference's vertical weights.  Whenever v is a multiple of
// 2^-23 with |v| <= 1 (always true for |py| >= 1, where float32 spacing is >= 2^-23 ... 2^-13)
// both weights are integers/2^23 below 2^24+1, a pixel is below 2^16, so
//     p_b*(1-v) + p_t*v  =  (p_b*A + p_t*B) / 2^23,   A = (1-v)*2^23, B = v*2^23
// has at most 41 significant bits: each fp64 product and their sum in the reference are EXACT,
// and equal the integer N = p_b*A + p_t*B scaled by 2^-23.  N is formed with two 64-bit integer
// multiply-adds and turned into the double N*2^-23 by writing it into the mantissa of 2^29 and
// subtracting 2^29 (one exact DADD).  Rows where the condition fails (0 <= py < 1 with a finer
// fraction, e.g. denormal shifts) take the plain fp64 column blend.  The horizontal blend keeps
// the reference's rounded fp64 operations: c_l*(1-u) + c_r*u.
__device__ __forceinline__ double int_to_double_scaled23(long long n)
{
    // n in [0, 2^41): double with exponent of 2^29 has ulp 2^-23 => bits = bits(2^29) + n
    const long long bits = 0x41C0000000000000LL + n;
    return __dsub_rn(__longlong_as_double(bits), 536870912.0);
}

constexpr int TR_PX = 4;  // destination pixels per thread

template <bool MOTION>
__global__ void __launch_bounds__(256)
translate_u16_kernel(const u16* __restrict__ src, u16* __restrict__ dst, int w, int h, long long nframes, size_t src_stride,
                     size_t dst_stride, const float* __restrict__ dxs, const float* __restrict__ dys, float dx0, float dy0,
                     int strategy, unsigned background)
{
    const int xg = blockIdx.x * blockDim.x + threadIdx.x;  // group of TR_PX pixels
    const int y = blockIdx.y * blockDim.y + threadIdx.y;
    const int x0 = xg * TR_PX;
    if (x0 >= w || y >= h) return;
    const float fw = (float)w, fh = (float)h;
    for (long long f = blockIdx.z; f < nframes; f += gridDim.z) {
        const float dx = dxs ? dxs[f] : dx0;
        const float dy = dys ? dys[f] : dy0;
        const u16* frame = src + f * src_stride;
        u16* orow = dst + f * dst_stride + (size_t)y * w + x0;
        const float py = (float)y - dy;
        const bool row_in = !(py < 0 || py >= fh);
        // fast path: whole group in range, source columns consecutive, v on the 2^-23 grid
        const float px_first = (float)x0 - dx;
        const float px_last = (float)(x0 + TR_PX - 1) - dx;
        bool fast = row_in && (x0 + TR_PX <= w) && !(px_first < 0) && (px_last < fw);
        long long l0 = 0;
        int t = 0, b = 0;
        float vf = 0.f;
        if (fast) {
            l0 = (long long)px_first;
            t = (int)py;
            b = (int)(py + 1.0f);
            if (b == h) b = t;
            vf = (float)b - py;
            const float vs = vf * 8388608.0f;
            fast = (vs == truncf(vs)) && (fabsf(vf) <= 1.0f);
#pragma unroll
            for (int i = 0; i < TR_PX; ++i) {  // l_i = l0+i and rt_i = l_i+1, as the reference would compute them
                const float pxi = (float)(x0 + i) - dx;
                fast = fast && ((long long)pxi == l0 + i) && ((long long)(pxi + 1.0f) == l0 + i + 1);
            }
        }
        if (fast) {
            const int B = (int)(vf * 8388608.0f);
            const int A = 8388608 - B;
            const u16* rb = frame + (size_t)b * w + l0;
            const u16* rt_ = frame + (size_t)t * w + l0;
            const int ncol = (l0 + TR_PX < w) ? TR_PX + 1 : TR_PX;  // right edge: rt clamps to l
            double c[TR_PX + 1];
#pragma unroll
            for (int i = 0; i <= TR_PX; ++i) {
                if (i < ncol) {
                    long long n = (long long)rb[i] * A + (long long)rt_[i] * B;
                    c[i] = int_to_double_scaled23(n);
                } else {
                    c[i] = c[i - 1];
                }
            }
            unsigned outv[TR_PX];
#pragma unroll
            for (int i = 0; i < TR_PX; ++i) {
                const float px = (float)(x0 + i) - dx;
                const double u = (double)(px - (float)(l0 + i));
                const double omu = __dsub_rn(1.0, u);
                const double val = __dadd_rn(__dmul_rn(c[i], omu), __dmul_rn(c[i + 1], u));
                outv[i] = MOTION ? (unsigned)(u16)(float)val : (unsigned)(u16)val;
            }
            if ((((uintptr_t)orow) & 7u) == 0) {
                uint2 o;
                o.x = outv[0] | (outv[1] << 16);
                o.y = outv[2] | (outv[3] << 16);
                *reinterpret_cast<uint2*>(orow) = o;
            } else {
#pragma unroll
                for (int i = 0; i < TR_PX; ++i) orow[i] = (u16)outv[i];
            }
        } else {
#pragma unroll
            for (int i = 0; i < TR_PX; ++i) {
                if (x0 + i < w) {
                    if (MOTION) {
                        float r;
                        if (translate_pixel<u16, float>(frame, w, h, x0 + i, y, dx, dy, strategy, (float)background, r))
                            orow[i] = (u16)r;
                    } else {
                        u16 r;
                        if (translate_pixel<u16, u16>(frame, w, h, x0 + i, y, dx, dy, strategy, (u16)background, r)) orow[i] = r;
                    }
                }
            }
        }
    }
}

// ------------------------------------------------------------------------------------------------
// uint16 hot path, TMA-tiled
// ------------------------------------------------------------------------------------------------
// Destination tile TT_W x TT_H; its source window is [x0+sx, x0+sx+TT_W+2) x [y0+sy, y0+sy+TT_H+2)
// with sx = floor(-dx), sy = floor(-dy): the real source coordinate x-dx lies in [x+sx, x+sx+1), its
// float32 rounding px in [x+sx, x+sx+1], so l = trunc(px) is x+sx (or x+sx+1 when px rounds up to
// the integer -- those rare groups take the per-pixel routine) and rt <= l+1.
// TMA wants the box's innermost start coordinate on a 16-byte boundary (measured: any other x
// traps, scripts/probes/tma_probe.cu), so the box starts at (x0+sx) rounded down to 8 pixels and
// every thread of the CTA applies the same residual offset XOFF = 0..7 when it unpacks its two
// 128-bit shared-memory reads: the row routine is instantiated for the 8 offsets and picked by a
// CTA-uniform switch.
//
// Per thread: 8 consecutive destination pixels of one row, validated through a few probe pixels:
//   * px_i = RN32(x_i - dx) sits on a grid g_i = ulp(px_i) that only gets coarser with i, and the
//     fraction it carries is u_i = RN_{g_i}(frac(-dx)).  If u is equal at both ends of a run of
//     pixels it is representable on both grids, hence on every grid in between: uniform on the run.
//   * the grid changes where px crosses a power of two P >= 8, i.e. at source column l = P, a
//     multiple of 8; a group starts at source column 8m + XOFF, so inside a group the change can
//     only sit between pixel 7-XOFF and pixel 8-XOFF -- a COMPILE-TIME position in the XOFF
//     instance.  A thread therefore carries two sets of horizontal weights, (a) from pixel 0 for
//     pixels < 8-XOFF and (b) from pixel 7 for the rest, checked at the two pixels next to the split.
//     (Groups that still fail -- source columns below 8, where grids change at 1, 2, 4 -- are slow.)
//   * a round-up of px_i (or of px_i + 1.0f, which decides rt) to the next integer needs
//     frac >= 1 - g/2; if it happens at some i it also happens at the coarser pixel 7 (ties go to
//     the even neighbour, which is the integer, on every grid < 1), so l_7 == l_0 + 7 and
//     trunc(px + 1) == l + 1 at pixel 7 and at the last pixel of run (a) exclude it for the group.
// With u uniform on a run, (1-u) and u are thread constants, and with M_j = 2^29 + c_j (c_j the exact
// column blend, see int_to_double_scaled23) the reference's RN(c_l*(1-u)) is one DFMA:
//   RN(M_l*(1-u) - 2^29*(1-u)) = RN((M_l - 2^29)*(1-u))      (the FMA product is exact, 2^29*(1-u) is exact)
// so a pixel costs 2 DFMA + 1 DADD + one DADD.RM with 2^52 that leaves trunc(val) in the low word
// (val >= 0): 4 fp64 instructions and no F2I/I2F/F2F (those issue at 16/clk/SM and were the limiter of
// the 4-pixel kernel: profiles/r1_v1_ncu_summary.md).
//
// Warp shape: 2 column groups x 16 rows, so that the slow groups (image edges, source columns < 8)
// are confined to the warps that own the edge columns instead of costing every warp of an edge tile
// a divergent detour.  Row pitch 288 B keeps the 128-bit reads of 4 rows x 2 groups conflict-free.
constexpr int TT_W = 128, TT_H = 64;
constexpr int TT_BW = TT_W + 16, TT_BH = TT_H + 2;  // box: thread c reads columns [8c, 8c+16); +2 rows
constexpr int TT_THREADS = 256;

struct HWeights {  // horizontal weights of a run of pixels with the same fraction u
    double u, omu, k_l, k_r;
};
__device__ __forceinline__ HWeights make_hweights(float uf)
{
    HWeights c;
    c.u = (double)uf;
    c.omu = __dsub_rn(1.0, c.u);
    c.k_l = __dmul_rn(-536870912.0, c.omu);
    c.k_r = __dmul_rn(-536870912.0, c.u);
    // keep them in registers: ptxas otherwise re-derives them with two DMULs per row
    asm volatile("" : "+d"(c.k_l), "+d"(c.k_r));
    return c;
}

// columns D .. D+8 of the 16 pixels held in two 128-bit words (little-endian pairs)
template <int D>
__device__ __forceinline__ void unpack9(const uint4& a, const uint4& b, unsigned (&p)[9])
{
    const unsigned wv[8] = {a.x, a.y, a.z, a.w, b.x, b.y, b.z, b.w};
#pragma unroll
    for (int j = 0; j < 9; ++j) {
        const int c = D + j;
        p[j] = (c & 1) ? (wv[c >> 1] >> 16) : (wv[c >> 1] & 0xFFFFu);
    }
}

// One fast group: 8 destination pixels from the two staged source rows.
__device__ __forceinline__ uint4 lds128(uint32_t addr)
{
    uint4 v;
    asm volatile("ld.shared.v4.u32 {%0,%1,%2,%3}, [%4];" : "=r"(v.x), "=r"(v.y), "=r"(v.z), "=r"(v.w) : "r"(addr));
    return v;
}

// rowb / rowt: shared-memory byte addresses of the thread's 16 staged pixels in the bottom / top row
template <int XOFF, bool MOTION>
__device__ __forceinline__ void blend_group(uint32_t rowb, uint32_t rowt, unsigned A, unsigned B, bool clamp_rt,
                                            const HWeights& ca, const HWeights& cb, unsigned long long magic, u16* orow)
{
    unsigned pb[9], pt[9];
    unpack9<XOFF>(lds128(rowb), lds128(rowb + 16), pb);
    unpack9<XOFF>(lds128(rowt), lds128(rowt + 16), pt);
    if (clamp_rt) {  // rt of the last pixel clamps to its l (Filters.h:309)
        pb[8] = pb[7];
        pt[8] = pt[7];
    }
    double m[9];
#pragma unroll
    for (int j = 0; j < 9; ++j) {  // bits(2^29) + N: the double 2^29 + N * 2^-23, N = p_b*A + p_t*B < 2^40 (two IMAD.WIDE.U32)
        unsigned long long n = (unsigned long long)pb[j] * A + magic;  // magic = bits(2^29), a register pair: one IMAD.WIDE
        n += (unsigned long long)pt[j] * B;
        m[j] = __longlong_as_double((long long)n);
    }
    unsigned o[8];
#pragma unroll
    for (int j = 0; j < 8; ++j) {
        const HWeights& c = (XOFF != 0 && j >= 8 - XOFF) ? cb : ca;  // static choice
        const double val = __dadd_rn(__fma_rn(m[j], c.omu, c.k_l), __fma_rn(m[j + 1], c.u, c.k_r));
        if (MOTION)
            o[j] = (unsigned)(u16)(float)val;  // double -> float (nearest) -> uint16 (truncation), IRFileLoader.cpp:624
                                               // (an fp64-only emulation of the two conversions measured slower: the kernel
                                               // is issue-bound, and it costs 5 instructions instead of 2)
        else
            o[j] = (unsigned)__double2loint(__dadd_rd(val, 4503599627370496.0));  // trunc(val), 0 <= val < 2^16
    }
    uint4 ov;
    ov.x = __byte_perm(o[0], o[1], 0x5410);
    ov.y = __byte_perm(o[2], o[3], 0x5410);
    ov.z = __byte_perm(o[4], o[5], 0x5410);
    ov.w = __byte_perm(o[6], o[7], 0x5410);
    st_stream(reinterpret_cast<uint4*>(orow), ov);
}

// Staged box first, global memory for the few source pixels outside it (clamped / wrapped borders).
struct TileSrc {
    const u16* tile;  // [TT_BH][TT_BW], box origin (xs, ys)
    const u16* __restrict__ frame;
    int xs, ys, w, h;
    __device__ __forceinline__ u16 operator()(long long row, long long col) const
    {
        const long long r = row - ys, c = col - xs;
        // col >= w / row >= h: the flat index of GlobalSrc (the box holds the hardware's zero fill there)
        if (col < w && row < h && r >= 0 && r < TT_BH && c >= 0 && c < TT_BW) return tile[r * TT_BW + c];
        const long long i = row * w + col, npx = (long long)w * h;
        return frame[i < npx ? i : npx - 1];
    }
};

// Per-row parameters, computed once per CTA (one thread per destination row, while the box is in
// flight) instead of by each of the 16 threads that share the row.
struct RowInfo {
    int B;       // v * 2^23 (0 when the bottom row is clamped onto the top row); < 0: the row is slow
    unsigned rows;  // byte offsets in the staged box of the top (low half) / bottom (high half) source row
};
__device__ __forceinline__ RowInfo make_row_info(int y, int h, float dy, int ys)
{
    RowInfo ri;
    ri.B = -1;
    ri.rows = 0;
    const float fh = (float)h;
    const float py = (float)y - dy;
    const int t = (int)py;
    int b = (int)(py + 1.0f);
    if (b == h) b = t;
    const float vf = (float)b - py;
    const float vs = vf * 8388608.0f;  // v on the 2^-23 grid -> the vertical blend is exact in 64-bit integers
    const int tr = t - ys, br = b - ys;
    if (y < h && !(py < 0) && (py < fh) && (vs == truncf(vs)) && (fabsf(vf) <= 1.0f) && (tr >= 0) && (br >= tr) && (br < TT_BH)) {
        ri.B = (br == tr) ? 0 : (int)vs;  // b == t (v = -frac): both rows are the same pixel, N = p * 2^23
        ri.rows = (unsigned)(tr * (TT_BW * 2)) | ((unsigned)(br * (TT_BW * 2)) << 16);
    }
    return ri;
}

static_assert(TT_BH * TT_BW * 2 <= 65536, "row byte offsets are packed in 16 bits");
static_assert(TT_H <= 64 && TT_W / 8 <= 16, "queue entries pack cx in 4 bits and the row in 6");

// ---- edge groups --------------------------------------------------------------------------------
// The first and the last 8-pixel group of an image row are where the regular structure breaks:
// some of their pixels have no source (px < 0 or px >= w: border strategy), and source columns
// below 8 change binade at 1, 2 and 4, so the fraction differs from pixel to pixel.  Their
// horizontal weights depend on (dx, x) only -- not on the row -- so the CTA that owns such a group
// tabulates them once per pixel in shared memory (EdgeTable) together with a mask of the pixels
// the table is valid for.  The groups still go through the CTA's queue (so that the work is
// spread over all threads instead of stalling the warp that owns the image edge), but a valid
// pixel of a regular row then costs the fast path's arithmetic instead of the literal routine.
struct EdgeTable {
    HWeights wt[8];
    unsigned valid;     // bit i: pixel i is in range, its source column is l0 + i and rt is l + 1 (or clamped)
    unsigned clamped;   // bit i: rt of pixel i clamps onto l (l == w - 1)
    unsigned outside;   // bit i: px of pixel i is < 0 or >= w: the border strategy decides (second-generation kernel only)
    unsigned below;     // bit i: px of pixel i is < 0 (an 8-pixel-wide image has both kinds in its one group)
};

// One pixel of an edge group in a regular row: the fast path's arithmetic with the pixel's own
// weights.  col: the pixel's source column l in the staged box.
template <bool MOTION>
__device__ __forceinline__ u16 blend_edge_pixel(const u16* tile, unsigned rows, unsigned A, unsigned B, int col, bool clamped,
                                                const HWeights& c)
{
    const u16* rt_ = tile + (rows & 0xFFFFu) / 2 + col;
    const u16* rb = tile + (rows >> 16) / 2 + col;
    const int r = clamped ? 0 : 1;
    const unsigned long long nl = (unsigned long long)rb[0] * A + (unsigned long long)rt_[0] * B + 0x41C0000000000000ULL;
    const unsigned long long nr = (unsigned long long)rb[r] * A + (unsigned long long)rt_[r] * B + 0x41C0000000000000ULL;
    const double val = __dadd_rn(__fma_rn(__longlong_as_double((long long)nl), c.omu, c.k_l),
                                 __fma_rn(__longlong_as_double((long long)nr), c.u, c.k_r));
    return MOTION ? (u16)(float)val : (u16)__double2loint(__dadd_rd(val, 4503599627370496.0));
}

// tbase: shared address of the thread's column slot in box row 0; rinfo: shared address of rowinfo[ry].
// Groups that cannot be done here are appended to the CTA's queue as cx | row << 4.
template <int XOFF, bool MOTION>
__device__ __forceinline__ void fast_rows(uint32_t tbase, uint32_t rinfo, bool xfast, bool clamp_rt, const HWeights& ca,
                                          const HWeights& cb, u16* ocol, size_t row_step, int cx, int ry, int rows_left,
                                          unsigned* slowq, unsigned* slow_count)
{
    unsigned long long magic = 0x41C0000000000000ULL;
    asm volatile("" : "+l"(magic));  // opaque: otherwise ptxas ORs the constant into every column's high word
#pragma unroll
    for (int k = 0; k < TT_H / 16; ++k) {
        int B;
        unsigned rows;
        asm volatile("ld.shared.v2.u32 {%0,%1}, [%2];" : "=r"(B), "=r"(rows) : "r"(rinfo + k * (16 * (int)sizeof(RowInfo))));
        if (xfast && B >= 0) {
            blend_group<XOFF, MOTION>(tbase + (rows >> 16), tbase + (rows & 0xFFFFu), 8388608u - (unsigned)B, (unsigned)B, clamp_rt, ca,
                                      cb, magic, ocol);
        } else if (ry + 16 * k < rows_left) {
            slowq[atomicAdd(slow_count, 1u)] = (unsigned)cx | ((unsigned)(ry + 16 * k) << 4);
        }
        ocol += row_step;
    }
}

// A CTA owns one 128-pixel column of tiles of one frame and walks down it: the horizontal weights
// depend on (dx, x) only and are computed once; the box of tile ty+1 is in flight (second shared
// memory stage, its own mbarrier) while tile ty is being blended.
constexpr int TT_STAGES = 2;
constexpr unsigned TT_STAGE_BYTES = (TT_BH * TT_BW * 2 + 127u) & ~127u;

// ---- fused reader front end (PLANES) --------------------------------------------------------------
// IRFileLoader::readImage's whole post-decode chain in ONE pass over HBM (SURVEY.md 8f-1): the source
// of a tile is not a uint16 frame but the decoder's two byte planes.  Per stage two TMA boxes (low
// bytes, high bytes; uint8 boxes start on 16-pixel boundaries) land in shared memory; the CTA merges
// them into the uint16 tile the blend reads (v = lo | hi << 8, h264.cpp:3030,3044; += min_T on the
// rows that ask for it, IRFileLoader.cpp:1174-1179), patches the flagged pixels of the tile with the
// loader's median (IRFileLoader.cpp:754-795) and then runs the motion translate (:617-627) exactly
// as the plain kernel does.  2 B/px read + 2 B/px written instead of three round trips.
constexpr int TP_BW = 160;                                      // plane box width (bytes = pixels)
constexpr unsigned TP_BOX_BYTES = TP_BW * TT_BH;                // one plane, one stage
constexpr unsigned TP_BOX_AL = (TP_BOX_BYTES + 127u) & ~127u;
constexpr unsigned TP_STAGE_BYTES = 2 * TP_BOX_AL;              // lo box + hi box
constexpr unsigned TP_SMEM_BYTES = TT_STAGES * TP_STAGE_BYTES + TT_STAGE_BYTES;  // + the merged uint16 tile

struct PlaneSrc {
    const u8* lo;            // [n][h_full][w] byte planes (global), for the medians and out-of-box reads
    const u8* hi;
    size_t plane_stride;     // h_full * w
    const int* xy;           // bad-pixel list of the w x h image (nullptr: no correction)
    const int* nbr;          // per entry: flagged cells of its shifted 3x3 window
    const int* row_off;      // first list entry of each row, h + 1 entries
    const u8* mask;          // bitmap (row stride (w + 7) / 8), used by out-of-box reads only
    unsigned min_t;          // added (mod 2^16) on rows < t_rows
    int t_rows;
    int h_full;              // rows of the stored frame; rows [h, h_full) are metadata: merged, not translated
};

__device__ __forceinline__ unsigned plane_px(const u8* __restrict__ lo, const u8* __restrict__ hi, int w, int x, int y, const PlaneSrc& ps)
{
    const size_t i = (size_t)y * w + x;
    return (((unsigned)lo[i] | ((unsigned)hi[i] << 8)) + (y < ps.t_rows ? ps.min_t : 0u)) & 0xFFFFu;
}
// the loader's median for flagged pixel (x, y) of the w x h image; false: no un-flagged cell (pixel stays)
__device__ __forceinline__ bool plane_median(const u8* __restrict__ lo, const u8* __restrict__ hi, int w, int h, int x, int y, int flags,
                                             const PlaneSrc& ps, unsigned& med)
{
    const int x0 = x == 0 ? 0 : (x == w - 1 ? w - 3 : x - 1);
    const int y0 = y == 0 ? 0 : (y == h - 1 ? h - 3 : y - 1);
    unsigned v[9];
    int c = 0;
#pragma unroll
    for (int k = 0; k < 9; ++k) {
        const unsigned val = plane_px(lo, hi, w, x0 + k / 3, y0 + k % 3, ps);
        const bool ok = !((flags >> k) & 1);
        v[k] = ok ? val : 0xFFFFFFFFu;
        c += ok;
    }
    if (c == 0) return false;
    sort9(v);
    med = pick_mid(v, c);
    return true;
}
// Source pixel of the corrected frame that is NOT in the staged tile (far clamped / wrapped reads): rebuilt from the planes.
__device__ __noinline__ unsigned plane_corrected_px(const u8* __restrict__ lo, const u8* __restrict__ hi, int w, int h, int x, int y,
                                                    const PlaneSrc& ps)
{
    unsigned v = plane_px(lo, hi, w, x, y, ps);
    if (ps.xy != nullptr) {
        const int mstride = (w + 7) >> 3;
        if (ps.mask[(size_t)y * mstride + (x >> 3)] & (1u << (x & 7))) {
            const int x0 = x == 0 ? 0 : (x == w - 1 ? w - 3 : x - 1);
            const int y0 = y == 0 ? 0 : (y == h - 1 ? h - 3 : y - 1);
            int flags = 0;
            for (int k = 0; k < 9; ++k) {
                const int xx = x0 + k / 3, yy = y0 + k % 3;
                if (ps.mask[(size_t)yy * mstride + (xx >> 3)] & (1u << (xx & 7))) flags |= 1 << k;
            }
            unsigned med;
            if (plane_median(lo, hi, w, h, x, y, flags, ps, med)) v = med;
        }
    }
    return v;
}
struct PlaneTileSrc {
    const u16* tile;  // merged [TT_BH][TT_BW], origin (xs, ys)
    const u8* __restrict__ lo;
    const u8* __restrict__ hi;
    const PlaneSrc* ps;
    int xs, ys, w, h;
    __device__ __forceinline__ u16 operator()(long long row, long long col) const
    {
        const long long r = row - ys, c = col - xs;
        if (col < w && row < h && r >= 0 && r < TT_BH && c >= 0 && c < TT_BW) return tile[r * TT_BW + c];
        long long i = row * w + col;  // flat meaning, clamped to the image (see GlobalSrc)
        const long long npx = (long long)w * h;
        i = i < npx ? i : npx - 1;
        return (u16)plane_corrected_px(lo, hi, w, h, (int)(i % w), (int)(i / w), *ps);
    }
};

// PLANES: tmap / tmap_hi describe the low / high byte planes and `src` is unused (see PlaneSrc).
template <bool MOTION, bool PLANES>
__global__ void __launch_bounds__(TT_THREADS, 3)
translate_u16_tma_kernel(const __grid_constant__ CUtensorMap tmap, const __grid_constant__ CUtensorMap tmap_hi,
                         const u16* __restrict__ src, u16* __restrict__ dst, int w, int h, size_t src_stride, size_t dst_stride,
                         const float* __restrict__ dxs, const float* __restrict__ dys, float dx0, float dy0, int strategy,
                         unsigned background, int tiles_y, const __grid_constant__ PlaneSrc ps)
{
    extern __shared__ __align__(128) unsigned char smem_raw[];
    __shared__ __align__(8) unsigned long long bar[TT_STAGES];
    __shared__ RowInfo rowinfo[2][TT_H];  // double-buffered with the queue counter: tile ty+1's are prepared
    __shared__ unsigned slow_count[2];    // between the two barriers of tile ty
    __shared__ unsigned slowq[(TT_W / 8) * TT_H];
    __shared__ EdgeTable edge_tab[2];  // [0]: the image's first group of a row, [1]: its last
    constexpr unsigned TILE_BYTES = PLANES ? 2 * TP_BOX_BYTES : TT_BH * TT_BW * 2;  // bytes one stage receives
    constexpr unsigned STAGE_BYTES = PLANES ? TP_STAGE_BYTES : TT_STAGE_BYTES;      // TMA destinations are 128-byte aligned
    const int f = blockIdx.y;
    const int x0t = blockIdx.x * TT_W;
    const float dx = dxs ? dxs[f] : dx0;
    const float dy = dys ? dys[f] : dy0;
    const float fw = (float)w, fh = (float)h;
    // integer part of the shift, kept in a range where the int arithmetic below cannot overflow
    // (a clamped value simply never matches l0, and the group takes the per-pixel routine)
    const int sx = (int)fminf(fmaxf(floorf(-dx), -fw - 16.f), fw + 16.f);
    const int sy = (int)fminf(fmaxf(floorf(-dy), -fh - 16.f), fh + 16.f);
    const int xs = (x0t + sx) & ~7;      // box origin: 16-byte aligned column
    const int xoff = (x0t + sx) - xs;    // 0..7, the same for every fast group of the CTA
    const int xs16 = (x0t + sx) & ~15;   // PLANES: the uint8 boxes start on 16-pixel boundaries; xs - xs16 is 0 or 8
    auto issue_boxes = [&](int s, int tile_row) {
        mbar_expect_tx(&bar[s], TILE_BYTES);
        if (PLANES) {
            tma_load_box(smem_raw + s * STAGE_BYTES, &tmap, &bar[s], xs16, tile_row * TT_H + sy, f);
            tma_load_box(smem_raw + s * STAGE_BYTES + TP_BOX_AL, &tmap_hi, &bar[s], xs16, tile_row * TT_H + sy, f);
        } else {
            tma_load_box(smem_raw + s * STAGE_BYTES, &tmap, &bar[s], xs, tile_row * TT_H + sy, f);
        }
    };
    if (threadIdx.x == 0) {
#pragma unroll
        for (int s = 0; s < TT_STAGES; ++s) mbar_init(&bar[s], 1);
        mbar_fence_init();
        slow_count[0] = 0;
    }
    if (threadIdx.x < TT_H) rowinfo[0][threadIdx.x] = make_row_info(threadIdx.x, h, dy, sy);
    if (threadIdx.x >= TT_THREADS - 32 && threadIdx.x < TT_THREADS - 16) {  // 16 lanes of the last warp: 2 tables x 8 pixels
        const int e = (threadIdx.x >> 3) & 1, i = threadIdx.x & 7;
        const int xe0 = e ? w - 8 : 0;
        const int x = xe0 + i;
        const float px = (float)x - dx;
        bool ok = (xe0 >= x0t) && (xe0 < x0t + TT_W) && !(px < 0) && (px < fw);
        const int l = (int)px;
        const int rt = (int)(px + 1.0f);
        const bool cl = ok && (rt == w) && (l == w - 1);
        ok = ok && (l == x + sx) && (cl || rt == l + 1);
        edge_tab[e].wt[i] = make_hweights(ok ? px - (float)l : 0.f);
        const unsigned vb = __ballot_sync(0x0000FFFFu, ok), cb2 = __ballot_sync(0x0000FFFFu, cl);
        if (i == 0) {
            edge_tab[e].valid = (vb >> (8 * e)) & 0xFFu;
            edge_tab[e].clamped = (cb2 >> (8 * e)) & 0xFFu;
        }
    }
    __syncthreads();
    if (threadIdx.x == 0) {
#pragma unroll
        for (int s = 0; s < TT_STAGES; ++s)
            if (s < tiles_y) issue_boxes(s, s);
    }

    // ---- per-thread column constants (while the first boxes are in flight) -----------------------
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int cx = 2 * warp + (lane & 1), ry = lane >> 1;
    const int x0 = x0t + 8 * cx;
    const int isplit = (8 - xoff) & 7;  // first pixel of run (b); 0: a single run
    const float pxf = (float)x0 - dx, pxl = (float)(x0 + 7) - dx;
    const int l0 = (int)pxf, l7 = (int)pxl;
    const float u0 = pxf - (float)l0, u7 = pxl - (float)l7;
    bool xfast = (x0 + 8 <= w) && !(pxf < 0) && (pxl < fw) && (l0 == x0 + sx) && (l7 == l0 + 7) && ((int)(pxl + 1.0f) == l7 + 1);
    if (isplit == 0) {
        xfast = xfast && (u0 == u7);
    } else {  // the two pixels either side of the only place where the grid of px may change
        const float pxa = (float)(x0 + isplit - 1) - dx, pxb = (float)(x0 + isplit) - dx;
        const int la = l0 + isplit - 1;
        xfast = xfast && (pxa - (float)la == u0) && (pxb - (float)(la + 1) == u7) && ((int)(pxa + 1.0f) == la + 1);
    }
    const bool clamp_rt = (l0 + 8 == w);
    const HWeights ca = make_hweights(u0), cb = make_hweights(u7);
    const u16* frame = PLANES ? nullptr : src + (size_t)f * src_stride;
    const u8* flo = PLANES ? ps.lo + (size_t)f * ps.plane_stride : nullptr;
    const u8* fhi = PLANES ? ps.hi + (size_t)f * ps.plane_stride : nullptr;
    u16* oframe = dst + (size_t)f * dst_stride;
    const uint32_t rinfo = smem_addr(&rowinfo[0][ry]);
    const size_t row_step = (size_t)16 * w;

#pragma unroll 1
    for (int ty = 0; ty < tiles_y; ++ty) {
        const int stage = ty % TT_STAGES;
        const unsigned parity = (unsigned)(ty / TT_STAGES) & 1u;
        const int y0t = ty * TT_H, ys = y0t + sy;
        const int pp = ty & 1;  // which rowinfo / queue counter this tile uses
        mbar_wait(&bar[stage], parity);
        const u16* tile = reinterpret_cast<const u16*>(smem_raw + (PLANES ? TT_STAGES * STAGE_BYTES : stage * STAGE_BYTES));
        if (PLANES) {
            // (1) merge the two byte boxes into the uint16 tile, 8 pixels per step
            u16* merged = reinterpret_cast<u16*>(smem_raw + TT_STAGES * STAGE_BYTES);
            const unsigned char* blo = smem_raw + stage * STAGE_BYTES + (xs - xs16);
            const unsigned char* bhi = blo + TP_BOX_AL;
            const unsigned t2 = ps.min_t | (ps.min_t << 16);
            for (int v = threadIdx.x; v < TT_BH * (TT_BW / 8); v += TT_THREADS) {
                const int r = v / (TT_BW / 8), c8 = v - r * (TT_BW / 8);
                const uint2 l = *reinterpret_cast<const uint2*>(blo + r * TP_BW + 8 * c8);
                const uint2 hh = *reinterpret_cast<const uint2*>(bhi + r * TP_BW + 8 * c8);
                const int gy = ys + r;
                const unsigned add = (gy >= 0 && gy < ps.t_rows) ? t2 : 0u;
                uint4 o;
                o.x = __vadd2(__byte_perm(l.x, hh.x, 0x5140), add);
                o.y = __vadd2(__byte_perm(l.x, hh.x, 0x7362), add);
                o.z = __vadd2(__byte_perm(l.y, hh.y, 0x5140), add);
                o.w = __vadd2(__byte_perm(l.y, hh.y, 0x7362), add);
                *reinterpret_cast<uint4*>(merged + r * TT_BW + 8 * c8) = o;
            }
            __syncthreads();
            // (2) the loader's bad-pixel medians for the flagged pixels that fall into the tile
            if (ps.xy != nullptr) {
                const int gy0 = max(ys, 0), gy1 = min(ys + TT_BH, h);
                if (gy0 < gy1) {
                    const int a = ps.row_off[gy0], b = ps.row_off[gy1];
                    for (int i = a + threadIdx.x; i < b; i += TT_THREADS) {
                        const int2 p = reinterpret_cast<const int2*>(ps.xy)[i];
                        const int cxl = p.x - xs;
                        unsigned med;
                        if (cxl >= 0 && cxl < TT_BW && plane_median(flo, fhi, w, h, p.x, p.y, ps.nbr[i], ps, med))
                            merged[(p.y - ys) * TT_BW + cxl] = (u16)med;
                    }
                }
            }
            __syncthreads();
        }
        u16* ocol = oframe + (size_t)(y0t + ry) * w + x0;
        const int rows_left = (x0 < w) ? h - y0t : 0;  // destination rows of this tile that exist (none for columns past the edge)

        const uint32_t tbase = smem_addr(tile + 8 * cx);
        switch (xoff) {  // CTA-uniform
        case 0: fast_rows<0, MOTION>(tbase, rinfo + pp * (int)sizeof(rowinfo[0]), xfast, clamp_rt, ca, cb, ocol, row_step, cx, ry, rows_left, slowq, &slow_count[pp]); break;
        case 1: fast_rows<1, MOTION>(tbase, rinfo + pp * (int)sizeof(rowinfo[0]), xfast, clamp_rt, ca, cb, ocol, row_step, cx, ry, rows_left, slowq, &slow_count[pp]); break;
        case 2: fast_rows<2, MOTION>(tbase, rinfo + pp * (int)sizeof(rowinfo[0]), xfast, clamp_rt, ca, cb, ocol, row_step, cx, ry, rows_left, slowq, &slow_count[pp]); break;
        case 3: fast_rows<3, MOTION>(tbase, rinfo + pp * (int)sizeof(rowinfo[0]), xfast, clamp_rt, ca, cb, ocol, row_step, cx, ry, rows_left, slowq, &slow_count[pp]); break;
        case 4: fast_rows<4, MOTION>(tbase, rinfo + pp * (int)sizeof(rowinfo[0]), xfast, clamp_rt, ca, cb, ocol, row_step, cx, ry, rows_left, slowq, &slow_count[pp]); break;
        case 5: fast_rows<5, MOTION>(tbase, rinfo + pp * (int)sizeof(rowinfo[0]), xfast, clamp_rt, ca, cb, ocol, row_step, cx, ry, rows_left, slowq, &slow_count[pp]); break;
        case 6: fast_rows<6, MOTION>(tbase, rinfo + pp * (int)sizeof(rowinfo[0]), xfast, clamp_rt, ca, cb, ocol, row_step, cx, ry, rows_left, slowq, &slow_count[pp]); break;
        default: fast_rows<7, MOTION>(tbase, rinfo + pp * (int)sizeof(rowinfo[0]), xfast, clamp_rt, ca, cb, ocol, row_step, cx, ry, rows_left, slowq, &slow_count[pp]); break;
        }
        __syncthreads();  // queue complete
        // row parameters and an empty queue for the next tile (nobody reads that half before the barrier below)
        if (threadIdx.x < TT_H) rowinfo[pp ^ 1][threadIdx.x] = make_row_info(y0t + TT_H + threadIdx.x, h, dy, ys + TT_H);
        if (threadIdx.x == 0) slow_count[pp ^ 1] = 0;

        // ---- slow groups (image edges, source columns < 8, rows with 0 <= py < 1), spread over the whole
        // CTA one PIXEL per thread, reading the staged box where they can -- instead of the few threads
        // that own them walking 8 pixels each through dependent loads while their CTA waits.
        const int nslow = (int)slow_count[pp] * 8;
#pragma unroll 1
        for (int i = threadIdx.x; i < nslow; i += TT_THREADS) {
            const unsigned g = slowq[i >> 3];
            const int gcx = (int)(g & 15u), grow = (int)(g >> 4), gi = i & 7;
            const int gx = x0t + 8 * gcx + gi;
            const int gy = y0t + grow;
            if (gx >= w) continue;
            u16* o = oframe + (size_t)gy * w + gx;
            const int gx0 = x0t + 8 * gcx;
            const int e = (gx0 == 0) ? 0 : ((gx0 == w - 8) ? 1 : -1);
            const RowInfo ri = rowinfo[pp][grow];
            if (e >= 0 && ri.B >= 0 && ((edge_tab[e].valid >> gi) & 1u)) {
                *o = blend_edge_pixel<MOTION>(tile, ri.rows, 8388608u - (unsigned)ri.B, (unsigned)ri.B, 8 * gcx + xoff + gi,
                                              (edge_tab[e].clamped >> gi) & 1u, edge_tab[e].wt[gi]);
                continue;
            }
            if (PLANES) {
                const PlaneTileSrc ts{tile, flo, fhi, &ps, xs, ys, w, h};
                float r;
                if (translate_pixel<u16, float>(ts, w, h, gx, gy, dx, dy, strategy, (float)background, r)) *o = (u16)r;
            } else {
                const TileSrc ts{tile, frame, xs, ys, w, h};
                if (MOTION) {
                    float r;
                    if (translate_pixel<u16, float>(ts, w, h, gx, gy, dx, dy, strategy, (float)background, r)) *o = (u16)r;
                } else {
                    u16 r;
                    if (translate_pixel<u16, u16>(ts, w, h, gx, gy, dx, dy, strategy, (u16)background, r)) *o = r;
                }
            }
        }
        __syncthreads();  // every warp is done with this stage and the queue; next tile's row parameters are visible
        if (threadIdx.x == 0 && ty + TT_STAGES < tiles_y) issue_boxes(stage, ty + TT_STAGES);
    }
    if (PLANES) {  // metadata rows [h, h_full): merged, never translated (IRFileLoader.cpp:1241-1243 pass h - 3)
        const int nmeta = (ps.h_full - h) * TT_W;
        for (int i = threadIdx.x; i < nmeta; i += TT_THREADS) {
            const int yy = h + i / TT_W, xx = x0t + i % TT_W;
            if (xx < w) oframe[(size_t)yy * w + xx] = (u16)plane_px(flo, fhi, w, xx, yy, ps);
        }
    }
}


// ------------------------------------------------------------------------------------------------
// uint16 hot path, second generation: warps that do not wait for each other
// ------------------------------------------------------------------------------------------------
// The kernel above spends its time waiting, not computing (ncu, profiles/r1_v11_ncu_summary.md: 58 % of the issue slots,
// two CTA-wide barriers per tile, a CTA-wide queue for the edge groups, every source row unpacked twice).  Same staging
// (one TMA box per 128 x 64 destination tile, two stages), same exact arithmetic (blend_group's), different schedule:
//   * a CTA is FOUR warps and there is no __syncthreads in the tile loop.  A warp waits for a stage's box on its mbarrier,
//     does ITS 16 rows of the tile -- fast groups, edge pixels and border rows alike -- and signs off on a per-stage
//     counter; the warp that signs off LAST prepares the next row table for that stage and issues the box of tile ty + 2
//     into it (its lanes' shared-memory writes are published by the mbarrier arrive of its lane 0).
//   * lanes 0-15 of a warp own the 16 column groups of rows [16w, 16w+8), lanes 16-31 those of rows [16w+8, 16w+16): a thread
//     walks down 8 CONSECUTIVE destination rows, so the source row that is the bottom of row y is carried in registers as
//     the top of row y + 1 -- 9 staged rows are read and unpacked for 8 destination rows instead of 16.  Each octet of
//     lanes reads 128 contiguous bytes of one staged row: conflict-free whatever the row pitch.
//   * what is not a fast group is done by the warp that owns the rows, one pixel per lane: pixels of the image's first /
//     last group with the tabulated per-pixel weights (EdgeTable), pixels of border rows and everything else with the
//     literal per-pixel routine reading the staged box.
// Measured on the B200 (profiles/r2_translate_notes.md): 0.848 of the copy bandwidth in bench.py (first generation 0.733),
// 14.8 instructions per pixel instead of 17.9.  What was tried on top of it and NOT kept, each measured: a 256-pixel-wide
// footprint per CTA (staging alone 0.865 -> 0.889, but the arithmetic hides worse: 0.81), full-width 16-row bands (0.71), a
// per-warp cp.async ring instead of TMA boxes (0.52-0.61: the copy loop's registers spill into the blend), a leaner edge
// path (no change), an L2 prefetch of the boxes two tiles ahead (no change), a suspend-time hint on the mbarrier wait (no
// change).  The eight row-routine instances must not be unrolled further: fully unrolled they fall out of the 32 KB
// instruction cache (1.5x slower).
constexpr int TW_WARPS = 4, TW_THREADS = 32 * TW_WARPS;
constexpr int TW_ROWS = 8;  // consecutive destination rows per thread
struct RowAB {       // vertical weights of a destination row on the 2^-23 grid: N = p_bottom * A + p_top * B
    unsigned A, B;   // B == ROW_SLOW: not a regular row (border rows, rows whose source rows are not y+sy / y+sy+1, fine fractions);
                     // A then says which: 1 = py < 0 (above the image), 2 = py >= h (below it), 0 = anything else
};
constexpr unsigned ROW_SLOW = 0xFFFFFFFFu;

// the regular case: top tap = image row y + sy (= t_expected), bottom tap = the row below it
__device__ __forceinline__ RowAB make_row_ab(int y, int h, float dy, int t_expected)
{
    RowAB r;
    r.A = 0;
    r.B = ROW_SLOW;
    const float fh = (float)h;
    const float py = (float)y - dy;
    const int t = (int)py;
    int b = (int)(py + 1.0f);
    const bool clamped = (b == h);
    if (clamped) b = t;
    const float vf = (float)b - py;
    const float vs = vf * 8388608.0f;
    if (y < h && py < 0) r.A = 1;
    if (y < h && !(py < fh)) r.A = 2;
    if (y < h && !(py < 0) && (py < fh) && t == t_expected + 1 && py == (float)t) {
        // -dy within half a float ulp below an integer: py has rounded UP to the integer t_expected + 1 and the reference
        // blends row t with weight 1 (or, clamped, with itself).  Seen from the regular taps (top t_expected, bottom
        // t_expected + 1) that is the bottom row alone -- the same value, and the row stays on the fast path.  Without
        // this, every row of the upper float binades of such a frame is a border row (one CTA column ran 50x longer).
        r.A = 8388608u;
        r.B = 0;
        return r;
    }
    if (y < h && !(py < 0) && (py < fh) && (vs == truncf(vs)) && (fabsf(vf) <= 1.0f) && t == t_expected && (clamped || b == t + 1)) {
        if (clamped) {  // both taps are the top pixel: N = p * 2^23 (see make_row_info)
            r.A = 0;
            r.B = 8388608u;
        } else {
            r.B = (unsigned)(int)vs;
            r.A = 8388608u - r.B;
        }
    }
    return r;
}

// 8 destination pixels from two unpacked source rows (pt: top, pb: bottom); the arithmetic of blend_group
template <int XOFF, bool MOTION>
__device__ __forceinline__ void blend_rows(const unsigned (&pb)[9], const unsigned (&pt)[9], unsigned A, unsigned B, const HWeights& ca,
                                           const HWeights& cb, unsigned long long magic, u16* orow)
{
    double m[9];
#pragma unroll
    for (int j = 0; j < 9; ++j) {
        unsigned long long n = (unsigned long long)pb[j] * A + magic;
        n += (unsigned long long)pt[j] * B;
        m[j] = __longlong_as_double((long long)n);
    }
    unsigned o[8];
#pragma unroll
    for (int j = 0; j < 8; ++j) {
        const HWeights& c = (XOFF != 0 && j >= 8 - XOFF) ? cb : ca;
        const double val = __dadd_rn(__fma_rn(m[j], c.omu, c.k_l), __fma_rn(m[j + 1], c.u, c.k_r));
        // MOTION: the reference's translate<u16, float> result narrowed to u16.  Emulating the two conversions on the
        // integer / fp64 side (floor(val + half a float ulp of val's binade)) was built and measured: +4.8 instructions per
        // pixel instead of +2 and 2 % slower; with one half-ulp per 8-pixel group, faster on smooth images but 20 % slower
        // on noise (profiles/r2_translate_notes.md).  The kernel's time follows its instruction count, not the conversion pipe.
        // MOTION: (u16)(float)val with the float -> integer truncation as FADD.RZ with 2^23 (the low 16 bits of the sum's
        // mantissa are trunc(f); the byte permutes below take exactly those): one conversion on the 16-lane pipe instead of two
        if (MOTION)
            o[j] = __float_as_uint(__fadd_rz((float)val, 8388608.0f));
        else
            o[j] = (unsigned)__double2loint(__dadd_rd(val, 4503599627370496.0));
    }
    uint4 ov;
    ov.x = __byte_perm(o[0], o[1], 0x5410);
    ov.y = __byte_perm(o[2], o[3], 0x5410);
    ov.z = __byte_perm(o[4], o[5], 0x5410);
    ov.w = __byte_perm(o[6], o[7], 0x5410);
    st_stream(reinterpret_cast<uint4*>(orow), ov);
}

// a thread's 8 rows of one tile.  srow: shared address of the thread's 16 staged pixels in the box row of its first
// destination row; rab: shared address of that row's RowAB
template <int XOFF, bool MOTION>
__device__ __forceinline__ void fast_column(uint32_t srow, uint32_t rab, bool clamp_rt, const HWeights& ca, const HWeights& cb,
                                            u16* orow, size_t w)
{
    unsigned long long magic = 0x41C0000000000000ULL;
    asm volatile("" : "+l"(magic));
    unsigned pt[9], pb[9];
    unpack9<XOFF>(lds128(srow), lds128(srow + 16), pt);
    if (clamp_rt) pt[8] = pt[7];
#pragma unroll 2  // not more: see the instruction-cache note above
    for (int k = 0; k < TW_ROWS; ++k) {
        srow += TT_BW * 2;
        unpack9<XOFF>(lds128(srow), lds128(srow + 16), pb);
        if (clamp_rt) pb[8] = pb[7];  // rt of the last pixel clamps to its l (Filters.h:309)
        unsigned A, B;
        asm volatile("ld.shared.v2.u32 {%0,%1}, [%2];" : "=r"(A), "=r"(B) : "r"(rab + k * (int)sizeof(RowAB)));
        if (B != ROW_SLOW) blend_rows<XOFF, MOTION>(pb, pt, A, B, ca, cb, magic, orow);
        orow += w;
#pragma unroll
        for (int j = 0; j < 9; ++j) pt[j] = pb[j];
    }
}

template <bool MOTION>
__global__ void __launch_bounds__(TW_THREADS, 5)
translate_u16_rows_kernel(const __grid_constant__ CUtensorMap tmap, const u16* __restrict__ src, u16* __restrict__ dst, int w, int h,
                          size_t src_stride, size_t dst_stride, const float* __restrict__ dxs, const float* __restrict__ dys,
                          float dx0, float dy0, int strategy, unsigned background, int tiles_y, const int* __restrict__ order)
{
    extern __shared__ __align__(128) unsigned char smem_raw[];
    __shared__ __align__(8) unsigned long long bar[TT_STAGES];
    __shared__ __align__(8) RowAB rowab[3][TT_H];  // row tables of three consecutive tiles (tile % 3): see make_table
    __shared__ unsigned done[TT_STAGES];  // warps that are through with the stage's current tile
    __shared__ EdgeTable edge_tab[2];     // [0]: the image's first group of a row, [1]: its last
    const int f = order ? order[blockIdx.y] : (int)blockIdx.y;  // frames grouped by column offset (translate_order_kernel)
    const int x0t = blockIdx.x * TT_W;
    const float dx = dxs ? dxs[f] : dx0;
    const float dy = dys ? dys[f] : dy0;
    const float fw = (float)w;
    const float fh = (float)h;
    const int sx = (int)fminf(fmaxf(floorf(-dx), -fw - 16.f), fw + 16.f);
    const int sy = (int)fminf(fmaxf(floorf(-dy), -fh - 16.f), fh + 16.f);
    // the box starts on a 32-byte sector (16 pixels): its 288-byte rows are then 9 sectors, never 10.  xoff = 0..15; the
    // row routines are instantiated for xoff & 7 and read 16 bytes further into the staged row when xoff >= 8
    const int xs = (x0t + sx) & ~15;
    const int xoff = (x0t + sx) - xs;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    // Weight of the RIGHT tap of destination pixel xp when its left tap is source column xp + sx: px - l in the regular case.
    // When -dx lies within half a float ulp below an integer, px rounds UP to the integer xp + sx + 1 in the upper float
    // binades of the row; the reference then takes l = px, u = 0, i.e. the value of column xp + sx + 1 alone -- which is the
    // regular taps with u = 1.  -1: neither (the pixel goes to the literal routine).
    auto tap_u = [&](float px, int xp) -> float {
        const int l = (int)px;
        const float u = px - (float)l;
        return (l == xp + sx) ? u : ((l == xp + sx + 1 && u == 0.f) ? 1.0f : -1.0f);
    };
    // The row table of a tile is made one tile EARLIER than its box is asked for, so that what stands between the last warp's
    // sign-off and the next box is a fence and the TMA instruction, not ~130 instructions of float arithmetic: the tables
    // of tiles 0, 1, 2 at the start, the table of tile t + 3 by the warp that signs tile t off last (slot t % 3 is free then).
    auto make_table = [&](int tile_row) {  // by one whole warp
        const int y0 = tile_row * TT_H;
        RowAB* tab = rowab[tile_row % 3];
#pragma unroll
        for (int k = 0; k < TT_H / 32; ++k) tab[lane + 32 * k] = make_row_ab(y0 + lane + 32 * k, h, dy, y0 + lane + 32 * k + sy);
        __syncwarp();
    };
    auto issue_box = [&](int s, int tile_row) {  // lane 0 of the calling warp; publishes the warp's earlier shared-memory writes too
        if (lane == 0) {
            done[s] = 0;
            asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
            mbar_expect_tx(&bar[s], TT_BH * TT_BW * 2);
            tma_load_box(smem_raw + s * TT_STAGE_BYTES, &tmap, &bar[s], xs, tile_row * TT_H + sy, f);
        }
    };
    if (threadIdx.x == 0) {
#pragma unroll
        for (int s = 0; s < TT_STAGES; ++s) mbar_init(&bar[s], 1);
        mbar_fence_init();
    }
    if (warp == TW_WARPS - 1 && lane < 16) {  // 2 tables x 8 pixels
        const int e = lane >> 3, i = lane & 7;
        const int xe0 = e ? w - 8 : 0;
        const int x = xe0 + i;
        const float px = (float)x - dx;
        bool ok = (xe0 >= x0t) && (xe0 < x0t + TT_W) && !(px < 0) && (px < fw);
        const int l = (int)px;
        const int rt = (int)(px + 1.0f);
        const float un = tap_u(px, x);
        const bool cl = ok && (rt == w) && (l == w - 1) && (l == x + sx);
        ok = ok && (un >= 0.f) && (cl || rt == l + 1);
        edge_tab[e].wt[i] = make_hweights(ok ? un : 0.f);
        const unsigned vb = __ballot_sync(0x0000FFFFu, ok), cb2 = __ballot_sync(0x0000FFFFu, cl);
        const unsigned ob = __ballot_sync(0x0000FFFFu, (px < 0) || !(px < fw)), lb = __ballot_sync(0x0000FFFFu, px < 0);
        if (i == 0) {
            edge_tab[e].valid = (vb >> (8 * e)) & 0xFFu;
            edge_tab[e].clamped = (cb2 >> (8 * e)) & 0xFFu;
            edge_tab[e].outside = (ob >> (8 * e)) & 0xFFu;
            edge_tab[e].below = (lb >> (8 * e)) & 0xFFu;
        }
    }
    if (warp < 3 && warp < tiles_y) make_table(warp);
    __syncthreads();  // barriers initialised, edge tables and the first three row tables written: the only CTA-wide barrier
    if (warp < TT_STAGES && warp < tiles_y) issue_box(warp, warp);

    // ---- per-thread column constants (while the first boxes are in flight) -----------------------
    const int cx = lane & 15, half = lane >> 4;
    const int r0 = 2 * TW_ROWS * warp + TW_ROWS * half;  // the thread's first row inside a tile
    const int x0 = x0t + 8 * cx;
    const int isplit = (8 - xoff) & 7;
    const float pxf = (float)x0 - dx, pxl = (float)(x0 + 7) - dx;
    const float u0 = tap_u(pxf, x0), u7 = tap_u(pxl, x0 + 7);
    bool xfast = (x0 + 8 <= w) && !(pxf < 0) && (pxl < fw) && (u0 >= 0.f) && (u7 >= 0.f) && ((int)(pxl + 1.0f) == (int)pxl + 1);
    if (isplit == 0) {
        xfast = xfast && (u0 == u7);
    } else {
        const float pxa = (float)(x0 + isplit - 1) - dx, pxb = (float)(x0 + isplit) - dx;
        xfast = xfast && (tap_u(pxa, x0 + isplit - 1) == u0) && (tap_u(pxb, x0 + isplit) == u7) && ((int)(pxa + 1.0f) == (int)pxa + 1);
    }
    const bool clamp_rt = (x0 + sx + 8 == w);
    const HWeights ca = make_hweights(u0), cb = make_hweights(u7);
    // column groups of this tile column that exist but are not fast: bit cx (the same in both halves of the warp)
    const unsigned slowcols = __ballot_sync(0xFFFFFFFFu, !xfast && x0 < w) & 0xFFFFu;
    const u16* frame = src + (size_t)f * src_stride;
    u16* oframe = dst + (size_t)f * dst_stride;

#pragma unroll 1
    for (int ty = 0; ty < tiles_y; ++ty) {
        const int stage = ty % TT_STAGES;
        const int tslot = ty % 3;
        const unsigned parity = (unsigned)(ty / TT_STAGES) & 1u;
        const int y0t = ty * TT_H, ys = y0t + sy;
        mbar_wait(&bar[stage], parity);
        const u16* tile = reinterpret_cast<const u16*>(smem_raw + stage * TT_STAGE_BYTES);
        if (xfast) {
            const uint32_t srow = smem_addr(tile + r0 * TT_BW + 8 * cx + (xoff & 8));
            const uint32_t rab = smem_addr(&rowab[tslot][r0]);
            u16* orow = oframe + (size_t)(y0t + r0) * w + x0;
            switch (xoff & 7) {  // CTA-uniform
            case 0: fast_column<0, MOTION>(srow, rab, clamp_rt, ca, cb, orow, (size_t)w); break;
            case 1: fast_column<1, MOTION>(srow, rab, clamp_rt, ca, cb, orow, (size_t)w); break;
            case 2: fast_column<2, MOTION>(srow, rab, clamp_rt, ca, cb, orow, (size_t)w); break;
            case 3: fast_column<3, MOTION>(srow, rab, clamp_rt, ca, cb, orow, (size_t)w); break;
            case 4: fast_column<4, MOTION>(srow, rab, clamp_rt, ca, cb, orow, (size_t)w); break;
            case 5: fast_column<5, MOTION>(srow, rab, clamp_rt, ca, cb, orow, (size_t)w); break;
            case 6: fast_column<6, MOTION>(srow, rab, clamp_rt, ca, cb, orow, (size_t)w); break;
            default: fast_column<7, MOTION>(srow, rab, clamp_rt, ca, cb, orow, (size_t)w); break;
            }
        }
        __syncwarp();
        // ---- the rest of the warp's 16 rows, one pixel per lane ----
        const int wr0 = 2 * TW_ROWS * warp;  // the warp's first row inside the tile
        const unsigned slowrows = __ballot_sync(0xFFFFFFFFu, lane < 16 && rowab[tslot][wr0 + (lane & 15)].B == ROW_SLOW) & 0xFFFFu;
        const TileSrc ts{tile, frame, xs, ys, w, h};
        auto slow_pixel = [&](int col, int row) {  // col: pixel inside the tile column, row: inside the tile
            const int gx = x0t + col, gy = y0t + row;
            if (gx >= w || gy >= h) return;
            u16* o = oframe + (size_t)gy * w + gx;
            const int gx0 = gx & ~7, gi = gx & 7;
            const int e = (gx0 == 0) ? 0 : ((gx0 == w - 8) ? 1 : -1);
            const RowAB ra = rowab[tslot][row];
            if (e >= 0 && ra.B != ROW_SLOW && ((edge_tab[e].valid >> gi) & 1u)) {
                const unsigned rows = (unsigned)(row * (TT_BW * 2)) | ((unsigned)((row + 1) * (TT_BW * 2)) << 16);
                *o = blend_edge_pixel<MOTION>(tile, rows, ra.A, ra.B, col + xoff, (edge_tab[e].clamped >> gi) & 1u, edge_tab[e].wt[gi]);
                return;
            }
            if (MOTION) {
                float r;
                if (translate_pixel<u16, float>(ts, w, h, gx, gy, dx, dy, strategy, (float)background, r)) *o = (u16)r;
            } else {
                u16 r;
                if (translate_pixel<u16, u16>(ts, w, h, gx, gy, dx, dy, strategy, (u16)background, r)) *o = r;
            }
        };
        // The image's first and last group of a row are slow column groups for nearly every shift (pixels left of / beyond
        // the image, a different weight per pixel where px < 8), i.e. in two of a 640-wide frame's five CTAs; one pixel per
        // lane through slow_pixel they cost those CTAs as much again as their fast groups (the divergent border / blend
        // branches, everything recomputed per pixel).  Here a lane takes 4 pixels of one regular row: 5 + 5 staged pixels,
        // the row's integer blend once per column, the tabulated weights (a broadcast read per pixel), the border
        // strategy decided from the table's `outside` bits without the literal routine.  Rows that are not regular are left
        // to the border-row pass below.
        auto edge_rows = [&](int g, int e) {
            const EdgeTable& et = edge_tab[e];
            const int row = wr0 + (lane & 15), j0 = 4 * (lane >> 4);
            const int gy = y0t + row;
            if (gy >= h) return;
            const RowAB ra = rowab[tslot][row];
            if (ra.B == ROW_SLOW) return;
            const u16* top = tile + row * TT_BW + 8 * g + xoff + j0;  // left tap of pixel j0, top source row
            const u16* bot = top + TT_BW;
            u16* o = oframe + (size_t)gy * w + x0t + 8 * g + j0;
            unsigned long long nn[5];
#pragma unroll
            for (int c = 0; c < 5; ++c) nn[c] = (unsigned long long)bot[c] * ra.A + (unsigned long long)top[c] * ra.B + 0x41C0000000000000ULL;
#pragma unroll
            for (int q = 0; q < 4; ++q) {
                const unsigned bit = 1u << (j0 + q);
                if (et.valid & bit) {
                    const HWeights c = et.wt[j0 + q];
                    const unsigned long long nr = (et.clamped & bit) ? nn[q] : nn[q + 1];
                    const double val = __dadd_rn(__fma_rn(__longlong_as_double((long long)nn[q]), c.omu, c.k_l),
                                                 __fma_rn(__longlong_as_double((long long)nr), c.u, c.k_r));
                    o[q] = MOTION ? (u16)__float_as_uint(__fadd_rz((float)val, 8388608.0f)) : (u16)__double2loint(__dadd_rd(val, 4503599627370496.0));
                } else {  // outside the image (the caller has checked that the table knows every pixel of the group)
                    // translate_pixel's border branch: src((long long)py, column 0 or w - 1).  (long long)py is the row of the
                    // top tap -- or, when py has rounded up to an integer (make_row_ab's B == 0 case), the one below it
                    if (strategy == STRAT_NEAREST)
                        o[q] = tile[(row + (ra.B == 0 ? 1 : 0)) * TT_BW + (((et.below & bit) ? 0 : w - 1) - xs)];
                    else if (strategy == STRAT_BACKGROUND)
                        o[q] = (u16)background;
                }
            }
        };
        unsigned generic_cols = 0;  // slow column groups done pixel by pixel, all 16 rows of the warp
        if (slowcols) {  // CTA-uniform
            for (unsigned m = slowcols; m; m &= m - 1) {
                const int g = __ffs(m) - 1;
                const int xg = x0t + 8 * g;
                const int e = (xg == 0) ? 0 : ((xg == w - 8) ? 1 : -1);
                if (e >= 0 && strategy != STRAT_WRAP) {
                    // every pixel either tabulated or outside the image, and the border column staged: else pixel by pixel
                    const unsigned below = edge_tab[e].below, above = edge_tab[e].outside & ~below;
                    const bool staged = (below == 0 || (-xs >= 0 && -xs < TT_BW)) && (above == 0 || (w - 1 - xs >= 0 && w - 1 - xs < TT_BW));
                    if (((edge_tab[e].valid | edge_tab[e].outside) & 0xFFu) == 0xFFu && staged) {
                        edge_rows(g, e);
                        continue;
                    }
                }
                generic_cols |= 1u << g;
#pragma unroll 1
                for (int rr = lane >> 3; rr < 2 * TW_ROWS; rr += 4) slow_pixel(8 * g + (lane & 7), wr0 + rr);  // 4 rows per pass
            }
        }
        if (slowrows) {  // warp-uniform: the pixels of border rows that the passes above have not done
            for (unsigned m = slowrows; m; m &= m - 1) {
                const int rr = __ffs(m) - 1;
                const RowAB ra = rowab[tslot][wr0 + rr];
                // rows above / below the image (up to |dy| of them per frame, in every CTA of the frame): the border strategy
                // alone decides -- for "nearest" a copy of the image's first / last row at the clamped source column,
                // translate_pixel's border branch without the routine around it (a quarter of its instructions)
                const int brow = (ra.A == 1 ? 0 : h - 1) - ys;  // that row in the staged box
                auto clamped_col = [&](int gx) {  // (long long)px clamped into the image, as a box column
                    const float px = (float)gx - dx;
                    return (px < 0 ? 0 : (px >= fw ? w - 1 : (int)px)) - xs;
                };
                // the source column is monotonic in gx: staged for the tile's first and last pixel = staged for all of them
                const int bc_a = clamped_col(x0t), bc_b = clamped_col(min(x0t + TT_W, w) - 1);
                if (ra.A != 0 && strategy != STRAT_WRAP && brow >= 0 && brow < TT_BH && bc_a >= 0 && bc_b < TT_BW) {
                    const int gy = y0t + wr0 + rr;
                    if (strategy == STRAT_NOBORDER) continue;
#pragma unroll 1
                    for (int c = lane; c < TT_W; c += 32) {
                        const int gx = x0t + c;
                        if (gx >= w || ((generic_cols >> (c >> 3)) & 1u)) continue;
                        const unsigned v = strategy == STRAT_NEAREST ? (unsigned)tile[brow * TT_BW + clamped_col(gx)] : background;
                        oframe[(size_t)gy * w + gx] = (u16)v;
                    }
                    continue;
                }
#pragma unroll 1
                for (int c = lane; c < TT_W; c += 32)
                    if (!((generic_cols >> (c >> 3)) & 1u)) slow_pixel(c, wr0 + rr);
            }
        }
        // ---- sign off; the last warp through refills the stage ----
        __syncwarp();
        unsigned last = 0;
        if (lane == 0) {
            unsigned old;
            asm volatile("atom.acq_rel.cta.shared.add.u32 %0, [%1], 1;" : "=r"(old) : "r"(smem_addr(&done[stage])) : "memory");
            last = (old == TW_WARPS - 1);
        }
        last = __shfl_sync(0xFFFFFFFFu, last, 0);
        if (last) {
            if (ty + TT_STAGES < tiles_y) issue_box(stage, ty + TT_STAGES);
            if (ty + 3 < tiles_y) make_table(ty + 3);
        }
    }
}

// The eight instances of the row routine (one per residual column offset) are ~3 KB of code each, and the offset follows the
// frame's shift: with per-frame shifts the CTAs resident on an SM run up to five different instances.  For the motion variant
// (more code per instance) handing the frames out grouped by offset is worth 4 %: order[i] = i-th frame of a counting sort by
// (floor(-dx) & 7).  (The plain variant loses 1.5 % to the indirection and is launched without it.)  One CTA; n <= 65535.
__global__ void __launch_bounds__(1024) translate_order_kernel(const float* __restrict__ dxs, int n, int w, int* __restrict__ order)
{
    __shared__ int count[8], start[8];
    const float fw = (float)w;
    if (threadIdx.x < 8) count[threadIdx.x] = 0;
    __syncthreads();
    auto key = [&](int f) { return (int)fminf(fmaxf(floorf(-dxs[f]), -fw - 16.f), fw + 16.f) & 7; };
    for (int f = threadIdx.x; f < n; f += blockDim.x) atomicAdd(&count[key(f)], 1);
    __syncthreads();
    if (threadIdx.x == 0) {
        int a = 0;
        for (int k = 0; k < 8; ++k) {
            start[k] = a;
            a += count[k];
        }
    }
    __syncthreads();
    for (int f = threadIdx.x; f < n; f += blockDim.x) order[atomicAdd(&start[key(f)], 1)] = f;
}

int launch_translate_u16(const u16* src, u16* dst, int w, int h, long long nframes, size_t src_stride, size_t dst_stride,
                         const float* dxs, const float* dys, float dx0, float dy0, int strategy, unsigned background, bool motion,
                         cudaStream_t st)
{
    if (nframes <= 0 || w <= 0 || h <= 0) return 0;
    const bool tma_enabled = option_enabled(OPT_TRANSLATE_TMA);  // "translate_tma" = 0 selects the plain kernel (A/B measurements)
    const int tiles_x = (int)ceil_div(w, TT_W), tiles_y = (int)ceil_div(h, TT_H);
    if (tma_enabled && (w % 8 == 0) && aligned16(dst) && (dst_stride % 8 == 0) && tma_compatible(src, (size_t)w * 2, src_stride * 2)) {
        const size_t smem = (size_t)TT_STAGES * TT_STAGE_BYTES;
        RIRB_SMEM_ATTR((translate_u16_tma_kernel<true, false>), smem);
        RIRB_SMEM_ATTR((translate_u16_tma_kernel<false, false>), smem);
        RIRB_SMEM_ATTR((translate_u16_rows_kernel<true>), smem);
        RIRB_SMEM_ATTR((translate_u16_rows_kernel<false>), smem);
        // per-frame shifts: the row kernel takes the frames grouped by their column offset (one order buffer for every launch)
        int* order_buf = nullptr;
        if (option_enabled(OPT_TRANSLATE_ROWS) && (motion || option_value(OPT_TRANSLATE_ROWS) >= 2) && dxs && nframes > 1) {
            order_buf = (int*)scratch_buffer(sizeof(int) * 65536);
            if (!order_buf) return -1;
        }
        // grid = (tile column, frame); gridDim.y <= 65535, so long movies go in several launches
        for (long long f0 = 0; f0 < nframes; f0 += 65535) {
            const long long n = min(nframes - f0, 65535LL);
            const u16* s0 = src + f0 * src_stride;
            u16* d0 = dst + f0 * dst_stride;
            const float* dx_p = dxs ? dxs + f0 : nullptr;
            const float* dy_p = dys ? dys + f0 : nullptr;
            CUtensorMap tmap;
            if (make_movie_tensor_map(&tmap, s0, 2, w, h, n, (size_t)w * 2, src_stride * 2, TT_BW, TT_BH) != 0) return -1;
            const dim3 tgrid((unsigned)tiles_x, (unsigned)n);
            const PlaneSrc none{};
            if (option_enabled(OPT_TRANSLATE_ROWS)) {  // "translate_rows" = 0: the first-generation tiled kernel (A/B)
                int* order = n > 1 ? order_buf : nullptr;
                if (order) RIRB_LAUNCH(translate_order_kernel, 1, 1024, 0, st, dx_p, (int)n, w, order);
                if (motion)
                    RIRB_LAUNCH((translate_u16_rows_kernel<true>), tgrid, TW_THREADS, smem, st, tmap, s0, d0, w, h, src_stride, dst_stride,
                                dx_p, dy_p, dx0, dy0, strategy, background, tiles_y, order);
                else
                    RIRB_LAUNCH((translate_u16_rows_kernel<false>), tgrid, TW_THREADS, smem, st, tmap, s0, d0, w, h, src_stride, dst_stride,
                                dx_p, dy_p, dx0, dy0, strategy, background, tiles_y, order);
                continue;
            }
            if (motion)
                RIRB_LAUNCH((translate_u16_tma_kernel<true, false>), tgrid, TT_THREADS, smem, st, tmap, tmap, s0, d0, w, h, src_stride,
                            dst_stride, dx_p, dy_p, dx0, dy0, strategy, background, tiles_y, none);
            else
                RIRB_LAUNCH((translate_u16_tma_kernel<false, false>), tgrid, TT_THREADS, smem, st, tmap, tmap, s0, d0, w, h, src_stride,
                            dst_stride, dx_p, dy_p, dx0, dy0, strategy, background, tiles_y, none);
        }
        return 0;
    }
    dim3 block(32, 8);
    dim3 grid((unsigned)ceil_div(ceil_div(w, TR_PX), 32), (unsigned)ceil_div(h, 8), (unsigned)min(nframes, 32768LL));
    if (motion)
        RIRB_LAUNCH(translate_u16_kernel<true>, grid, block, 0, st, src, dst, w, h, nframes, src_stride, dst_stride, dxs, dys, dx0,
                    dy0, strategy, background);
    else
        RIRB_LAUNCH(translate_u16_kernel<false>, grid, block, 0, st, src, dst, w, h, nframes, src_stride, dst_stride, dxs, dys,
                    dx0, dy0, strategy, background);
    return 0;
}

// The reader's chain in one pass: byte planes [n][h_full][w] -> corrected, registered uint16 frames.
// Returns 1 when the layout cannot take this path (the caller then runs the two-pass chain), 0 / -1 otherwise.
int launch_loader_fused(const u8* lo, const u8* hi, u16* out, int w, int h_full, int hb, long long nframes, int min_t, int t_rows,
                        const int* xy_dev, const int* nbr_dev, const int* row_off_dev, const u8* mask_dev, const float* dxs,
                        const float* dys, cudaStream_t st)
{
    // Off by default: measured on B200 (profiles/r1_loader_fused_ab.md) the one-pass kernel is instruction-bound
    // (merge + medians + blend in one CTA) and only ties the two-pass chain at 640x512, losing on larger frames.
    const bool enabled = option_enabled(OPT_LOADER_FUSED);
    const size_t fpx = (size_t)w * h_full;
    if (!enabled || (w % 16) != 0 || hb < 3 || !aligned16(out) || !tma_compatible(lo, (size_t)w, fpx) ||
        !tma_compatible(hi, (size_t)w, fpx))
        return 1;
    RIRB_SMEM_ATTR((translate_u16_tma_kernel<true, true>), TP_SMEM_BYTES);
    const int tiles_x = (int)ceil_div(w, TT_W), tiles_y = (int)ceil_div(hb, TT_H);
    for (long long f0 = 0; f0 < nframes; f0 += 65535) {
        const long long n = min(nframes - f0, 65535LL);
        CUtensorMap map_lo, map_hi;
        // the translated image is the first hb rows of every stored frame: rows >= hb must read as "outside"
        if (make_movie_tensor_map(&map_lo, lo + f0 * fpx, 1, w, hb, n, (size_t)w, fpx, TP_BW, TT_BH) != 0 ||
            make_movie_tensor_map(&map_hi, hi + f0 * fpx, 1, w, hb, n, (size_t)w, fpx, TP_BW, TT_BH) != 0)
            return -1;
        PlaneSrc ps;
        ps.lo = lo + f0 * fpx;
        ps.hi = hi + f0 * fpx;
        ps.plane_stride = fpx;
        ps.xy = xy_dev;
        ps.nbr = nbr_dev;
        ps.row_off = row_off_dev;
        ps.mask = mask_dev;
        ps.min_t = (unsigned)min_t & 0xFFFFu;
        ps.t_rows = t_rows;
        ps.h_full = h_full;
        const dim3 tgrid((unsigned)tiles_x, (unsigned)n);
        RIRB_LAUNCH((translate_u16_tma_kernel<true, true>), tgrid, TT_THREADS, TP_SMEM_BYTES, st, map_lo, map_hi, (const u16*)nullptr,
                    out + f0 * fpx, w, hb, fpx, fpx, dxs + f0, dys + f0, 0.f, 0.f, STRAT_NEAREST, 0u, tiles_y, ps);
    }
    return 0;
}

int launch_translate(int type, const void* src, void* dst, int w, int h, long long nframes, const float* dxs, const float* dys,
                     float dx0, float dy0, int strategy, const void* background_host, cudaStream_t st)
{
    if (nframes <= 0 || w <= 0 || h <= 0) return 0;
    switch (type) {
    case '?': return launch_generic<BoolPix>(src, dst, w, h, nframes, dxs, dys, dx0, dy0, strategy, background_host, st);
    case 'b': return launch_generic<signed char>(src, dst, w, h, nframes, dxs, dys, dx0, dy0, strategy, background_host, st);
    case 'B': return launch_generic<unsigned char>(src, dst, w, h, nframes, dxs, dys, dx0, dy0, strategy, background_host, st);
    case 'h': return launch_generic<short>(src, dst, w, h, nframes, dxs, dys, dx0, dy0, strategy, background_host, st);
    case 'H':
        return launch_translate_u16((const u16*)src, (u16*)dst, w, h, nframes, (size_t)w * h, (size_t)w * h, dxs, dys, dx0, dy0,
                                    strategy, *(const u16*)background_host, false, st);
    case 'i': return launch_generic<int>(src, dst, w, h, nframes, dxs, dys, dx0, dy0, strategy, background_host, st);
    case 'I': return launch_generic<unsigned int>(src, dst, w, h, nframes, dxs, dys, dx0, dy0, strategy, background_host, st);
    case 'l': return launch_generic<long long>(src, dst, w, h, nframes, dxs, dys, dx0, dy0, strategy, background_host, st);
    case 'L': return launch_generic<unsigned long long>(src, dst, w, h, nframes, dxs, dys, dx0, dy0, strategy, background_host, st);
    case 'f': return launch_generic<float>(src, dst, w, h, nframes, dxs, dys, dx0, dy0, strategy, background_host, st);
    case 'd': return launch_generic<double>(src, dst, w, h, nframes, dxs, dys, dx0, dy0, strategy, background_host, st);
    default: set_error("translate: unknown dtype code %d", type); return -1;
    }
}

}  // namespace rirb
