// librir_b200/csrc/lossy.cu -- the lossy "bounded-error" pre-conditioner of the H.264 saver (SURVEY.md 8f-2).
//
// Reference: H264_Saver::addImageLossyNoCamera, h264.cpp:2253-2424 (input already in temperature; behind
// h264_add_image_lossy) and H264_Saver::addLoss, :2426-2607 (behind h264_add_loss; `variant` 1: the bounds only
// tighten when the spread is ABOVE its running mean, and there is no integration-time test),
// with RunningAverage2 (:1526-1615), get_background (:1955-1991) and stdDev (:1993-2036).  Per frame:
//   tmp  = bad-pixel-corrected input (optional)                                   :2259-2271
//   tmpT = tmp - min (saturating, lossy rows only, optional)                      :2314-2328
//   background = mode of the 16,384-bin histogram of tmp >> 2                      :2331
//   (sd_back, sd_fore) = spread of |tmpT - prevT|, split by img > background once 40 frames are in   :2337-2340
//   lowError / highError = defaults minus round(|sd - running mean| * stdFactor)   :2353-2376
//   per pixel: if |tmpT - refT| <= error(class) and the integration-time bits did not change, the pixel is
//              replaced by the running average (or refT), else refT restarts from it                :2392-2413
//   prevT = output, lastDL = tmp, metadata rows copied                              :2415-2421
// Time is sequential (every frame needs the previous frame's state and two global reductions of its
// own), pixels are parallel: three small launches per frame on one stream (the two scalar steps run in the
// last CTA of the reduction that feeds them).  All sums are exact integers
// (the reference adds int products into doubles, exact below 2^53; its products wrap, see lossy_wrapped_square), the
// scalar decision is evaluated in non-contracted fp64 by one thread with x86's float -> int conversion (lossy_sub_rounded),
// so the outputs are bit-identical to the COMPILED reference (oracle/_ref/libs/
// libvideo_io.so; tests/golden/vio_golden.npz) -- including what its overlapping memcpy at :2347 does to the window of
// spreads (see lossy_window_quirk below).
// State per pixel: sums u32, const (value u16, count i16), refT, prevT, lastDL u16 and a ring of
// `running_average` frames -- 12 + 2 * running_average bytes.
#include <cooperative_groups.h>

#include "common.cuh"
#include "kernels.h"

namespace rirb {

constexpr int LOSSY_MAX_CTAS = 256;  // CTAs of lossy_run_kernel (one per SM)
constexpr int LOSSY_MAX_RUN = 64;    // frames per launch of it

struct LossyScalars {
    unsigned minv;                  // m_data->min
    unsigned background;
    int low_error, high_error;      // of the current frame
    unsigned long long sum[4];      // fore: sum_diff, sum_diff2; back: b_sum_diff, b_sum_diff2
    unsigned cnt[2];                // fore, back pixel counts
    double first[2];                // firstStdDevs[0]
    double stds[40][2];             // stdDevs window, circular: the oldest entry is stds[head] once 40 are in
    alignas(16) unsigned hist[16384];
    unsigned ticket[2];             // "last CTA done" counters of the two reduction kernels
    // lossy_run_kernel (several frames per launch): per-CTA partial sums of stdDev, two sets used alternately by frame
    // parity (written while the previous frame is updated, read after the grid barrier: nothing to clear, no atomics),
    // the grid barrier's counter, the backgrounds of the run's frames and the tickets of the pass that finds them
    alignas(16) unsigned long long psum[2][LOSSY_MAX_CTAS][4];
    unsigned pcnt[2][LOSSY_MAX_CTAS][2];
    unsigned barrier;
    unsigned back_run[LOSSY_MAX_RUN];
    unsigned back_ticket[LOSSY_MAX_RUN];
};

// h264.cpp:2347 (and :2538 in addLoss) shifts the full window of 40 (background, foreground) spreads with
// memcpy(data, data + 1, 39 pairs): overlapping, i.e. undefined behaviour.  As compiled with the reference's stock flags
// (g++ -O3, x86-64) the copy moves the LAST 8 bytes first and the rest front to back, so after every shift the pair that
// is now third from the end carries the old last pair's .second (its own is lost); every .first is right.  win[] is the
// window in time order BEFORE the shift: the shifted window is win[1..39] + the new pair, so the smear lands on win[38].
// quirk == 0 gives the memmove the author meant.
__device__ __forceinline__ void lossy_window_quirk(double (*win)[2], int nstds, int quirk)
{
    if (quirk && nstds == 40) win[38][1] = win[39][1];
}

// stdDev's `sum_diff2 += diff * diff` (:1993-2036) multiplies ints: for |diff| >= 46341 the product wraps modulo
// 2^32 (undefined in C++, a wrap as x86-64 builds it), and the wrapped, possibly negative value is what the reference adds
// into its double sum.  Here the wrapped products are added in signed 64-bit two's complement (carried in the unsigned long
// long sums and slots) and converted to double once.  That equals the reference's sequential double sum as long as every
// partial sum stays exact in a double: |product| <= 2^31, so up to 2^22 lossy pixels (DESIGN.md section 4).
__device__ __forceinline__ unsigned long long lossy_wrapped_square(int d)
{
    return (unsigned long long)(long long)(int)((unsigned)d * (unsigned)d);
}

__global__ void lossy_min_kernel(const u16* __restrict__ tmp, int ns, LossyScalars* sc)
{
    unsigned m = 65535u;
    for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < ns; i += gridDim.x * blockDim.x) m = min(m, (unsigned)tmp[i]);
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) m = min(m, __shfl_xor_sync(0xFFFFFFFFu, m, o));
    if ((threadIdx.x & 31) == 0) atomicMin(&sc->minv, m);
}

// first image (:2273-2311): lastDL = tmp, tmp -= min, out = tmp, refT = prevT = tmp
__global__ void lossy_first_kernel(const u16* __restrict__ tmp, u16* __restrict__ out, u16* __restrict__ lastDL, u16* __restrict__ refT,
                                   u16* __restrict__ prevT, int n, int ns, int subtract_min, const LossyScalars* __restrict__ sc)
{
    const unsigned mn = subtract_min ? sc->minv : 0u;
    for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) {
        const unsigned v = tmp[i];
        lastDL[i] = (u16)v;
        unsigned t = v;
        if (i < ns) {
            t = v < mn ? 0u : v - mn;
            refT[i] = (u16)t;
            prevT[i] = (u16)t;
        }
        out[i] = (u16)t;
    }
}

// background = (first maximum bin << 2) + 1 (:1974-1990); clears the histogram and the sums for the next steps.
// Run by all 1024 threads of ONE CTA: the last CTA of lossy_prep_kernel to finish (no separate launch).
__device__ __forceinline__ void lossy_background_body(LossyScalars* sc)
{
    __shared__ unsigned bv[1024];
    __shared__ int bi[1024];
    const int t = threadIdx.x;
    // 16 consecutive bins per thread: four independent 128-bit loads at L2 (the counts were written by other
    // CTAs' atomics), then the zeroing stores -- interleaving them would serialise sixteen L2 round trips
    uint4* hv = reinterpret_cast<uint4*>(&sc->hist[t * 16]);
    uint4 q[4];
#pragma unroll
    for (int k = 0; k < 4; ++k) q[k] = __ldcg(hv + k);
#pragma unroll
    for (int k = 0; k < 4; ++k) hv[k] = make_uint4(0u, 0u, 0u, 0u);
    const unsigned c16[16] = {q[0].x, q[0].y, q[0].z, q[0].w, q[1].x, q[1].y, q[1].z, q[1].w,
                              q[2].x, q[2].y, q[2].z, q[2].w, q[3].x, q[3].y, q[3].z, q[3].w};
    unsigned best = c16[0];
    int idx = t * 16;
#pragma unroll
    for (int k = 1; k < 16; ++k)
        if (c16[k] > best) {  // strict: the first maximum wins, like the reference's scan (:1976-1983)
            best = c16[k];
            idx = t * 16 + k;
        }
    bv[t] = best;
    bi[t] = idx;
    __syncthreads();
    for (int s = 512; s > 0; s >>= 1) {
        if (t < s && (bv[t + s] > bv[t] || (bv[t + s] == bv[t] && bi[t + s] < bi[t]))) {
            bv[t] = bv[t + s];
            bi[t] = bi[t + s];
        }
        __syncthreads();
    }
    if (t == 0) {
        sc->background = ((unsigned)bi[0] << 2) + 1u;
        sc->sum[0] = sc->sum[1] = sc->sum[2] = sc->sum[3] = 0ull;
        sc->cnt[0] = sc->cnt[1] = 0u;
    }
}

// true in every thread of the CTA that finishes last (its global writes being ordered before the ticket)
__device__ __forceinline__ bool lossy_last_cta(unsigned* ticket)
{
    __shared__ bool last;
    __threadfence();
    __syncthreads();
    if (threadIdx.x == 0) {
        const unsigned t = atomicAdd(ticket, 1u);
        last = (t == gridDim.x - 1);
        if (last) *ticket = 0;  // ready for the next frame
    }
    __syncthreads();
    if (last) __threadfence();
    return last;
}

// tmpT = tmp - min on the lossy rows; histogram of tmp >> 2 (get_background's, :1958-1962)
__global__ void __launch_bounds__(1024) lossy_prep_kernel(const u16* __restrict__ tmp, u16* __restrict__ tmpT, int ns, int subtract_min, LossyScalars* sc)
{
    extern __shared__ unsigned sh[];  // 16,384 bins = 64 KB (dynamic: above the 48 KB static limit)
    for (int i = threadIdx.x; i < 16384; i += blockDim.x) sh[i] = 0;
    __syncthreads();
    const unsigned mn = subtract_min ? sc->minv : 0u;
    for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < ns; i += gridDim.x * blockDim.x) {
        const unsigned v = tmp[i];
        tmpT[i] = (u16)(v < mn ? 0u : v - mn);
        atomicAdd(&sh[v >> 2], 1u);
    }
    __syncthreads();
    for (int i = threadIdx.x; i < 16384; i += blockDim.x) {
        const unsigned c = sh[i];
        if (c) atomicAdd(&sc->hist[i], c);
    }
    if (lossy_last_cta(&sc->ticket[0])) lossy_background_body(sc);
}

// The scalar part of the frame (:2337-2376), run by the last CTA of lossy_sums_kernel to finish: the reference's
// operation order in plain fp64, by ONE thread -- the others only fetch the window into shared memory with independent loads (a lone thread walking global
// memory pays a full round trip per entry: 40 us per frame in the first version of this kernel).
// nstds: size of the stdDevs window BEFORE this frame (0..40); head: slot of its oldest entry when full;
// first: this is the first non-initial frame.
// `error -= (int)round(x)` (:2367-2368, :2559-2563) as the reference's x86-64 build evaluates it: cvttsd2si gives INT_MIN
// for NaN -- an empty background / foreground split makes a spread 0 / 0 -- and for values beyond int range, and the int
// subtraction wraps.  A plain (int) here would be cvt.rzi, which saturates and turns NaN into 0.
__device__ __forceinline__ int lossy_sub_rounded(int error, double x)
{
    const double r = round(x);
    const int k = (r >= -2147483648.0 && r <= 2147483647.0) ? (int)r : INT_MIN;
    return (int)((unsigned)error - (unsigned)k);
}

__device__ __forceinline__ void lossy_bounds(double sd0, double sd1, double m0, double m1, double std_factor, int variant, int low0,
                                             int high0, int* low_out, int* high_out)
{
    double dh, dl;
    if (variant == 0) {  // addImageLossyNoCamera :2367-2368
        dh = fabs(__dsub_rn(sd1, m1));
        dl = fabs(__dsub_rn(sd0, m0));
    } else {  // addLoss :2559-2563
        dh = sd1 < m1 ? 0.0 : __dsub_rn(sd1, m1);
        dl = sd0 < m0 ? 0.0 : __dsub_rn(sd0, m0);
    }
    int high = lossy_sub_rounded(high0, __dmul_rn(dh, std_factor));
    int low = lossy_sub_rounded(low0, __dmul_rn(dl, std_factor));
    if (high < 0) high = 0;
    if (low < high) low = high;
    *low_out = low;
    *high_out = high;
}

__device__ __forceinline__ void lossy_decide_body(LossyScalars* sc, int ns, int nstds, int head, int first, int low0, int high0,
                                                  double std_factor, int variant, int quirk, int* __restrict__ errors_out)
{
    __shared__ double win[40][2];
    __shared__ unsigned long long sums[4];
    __shared__ unsigned cnts[2];
    const int t = threadIdx.x;
    if (t < 40) {  // window in time order: oldest first
        const int slot = nstds < 40 ? t : (head + t) % 40;
        win[t][0] = sc->stds[slot][0];
        win[t][1] = sc->stds[slot][1];
    } else if (t < 44) {
        sums[t - 40] = __ldcg(&sc->sum[t - 40]);  // other CTAs' atomics: read at L2
    } else if (t < 46) {
        cnts[t - 44] = __ldcg(&sc->cnt[t - 44]);
    }
    __syncthreads();
    if (t != 0) return;
    lossy_window_quirk(win, nstds, quirk);
    if (quirk && nstds == 40) sc->stds[(head + 38) % 40][1] = win[38][1];
    double sd0, sd1;
    if (nstds < 40) {
        const double s = (double)(sums[0] + sums[2]), s2 = (double)(long long)(sums[1] + sums[3]);
        sd0 = sd1 = __ddiv_rn(__dsqrt_rn(__dsub_rn(__dmul_rn(s, s), s2)), (double)ns);
    } else {
        const double s = (double)sums[0], s2 = (double)(long long)sums[1], b = (double)sums[2], b2 = (double)(long long)sums[3];
        sd0 = __ddiv_rn(__dsqrt_rn(__dsub_rn(__dmul_rn(b, b), b2)), (double)(int)cnts[1]);
        sd1 = __ddiv_rn(__dsqrt_rn(__dsub_rn(__dmul_rn(s, s), s2)), (double)(int)cnts[0]);
    }
    double f0 = sc->first[0], f1 = sc->first[1];
    if (first) {
        sc->first[0] = f0 = sd0;
        sc->first[1] = f1 = sd1;
    }
    // push (window not full) or drop the oldest and append (:2343-2351); the sum below runs oldest -> newest
    int n, from;
    if (nstds < 40) {
        sc->stds[nstds][0] = sd0;
        sc->stds[nstds][1] = sd1;
        n = nstds + 1;
        from = 0;
    } else {
        sc->stds[head][0] = sd0;  // the oldest slot becomes the newest
        sc->stds[head][1] = sd1;
        n = 40;
        from = 1;
    }
    double m0 = f0, m1 = f1;
    for (int i = from; i < (nstds < 40 ? nstds : 40); ++i) {
        m0 = __dadd_rn(m0, win[i][0]);
        m1 = __dadd_rn(m1, win[i][1]);
    }
    m0 = __dadd_rn(m0, sd0);
    m1 = __dadd_rn(m1, sd1);
    m0 = __ddiv_rn(m0, (double)(n + 1));
    m1 = __ddiv_rn(m1, (double)(n + 1));
    int high, low;
    lossy_bounds(sd0, sd1, m0, m1, std_factor, variant, low0, high0, &low, &high);
    sc->low_error = low;
    sc->high_error = high;
    errors_out[0] = low;
    errors_out[1] = high;
}

// stdDev's sums (:1993-2036), always split by img > background (the un-split case is the sum of both halves)
__global__ void __launch_bounds__(1024)
lossy_sums_kernel(const u16* __restrict__ prevT, const u16* __restrict__ tmpT, const u16* __restrict__ img, int ns, LossyScalars* sc,
                  int nstds, int head, int first, int low0, int high0, double std_factor, int variant, int quirk,
                  int* __restrict__ errors_out)
{
    const unsigned back = sc->background;
    unsigned long long sd = 0, sd2 = 0, bd = 0, bd2 = 0;
    unsigned nf = 0, nb = 0;
    for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < ns; i += gridDim.x * blockDim.x) {
        const int d = abs((int)tmpT[i] - (int)prevT[i]);
        const unsigned long long d2 = lossy_wrapped_square(d);
        if ((unsigned)img[i] > back) {
            sd += d; sd2 += d2; ++nf;
        } else {
            bd += d; bd2 += d2; ++nb;
        }
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        sd += __shfl_xor_sync(0xFFFFFFFFu, sd, o);
        sd2 += __shfl_xor_sync(0xFFFFFFFFu, sd2, o);
        bd += __shfl_xor_sync(0xFFFFFFFFu, bd, o);
        bd2 += __shfl_xor_sync(0xFFFFFFFFu, bd2, o);
        nf += __shfl_xor_sync(0xFFFFFFFFu, nf, o);
        nb += __shfl_xor_sync(0xFFFFFFFFu, nb, o);
    }
    // one set of global atomics per CTA, not per warp: they all land on the same six words
    __shared__ unsigned long long part[32][4];
    __shared__ unsigned pcnt[32][2];
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31, nwarps = blockDim.x >> 5;
    if (lane == 0) {
        part[warp][0] = sd; part[warp][1] = sd2; part[warp][2] = bd; part[warp][3] = bd2;
        pcnt[warp][0] = nf; pcnt[warp][1] = nb;
    }
    __syncthreads();
    if (threadIdx.x < 4) {
        unsigned long long a = 0;
        for (int k = 0; k < nwarps; ++k) a += part[k][threadIdx.x];
        atomicAdd(&sc->sum[threadIdx.x], a);
    } else if (threadIdx.x < 6) {
        unsigned a = 0;
        for (int k = 0; k < nwarps; ++k) a += pcnt[k][threadIdx.x - 4];
        atomicAdd(&sc->cnt[threadIdx.x - 4], a);
    }
    if (lossy_last_cta(&sc->ticket[1])) lossy_decide_body(sc, ns, nstds, head, first, low0, high0, std_factor, variant, quirk, errors_out);
}

// Per-pixel update (:2392-2421) with RunningAverage2::addImage / pixel / resetPixel folded in.
// len_before: frames in the ring before this one; slot_new: ring slot this frame is written to;
// slot_old: slot of the oldest frame (read only when the ring is full).
__global__ void lossy_update_kernel(const u16* __restrict__ tmp, const u16* __restrict__ tmpT, u16* __restrict__ out,
                                    u16* __restrict__ lastDL, u16* __restrict__ refT, u16* __restrict__ prevT, unsigned* __restrict__ sums,
                                    u16* __restrict__ cvalue, short* __restrict__ ccount, u16* __restrict__ ring, int n, int ns, int ra,
                                    int len_before, int slot_new, int slot_old, int variant, const LossyScalars* __restrict__ sc)
{
    const unsigned back = sc->background;
    const int low = sc->low_error, high = sc->high_error;
    const unsigned len_after = (unsigned)(len_before < ra ? len_before + 1 : ra);
    for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) {
        const unsigned v = tmp[i];
        if (i >= ns) {  // metadata rows: copied (:2419)
            out[i] = (u16)v;
            lastDL[i] = (u16)v;
            continue;
        }
        const unsigned t = tmpT[i];
        unsigned s = 0;
        short cc = 0;
        if (ra > 0) {
            s = sums[i] + t;
            cc = ccount[i];
            if (len_before == ra) {
                if (cc) {
                    --cc;
                    s -= cvalue[i];
                } else {
                    s -= ring[(size_t)slot_old * ns + i];
                }
            }
            ring[(size_t)slot_new * ns + i] = (u16)t;
        }
        const unsigned r = refT[i];
        const int diff = abs((int)t - (int)r);
        const int max_error = v > back ? high : low;
        unsigned o;
        if (diff <= max_error && (variant == 1 || ((unsigned)lastDL[i] >> 13) == (v >> 13))) {
            o = ra > 0 ? ((s / len_after) & 0xFFFFu) : r;
        } else {
            o = t;
            refT[i] = (u16)t;
            if (ra > 0) {
                cvalue[i] = (u16)t;
                cc = (short)len_after;
                s = t * len_after;
            }
        }
        if (ra > 0) {
            sums[i] = s;
            ccount[i] = cc;
        }
        out[i] = (u16)o;
        prevT[i] = (u16)o;
        lastDL[i] = (u16)v;
    }
}

// ---- several frames per launch ------------------------------------------------------------------
// The three launches per frame above cost more in launch latency than in work (0.65 MB per frame).  A run of frames
// goes through two launches instead:
//   1. lossy_back_kernel: get_background of EVERY frame of the run at once -- it depends on the input frame only
//      (h264.cpp:2331), so it does not belong in the sequential loop;
//   2. lossy_run_kernel: one cooperative launch, one 1024-thread CTA per SM, ONE grid barrier per frame.  The spread of
//      frame f+1 is |tmpT[f+1] - prevT| with prevT = the OUTPUT of frame f, so a thread adds its pixels' share of frame
//      f+1's sums right after it has produced them in frame f's update pass (each CTA stores its partial sums in its own
//      slot: no atomics, nothing to clear).  After the barrier every CTA adds the slots in the same order and evaluates
//      the error bounds itself (CTA 0 also records them), then updates its pixels of frame f+1, and so on.
// A pixel is always handled by the same thread (same grid-stride mapping in every frame), so the per-pixel state needs
// no barrier at all.  All reductions are integer sums: any order gives the same bits.
struct LossyRun {
    const u16* img;      // [m][n] frames as given (the "> background" test reads them)
    const u16* cur;      // [m][n] the reference's tmp: the same frames, bad-pixel-corrected when that is enabled
    u16* out;            // [m][n]
    u16 *lastDL, *refT, *prevT, *cvalue, *ring;
    unsigned* sums;
    short* ccount;
    LossyScalars* sc;
    int* errors_out;     // [m][2]
    int n, ns, ra, subtract_min, low0, high0, m, variant, quirk;
    long long frame_index;  // of the first frame of the run (>= 1)
    double std_factor;
};

// first-maximum bin of a 16,384-bin histogram (:1974-1990), by the 1024 threads of a CTA; bins in shared or global memory
__device__ __forceinline__ unsigned lossy_mode_of(const unsigned* hist, bool global, unsigned* bv, int* bi)
{
    const int t = threadIdx.x;
    const uint4* hv = reinterpret_cast<const uint4*>(hist + t * 16);
    uint4 q[4];
#pragma unroll
    for (int k = 0; k < 4; ++k) q[k] = global ? __ldcg(hv + k) : hv[k];
    const unsigned c16[16] = {q[0].x, q[0].y, q[0].z, q[0].w, q[1].x, q[1].y, q[1].z, q[1].w,
                              q[2].x, q[2].y, q[2].z, q[2].w, q[3].x, q[3].y, q[3].z, q[3].w};
    unsigned best = c16[0];
    int idx = t * 16;
#pragma unroll
    for (int k = 1; k < 16; ++k)
        if (c16[k] > best) {  // strict: the first maximum wins
            best = c16[k];
            idx = t * 16 + k;
        }
    // warp level first, then one value per warp
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        const unsigned ob = __shfl_xor_sync(0xFFFFFFFFu, best, o);
        const int oi = __shfl_xor_sync(0xFFFFFFFFu, idx, o);
        if (ob > best || (ob == best && oi < idx)) {
            best = ob;
            idx = oi;
        }
    }
    __syncthreads();  // bv / bi may still be read from a previous call
    if ((t & 31) == 0) {
        bv[t >> 5] = best;
        bi[t >> 5] = idx;
    }
    __syncthreads();
    if (t < 32) {
        best = bv[t];
        idx = bi[t];
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) {
            const unsigned ob = __shfl_xor_sync(0xFFFFFFFFu, best, o);
            const int oi = __shfl_xor_sync(0xFFFFFFFFu, idx, o);
            if (ob > best || (ob == best && oi < idx)) {
                best = ob;
                idx = oi;
            }
        }
        if (t == 0) bi[32] = idx;
    }
    __syncthreads();
    return ((unsigned)bi[32] << 2) + 1u;
}

// get_background of frames [0, m) of `cur` (lossy rows): grid = (parts, m).  parts == 1: the CTA's shared histogram is
// the frame's; otherwise the parts meet in hist_scratch[f] and the last one to arrive takes the mode (and clears it).
__global__ void __launch_bounds__(1024)
lossy_back_kernel(const u16* __restrict__ cur, int n, int ns, unsigned* __restrict__ hist_scratch, LossyScalars* sc)
{
    extern __shared__ unsigned sh[];  // 16,384 bins
    __shared__ unsigned bv[32];
    __shared__ int bi[33];
    __shared__ bool last;
    const int t = threadIdx.x, f = blockIdx.y, parts = gridDim.x;
    const u16* tmp = cur + (size_t)f * n;
    for (int i = t; i < 16384; i += 1024) sh[i] = 0;
    __syncthreads();
    if ((ns & 7) == 0) {  // 8 pixels per 128-bit load
        const uint4* v4 = reinterpret_cast<const uint4*>(tmp);
        for (int i = blockIdx.x * 1024 + t; i < ns / 8; i += parts * 1024) {
            const uint4 q = __ldg(v4 + i);
            const unsigned wds[4] = {q.x, q.y, q.z, q.w};
#pragma unroll
            for (int k = 0; k < 4; ++k) {
                atomicAdd(&sh[(wds[k] & 0xFFFFu) >> 2], 1u);
                atomicAdd(&sh[wds[k] >> 18], 1u);
            }
        }
    } else {
        for (int i = blockIdx.x * 1024 + t; i < ns; i += parts * 1024) atomicAdd(&sh[tmp[i] >> 2], 1u);
    }
    __syncthreads();
    if (parts == 1) {
        const unsigned b = lossy_mode_of(sh, false, bv, bi);
        if (t == 0) sc->back_run[f] = b;
        return;
    }
    unsigned* gh = hist_scratch + (size_t)f * 16384;
    for (int i = t; i < 16384; i += 1024) {
        const unsigned c = sh[i];
        if (c) atomicAdd(&gh[i], c);
    }
    __threadfence();
    __syncthreads();
    if (t == 0) {
        const unsigned k = atomicAdd(&sc->back_ticket[f], 1u);
        last = (k == (unsigned)parts - 1);
        if (last) sc->back_ticket[f] = 0;
    }
    __syncthreads();
    if (!last) return;
    __threadfence();
    const unsigned b = lossy_mode_of(gh, true, bv, bi);
    for (int i = t; i < 16384; i += 1024) gh[i] = 0;  // ready for the next run
    if (t == 0) sc->back_run[f] = b;
}

// all CTAs of a cooperative launch meet here; `target` counts arrivals since the launch (the counter starts at 0)
__device__ __forceinline__ void lossy_grid_barrier(unsigned* counter, unsigned& target)
{
    __syncthreads();
    if (threadIdx.x == 0) {
        target += gridDim.x;
        __threadfence();
        atomicAdd(counter, 1u);
        unsigned v;
        do {
            asm volatile("ld.acquire.gpu.u32 %0, [%1];" : "=r"(v) : "l"(counter) : "memory");
        } while ((int)(v - target) < 0);
    }
    __syncthreads();
}

__global__ void __launch_bounds__(1024) lossy_run_kernel(const __grid_constant__ LossyRun p)
{
    __shared__ unsigned long long part[32][4];
    __shared__ unsigned pcnt[32][2];
    __shared__ double win[40][2];
    __shared__ int decided[2];
    LossyScalars* sc = p.sc;
    const int t = threadIdx.x, gt = blockIdx.x * 1024 + t, gstride = gridDim.x * 1024;
    const int warp = t >> 5, lane = t & 31;
    const int n = p.n, ns = p.ns, ra = p.ra, G = gridDim.x;
    const unsigned mn = p.subtract_min ? sc->minv : 0u;
    unsigned bar_target = 0;

    // this CTA's share of stdDev's sums for frame `f`, given the pixel value `prev` it is compared with; stored in the
    // CTA's slot of set `par`
    unsigned long long sd = 0, sd2 = 0, bd = 0, bd2 = 0;
    unsigned nf = 0, nb = 0;
    auto add_pixel = [&](unsigned tv1, unsigned prev, bool fore) {
        const int d = abs((int)tv1 - (int)prev);
        const unsigned long long d2 = lossy_wrapped_square(d);
        if (fore) {
            sd += d; sd2 += d2; ++nf;
        } else {
            bd += d; bd2 += d2; ++nb;
        }
    };
    auto store_partials = [&](int par) {
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) {
            sd += __shfl_xor_sync(0xFFFFFFFFu, sd, o);
            sd2 += __shfl_xor_sync(0xFFFFFFFFu, sd2, o);
            bd += __shfl_xor_sync(0xFFFFFFFFu, bd, o);
            bd2 += __shfl_xor_sync(0xFFFFFFFFu, bd2, o);
            nf += __shfl_xor_sync(0xFFFFFFFFu, nf, o);
            nb += __shfl_xor_sync(0xFFFFFFFFu, nb, o);
        }
        if (lane == 0) {
            part[warp][0] = sd; part[warp][1] = sd2; part[warp][2] = bd; part[warp][3] = bd2;
            pcnt[warp][0] = nf; pcnt[warp][1] = nb;
        }
        __syncthreads();
        if (warp < 6) {  // warp w adds the 32 warps' entries of value w: a shuffle tree instead of 32 serial additions
            unsigned long long a = warp < 4 ? part[lane][warp] : (unsigned long long)pcnt[lane][warp - 4];
#pragma unroll
            for (int o = 16; o > 0; o >>= 1) a += __shfl_xor_sync(0xFFFFFFFFu, a, o);
            if (lane == 0) {
                if (warp < 4) sc->psum[par][blockIdx.x][warp] = a;
                else sc->pcnt[par][blockIdx.x][warp - 4] = (unsigned)a;
            }
        }
        sd = sd2 = bd = bd2 = 0;
        nf = nb = 0;
    };

    // ---- sums of the run's first frame against the state's prevT ----
    {
        const unsigned back0 = __ldcg(&sc->back_run[0]);
        for (int i = gt; i < ns; i += gstride) {
            const unsigned v = p.cur[i];
            add_pixel(v < mn ? 0u : v - mn, p.prevT[i], (unsigned)p.img[i] > back0);
        }
        store_partials((int)(p.frame_index & 1));
    }
    for (int f = 0; f < p.m; ++f) {
        lossy_grid_barrier(&sc->barrier, bar_target);
        const long long prior = p.frame_index + f - 1;  // non-initial frames before this one
        const int par = (int)((p.frame_index + f) & 1);
        const int nstds = (int)min(prior, 40LL), head = (int)(prior % 40), first = prior == 0;
        const int len_before = (int)min(prior, (long long)ra), slot = ra > 0 ? (int)(prior % ra) : 0;
        const u16* tmp = p.cur + (size_t)f * n;
        u16* out = p.out + (size_t)f * n;
        const unsigned back = __ldcg(&sc->back_run[f]);
        // ---- error bounds of this frame (:2337-2376): every CTA adds the slots and runs the reference's fp64 operation
        //      order in one thread ----
        {
            unsigned long long su[4] = {0, 0, 0, 0};
            unsigned cn[2] = {0, 0};
            if (t < G) {
                const ulonglong2* ps = reinterpret_cast<const ulonglong2*>(&sc->psum[par][t][0]);
                const ulonglong2 a = __ldcg(ps), b = __ldcg(ps + 1);
                const uint2 c = __ldcg(reinterpret_cast<const uint2*>(&sc->pcnt[par][t][0]));
                su[0] = a.x; su[1] = a.y; su[2] = b.x; su[3] = b.y;
                cn[0] = c.x; cn[1] = c.y;
            }
            if (t < 256) {  // LOSSY_MAX_CTAS slots: the first eight warps
#pragma unroll
                for (int o = 16; o > 0; o >>= 1) {
#pragma unroll
                    for (int k = 0; k < 4; ++k) su[k] += __shfl_xor_sync(0xFFFFFFFFu, su[k], o);
                    cn[0] += __shfl_xor_sync(0xFFFFFFFFu, cn[0], o);
                    cn[1] += __shfl_xor_sync(0xFFFFFFFFu, cn[1], o);
                }
                if (lane == 0) {
#pragma unroll
                    for (int k = 0; k < 4; ++k) part[warp][k] = su[k];
                    pcnt[warp][0] = cn[0];
                    pcnt[warp][1] = cn[1];
                }
            } else if (t >= 512 && t < 552) {  // window in time order: oldest first
                const int e = t - 512;
                const int s2 = nstds < 40 ? e : (head + e) % 40;
                win[e][0] = __ldcg(&sc->stds[s2][0]);
                win[e][1] = __ldcg(&sc->stds[s2][1]);
            }
            __syncthreads();
            if (t == 0) {
                for (int k = 0; k < 4; ++k) su[k] = 0;
                cn[0] = cn[1] = 0;
                for (int wv = 0; wv < 8; ++wv) {
                    for (int k = 0; k < 4; ++k) su[k] += part[wv][k];
                    cn[0] += pcnt[wv][0];
                    cn[1] += pcnt[wv][1];
                }
                lossy_window_quirk(win, nstds, p.quirk);
                double sd0, sd1;
                if (nstds < 40) {
                    const double s1 = (double)(su[0] + su[2]), s2 = (double)(long long)(su[1] + su[3]);
                    sd0 = sd1 = __ddiv_rn(__dsqrt_rn(__dsub_rn(__dmul_rn(s1, s1), s2)), (double)ns);
                } else {
                    const double s1 = (double)su[0], s2 = (double)(long long)su[1], b1 = (double)su[2], b2 = (double)(long long)su[3];
                    sd0 = __ddiv_rn(__dsqrt_rn(__dsub_rn(__dmul_rn(b1, b1), b2)), (double)(int)cn[1]);
                    sd1 = __ddiv_rn(__dsqrt_rn(__dsub_rn(__dmul_rn(s1, s1), s2)), (double)(int)cn[0]);
                }
                const double f0 = first ? sd0 : __ldcg(&sc->first[0]), f1 = first ? sd1 : __ldcg(&sc->first[1]);
                const int cnt = nstds < 40 ? nstds + 1 : 40, from = nstds < 40 ? 0 : 1;
                double m0 = f0, m1 = f1;
                for (int i = from; i < (nstds < 40 ? nstds : 40); ++i) {
                    m0 = __dadd_rn(m0, win[i][0]);
                    m1 = __dadd_rn(m1, win[i][1]);
                }
                m0 = __ddiv_rn(__dadd_rn(m0, sd0), (double)(cnt + 1));
                m1 = __ddiv_rn(__dadd_rn(m1, sd1), (double)(cnt + 1));
                int low, high;
                lossy_bounds(sd0, sd1, m0, m1, p.std_factor, p.variant, p.low0, p.high0, &low, &high);
                decided[0] = low;
                decided[1] = high;
                if (blockIdx.x == 0) {  // the state that outlives the frame is written once
                    if (first) {
                        sc->first[0] = sd0;
                        sc->first[1] = sd1;
                    }
                    // the other CTAs read the window in this same interval: the smeared value is what they compute for
                    // themselves, and the slot of the new entry is the one nobody uses (the oldest, or beyond the end)
                    if (p.quirk && nstds == 40) sc->stds[(head + 38) % 40][1] = win[38][1];
                    const int dst = nstds < 40 ? nstds : head;  // push, or the oldest slot becomes the newest
                    sc->stds[dst][0] = sd0;
                    sc->stds[dst][1] = sd1;
                    sc->background = back;
                    sc->low_error = low;
                    sc->high_error = high;
                    p.errors_out[2 * f] = low;
                    p.errors_out[2 * f + 1] = high;
                }
            }
            __syncthreads();
        }
        const int low = decided[0], high = decided[1];
        // ---- per-pixel update (:2392-2421), and this CTA's share of the next frame's spread ----
        const bool more = f + 1 < p.m;
        const u16* tmp1 = tmp + n;
        const u16* img1 = p.img + (size_t)(f + 1) * n;
        const unsigned back1 = more ? __ldcg(&sc->back_run[f + 1]) : 0u;
        const unsigned len_after = (unsigned)(len_before < ra ? len_before + 1 : ra);
        // Three pixels of the thread at a time, ALL their loads first: the state arrays may alias each other as far as the
        // compiler knows, so a plain grid-stride loop waits for one pixel's stores before it issues the next pixel's loads --
        // three serial trips to L2 per frame at 640 x 512 (2.2 pixels per thread).
        constexpr int PP = 3;
        for (int base = gt; base < n; base += PP * gstride) {
            unsigned v[PP], sm[PP], rv[PP], ld[PP], cvv[PP], rg[PP], v1[PP], im1[PP];
            short ccv[PP];
#pragma unroll
            for (int q = 0; q < PP; ++q) {
                const int i = base + q * gstride;
                v[q] = sm[q] = rv[q] = ld[q] = cvv[q] = rg[q] = v1[q] = im1[q] = 0;
                ccv[q] = 0;
                if (i < n) {
                    v[q] = tmp[i];
                    if (i < ns) {
                        if (ra > 0) {
                            sm[q] = p.sums[i];
                            ccv[q] = p.ccount[i];
                            if (len_before == ra) {
                                cvv[q] = p.cvalue[i];
                                rg[q] = p.ring[(size_t)slot * ns + i];
                            }
                        }
                        rv[q] = p.refT[i];
                        ld[q] = p.lastDL[i];
                        if (more) {
                            v1[q] = tmp1[i];
                            im1[q] = img1[i];
                        }
                    }
                }
            }
#pragma unroll
            for (int q = 0; q < PP; ++q) {
                const int i = base + q * gstride;
                if (i >= n) break;
                if (i >= ns) {
                    out[i] = (u16)v[q];
                    p.lastDL[i] = (u16)v[q];
                    continue;
                }
                const unsigned tv = v[q] < mn ? 0u : v[q] - mn;
                unsigned sacc = 0;
                short cc = 0;
                if (ra > 0) {
                    sacc = sm[q] + tv;
                    cc = ccv[q];
                    if (len_before == ra) {
                        if (cc) {
                            --cc;
                            sacc -= cvv[q];
                        } else {
                            sacc -= rg[q];
                        }
                    }
                    p.ring[(size_t)slot * ns + i] = (u16)tv;
                }
                const unsigned r = rv[q];
                const int diff = abs((int)tv - (int)r);
                const int max_error = v[q] > back ? high : low;
                unsigned o;
                if (diff <= max_error && (p.variant == 1 || (ld[q] >> 13) == (v[q] >> 13))) {
                    o = ra > 0 ? ((sacc / len_after) & 0xFFFFu) : r;
                } else {
                    o = tv;
                    p.refT[i] = (u16)tv;
                    if (ra > 0) {
                        p.cvalue[i] = (u16)tv;
                        cc = (short)len_after;
                        sacc = tv * len_after;
                    }
                }
                if (ra > 0) {
                    p.sums[i] = sacc;
                    p.ccount[i] = cc;
                }
                out[i] = (u16)o;
                p.lastDL[i] = (u16)v[q];
                if (more) {
                    add_pixel(v1[q] < mn ? 0u : v1[q] - mn, o, im1[q] > back1);
                } else {
                    p.prevT[i] = (u16)o;  // the state the next call starts from
                }
            }
        }
        if (more) store_partials(par ^ 1);
    }
}

// frames [0, m) of img / cur / out are consecutive non-initial frames, the first of them frame number frame_index.
// hist_scratch: LOSSY_MAX_RUN x 16,384 zeroed counters.  Returns 1 when the device cannot launch cooperatively (the caller
// then goes frame by frame).
int launch_lossy_run(const u16* img, const u16* cur, u16* out, u16* lastDL, u16* refT, u16* prevT, unsigned* sums, u16* cvalue,
                     short* ccount, u16* ring, int n, int ns, int ra, int subtract_min, long long frame_index, int m, int low0,
                     int high0, double std_factor, int variant, int quirk, void* scalars, unsigned* hist_scratch, int* errors_out_dev,
                     cudaStream_t st)
{
    if (m <= 0) return 0;
    if (m > LOSSY_MAX_RUN) {
        set_error("lossy_run: at most %d frames per launch", LOSSY_MAX_RUN);
        return -1;
    }
    int dev = 0, coop = 0, per_sm = 0;
    RIRB_CUDA_OK(cudaGetDevice(&dev));
    if (cudaDeviceGetAttribute(&coop, cudaDevAttrCooperativeLaunch, dev) != cudaSuccess || !coop ||
        cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, lossy_run_kernel, 1024, 0) != cudaSuccess || per_sm < 1) {
        cudaGetLastError();
        return 1;
    }
    LossyRun p;
    p.img = img; p.cur = cur; p.out = out; p.lastDL = lastDL; p.refT = refT; p.prevT = prevT; p.cvalue = cvalue;
    p.ring = ring; p.sums = sums; p.ccount = ccount; p.sc = (LossyScalars*)scalars; p.errors_out = errors_out_dev;
    p.n = n; p.ns = ns; p.ra = ra; p.subtract_min = subtract_min; p.low0 = low0; p.high0 = high0; p.m = m;
    p.variant = variant; p.quirk = quirk;
    p.frame_index = frame_index; p.std_factor = std_factor;
    // backgrounds of the whole run: enough CTAs per frame to fill the machine once
    RIRB_SMEM_ATTR(lossy_back_kernel, 16384 * 4);
    int parts = (int)max(1LL, min((long long)ceil_div(ns, 1024 * 8 * 4), (long long)(2 * sm_count() / m)));
    RIRB_LAUNCH(lossy_back_kernel, dim3((unsigned)parts, (unsigned)m), 1024, 16384 * 4, st, cur, n, ns, hist_scratch, p.sc);
    const int grid = (int)max(1LL, min(min((long long)ceil_div(n, 1024 * 2), (long long)sm_count()), (long long)LOSSY_MAX_CTAS));
    RIRB_CUDA_OK(cudaMemsetAsync(&p.sc->barrier, 0, sizeof(unsigned), st));
    void* args[] = {&p};
    RIRB_CUDA_OK(cudaLaunchCooperativeKernel((const void*)lossy_run_kernel, dim3((unsigned)grid), dim3(1024), args, 0, st));
    g_launches.fetch_add(1, std::memory_order_relaxed);
    return 0;
}

size_t lossy_hist_scratch_bytes() { return (size_t)LOSSY_MAX_RUN * 16384 * sizeof(unsigned); }
int lossy_max_run() { return LOSSY_MAX_RUN; }

// ---- launchers ----------------------------------------------------------------------------------
size_t lossy_scalars_bytes() { return sizeof(LossyScalars); }

int launch_lossy_first(const u16* tmp, u16* out, u16* lastDL, u16* refT, u16* prevT, int n, int ns, int subtract_min, void* scalars,
                       int* errors_out_dev, int low0, int high0, cudaStream_t st)
{
    LossyScalars* sc = (LossyScalars*)scalars;
    RIRB_CUDA_OK(cudaMemsetAsync(sc, 0, sizeof(LossyScalars), st));
    const int grid = (int)min((long long)ceil_div(n, 256), (long long)sm_count() * 8);
    if (subtract_min) {
        const unsigned init = 65535u;
        RIRB_CUDA_OK(cudaMemcpyAsync(&sc->minv, &init, sizeof(unsigned), cudaMemcpyHostToDevice, st));
        if (ns > 0) RIRB_LAUNCH(lossy_min_kernel, grid, 256, 0, st, tmp, ns, sc);
    }
    RIRB_LAUNCH(lossy_first_kernel, grid, 256, 0, st, tmp, out, lastDL, refT, prevT, n, ns, subtract_min, sc);
    const int e[2] = {low0, high0};
    RIRB_CUDA_OK(cudaMemcpyAsync(errors_out_dev, e, sizeof(e), cudaMemcpyHostToDevice, st));
    return 0;
}

int launch_lossy_frame(const u16* img, const u16* tmp, u16* tmpT, u16* out, u16* lastDL, u16* refT, u16* prevT, unsigned* sums,
                       u16* cvalue, short* ccount, u16* ring, int n, int ns, int ra, int subtract_min, long long frame_index,
                       int low0, int high0, double std_factor, int variant, int quirk, void* scalars, int* errors_out_dev, cudaStream_t st)
{
    LossyScalars* sc = (LossyScalars*)scalars;
    const int grid_s = (int)max(1LL, min((long long)ceil_div(ns, 256), (long long)sm_count() * 8));
    const int grid_n = (int)max(1LL, min((long long)ceil_div(n, 256), (long long)sm_count() * 8));
    // frame_index >= 1: frames already stored.  Window / ring sizes follow from it.
    const long long prior = frame_index - 1;                 // non-initial frames before this one
    const int nstds = (int)min(prior, 40LL);
    const int len_before = (int)min(prior, (long long)ra);
    const int slot_new = ra > 0 ? (int)(prior % ra) : 0;     // circular: the slot of the oldest frame once full
    const int slot_old = slot_new;
    RIRB_SMEM_ATTR(lossy_prep_kernel, 16384 * 4);
    const int grid_r = (int)max(1LL, min((long long)ceil_div(ns, 1024 * 4), (long long)sm_count()));  // reductions: few, fat CTAs
    const int head = (int)(prior % 40);  // circular stdDevs window: slot of the oldest entry once 40 are in
    // three launches per frame: the two scalar steps run in the last CTA of the reduction before them
    RIRB_LAUNCH(lossy_prep_kernel, grid_r, 1024, 16384 * 4, st, tmp, tmpT, ns, subtract_min, sc);
    RIRB_LAUNCH(lossy_sums_kernel, grid_r, 1024, 0, st, prevT, tmpT, img, ns, sc, nstds, head, prior == 0 ? 1 : 0, low0, high0, std_factor,
                variant, quirk, errors_out_dev);
    RIRB_LAUNCH(lossy_update_kernel, grid_n, 256, 0, st, tmp, tmpT, out, lastDL, refT, prevT, sums, cvalue, ccount, ring, n, ns, ra,
                len_before, slot_new, slot_old, variant, sc);
    return 0;
}

}  // namespace rirb
