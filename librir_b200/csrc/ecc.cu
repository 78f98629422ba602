// librir_b200/csrc/ecc.cu -- the registration front end on the GPU (SURVEY.md 8f-4).
//
// Reference: MaskedRegistratorECC.compute, librir/registration/masked_registration_ecc.py:105-191 --
//   crop of the Gaussian-filtered frame, optional quantile clamp of template and image (:143-151),
//   min/max normalisation of both (:153-160), then
//   cv2.findTransformECC(template, image, warp, MOTION_TRANSLATION, (COUNT|EPS, 500, 1e-3), mask, 1) (:165-167).
// The ECC iteration is OpenCV's (4.13.0, video/src/ecc.cpp), third-party to librir: restated in
// oracle/ecc.py, which is pinned against cv2 itself; this file follows that restatement.
//
// What OpenCV does per iteration, and what it becomes here:
//   warpAffine x4 (image, d/dx, d/dy bilinear; mask nearest)   -> for a pure translation warpAffine's fixed-point
//       coordinates (10 fractional bits, rounded to 1/32 px) give EVERY pixel the same integer offset and the same four
//       float weights, so the warp is a 4-tap stencil with launch-constant weights, evaluated on the fly;
//   meanStdDev x2, subtract x2, 7 dot products over full images   -> ONE pass that accumulates 15 raw sums in fp64
//       (products of two floats are exact in fp64) from which every masked, zero-meaned quantity follows
//       algebraically; no intermediate image is ever written; per-CTA partial sums are added in a fixed order (no
//       atomics), so results are reproducible bit for bit;
//   2x2 inverse, lambda, parameter update                         -> one thread, in the float / double types of OpenCV's
//       Mats.
// The whole solve (min/max, normalisation + gradients, all iterations) is ONE cooperative launch with grid barriers
// between the phases (ecc_solve_kernel); a launch-per-iteration driver (ecc_iter_kernel, "last CTA done" epilogue) is
// the fallback.  The host reads 40 bytes back per frame; nothing else crosses PCIe.
// Traffic per iteration: template, image, two gradients (float) + mask, all L2-resident (3 MB at 448 x 358): the loop
// is bound by launch / barrier latency, not by memory.
#include <cooperative_groups.h>
#include <math.h>
#include <string.h>

#include <memory>
#include <mutex>
#include <vector>

#include "../../include/librir_b200.h"
#include "common.cuh"
#include "handles.h"
#include "kernels.h"

namespace rirb {

enum { A_N, A_I, A_T, A_II, A_TT, A_IT, A_H11, A_H12, A_H22, A_B1, A_B2, A_C1, A_C2, A_D1, A_D2, NACC };

struct EccDev {
    double rho, last_rho, eps;
    unsigned ticket;
    unsigned mm[4];  // order-preserving keys: template min, max, image min, max
    float tx, ty;
    int it, max_it, done, status;  // status: 0 ok, 1 NaN (cv2: "NaN encountered."), 2 correlation about to be minimised
    // a run of solves queued back to back (rirb_ecc_track): the solve after this one must not run -- this one failed, or its
    // correlation fell under the confidence threshold and the host will replace the reference image; skipped = this slot's
    // solve did not run for that reason
    int stop, skipped;
};

struct EccResult {  // what the host reads back
    double rho;
    float tx, ty;
    int it, done, status;
};

__device__ __forceinline__ unsigned fkey(float f)
{
    const unsigned b = __float_as_uint(f);
    return b ^ ((b >> 31) ? 0xFFFFFFFFu : 0x80000000u);
}
__device__ __forceinline__ float fkey_inv(unsigned k)
{
    return __uint_as_float(k ^ ((k >> 31) ? 0x80000000u : 0xFFFFFFFFu));
}

// masked_registration_ecc.py:147-151: where EITHER image exceeds the threshold, BOTH are set to it
__device__ __forceinline__ float clamp_pair(float own, float other, float th) { return (own > th || other > th) ? th : own; }

__global__ void ecc_begin_kernel(EccDev* d, float tx, float ty, int max_it, double eps)
{
    d->ticket = 0;
    d->mm[0] = d->mm[2] = 0xFFFFFFFFu;
    d->mm[1] = d->mm[3] = 0u;
    d->tx = tx;
    d->ty = ty;
    d->rho = -1.0;        // ecc.cpp: rho = -1, last_rho = -termination_eps
    d->last_rho = -eps;
    d->eps = eps;
    d->it = 0;
    d->max_it = max_it;
    d->done = (max_it <= 0) || !(fabs(-1.0 + eps) >= eps);
    d->status = 0;
    d->stop = d->skipped = 0;
}

constexpr int ECC_THREADS = 256;  // 512 and 1024 were measured: no consistent gain (profiles/r2_ecc_bench.jsonl), 1024 spills

__global__ void __launch_bounds__(ECC_THREADS) ecc_minmax_kernel(const float* __restrict__ ref, const float* __restrict__ cur, int n,
                                                                  float thresh, EccDev* d)
{
    unsigned k[4] = {0xFFFFFFFFu, 0u, 0xFFFFFFFFu, 0u};
    for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) {
        const float r = ref[i], c = cur[i];
        const unsigned kr = fkey(clamp_pair(r, c, thresh)), kc = fkey(clamp_pair(c, r, thresh));
        k[0] = min(k[0], kr);
        k[1] = max(k[1], kr);
        k[2] = min(k[2], kc);
        k[3] = max(k[3], kc);
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        k[0] = min(k[0], __shfl_down_sync(0xFFFFFFFFu, k[0], o));
        k[1] = max(k[1], __shfl_down_sync(0xFFFFFFFFu, k[1], o));
        k[2] = min(k[2], __shfl_down_sync(0xFFFFFFFFu, k[2], o));
        k[3] = max(k[3], __shfl_down_sync(0xFFFFFFFFu, k[3], o));
    }
    __shared__ unsigned kred[ECC_THREADS / 32][4];
    if ((threadIdx.x & 31) == 0)
#pragma unroll
        for (int q = 0; q < 4; ++q) kred[threadIdx.x >> 5][q] = k[q];
    __syncthreads();
    if (threadIdx.x < 4) {  // one atomic per value and CTA
        unsigned v = kred[0][threadIdx.x];
        for (int q = 1; q < ECC_THREADS / 32; ++q) v = (threadIdx.x & 1) ? max(v, kred[q][threadIdx.x]) : min(v, kred[q][threadIdx.x]);
        if (threadIdx.x & 1) atomicMax(&d->mm[threadIdx.x], v); else atomicMin(&d->mm[threadIdx.x], v);
    }
}

// numpy float32: (im - mi) / (ma - mi), two roundings
__device__ __forceinline__ float normalise(float v, float mi, float span) { return __fdiv_rn(__fsub_rn(v, mi), span); }

// T = normalised template, I = normalised image, gx / gy = its [-0.5 0 0.5] derivatives (reflect-101 at the window's
// edge, ecc.cpp's filter2D) times the 0/1 mask.
__global__ void __launch_bounds__(ECC_THREADS)
ecc_normalise_kernel(const float* __restrict__ ref, const float* __restrict__ cur, const u8* __restrict__ mask, int w, int h,
                     float thresh, const EccDev* __restrict__ d, float* __restrict__ T, float* __restrict__ I, float* __restrict__ gx,
                     float* __restrict__ gy)
{
    const int x = blockIdx.x * blockDim.x + threadIdx.x;
    const int y = blockIdx.y;
    if (x >= w) return;
    const float mi_t = fkey_inv(d->mm[0]), span_t = __fsub_rn(fkey_inv(d->mm[1]), mi_t);
    const float mi_i = fkey_inv(d->mm[2]), span_i = __fsub_rn(fkey_inv(d->mm[3]), mi_i);
    auto img = [&](int xx, int yy) {
        const int i = yy * w + xx;
        return normalise(clamp_pair(cur[i], ref[i], thresh), mi_i, span_i);
    };
    const int i = y * w + x;
    T[i] = normalise(clamp_pair(ref[i], cur[i], thresh), mi_t, span_t);
    I[i] = img(x, y);
    const int xm = x == 0 ? (w > 1 ? 1 : 0) : x - 1, xp = x == w - 1 ? (w > 1 ? w - 2 : 0) : x + 1;
    const int ym = y == 0 ? (h > 1 ? 1 : 0) : y - 1, yp = y == h - 1 ? (h > 1 ? h - 2 : 0) : y + 1;
    const float m = (mask == nullptr || mask[i] != 0) ? 1.0f : 0.0f;
    gx[i] = __fmul_rn(__fsub_rn(__fmul_rn(0.5f, img(xp, y)), __fmul_rn(0.5f, img(xm, y))), m);
    gy[i] = __fmul_rn(__fsub_rn(__fmul_rn(0.5f, img(x, yp)), __fmul_rn(0.5f, img(x, ym))), m);
}

__global__ void ecc_u16_to_f32_kernel(const u16* __restrict__ src, float* __restrict__ dst, int n)
{
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) dst[i] = (float)src[i];
}

__global__ void ecc_cast_u16_kernel(const float* __restrict__ src, u16* __restrict__ dst, int n)
{
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    // numpy's astype(uint16) on x86-64: cvttss2si to int32, low 16 bits kept.  NaN and values beyond int range give
    // INT_MIN, i.e. 0 -- where __float2int_rz would saturate +inf and values >= 2^31 to 65,535
    const float v = src[i];
    dst[i] = (v >= -2147483648.0f && v < 2147483648.0f) ? (u16)__float2int_rz(v) : (u16)0;
}

// ---- one ECC iteration (ecc.cpp, the body of the for loop), in pieces shared by the two drivers below -----------
struct EccShift {  // warpAffine's fixed point (imgwarp.cpp): AB_BITS = 10, INTER_BITS = 5; M = [1 0 tx; 0 1 ty], WARP_INVERSE_MAP
    int ox, oy, oxn, oyn;
    float w00, w01, w10, w11;
    __device__ EccShift(float tx, float ty)
    {
        const int SX = __double2int_rn((double)tx * 1024.0), SY = __double2int_rn((double)ty * 1024.0);
        ox = (SX + 16) >> 10;  // bilinear: round_delta = 1024 / 32 / 2, then 5 fractional bits
        oy = (SY + 16) >> 10;
        const float fx = (float)(((SX + 16) >> 5) & 31) * 0.03125f, fy = (float)(((SY + 16) >> 5) & 31) * 0.03125f;
        oxn = (SX + 512) >> 10;  // nearest: round_delta = 1024 / 2
        oyn = (SY + 512) >> 10;
        w00 = __fmul_rn(1.0f - fy, 1.0f - fx);
        w01 = __fmul_rn(1.0f - fy, fx);
        w10 = __fmul_rn(fy, 1.0f - fx);
        w11 = __fmul_rn(fy, fx);
    }
};

// the 15 sums of pixels p0, p0 + stride, ... < w * h
__device__ __forceinline__ void ecc_accumulate(const float* __restrict__ T, const float* __restrict__ I, const float* __restrict__ gx,
                                               const float* __restrict__ gy, const u8* __restrict__ mask, int w, int h, const EccShift& sh,
                                               int p0, int stride, double (&a)[NACC])
{
    const int npx = w * h;
    for (int p = p0; p < npx; p += stride) {
        const int y = p / w, x = p - y * w;
        const int ix = x + sh.ox, iy = y + sh.oy;
        const bool x0 = ix >= 0 && ix < w, x1 = ix + 1 >= 0 && ix + 1 < w, y0 = iy >= 0 && iy < h, y1 = iy + 1 >= 0 && iy + 1 < h;
        const int i00 = iy * w + ix;
        auto warp = [&](const float* __restrict__ s) {  // remapBilinear: S[0]*w0 + S[1]*w1 + S[step]*w2 + S[step+1]*w3, border 0
            const float s00 = (x0 && y0) ? s[i00] : 0.f, s01 = (x1 && y0) ? s[i00 + 1] : 0.f;
            const float s10 = (x0 && y1) ? s[i00 + w] : 0.f, s11 = (x1 && y1) ? s[i00 + w + 1] : 0.f;
            return __fadd_rn(__fadd_rn(__fadd_rn(__fmul_rn(s00, sh.w00), __fmul_rn(s01, sh.w01)), __fmul_rn(s10, sh.w10)),
                             __fmul_rn(s11, sh.w11));
        };
        const double Iw = warp(I), Gx = warp(gx), Gy = warp(gy);
        const int mx = x + sh.oxn, my = y + sh.oyn;
        const bool m = mx >= 0 && mx < w && my >= 0 && my < h && (mask == nullptr || mask[my * w + mx] != 0);
        const double t = T[p];
        a[A_H11] += Gx * Gx;
        a[A_H12] += Gx * Gy;
        a[A_H22] += Gy * Gy;
        a[A_B1] += Gx * Iw;
        a[A_B2] += Gy * Iw;
        if (m) {
            a[A_N] += 1.0;
            a[A_I] += Iw;
            a[A_T] += t;
            a[A_II] += Iw * Iw;
            a[A_TT] += t * t;
            a[A_IT] += Iw * t;
            a[A_C1] += Gx;
            a[A_C2] += Gy;
            a[A_D1] += Gx * t;
            a[A_D2] += Gy * t;
        }
    }
}

// CTA-wide sum of the 15 values into this CTA's slot of `partials` ([gridDim.x][NACC]).  No atomics anywhere on the way to
// the result: the order of every addition is fixed, so a frame gives the same bits on every run and in every batching.
__device__ __forceinline__ void ecc_block_partial(double (&a)[NACC], double (*red)[NACC], double* partials)
{
#pragma unroll
    for (int k = 0; k < NACC; ++k)
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) a[k] += __shfl_down_sync(0xFFFFFFFFu, a[k], o);
    const int lane = threadIdx.x & 31, wi = threadIdx.x >> 5;
    if (lane == 0)
#pragma unroll
        for (int k = 0; k < NACC; ++k) red[wi][k] = a[k];
    __syncthreads();
    if (threadIdx.x < NACC) {
        double s = 0.0;
        for (int q = 0; q < ECC_THREADS / 32; ++q) s += red[q][threadIdx.x];
        partials[(size_t)blockIdx.x * NACC + threadIdx.x] = s;
    }
}

// Sum of all CTAs' slots, 8 threads per value (strided, then a fixed shuffle tree); result in sums[NACC] (shared).
// The slots come down first, every thread of the CTA fetching its share in ONE round trip to L2 (the strided loop used to
// be ~19 dependent round trips for the 120 adding threads: a third of an iteration); the order of the additions is the
// old one, so the sums are the same bits.
constexpr int ECC_MAX_SLOTS = 320;  // >= the largest grid either driver launches (2 CTAs per SM)
__device__ __forceinline__ void ecc_sum_partials(const double* partials, int nblk, double* sums, double* stage)
{
    static_assert(NACC * 8 <= ECC_THREADS, "8 threads per accumulated value");
    const int total = nblk * NACC;
    constexpr int PER = 10;
    for (int base = 0; base < total; base += PER * ECC_THREADS) {
        double v[PER];
#pragma unroll
        for (int q = 0; q < PER; ++q) {
            const int i = base + q * ECC_THREADS + (int)threadIdx.x;
            v[q] = i < total ? __ldcg(&partials[i]) : 0.0;
        }
#pragma unroll
        for (int q = 0; q < PER; ++q) {
            const int i = base + q * ECC_THREADS + (int)threadIdx.x;
            if (i < total) stage[i] = v[q];
        }
    }
    __syncthreads();
    const bool active = threadIdx.x < NACC * 8;
    const int k = threadIdx.x >> 3, j = threadIdx.x & 7;
    double v = 0.0;
    if (active)
        for (int b = j; b < nblk; b += 8) v += stage[b * NACC + k];
    v += __shfl_down_sync(0xFFFFFFFFu, v, 4, 8);
    v += __shfl_down_sync(0xFFFFFFFFu, v, 2, 8);
    v += __shfl_down_sync(0xFFFFFFFFu, v, 1, 8);
    if (active && j == 0) sums[k] = v;
    __syncthreads();
}

struct EccIterate {  // the scalar state of the loop
    float tx, ty;
    double rho, last_rho;
    int it, status, done;
};

// From the sums to the next shift: means / norms under the warped mask, 2 x 2 Hessian inverse, rho, lambda, update --
// in the float / double types OpenCV's Mats have.
__device__ __forceinline__ void ecc_update(const double* acc, EccIterate& s, int max_it, double eps)
{
    const double n = acc[A_N], sI = acc[A_I], sT = acc[A_T], sII = acc[A_II], sTT = acc[A_TT], sIT = acc[A_IT];
    const double h11 = acc[A_H11], h12 = acc[A_H12], h22 = acc[A_H22], b1 = acc[A_B1], b2 = acc[A_B2];
    const double c1 = acc[A_C1], c2 = acc[A_C2], d1 = acc[A_D1], d2 = acc[A_D2];
    s.it += 1;
    s.status = 0;
    if (n <= 0.0) {
        s.status = 1;
    } else {
        // meanStdDev under the warped mask; subtract(image, mean) works in the image's type: the mean is rounded to float
        const double meanI = sI / n, meanT = sT / n;
        const double varI = fmax(sII / n - meanI * meanI, 0.0), varT = fmax(sTT / n - meanT * meanT, 0.0);
        const double img_norm = sqrt(n * varI), tmp_norm = sqrt(n * varT);
        const double muI = (double)(float)meanI, muT = (double)(float)meanT;
        const float H11 = (float)h11, H12 = (float)h12, H22 = (float)h22;  // Mat hessian is CV_32F
        // cv::invert of a 2 x 2 float matrix: closed form evaluated in double
        const double det = (double)H11 * H22 - (double)H12 * H12;
        const double id = det != 0.0 ? 1.0 / det : 0.0;
        const float Hi11 = (float)(H22 * id), Hi22 = (float)(H11 * id), Hi12 = (float)(-(double)H12 * id);
        const double corr = sIT - muT * sI - muI * sT + muI * muT * n;  // templateZM . imageWarped
        s.last_rho = s.rho;
        s.rho = corr / (img_norm * tmp_norm);
        if (isnan(s.rho) || det == 0.0) {
            s.status = 1;
        } else {
            const double pI1 = b1 - muI * c1, pI2 = b2 - muI * c2;  // J^T (I - mean), exact sums
            const double pT1 = d1 - muT * c1, pT2 = d2 - muT * c2;  // J^T (T - mean)
            const float ip1 = (float)pI1, ip2 = (float)pI2, tp1 = (float)pT1, tp2 = (float)pT2;  // CV_32F projections
            const float iph1 = (float)((double)Hi11 * ip1 + (double)Hi12 * ip2), iph2 = (float)((double)Hi12 * ip1 + (double)Hi22 * ip2);
            const double lam_n = img_norm * img_norm - ((double)ip1 * iph1 + (double)ip2 * iph2);
            const double lam_d = corr - ((double)tp1 * iph1 + (double)tp2 * iph2);
            if (lam_d <= 0.0) {
                s.rho = -1.0;
                s.status = 2;
            } else {
                const double lam = lam_n / lam_d;
                const float e1 = (float)(lam * pT1 - pI1), e2 = (float)(lam * pT2 - pI2);  // J^T (lambda T - I)
                const float dp1 = (float)((double)Hi11 * e1 + (double)Hi12 * e2), dp2 = (float)((double)Hi12 * e1 + (double)Hi22 * e2);
                s.tx = __fadd_rn(s.tx, dp1);
                s.ty = __fadd_rn(s.ty, dp2);
            }
        }
    }
    s.done = s.status != 0 || s.it >= max_it || !(fabs(s.rho - s.last_rho) >= eps);
}

// Driver 1: one launch per iteration; the last CTA to finish adds up the slots and runs the update (used when a
// cooperative launch is not possible).
__global__ void __launch_bounds__(ECC_THREADS)
ecc_iter_kernel(const float* __restrict__ T, const float* __restrict__ I, const float* __restrict__ gx, const float* __restrict__ gy,
                const u8* __restrict__ mask, int w, int h, EccDev* d, double* partials)
{
    if (d->done) return;  // written by the previous launch's last CTA only
    __shared__ double red[ECC_THREADS / 32][NACC];
    __shared__ double sums[NACC];
    __shared__ double stage[ECC_MAX_SLOTS * NACC];
    __shared__ bool last;
    const EccShift sh(d->tx, d->ty);
    double a[NACC];
#pragma unroll
    for (int k = 0; k < NACC; ++k) a[k] = 0.0;
    ecc_accumulate(T, I, gx, gy, mask, w, h, sh, blockIdx.x * ECC_THREADS + threadIdx.x, gridDim.x * ECC_THREADS, a);
    ecc_block_partial(a, red, partials);
    __threadfence();
    __syncthreads();
    if (threadIdx.x == 0) last = atomicAdd(&d->ticket, 1u) == gridDim.x - 1;
    __syncthreads();
    if (!last) return;
    __threadfence();
    ecc_sum_partials(partials, (int)gridDim.x, sums, stage);
    if (threadIdx.x != 0) return;
    EccIterate s{d->tx, d->ty, d->rho, d->last_rho, d->it, 0, 0};
    ecc_update(sums, s, d->max_it, d->eps);
    d->ticket = 0;
    d->tx = s.tx;
    d->ty = s.ty;
    d->rho = s.rho;
    d->last_rho = s.last_rho;
    d->it = s.it;
    d->status = s.status;
    d->done = s.done;
    __threadfence();
}

// Driver 2: the whole solve in ONE cooperative launch (one CTA per SM, all co-resident): min/max -> grid barrier ->
// normalisation + gradients -> grid barrier -> iterations, one grid barrier each.  After the barrier every CTA reads
// every CTA's 15 partial sums in the same fixed order and runs the same scalar update itself (identical inputs, identical
// arithmetic, identical result), so no second barrier is needed to publish the new shift.  The slots are double-buffered
// by iteration parity: a fast CTA writes iteration it + 1's sums into the other buffer while a slow one still reads it's.
__global__ void __launch_bounds__(ECC_THREADS)
ecc_solve_kernel(const float* __restrict__ ref, float* cur, const float* cur_src0, int cur_stride, const u8* __restrict__ mask, int w, int h,
                 float thresh, float* __restrict__ T, float* __restrict__ I, float* __restrict__ gx, float* __restrict__ gy, EccDev* d0,
                 double* partials, float tx0, float ty0, int max_it, double eps, int nrun, size_t frame_stride, double conf_thresh,
                 int have_thresh)
{
    namespace cg = cooperative_groups;
    cg::grid_group grid = cg::this_grid();
    __shared__ double red[ECC_THREADS / 32][NACC];
    __shared__ double sums[NACC];
    __shared__ double stage[ECC_MAX_SLOTS * NACC];
    __shared__ unsigned kred[ECC_THREADS / 32][4];
    __shared__ EccIterate shared_state;
    const int npx = w * h;
    const int gtid = blockIdx.x * ECC_THREADS + threadIdx.x, gthreads = gridDim.x * ECC_THREADS;
    const int lane = threadIdx.x & 31, wi = threadIdx.x >> 5;

    // nrun > 1: a RUN of frames (rirb_ecc_track, frames in device memory) without the host in between.  Frame r's window is
    // cur_src0 + r * frame_stride, its state d0[r]; its warm start is frame r - 1's shift, and the run ends behind a frame
    // that failed or whose correlation fell under the confidence threshold (the host then replaces the reference image):
    // the slots behind it keep `skipped`.  Every CTA holds the same scalar state, so all of them leave together.  No barrier
    // is needed between two frames: the first thing a frame writes that another phase reads (cur, then d0[r + 1].mm) is read
    // again only behind the frame's own first barrier.
    if (blockIdx.x == 0 && threadIdx.x == 0)
        for (int r = 0; r < nrun; ++r) d0[r].skipped = 1;
    // CTA-wide min / max of four keys, then one atomic per word into dst->mm
    auto publish_minmax = [&](unsigned (&k)[4], EccDev* dst) {
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) {
            k[0] = min(k[0], __shfl_down_sync(0xFFFFFFFFu, k[0], o));
            k[1] = max(k[1], __shfl_down_sync(0xFFFFFFFFu, k[1], o));
            k[2] = min(k[2], __shfl_down_sync(0xFFFFFFFFu, k[2], o));
            k[3] = max(k[3], __shfl_down_sync(0xFFFFFFFFu, k[3], o));
        }
        __syncthreads();  // kred may still be read from the previous use
        if (lane == 0)
#pragma unroll
            for (int q = 0; q < 4; ++q) kred[wi][q] = k[q];
        __syncthreads();
        if (threadIdx.x < 4) {
            unsigned v = kred[0][threadIdx.x];
            for (int q = 1; q < ECC_THREADS / 32; ++q) v = (threadIdx.x & 1) ? max(v, kred[q][threadIdx.x]) : min(v, kred[q][threadIdx.x]);
            if (threadIdx.x & 1) atomicMax(&dst->mm[threadIdx.x], v); else atomicMin(&dst->mm[threadIdx.x], v);
        }
    };
    for (int r = 0; r < nrun; ++r) {
    EccDev* d = d0 + r;
    const float* cur_src = cur_src0 + (size_t)r * frame_stride;
    // ---- min / max of the clamped windows (d->mm is in its initial state: rirb_ecc_open, then the end of every solve).
    //      Only the first frame of a run pays a phase of its own for it: frame r + 1's are taken while frame r is
    //      normalised (they do not depend on frame r's solution), which saves a pass and a grid barrier per frame ----
    if (r == 0) {
        unsigned k[4] = {0xFFFFFFFFu, 0u, 0xFFFFFFFFu, 0u};
        for (int i = gtid; i < npx; i += gthreads) {
            const int yy = i / w, xx = i - yy * w;
            const float rv = ref[i], c = cur_src[(size_t)yy * cur_stride + xx];
            const unsigned kr = fkey(clamp_pair(rv, c, thresh)), kc = fkey(clamp_pair(c, rv, thresh));
            k[0] = min(k[0], kr);
            k[1] = max(k[1], kr);
            k[2] = min(k[2], kc);
            k[3] = max(k[3], kc);
        }
        publish_minmax(k, d);
        grid.sync();
    }
    // ---- normalisation + gradients; the window is picked out of the filtered frame (cur_src, rows cur_stride floats
    //      apart) and its compact copy left in `cur` for the host (rirb_ecc_reset_reference, quantiles) ----
    {
        const float mi_t = fkey_inv(d->mm[0]), span_t = __fsub_rn(fkey_inv(d->mm[1]), mi_t);
        const float mi_i = fkey_inv(d->mm[2]), span_i = __fsub_rn(fkey_inv(d->mm[3]), mi_i);
        const bool more = r + 1 < nrun;
        const float* next_src = cur_src + frame_stride;
        unsigned k[4] = {0xFFFFFFFFu, 0u, 0xFFFFFFFFu, 0u};
        auto img = [&](int xx, int yy) {
            return normalise(clamp_pair(cur_src[(size_t)yy * cur_stride + xx], ref[yy * w + xx], thresh), mi_i, span_i);
        };
        for (int i = gtid; i < npx; i += gthreads) {
            const int y = i / w, x = i - y * w;
            const float rv = ref[i], c = cur_src[(size_t)y * cur_stride + x];
            if (cur != cur_src) cur[i] = c;
            T[i] = normalise(clamp_pair(rv, c, thresh), mi_t, span_t);
            I[i] = normalise(clamp_pair(c, rv, thresh), mi_i, span_i);
            const int xm = x == 0 ? 1 : x - 1, xp = x == w - 1 ? w - 2 : x + 1;  // w, h >= 2 (rirb_ecc_open)
            const int ym = y == 0 ? 1 : y - 1, yp = y == h - 1 ? h - 2 : y + 1;
            const float m = (mask == nullptr || mask[i] != 0) ? 1.0f : 0.0f;
            gx[i] = __fmul_rn(__fsub_rn(__fmul_rn(0.5f, img(xp, y)), __fmul_rn(0.5f, img(xm, y))), m);
            gy[i] = __fmul_rn(__fsub_rn(__fmul_rn(0.5f, img(x, yp)), __fmul_rn(0.5f, img(x, ym))), m);
            if (more) {
                const float cn = next_src[(size_t)y * cur_stride + x];
                const unsigned kr = fkey(clamp_pair(rv, cn, thresh)), kc = fkey(clamp_pair(cn, rv, thresh));
                k[0] = min(k[0], kr);
                k[1] = max(k[1], kr);
                k[2] = min(k[2], kc);
                k[3] = max(k[3], kc);
            }
        }
        if (more) publish_minmax(k, d + 1);
    }
    grid.sync();
    // ---- iterations ----
    EccIterate s{tx0, ty0, -1.0, -eps, 0, 0, 0};  // ecc.cpp: rho = -1, last_rho = -termination_eps
    s.done = (max_it <= 0) || !(fabs(s.rho - s.last_rho) >= eps);
    while (!s.done) {
        double* slots = partials + (size_t)(s.it & 1) * gridDim.x * NACC;
        const EccShift sh(s.tx, s.ty);
        double a[NACC];
#pragma unroll
        for (int k = 0; k < NACC; ++k) a[k] = 0.0;
        ecc_accumulate(T, I, gx, gy, mask, w, h, sh, gtid, gthreads, a);
        ecc_block_partial(a, red, slots);
        grid.sync();
        ecc_sum_partials(slots, (int)gridDim.x, sums, stage);
        if (threadIdx.x == 0) {
            ecc_update(sums, s, max_it, eps);
            shared_state = s;
        }
        __syncthreads();
        s = shared_state;
    }
    const bool stop = (s.status != 0) || (have_thresh && s.rho < conf_thresh);
    if (blockIdx.x == 0 && threadIdx.x == 0) {
        d->tx = s.tx;
        d->ty = s.ty;
        d->rho = s.rho;
        d->last_rho = s.last_rho;
        d->it = s.it;
        d->status = s.status;
        d->done = 1;
        d->skipped = 0;
        d->stop = stop ? 1 : 0;
        d->mm[0] = d->mm[2] = 0xFFFFFFFFu;  // ready for the next solve: every CTA read them two barriers ago
        d->mm[1] = d->mm[3] = 0u;
        if (stop && r + 1 < nrun) {  // the next frame's min / max were taken on the way and will not be used
            d[1].mm[0] = d[1].mm[2] = 0xFFFFFFFFu;
            d[1].mm[1] = d[1].mm[3] = 0u;
        }
    }
    if (stop) break;
    tx0 = s.tx;
    ty0 = s.ty;
    }
}

// ---- host side ------------------------------------------------------------------------------------
struct EccState {
    int w = 0, h = 0, dev = 0;
    float *ref = nullptr, *cur = nullptr, *T = nullptr, *I = nullptr, *gx = nullptr, *gy = nullptr;
    u8 *mask = nullptr, *qmask = nullptr;  // ECC mask; mask of the quantile thresholds (see rirb_ecc_set_mask)
    bool have_mask = false, have_qmask = false, have_ref = false, have_cur = false;
    bool mm_clean = false;  // the min/max words of `d` are in their initial state (the one-launch solver leaves them so)
    u16* q16 = nullptr;               // quantile scratch: the crop cast to uint16
    unsigned long long* hist = nullptr;
    unsigned* mm = nullptr;
    int* qout = nullptr;
    EccDev* d = nullptr;
    double* partials = nullptr;  // per-CTA partial sums, two buffers of [max grid][NACC]
    int max_grid = 0;
    int coop_grid = 0;       // CTAs of the cooperative launch (0: not available)
    // ---- tracking state of MaskedRegistratorECC (rirb_ecc_track*) ----
    bool started = false, fixed_ref = false, have_thresh = false;
    float sigma = 0.5f;
    double median = 1.0, conf_thresh = 0.0, last_x = 0.0, last_y = 0.0, last_conf = 1.0;
    float start[2] = {0.f, 0.f};  // warp_matrix[0,2], warp_matrix[1,2]: the warm start of the next frame
    std::vector<double> confs;
    EccDev* result = nullptr;     // pinned host copy of the device state
    EccDev* dq = nullptr;         // device states of a run of solves queued back to back (ECC_BATCH slots) ...
    EccDev* resultq = nullptr;    // ... and their pinned host copies
    const char* filt_src = nullptr;  // within one rirb_ecc_track call: s.filtered holds the filtered frames filt_src + i * frame bytes,
    int filt_n = 0;                  // i < filt_n (a run that stopped early does not filter its tail again)
    size_t filt_frame = 0, filt_off = 0;  // floats per filtered frame in s.filtered, offset of the window's first pixel in it
    int filt_stride = 0;                  // floats per row of it
    int launched = 0;             // iteration launches enqueued for the solve in flight
    cudaStream_t copy_stream = nullptr;
    cudaEvent_t copied[2] = {nullptr, nullptr};
    void* pinned[2] = {nullptr, nullptr};  // host frames: pinned staging ...
    void* stage2[2] = {nullptr, nullptr};  // ... and their device copies (double-buffered)
    size_t pin_cap[2] = {0, 0};
    float* filtered = nullptr;    // one full frame, Gaussian-filtered / converted to float
    size_t filtered_cap = 0;
    std::recursive_mutex mu;
    ~EccState()
    {
        void* ptrs[] = {ref, cur, T, I, gx, gy, mask, qmask, q16, hist, mm, qout, d, partials, filtered};
        for (void* p : ptrs)
            if (p) cudaFree(p);
        for (int i = 0; i < 2; ++i) {
            if (stage2[i]) cudaFree(stage2[i]);
            if (pinned[i]) cudaFreeHost(pinned[i]);
            if (copied[i]) cudaEventDestroy(copied[i]);
        }
        if (result) cudaFreeHost(result);
        if (dq) cudaFree(dq);
        if (resultq) cudaFreeHost(resultq);
        if (copy_stream) cudaStreamDestroy(copy_stream);
    }
};
static Table<EccState> g_ecc;

// Buffers live on the device the handle was opened on: refuse calls from a thread that is on another one.
static std::shared_ptr<EccState> ecc_get(int handle, const char* what)
{
    auto s = g_ecc.get(handle);
    if (!s) {
        set_error("%s: unknown handle %d", what, handle);
        return nullptr;
    }
    int dev = -1;
    if (cudaGetDevice(&dev) != cudaSuccess) cudaGetLastError();
    if (dev != s->dev) {
        set_error("%s: handle %d belongs to CUDA device %d, the calling thread is on device %d", what, handle, s->dev, dev);
        return nullptr;
    }
    return s;
}

static int ecc_need_device()
{
    int n = 0;
    if (cudaGetDeviceCount(&n) != cudaSuccess || n <= 0) {
        cudaGetLastError();
        set_error("no usable CUDA device: librir_b200 computes on the GPU only and has no CPU fallback");
        return -1;
    }
    return 0;
}

static bool is_device_pointer(const void* p)
{
    cudaPointerAttributes a;
    if (cudaPointerGetAttributes(&a, p) != cudaSuccess) {
        cudaGetLastError();
        return false;
    }
    return a.type == cudaMemoryTypeDevice || a.type == cudaMemoryTypeManaged;
}

static int ecc_load_window(EccState& s, float* dst, const float* src, int stride, cudaStream_t st)
{
    if (!src || stride < s.w) {
        set_error("ecc: bad image pointer or row stride");
        return -1;
    }
    RIRB_CUDA_OK(cudaMemcpy2DAsync(dst, (size_t)s.w * 4, src, (size_t)stride * 4, (size_t)s.w * 4, (size_t)s.h, cudaMemcpyDefault, st));
    return 0;
}

// The solve in two halves, so that a caller can do host work (fetching the next frame) while the GPU is busy.
// enqueue: everything up to and including the copy of the result towards the host; collect: wait, and for the
// launch-per-iteration driver keep launching until the problem reports done.
static int ecc_enqueue(EccState& s, float thresh, int use_mask, int max_iterations, double eps, const float* shift,
                       const float* cur_src = nullptr, int cur_stride = 0)
{
    cudaStream_t st = current_stream();
    const int n = s.w * s.h;
    const float th = isnan(thresh) ? INFINITY : thresh;
    const u8* mask = (use_mask && s.have_mask) ? s.mask : nullptr;
    if (!s.result) RIRB_CUDA_OK(cudaMallocHost((void**)&s.result, sizeof(EccDev)));  // pinned: the copy back does not stall the host
    s.launched = 0;
    if (s.coop_grid > 0 && option_enabled(OPT_ECC_FUSED)) {
        // the whole solve in one cooperative launch ("ecc_fused" = 0 selects the launch-per-iteration driver); it leaves
        // the min/max words in their initial state, so no preparing launch is needed unless the other driver ran last
        if (!s.mm_clean) RIRB_LAUNCH(ecc_begin_kernel, 1, 1, 0, st, s.d, shift[0], shift[1], max_iterations, eps);
        s.mm_clean = true;
        const float* ref = s.ref;
        float* cur = s.cur;
        const float* src = cur_src ? cur_src : s.cur;
        int stride = cur_src ? cur_stride : s.w;
        int w = s.w, h = s.h;
        float th_arg = th, tx0 = shift[0], ty0 = shift[1];
        int nrun = 1, have_thresh = 0;
        size_t frame_stride = 0;
        double no_thresh = 0.0;
        void* args[] = {&ref, &cur, &src, &stride, &mask, &w, &h, &th_arg, &s.T, &s.I, &s.gx, &s.gy, &s.d, &s.partials, &tx0, &ty0,
                        &max_iterations, &eps, &nrun, &frame_stride, &no_thresh, &have_thresh};
        RIRB_CUDA_OK(cudaLaunchCooperativeKernel((const void*)ecc_solve_kernel, dim3((unsigned)s.coop_grid), dim3(ECC_THREADS), args, 0, st));
        g_launches.fetch_add(1);
        s.launched = max_iterations;
    } else {
        if (cur_src && ecc_load_window(s, s.cur, cur_src, cur_stride, st) != 0) return -1;
        RIRB_LAUNCH(ecc_begin_kernel, 1, 1, 0, st, s.d, shift[0], shift[1], max_iterations, eps);
        s.mm_clean = false;
        const int blocks = (int)min((long long)ceil_div(n, ECC_THREADS), (long long)s.max_grid);
        RIRB_LAUNCH(ecc_minmax_kernel, (unsigned)blocks, ECC_THREADS, 0, st, s.ref, s.cur, n, th, s.d);
        RIRB_LAUNCH(ecc_normalise_kernel, dim3((unsigned)ceil_div(s.w, ECC_THREADS), (unsigned)s.h), ECC_THREADS, 0, st, s.ref, s.cur, mask,
                    s.w, s.h, th, s.d, s.T, s.I, s.gx, s.gy);
        const int burst = min(4, max_iterations);  // a converged problem turns the rest into no-ops
        for (int k = 0; k < burst; ++k)
            RIRB_LAUNCH(ecc_iter_kernel, (unsigned)blocks, ECC_THREADS, 0, st, s.T, s.I, s.gx, s.gy, mask, s.w, s.h, s.d, s.partials);
        s.launched = burst;
    }
    RIRB_CUDA_OK(cudaMemcpyAsync(s.result, s.d, sizeof(EccDev), cudaMemcpyDeviceToHost, st));
    return 0;
}

static int ecc_collect(EccState& s, int use_mask, int max_iterations, float* shift, double* rho, int* iterations)
{
    cudaStream_t st = current_stream();
    const u8* mask = (use_mask && s.have_mask) ? s.mask : nullptr;
    RIRB_CUDA_OK(cudaStreamSynchronize(st));
    while (!s.result->done && s.launched < max_iterations) {  // launch-per-iteration driver only
        const int blocks = (int)min((long long)ceil_div(s.w * s.h, ECC_THREADS), (long long)s.max_grid);
        const int burst = min(12, max_iterations - s.launched);
        for (int k = 0; k < burst; ++k)
            RIRB_LAUNCH(ecc_iter_kernel, (unsigned)blocks, ECC_THREADS, 0, st, s.T, s.I, s.gx, s.gy, mask, s.w, s.h, s.d, s.partials);
        s.launched += burst;
        RIRB_CUDA_OK(cudaMemcpyAsync(s.result, s.d, sizeof(EccDev), cudaMemcpyDeviceToHost, st));
        RIRB_CUDA_OK(cudaStreamSynchronize(st));
    }
    const EccDev& r = *s.result;
    if (iterations) *iterations = r.it;
    if (rho) *rho = r.rho;
    if (r.status == 0) {
        shift[0] = r.tx;
        shift[1] = r.ty;
    }
    return r.status;
}

// Frames that live in host memory: frame t + 1 is copied into a pinned buffer and sent on its own stream while the GPU
// solves frame t (two buffers, two events).
static int ecc_prefetch(EccState& s, const void* src, size_t bytes, int slot)
{
    if (!s.copy_stream) {
        RIRB_CUDA_OK(cudaStreamCreateWithFlags(&s.copy_stream, cudaStreamNonBlocking));
        for (int i = 0; i < 2; ++i) RIRB_CUDA_OK(cudaEventCreateWithFlags(&s.copied[i], cudaEventDisableTiming));
    }
    for (int i = 0; i < 2; ++i)
        if (s.pin_cap[i] < bytes) {
            if (s.pinned[i]) cudaFreeHost(s.pinned[i]);
            if (s.stage2[i]) cudaFree(s.stage2[i]);
            s.pinned[i] = s.stage2[i] = nullptr;
            s.pin_cap[i] = 0;
            RIRB_CUDA_OK(cudaMallocHost(&s.pinned[i], bytes));
            RIRB_CUDA_OK(cudaMalloc(&s.stage2[i], bytes));
            s.pin_cap[i] = bytes;
        }
    memcpy(s.pinned[slot], src, bytes);
    RIRB_CUDA_OK(cudaMemcpyAsync(s.stage2[slot], s.pinned[slot], bytes, cudaMemcpyHostToDevice, s.copy_stream));
    RIRB_CUDA_OK(cudaEventRecord(s.copied[slot], s.copy_stream));
    return 0;
}

// ---- a run of frames that are already in device memory, solved without the host in between ----------------------
// rirb_ecc_track's loop costs a launch, a copy back and a synchronisation per frame, about as long as the solve itself.
// Nothing in frame t + 1's solve needs the host: its warm start is frame t's shift and the one thing the host decides
// between two frames -- replace the reference image when the correlation falls under the confidence threshold
// (masked_registration_ecc.py:176-186), or deal with a failed frame -- only ever ENDS a run.  So up to ECC_BATCH frames are
// filtered in one Gaussian launch and ONE cooperative launch walks them (ecc_solve_kernel, nrun > 1), leaving behind the
// frame that ends the run.  The host then walks the results in order and applies the class's rules as before; the frames
// that were filtered but not reached stay in s.filtered for the next run.  Same arithmetic, same results as frame by frame.
// (Queuing one cooperative launch per frame instead was measured first: 5,000 frames/s against 14,400 frame by frame --
// a cooperative launch behind a running kernel is expensive.)
// Gaussian of K frames (device memory) into s.filtered -- of what the window needs of them: the window grown by the kernel
// radius, clipped to the frame, its left / right edge moved out to whole 16-byte vectors.  Filtering the region as an image of
// its own is exact inside the window (a region border that is not a frame border only spoils the `radius` pixels next to it),
// and a 448 x 358 window of a 640 x 512 frame is half the work.  Sets s.filt_frame / filt_off / filt_stride.
static int ecc_filter_frames(EccState& s, int type, const char* src0, int K, size_t fpx, int full_w, int full_h, int x0, int y0,
                             const GaussTaps& taps, cudaStream_t st)
{
    const int r = taps.radius, al = type == 'H' ? 8 : 4;
    const int rx0 = std::max(0, x0 - r) / al * al, ry0 = std::max(0, y0 - r);
    const int rx1 = std::min(full_w, (x0 + s.w + r + al - 1) / al * al), ry1 = std::min(full_h, y0 + s.h + r);
    const int wr = rx1 - rx0, hr = ry1 - ry0;
    if ((long long)wr * hr * 10 < (long long)full_w * full_h * 9) {  // worth it
        const size_t off = (size_t)ry0 * full_w + rx0;
        const int rc = type == 'H' ? launch_gaussian_u16_region((const u16*)src0 + off, (size_t)full_w, fpx, s.filtered, wr, hr, K, taps, st)
                                   : launch_gaussian_f32_region((const float*)src0 + off, (size_t)full_w, fpx, s.filtered, wr, hr, K, taps, st);
        if (rc < 0) return -1;
        if (rc == 0) {
            s.filt_frame = (size_t)wr * hr;
            s.filt_stride = wr;
            s.filt_off = (size_t)(y0 - ry0) * wr + (x0 - rx0);
            return 0;
        }
    }
    if ((type == 'H' ? launch_gaussian_u16((const u16*)src0, s.filtered, full_w, full_h, K, taps, st)
                     : launch_gaussian_f32((const float*)src0, s.filtered, full_w, full_h, K, taps, st)) != 0)
        return -1;
    s.filt_frame = fpx;
    s.filt_stride = full_w;
    s.filt_off = (size_t)y0 * full_w + x0;
    return 0;
}

constexpr int ECC_BATCH = 16;

// frames [0, K) at src0 (device); *done = frames fully handled (>= 0; 0: frame 0 failed, the caller redoes it the slow way)
static int ecc_track_run(EccState& s, int handle, int type, const char* src0, int K, size_t fpx, size_t esz, int full_w, int full_h,
                         int x0, int y0, int use_mask, const GaussTaps& taps, double* x, double* y, double* conf, int* iters, int* done)
{
    cudaStream_t st = current_stream();
    *done = 0;
    if (!s.dq) {
        RIRB_CUDA_OK(cudaMalloc((void**)&s.dq, sizeof(EccDev) * ECC_BATCH));
        RIRB_CUDA_OK(cudaMallocHost((void**)&s.resultq, sizeof(EccDev) * ECC_BATCH));
        for (int k = 0; k < ECC_BATCH; ++k) RIRB_LAUNCH(ecc_begin_kernel, 1, 1, 0, st, s.dq + k, 0.f, 0.f, 500, 1e-3);  // clean min / max words
    }
    if (s.filtered_cap < fpx * 4 * (size_t)K) {
        if (s.filtered) cudaFree(s.filtered);
        s.filtered = nullptr;
        s.filtered_cap = 0;
        RIRB_CUDA_OK(cudaMalloc((void**)&s.filtered, fpx * 4 * (size_t)ECC_BATCH));
        s.filtered_cap = fpx * 4 * (size_t)ECC_BATCH;
        s.filt_src = nullptr;
    }
    const size_t fbytes = fpx * esz;
    const float* win0;   // the window of the run's first frame, rows win_stride floats and frames win_frame floats apart
    int win_stride;
    size_t win_frame;
    if (s.filt_src && src0 >= s.filt_src && src0 < s.filt_src + (size_t)s.filt_n * fbytes && (size_t)(src0 - s.filt_src) % fbytes == 0) {
        const int j = (int)((size_t)(src0 - s.filt_src) / fbytes);  // already filtered by the run that stopped before this frame
        win0 = s.filtered + (size_t)j * s.filt_frame + s.filt_off;
        win_stride = s.filt_stride;
        win_frame = s.filt_frame;
        K = std::min(K, s.filt_n - j);
    } else if (s.sigma > 0.f) {
        s.filt_src = nullptr;
        if (ecc_filter_frames(s, type, src0, K, fpx, full_w, full_h, x0, y0, taps, st) != 0) return -1;
        s.filt_src = src0;
        s.filt_n = K;
        win0 = s.filtered + s.filt_off;
        win_stride = s.filt_stride;
        win_frame = s.filt_frame;
    } else {
        s.filt_src = nullptr;
        const float* full = (const float*)src0;
        if (type == 'H') {
            RIRB_LAUNCH(ecc_u16_to_f32_kernel, (unsigned)ceil_div((long long)(fpx * K), 256), 256, 0, st, (const u16*)src0, s.filtered, (int)(fpx * K));
            full = s.filtered;
            s.filt_src = src0;
            s.filt_n = K;
            s.filt_frame = fpx;
            s.filt_stride = full_w;
            s.filt_off = (size_t)y0 * full_w + x0;
        }
        win0 = full + (size_t)y0 * full_w + x0;
        win_stride = full_w;
        win_frame = fpx;
    }
    const int Kq = K;  // frames behind the one that ends the run cost nothing: the kernel leaves
    const u8* mask = (use_mask && s.have_mask) ? s.mask : nullptr;
    const bool may_reset = !s.fixed_ref;
    {
        const float* ref = s.ref;
        float* cur = s.cur;
        const float* src = win0;
        int stride = win_stride, w = s.w, h = s.h, max_it = 500, have_thresh = (may_reset && s.have_thresh) ? 1 : 0, nrun = Kq;
        float th = INFINITY, tx0 = s.start[0], ty0 = s.start[1];
        double eps = 1e-3, conf_thresh = s.conf_thresh;
        size_t frame_stride = win_frame;
        EccDev* d = s.dq;
        void* args[] = {&ref, &cur, &src, &stride, &mask, &w, &h, &th, &s.T, &s.I, &s.gx, &s.gy, &d, &s.partials, &tx0, &ty0,
                        &max_it, &eps, &nrun, &frame_stride, &conf_thresh, &have_thresh};
        RIRB_CUDA_OK(cudaLaunchCooperativeKernel((const void*)ecc_solve_kernel, dim3((unsigned)s.coop_grid), dim3(ECC_THREADS), args, 0, st));
        g_launches.fetch_add(1);
    }
    RIRB_CUDA_OK(cudaMemcpyAsync(s.resultq, s.dq, sizeof(EccDev) * (size_t)Kq, cudaMemcpyDeviceToHost, st));
    RIRB_CUDA_OK(cudaStreamSynchronize(st));
    s.have_cur = true;
    bool ended = false;
    for (int k = 0; k < Kq; ++k) {
        const EccDev& r = s.resultq[k];
        if (r.skipped || r.status != 0) {  // a failed frame is redone by the caller's frame-by-frame path (retries, error codes)
            ended = true;
            break;
        }
        s.start[0] = r.tx;
        s.start[1] = r.ty;
        x[k] = s.last_x = (double)r.tx;
        y[k] = s.last_y = (double)r.ty;
        conf[k] = s.last_conf = r.rho;
        if (iters) iters[k] = r.it;
        s.confs.push_back(r.rho);
        *done = k + 1;
        if (s.confs.size() > 20 && may_reset) {  // :176-186, as in rirb_ecc_track
            if (!s.have_thresh) {
                double mn = s.confs[0], mean = 0.0, var = 0.0;
                for (double c : s.confs) {
                    mn = c < mn ? c : mn;
                    mean += c;
                }
                mean /= (double)s.confs.size();
                for (double c : s.confs) var += (c - mean) * (c - mean);
                s.conf_thresh = mn - 2.0 * sqrt(var / (double)s.confs.size());
                s.have_thresh = true;
            }
            if (r.rho < s.conf_thresh) {  // s.cur holds this frame's window: the solves queued after it did not run
                if (rirb_ecc_reset_reference(handle, -r.tx, -r.ty) != 0) return -1;
                s.start[0] = s.start[1] = 0.f;
                ended = true;
                break;
            }
        }
    }
    (void)ended;
    return 0;
}

}  // namespace rirb

using namespace rirb;

extern "C" {

int rirb_ecc_open(int width, int height)
{
    if (width < 2 || height < 2 || (long long)width * height > (1LL << 28)) {
        set_error("ecc_open: bad window size %d x %d", width, height);
        return 0;
    }
    if (ecc_need_device() != 0) return 0;
    auto s = std::make_shared<EccState>();
    s->w = width;
    s->h = height;
    cudaGetDevice(&s->dev);
    const size_t n = (size_t)width * height;
    bool ok = true;
    for (float** p : {&s->ref, &s->cur, &s->T, &s->I, &s->gx, &s->gy}) ok = ok && cudaMalloc((void**)p, n * 4) == cudaSuccess;
    ok = ok && cudaMalloc((void**)&s->mask, n) == cudaSuccess && cudaMalloc((void**)&s->qmask, n) == cudaSuccess &&
         cudaMalloc((void**)&s->q16, n * 2) == cudaSuccess &&
         cudaMalloc((void**)&s->hist, 65536 * sizeof(unsigned long long)) == cudaSuccess &&
         cudaMalloc((void**)&s->mm, 2 * sizeof(unsigned)) == cudaSuccess && cudaMalloc((void**)&s->qout, sizeof(int)) == cudaSuccess &&
         cudaMalloc((void**)&s->d, sizeof(EccDev)) == cudaSuccess;
    s->max_grid = std::min(sm_count() * 2, ECC_MAX_SLOTS);
    ok = ok && cudaMalloc((void**)&s->partials, (size_t)2 * s->max_grid * NACC * sizeof(double)) == cudaSuccess;
    if (!ok) {
        cudaGetLastError();
        set_error("ecc_open: out of device memory");
        return 0;
    }
    // the one-launch solver needs every CTA resident at once: one per SM, if the device can launch cooperatively
    int coop = 0, per_sm = 0;
    if (cudaDeviceGetAttribute(&coop, cudaDevAttrCooperativeLaunch, s->dev) == cudaSuccess && coop &&
        cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, ecc_solve_kernel, ECC_THREADS, 0) == cudaSuccess && per_sm >= 1)
        s->coop_grid = (int)min((long long)sm_count(), (long long)ceil_div((long long)n, ECC_THREADS));
    cudaGetLastError();
    return g_ecc.add(s);
}

void rirb_ecc_close(int handle) { g_ecc.remove(handle); }

// mask: w x h bytes (non-zero = use), host or device; NULL removes it.  which = 0: the mask findTransformECC gets;
// which = 1: the mask of the quantile thresholds.  They are two because the reference hands find_median_pixel a
// non-contiguous view of the full-size mask without compacting it (rir_signal_processing.py:134-136), so with a
// uint8 mask its thresholds are taken under a different pixel set than the one ECC uses; the Python mirror reproduces that.
int rirb_ecc_set_mask(int handle, int which, const unsigned char* mask)
{
    auto s = ecc_get(handle, "ecc_set_mask");
    if (!s) return -1;
    if (!s || (which != 0 && which != 1)) {
        set_error("ecc: unknown handle %d or mask selector", handle);
        return -1;
    }
    std::lock_guard<std::recursive_mutex> lock(s->mu);
    (which ? s->have_qmask : s->have_mask) = mask != nullptr;
    if (mask) RIRB_CUDA_OK(cudaMemcpyAsync(which ? s->qmask : s->mask, mask, (size_t)s->w * s->h, cudaMemcpyDefault, current_stream()));
    return 0;
}

// which: 0 = the reference window, 1 = the current image window.  img points at the window's first pixel inside a
// float image whose rows are `stride` floats apart (host or device).
int rirb_ecc_set_image(int handle, int which, const float* img, int stride)
{
    auto s = ecc_get(handle, "ecc_set_image");
    if (!s) return -1;
    if (!s || (which != 0 && which != 1)) {
        set_error("ecc: unknown handle %d or image selector", handle);
        return -1;
    }
    std::lock_guard<std::recursive_mutex> lock(s->mu);
    if (ecc_load_window(*s, which ? s->cur : s->ref, img, stride, current_stream()) != 0) return -1;
    (which ? s->have_cur : s->have_ref) = true;
    return 0;
}

// The reference-image reset of MaskedRegistratorECC.compute (:182-185): reference = translate(current, dx, dy)
// with translate's default ("noborder") strategy, on the un-normalised float window.
int rirb_ecc_reset_reference(int handle, float dx, float dy)
{
    auto s = ecc_get(handle, "ecc_reset_reference");
    if (!s) return -1;
    if (!s || !s->have_cur) {
        set_error("ecc_reset_reference: unknown handle or no current image");
        return -1;
    }
    std::lock_guard<std::recursive_mutex> lock(s->mu);
    cudaStream_t st = current_stream();
    const size_t bytes = (size_t)s->w * s->h * 4;
    RIRB_CUDA_OK(cudaMemcpyAsync(s->ref, s->cur, bytes, cudaMemcpyDeviceToDevice, st));  // untouched pixels keep the source value
    const float zero = 0.f;
    if (launch_translate('f', s->cur, s->ref, s->w, s->h, 1, nullptr, nullptr, dx, dy, STRAT_NOBORDER, &zero, st) != 0) return -1;
    s->have_ref = true;
    return 0;
}

// find_median_pixel(window.astype(uint16), percent, mask) of the reference (0) or current (1) window (:144-145)
int rirb_ecc_quantile(int handle, int which, float percent, int use_mask)
{
    auto s = ecc_get(handle, "ecc_quantile");
    if (!s) return -1;
    if (!s || (which != 0 && which != 1) || !(which ? s->have_cur : s->have_ref)) {
        set_error("ecc_quantile: unknown handle or image not set");
        return -1;
    }
    std::lock_guard<std::recursive_mutex> lock(s->mu);
    cudaStream_t st = current_stream();
    const int n = s->w * s->h;
    RIRB_LAUNCH(ecc_cast_u16_kernel, (unsigned)ceil_div(n, 256), 256, 0, st, which ? s->cur : s->ref, s->q16, n);
    const bool masked = use_mask && s->have_qmask;
    if (launch_stats_init(s->mm, s->hist, st) != 0) return -1;
    if (launch_movie_stats(s->q16, (size_t)n, masked ? s->qmask : nullptr, s->mm, s->hist, st) != 0) return -1;
    if (launch_hist_quantile(s->hist, masked ? -1 : (long long)n, percent, masked ? 1 : 0, s->qout, st) != 0) return -1;
    int r = 0;
    RIRB_CUDA_OK(cudaMemcpyAsync(&r, s->qout, sizeof(int), cudaMemcpyDeviceToHost, st));
    RIRB_CUDA_OK(cudaStreamSynchronize(st));
    return r;
}

// cv2.findTransformECC(reference, current, [[1,0,tx],[0,1,ty]], MOTION_TRANSLATION, (COUNT|EPS, max_iterations, eps), mask, 1)
// after the quantile clamp (thresh; pass +inf or NaN for none) and the min/max normalisation of both windows.
// shift[2] = {tx, ty}: warm start in, result out (unchanged on failure).  Returns 0; 1 = "NaN encountered";
// 2 = "the correlation is going to be minimized" (both are cv2.error in the reference); -1 = bad call.
int rirb_ecc_compute(int handle, float thresh, int use_mask, int max_iterations, double eps, float* shift, double* rho, int* iterations)
{
    auto s = ecc_get(handle, "ecc_compute");
    if (!s) return -1;
    if (!s || !s->have_ref || !s->have_cur || !shift) {
        set_error("ecc_compute: unknown handle, or reference / current image not set");
        return -1;
    }
    std::lock_guard<std::recursive_mutex> lock(s->mu);
    if (ecc_enqueue(*s, thresh, use_mask, max_iterations, eps, shift) != 0) return -1;
    return ecc_collect(*s, use_mask, max_iterations, shift, rho, iterations);
}

// ---- the tracking loop of MaskedRegistratorECC, frame after frame, without leaving the library ---------------------
// (masked_registration_ecc.py: start :89-103, compute :105-191, manage_computation_and_tries :229-260)

// sigma / median as in the class constructor; fixed_ref != 0: the reference window set with rirb_ecc_set_image(0) is kept
// for good (the class's `ref` argument) and the confidence rule never replaces it.  Clears the tracking history.
int rirb_ecc_track_config(int handle, float sigma, double median, int fixed_ref)
{
    auto s = g_ecc.get(handle);
    if (!s || !(sigma >= 0.f)) {
        set_error("ecc_track_config: unknown handle or negative sigma");
        return -1;
    }
    std::lock_guard<std::recursive_mutex> lock(s->mu);
    s->sigma = sigma;
    s->median = median;
    s->fixed_ref = fixed_ref != 0;
    s->started = false;
    s->have_thresh = false;
    s->confs.clear();
    s->start[0] = s->start[1] = 0.f;
    s->last_x = s->last_y = 0.0;
    s->last_conf = 1.0;
    return 0;
}

// The class's `median` attribute is public: a caller may change it between frames without losing the history.
int rirb_ecc_track_set_median(int handle, double median)
{
    auto s = g_ecc.get(handle);
    if (!s) {
        set_error("ecc_track_set_median: unknown handle");
        return -1;
    }
    std::lock_guard<std::recursive_mutex> lock(s->mu);
    s->median = median;
    return 0;
}

// median (the manage rule changes it), conf_thresh (NaN until it exists), start[2], frames seen so far
int rirb_ecc_track_state(int handle, double* median, double* conf_thresh, float* start, long long* count)
{
    auto s = g_ecc.get(handle);
    if (!s) {
        set_error("ecc_track_state: unknown handle");
        return -1;
    }
    std::lock_guard<std::recursive_mutex> lock(s->mu);
    if (median) *median = s->median;
    if (conf_thresh) *conf_thresh = s->have_thresh ? s->conf_thresh : NAN;
    if (start) {
        start[0] = s->start[0];
        start[1] = s->start[1];
    }
    if (count) *count = (long long)s->confs.size();
    return 0;
}

// frames[nframes][full_h][full_w], type 'H' (uint16) or 'f' (float32), host or device, IN TIME ORDER; the registration
// window starts at (x0, y0).  The first frame the handle ever sees is the class's start() (outputs 0, 0, 1); every other
// frame is compute().  max_try = 0: a frame on which ECC fails stops the call, which returns the failure's status (1 / 2)
// with *processed = frames done before it.  max_try > 0: manage_computation_and_tries -- up to max_try attempts with the
// median lowered by 0.01 each time, then the previous estimate is repeated; after a success a median < 1 goes back to 1.
// x / y / conf / iters: nframes entries each (iters may be NULL; 0 for the start frame, -1 for a repeated estimate).
int rirb_ecc_track(int handle, int type, const void* frames, long long nframes, int full_w, int full_h, int x0, int y0, int use_mask,
                   int max_try, double* x, double* y, double* conf, int* iters, long long* processed)
{
    auto s = ecc_get(handle, "ecc_track");
    if (!s) return -1;
    if (processed) *processed = 0;
    if (!s || !frames || nframes < 0 || !x || !y || !conf || (type != 'H' && type != 'f') || x0 < 0 || y0 < 0 || x0 + s->w > full_w ||
        y0 + s->h > full_h) {
        set_error("ecc_track: unknown handle, bad pointers / dtype, or the window does not fit the frame");
        return -1;
    }
    std::lock_guard<std::recursive_mutex> lock(s->mu);
    if (s->fixed_ref && s->median < 1.0) {
        set_error("ecc_track: median < 1 together with a fixed reference image is not supported");
        return -1;
    }
    cudaStream_t st = current_stream();
    const size_t fpx = (size_t)full_w * full_h, esz = type == 'H' ? 2 : 4;
    const bool on_device = is_device_pointer(frames);
    if (!on_device && nframes > 0 && ecc_prefetch(*s, frames, fpx * esz, 0) != 0) return -1;
    if (s->filtered_cap < fpx * 4) {
        if (s->filtered) cudaFree(s->filtered);
        s->filtered = nullptr;
        s->filtered_cap = 0;
        RIRB_CUDA_OK(cudaMalloc((void**)&s->filtered, fpx * 4));
        s->filtered_cap = fpx * 4;
    }
    GaussTaps taps;
    if (s->sigma > 0.f && gaussian_taps_host(s->sigma, &taps) != 0) return -1;
    s->filt_src = nullptr;   // the caller's frames may have changed since the last call
    s->filt_n = 0;
    bool slow_once = false;  // the frame a queued run stopped at with a failure goes through the frame-by-frame path
    for (long long t = 0; t < nframes; ++t) {
        const char* src = (const char*)frames + (size_t)t * fpx * esz;
        if (on_device && s->started && !slow_once && s->median >= 1.0 && s->coop_grid > 0 && option_enabled(OPT_ECC_FUSED) &&
            option_enabled(OPT_ECC_QUEUE)) {
            long long K = std::min<long long>(ECC_BATCH, nframes - t);
            // the confidence threshold is fixed by the host when the 21st confidence arrives, and applies to that frame
            if (!s->fixed_ref && !s->have_thresh) K = std::min<long long>(K, std::max<long long>(1, 21 - (long long)s->confs.size()));
            int did = 0;
            if (ecc_track_run(*s, handle, type, src, (int)K, fpx, esz, full_w, full_h, x0, y0, use_mask, taps, x + t, y + t, conf + t,
                              iters ? iters + t : nullptr, &did) != 0)
                return -1;
            if (processed) *processed = t + did;
            if (did == 0) slow_once = true;
            t += did - 1;  // did == 0: the same frame again, frame by frame
            continue;
        }
        slow_once = false;
        s->filt_src = nullptr;  // this path filters into the first slot
        bool next_fetched = on_device || t + 1 >= nframes;
        auto fetch_next = [&]() -> int {  // called once per frame, as soon as the GPU has work queued
            if (next_fetched) return 0;
            next_fetched = true;
            return ecc_prefetch(*s, (const char*)frames + (size_t)(t + 1) * fpx * esz, fpx * esz, (int)((t + 1) & 1));
        };
        if (!on_device) {
            RIRB_CUDA_OK(cudaStreamWaitEvent(st, s->copied[t & 1], 0));
            src = (const char*)s->stage2[t & 1];
        }
        const float* window;  // the frame's window, rows wstride floats apart
        int wstride = full_w;
        if (s->sigma > 0.f) {
            if (ecc_filter_frames(*s, type, src, 1, fpx, full_w, full_h, x0, y0, taps, st) != 0) return -1;
            window = s->filtered + s->filt_off;
            wstride = s->filt_stride;
        } else if (type == 'H') {
            RIRB_LAUNCH(ecc_u16_to_f32_kernel, (unsigned)ceil_div((long long)fpx, 256), 256, 0, st, (const u16*)src, s->filtered, (int)fpx);
            window = s->filtered + (size_t)y0 * full_w + x0;
        } else {
            window = (const float*)src + (size_t)y0 * full_w + x0;
        }
        if (!s->started) {  // start(): the first window is the reference (unless one was given), shifts 0, confidence 1
            if (ecc_load_window(*s, s->fixed_ref ? s->cur : s->ref, window, wstride, st) != 0) return -1;
            (s->fixed_ref ? s->have_cur : s->have_ref) = true;
            s->started = true;
            s->confs.push_back(1.0);
            x[t] = y[t] = 0.0;
            conf[t] = 1.0;
            if (iters) iters[t] = 0;
            if (processed) *processed = t + 1;
            if (fetch_next() != 0) return -1;
            RIRB_CUDA_OK(cudaStreamSynchronize(st));  // the staged frame is free again
            continue;
        }
        // the one-launch solver picks the window out of the filtered frame itself; the quantile thresholds (median < 1)
        // read the compact copy first, so they get an explicit one
        bool window_loaded = false;
        if (s->median < 1.0) {
            if (ecc_load_window(*s, s->cur, window, wstride, st) != 0) return -1;
            window_loaded = true;
        }
        s->have_cur = true;
        int tries = 0, status = 0, its = 0;
        double rho = 0.0;
        float shift[2];
        for (;;) {
            float thresh = INFINITY;
            if (s->median < 1.0) {
                const int t1 = rirb_ecc_quantile(handle, 1, (float)s->median, use_mask);
                const int t2 = rirb_ecc_quantile(handle, 0, (float)s->median, use_mask);
                if (t1 < 0 || t2 < 0) return -1;
                thresh = (float)(t1 > t2 ? t1 : t2);
            }
            shift[0] = s->start[0];
            shift[1] = s->start[1];
            if (ecc_enqueue(*s, thresh, use_mask, 500, 1e-3, shift, window_loaded ? nullptr : window, wstride) != 0) return -1;
            window_loaded = true;  // a retry works on the compact copy
            if (fetch_next() != 0) return -1;  // host memcpy + upload of frame t + 1 while the GPU solves frame t
            status = ecc_collect(*s, use_mask, 500, shift, &rho, &its);
            if (status < 0) return -1;
            if (status == 0) {
                if (max_try > 0 && s->median < 1.0) s->median = 1.0;
                break;
            }
            if (max_try <= 0) return status;
            s->median -= 0.01;
            if (++tries >= max_try) break;
        }
        if (status != 0) {  // append_last_coordinates_and_confidence
            x[t] = s->last_x;
            y[t] = s->last_y;
            conf[t] = s->last_conf;
            s->confs.push_back(s->last_conf);
            if (iters) iters[t] = -1;
            if (processed) *processed = t + 1;
            continue;
        }
        s->start[0] = shift[0];
        s->start[1] = shift[1];
        x[t] = s->last_x = (double)shift[0];
        y[t] = s->last_y = (double)shift[1];
        conf[t] = s->last_conf = rho;
        if (iters) iters[t] = its;
        s->confs.push_back(rho);
        if (s->confs.size() > 20 && !s->fixed_ref) {  // :176-186
            if (!s->have_thresh) {  // np.min(c) - 2 * np.std(c), population std, once
                double mn = s->confs[0], mean = 0.0, var = 0.0;
                for (double c : s->confs) {
                    mn = c < mn ? c : mn;
                    mean += c;
                }
                mean /= (double)s->confs.size();
                for (double c : s->confs) var += (c - mean) * (c - mean);
                s->conf_thresh = mn - 2.0 * sqrt(var / (double)s->confs.size());
                s->have_thresh = true;
            }
            if (rho < s->conf_thresh) {
                if (rirb_ecc_reset_reference(handle, -shift[0], -shift[1]) != 0) return -1;
                s->start[0] = s->start[1] = 0.f;
            }
        }
        if (processed) *processed = t + 1;
    }
    return 0;
}

}  // extern "C"
