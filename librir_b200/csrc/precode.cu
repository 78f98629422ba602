// librir_b200/csrc/precode.cu -- the lossless writer's pre-coder: byte-plane split (+ temporal delta).
//
// Reference semantics: H264Capture::AddFrame h264.cpp:1022-1131 (split loops :1066-1103, the
// integration-time overload :1133-1238), inverse VideoGrabber::toArray h264.cpp:3016-3051,
// key-frame rule h264.cpp:1050-1061.  The split is exactly a type-size-2 byte shuffle:
// low bytes -> one plane, high bytes -> another.  The temporal delta is THIS REPO's addition
// (no reference counterpart; parity unpinned, DESIGN.md): a non-key frame is replaced by
// (frame[t] - frame[t-1]) mod 2^16 before the split, key frames every `gop` frames stay raw.
//
// Kernels (4 B/px algorithmic: 2 read + 2 written):
//   split_flat / merge_flat    whole movie as one flat array, 16 px (256-bit) per load, the two
//                              byte planes written as 128-bit vectors (__byte_perm transposes).
//   delta_split / delta_merge  a thread owns 16 pixel positions and walks them through the
//                              frames of one GOP with the previous frame kept in registers, so
//                              every frame is read from HBM once although it is used twice.
//   split_rows / merge_rows    the per-frame AVFrame layouts with row padding (linesize).
#include "common.cuh"
#include "hist.cuh"
#include "kernels.h"

namespace rirb {

struct LoHi {
    uint4 lo, hi;
};

// 16 pixels (8 words of 2 px) -> 16 low bytes + 16 high bytes
__device__ __forceinline__ LoHi split16(const U32x8& p)
{
    LoHi r;
    r.lo.x = __byte_perm(p.v[0], p.v[1], 0x6420);
    r.lo.y = __byte_perm(p.v[2], p.v[3], 0x6420);
    r.lo.z = __byte_perm(p.v[4], p.v[5], 0x6420);
    r.lo.w = __byte_perm(p.v[6], p.v[7], 0x6420);
    r.hi.x = __byte_perm(p.v[0], p.v[1], 0x7531);
    r.hi.y = __byte_perm(p.v[2], p.v[3], 0x7531);
    r.hi.z = __byte_perm(p.v[4], p.v[5], 0x7531);
    r.hi.w = __byte_perm(p.v[6], p.v[7], 0x7531);
    return r;
}

__device__ __forceinline__ U32x8 merge16(const uint4& lo, const uint4& hi)
{
    U32x8 p;
    p.v[0] = __byte_perm(lo.x, hi.x, 0x5140);
    p.v[1] = __byte_perm(lo.x, hi.x, 0x7362);
    p.v[2] = __byte_perm(lo.y, hi.y, 0x5140);
    p.v[3] = __byte_perm(lo.y, hi.y, 0x7362);
    p.v[4] = __byte_perm(lo.z, hi.z, 0x5140);
    p.v[5] = __byte_perm(lo.z, hi.z, 0x7362);
    p.v[6] = __byte_perm(lo.w, hi.w, 0x5140);
    p.v[7] = __byte_perm(lo.w, hi.w, 0x7362);
    return p;
}

constexpr int PC_THREADS = 256;
constexpr int PC_UNROLL = 4;

// ---- flat split / merge (no delta) -------------------------------------------------------------
__global__ void __launch_bounds__(PC_THREADS)
split_flat_kernel(const u16* __restrict__ in, u8* __restrict__ lo, u8* __restrict__ hi, size_t nvec)
{
    // a CTA owns PC_UNROLL*PC_THREADS consecutive vectors; each thread issues PC_UNROLL loads first
    size_t base = (size_t)blockIdx.x * (PC_THREADS * PC_UNROLL) + threadIdx.x;
    U32x8 p[PC_UNROLL];
#pragma unroll
    for (int k = 0; k < PC_UNROLL; ++k) {
        size_t i = base + (size_t)k * PC_THREADS;
        if (i < nvec) p[k] = ld_stream256(in + i * 16);
    }
#pragma unroll
    for (int k = 0; k < PC_UNROLL; ++k) {
        size_t i = base + (size_t)k * PC_THREADS;
        if (i < nvec) {
            LoHi r = split16(p[k]);
            st_stream(reinterpret_cast<uint4*>(lo) + i, r.lo);
            st_stream(reinterpret_cast<uint4*>(hi) + i, r.hi);
        }
    }
}

__global__ void __launch_bounds__(PC_THREADS)
merge_flat_kernel(const u8* __restrict__ lo, const u8* __restrict__ hi, u16* __restrict__ out, size_t nvec)
{
    size_t base = (size_t)blockIdx.x * (PC_THREADS * PC_UNROLL) + threadIdx.x;
    uint4 l[PC_UNROLL], h[PC_UNROLL];
#pragma unroll
    for (int k = 0; k < PC_UNROLL; ++k) {
        size_t i = base + (size_t)k * PC_THREADS;
        if (i < nvec) {
            l[k] = ld_stream(reinterpret_cast<const uint4*>(lo) + i);
            h[k] = ld_stream(reinterpret_cast<const uint4*>(hi) + i);
        }
    }
#pragma unroll
    for (int k = 0; k < PC_UNROLL; ++k) {
        size_t i = base + (size_t)k * PC_THREADS;
        if (i < nvec) st_stream256(out + i * 16, merge16(l[k], h[k]));
    }
}

// scalar tails / unaligned movies
__global__ void split_scalar_kernel(const u16* __restrict__ in, u8* __restrict__ lo, u8* __restrict__ hi, size_t first, size_t n)
{
    size_t i = first + (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) {
        unsigned v = in[i];
        lo[i] = (u8)(v & 0xFF);
        hi[i] = (u8)(v >> 8);
    }
}
__global__ void merge_scalar_kernel(const u8* __restrict__ lo, const u8* __restrict__ hi, u16* __restrict__ out, size_t first,
                                    size_t n)
{
    size_t i = first + (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) out[i] = (u16)(lo[i] | (hi[i] << 8));
}

// ---- temporal delta: a thread walks its 16 pixel positions through one GOP -----------------------
__device__ __forceinline__ U32x8 sub16(const U32x8& a, const U32x8& b)
{
    U32x8 r;
#pragma unroll
    for (int i = 0; i < 8; ++i) r.v[i] = __vsub2(a.v[i], b.v[i]);
    return r;
}
__device__ __forceinline__ U32x8 add16(const U32x8& a, const U32x8& b)
{
    U32x8 r;
#pragma unroll
    for (int i = 0; i < 8; ++i) r.v[i] = __vadd2(a.v[i], b.v[i]);
    return r;
}

__global__ void __launch_bounds__(PC_THREADS)
delta_split_kernel(const u16* __restrict__ mov, u8* __restrict__ lo, u8* __restrict__ hi, size_t vec_per_frame, long long nframes,
                   int gop)
{
    const size_t i = (size_t)blockIdx.x * PC_THREADS + threadIdx.x;  // vector position inside a frame
    if (i >= vec_per_frame) return;
    const long long t0 = (long long)blockIdx.y * gop;
    const long long t1 = min(nframes, t0 + gop);
    U32x8 prev;
#pragma unroll
    for (int k = 0; k < 8; ++k) prev.v[k] = 0;  // key frame: residual = frame - 0
    for (long long t = t0; t < t1; t += PC_UNROLL) {
        U32x8 cur[PC_UNROLL];
#pragma unroll
        for (int k = 0; k < PC_UNROLL; ++k)
            if (t + k < t1) cur[k] = ld_stream256(mov + ((size_t)(t + k) * vec_per_frame + i) * 16);
#pragma unroll
        for (int k = 0; k < PC_UNROLL; ++k)
            if (t + k < t1) {
                LoHi r = split16(sub16(cur[k], prev));
                prev = cur[k];
                const size_t o = (size_t)(t + k) * vec_per_frame + i;
                st_stream(reinterpret_cast<uint4*>(lo) + o, r.lo);
                st_stream(reinterpret_cast<uint4*>(hi) + o, r.hi);
            }
    }
}

__global__ void __launch_bounds__(PC_THREADS)
delta_merge_kernel(const u8* __restrict__ lo, const u8* __restrict__ hi, u16* __restrict__ mov, size_t vec_per_frame,
                   long long nframes, int gop)
{
    const size_t i = (size_t)blockIdx.x * PC_THREADS + threadIdx.x;
    if (i >= vec_per_frame) return;
    const long long t0 = (long long)blockIdx.y * gop;
    const long long t1 = min(nframes, t0 + gop);
    U32x8 prev;
#pragma unroll
    for (int k = 0; k < 8; ++k) prev.v[k] = 0;
    for (long long t = t0; t < t1; t += PC_UNROLL) {
        uint4 l[PC_UNROLL], h[PC_UNROLL];
#pragma unroll
        for (int k = 0; k < PC_UNROLL; ++k)
            if (t + k < t1) {
                const size_t o = (size_t)(t + k) * vec_per_frame + i;
                l[k] = ld_stream(reinterpret_cast<const uint4*>(lo) + o);
                h[k] = ld_stream(reinterpret_cast<const uint4*>(hi) + o);
            }
#pragma unroll
        for (int k = 0; k < PC_UNROLL; ++k)
            if (t + k < t1) {
                prev = add16(merge16(l[k], h[k]), prev);
                st_stream256(mov + ((size_t)(t + k) * vec_per_frame + i) * 16, prev);
            }
    }
}

// generic (any size / alignment) delta kernels: one thread per pixel position, walks a GOP
__global__ void delta_split_scalar_kernel(const u16* __restrict__ mov, u8* __restrict__ lo, u8* __restrict__ hi, size_t npx,
                                          long long nframes, int gop)
{
    const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= npx) return;
    const long long t0 = (long long)blockIdx.y * gop;
    const long long t1 = min(nframes, t0 + gop);
    unsigned prev = 0;
    for (long long t = t0; t < t1; ++t) {
        unsigned cur = mov[(size_t)t * npx + i];
        unsigned r = (cur - prev) & 0xFFFFu;
        prev = cur;
        lo[(size_t)t * npx + i] = (u8)(r & 0xFF);
        hi[(size_t)t * npx + i] = (u8)(r >> 8);
    }
}
__global__ void delta_merge_scalar_kernel(const u8* __restrict__ lo, const u8* __restrict__ hi, u16* __restrict__ mov, size_t npx,
                                          long long nframes, int gop)
{
    const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= npx) return;
    const long long t0 = (long long)blockIdx.y * gop;
    const long long t1 = min(nframes, t0 + gop);
    unsigned prev = 0;
    for (long long t = t0; t < t1; ++t) {
        unsigned r = lo[(size_t)t * npx + i] | (hi[(size_t)t * npx + i] << 8);
        prev = (r + prev) & 0xFFFFu;
        mov[(size_t)t * npx + i] = (u16)prev;
    }
}

constexpr long long MAX_GOPS_PER_LAUNCH = 65535;  // the delta kernels put the GOP index in gridDim.y

static bool movie_vectorizable(const void* mov, const void* lo, const void* hi, size_t npx)
{
    return (npx % 16 == 0) && aligned32(mov) && aligned16(lo) && aligned16(hi);
}

// ---- pre-coder fused with the movie statistics ---------------------------------------------------
// The frames the pre-coder reads are the frames the statistics are taken of (the registered movie), and
// the pre-coder leaves four fifths of the issue slots idle (it is purely bandwidth-bound), so one kernel
// does both: persistent, one 1024-thread CTA per SM with the 49,152-bin shared histogram of stats.cu,
// work items = (1024 vector positions, one GOP).  4 B/px for both results instead of 4 + 2.
constexpr int PS_THREADS = 1024;

template <bool DELTA>
__global__ void __launch_bounds__(PS_THREADS, 1)
split_stats_kernel(const u16* __restrict__ mov, u8* __restrict__ lo, u8* __restrict__ hi, size_t vec_per_frame, long long nframes,
                   int gop, unsigned* __restrict__ minmax, unsigned long long* __restrict__ hist)
{
    extern __shared__ unsigned sh[];
    for (unsigned i = threadIdx.x; i < HIST_SMEM_BINS; i += PS_THREADS) sh[i] = 0;
    __syncthreads();
    const long long ngop = (nframes + gop - 1) / gop;
    const long long blocks = (long long)((vec_per_frame + PS_THREADS - 1) / PS_THREADS);
    unsigned lo2 = 0xFFFFFFFFu, hi2 = 0u;  // packed per-halfword min / max
    for (long long item = blockIdx.x; item < blocks * ngop; item += gridDim.x) {
        const long long g = item / blocks;
        const size_t i = (size_t)(item - g * blocks) * PS_THREADS + threadIdx.x;
        if (i >= vec_per_frame) continue;
        const long long t0 = g * gop, t1 = min(nframes, t0 + gop);
        U32x8 prev;
#pragma unroll
        for (int k = 0; k < 8; ++k) prev.v[k] = 0;
        for (long long t = t0; t < t1; t += PC_UNROLL) {
            U32x8 cur[PC_UNROLL];
#pragma unroll
            for (int k = 0; k < PC_UNROLL; ++k)
                if (t + k < t1) cur[k] = ld_stream256(mov + ((size_t)(t + k) * vec_per_frame + i) * 16);
#pragma unroll
            for (int k = 0; k < PC_UNROLL; ++k)
                if (t + k < t1) {
                    const LoHi r = split16(DELTA ? sub16(cur[k], prev) : cur[k]);
                    if (DELTA) prev = cur[k];
                    const size_t o = (size_t)(t + k) * vec_per_frame + i;
                    st_stream(reinterpret_cast<uint4*>(lo) + o, r.lo);
                    st_stream(reinterpret_cast<uint4*>(hi) + o, r.hi);
#pragma unroll
                    for (int q = 0; q < 8; ++q) {
                        const unsigned w2 = cur[k].v[q];
                        lo2 = __vminu2(lo2, w2);
                        hi2 = __vmaxu2(hi2, w2);
                        count_px(w2 & 0xFFFFu, sh, hist);
                        count_px(w2 >> 16, sh, hist);
                    }
                }
        }
    }
    hist_flush(min(lo2 & 0xFFFFu, lo2 >> 16), max(hi2 & 0xFFFFu, hi2 >> 16), sh, minmax, hist, true);
}

// returns 1 when the layout cannot take the fused kernel (caller runs the two kernels)
int launch_precode_movie_stats(const u16* mov, long long nframes, int w, int h, int gop, int delta, long long first_frame, u8* lo,
                               u8* hi, unsigned* minmax, unsigned long long* hist, cudaStream_t st)
{
    if (nframes <= 0 || w <= 0 || h <= 0) return 0;
    const size_t npx = (size_t)w * h;
    if (gop < 1) gop = 1;
    if (!movie_vectorizable(mov, lo, hi, npx) || !hist || !minmax) return 1;
    if (delta && first_frame % gop != 0) {
        set_error("precode: with delta on, a shard must start on a key frame (first_frame %lld, GOP %d)", first_frame, gop);
        return -1;
    }
    const size_t vpf = npx / 16;
    const size_t smem = HIST_SMEM_BINS * sizeof(unsigned);
    const long long items = ceil_div((long long)vpf, PS_THREADS) * ceil_div(nframes, gop);
    const unsigned grid = (unsigned)min((long long)sm_count(), items);
    if (delta) {
        RIRB_SMEM_ATTR(split_stats_kernel<true>, smem);
        RIRB_LAUNCH(split_stats_kernel<true>, grid, PS_THREADS, smem, st, mov, lo, hi, vpf, nframes, gop, minmax, hist);
    } else {
        RIRB_SMEM_ATTR(split_stats_kernel<false>, smem);
        RIRB_LAUNCH(split_stats_kernel<false>, grid, PS_THREADS, smem, st, mov, lo, hi, vpf, nframes, gop, minmax, hist);
    }
    return 0;
}

int launch_precode_movie(const u16* mov, long long nframes, int w, int h, int gop, int delta, long long first_frame, u8* lo,
                         u8* hi, cudaStream_t st)
{
    if (nframes <= 0 || w <= 0 || h <= 0) return 0;
    const size_t npx = (size_t)w * h;
    if (gop < 1) gop = 1;
    if (!delta) {
        const size_t n = npx * (size_t)nframes;
        size_t done = 0;
        if (aligned32(mov) && aligned16(lo) && aligned16(hi) && n >= 16) {
            const size_t nvec = n / 16;
            RIRB_LAUNCH(split_flat_kernel, (unsigned)ceil_div((long long)nvec, PC_THREADS * PC_UNROLL), PC_THREADS, 0, st, mov, lo,
                        hi, nvec);
            done = nvec * 16;
        }
        if (done < n)
            RIRB_LAUNCH(split_scalar_kernel, (unsigned)ceil_div((long long)(n - done), 256), 256, 0, st, mov, lo, hi, done, n);
        return 0;
    }
    if (first_frame % gop != 0) {
        set_error("precode: with delta on, a shard must start on a key frame (first_frame %lld, GOP %d)", first_frame, gop);
        return -1;
    }
    // grid = (pixel block, GOP); gridDim.y <= 65535, so long movies go in several launches of whole GOPs (whole frames
    // keep the vector alignment, as npx % 16 == 0 on that path) -- the fused split_stats_kernel has no such limit
    const bool vec = movie_vectorizable(mov, lo, hi, npx);
    const long long span = (long long)MAX_GOPS_PER_LAUNCH * gop;
    for (long long f0 = 0; f0 < nframes; f0 += span) {
        const long long n = min(nframes - f0, span);
        const size_t off = (size_t)f0 * npx;
        const unsigned ngop = (unsigned)ceil_div(n, gop);
        if (vec) {
            const size_t vpf = npx / 16;
            dim3 grid((unsigned)ceil_div((long long)vpf, PC_THREADS), ngop);
            RIRB_LAUNCH(delta_split_kernel, grid, PC_THREADS, 0, st, mov + off, lo + off, hi + off, vpf, n, gop);
        } else {
            dim3 grid((unsigned)ceil_div((long long)npx, 256), ngop);
            RIRB_LAUNCH(delta_split_scalar_kernel, grid, 256, 0, st, mov + off, lo + off, hi + off, npx, n, gop);
        }
    }
    return 0;
}

int launch_decode_movie(const u8* lo, const u8* hi, long long nframes, int w, int h, int gop, int delta, long long first_frame,
                        u16* mov, cudaStream_t st)
{
    if (nframes <= 0 || w <= 0 || h <= 0) return 0;
    const size_t npx = (size_t)w * h;
    if (gop < 1) gop = 1;
    if (!delta) {
        const size_t n = npx * (size_t)nframes;
        size_t done = 0;
        if (aligned32(mov) && aligned16(lo) && aligned16(hi) && n >= 16) {
            const size_t nvec = n / 16;
            RIRB_LAUNCH(merge_flat_kernel, (unsigned)ceil_div((long long)nvec, PC_THREADS * PC_UNROLL), PC_THREADS, 0, st, lo, hi,
                        mov, nvec);
            done = nvec * 16;
        }
        if (done < n)
            RIRB_LAUNCH(merge_scalar_kernel, (unsigned)ceil_div((long long)(n - done), 256), 256, 0, st, lo, hi, mov, done, n);
        return 0;
    }
    if (first_frame % gop != 0) {
        set_error("decode: with delta on, a shard must start on a key frame (first_frame %lld, GOP %d)", first_frame, gop);
        return -1;
    }
    const bool vec = movie_vectorizable(mov, lo, hi, npx);
    const long long span = (long long)MAX_GOPS_PER_LAUNCH * gop;  // as in launch_precode_movie
    for (long long f0 = 0; f0 < nframes; f0 += span) {
        const long long n = min(nframes - f0, span);
        const size_t off = (size_t)f0 * npx;
        const unsigned ngop = (unsigned)ceil_div(n, gop);
        if (vec) {
            const size_t vpf = npx / 16;
            dim3 grid((unsigned)ceil_div((long long)vpf, PC_THREADS), ngop);
            RIRB_LAUNCH(delta_merge_kernel, grid, PC_THREADS, 0, st, lo + off, hi + off, mov + off, vpf, n, gop);
        } else {
            dim3 grid((unsigned)ceil_div((long long)npx, 256), ngop);
            RIRB_LAUNCH(delta_merge_scalar_kernel, grid, 256, 0, st, lo + off, hi + off, mov + off, npx, n, gop);
        }
    }
    return 0;
}

// ---- per-frame AVFrame layouts (row padding) ----------------------------------------------------
// lo/hi/aux planes with their own line sizes; aux (the Y plane of YUV444P, or the U plane of the
// YUV420P integration-time variant) receives it[] or 0.  Null plane pointers are skipped.
__global__ void split_rows_kernel(const u16* __restrict__ img, const u8* __restrict__ it, int w, int h, u8* __restrict__ lo,
                                  int ls_lo, u8* __restrict__ hi, int ls_hi, u8* __restrict__ aux, int ls_aux)
{
    const int x = blockIdx.x * blockDim.x + threadIdx.x;
    const int y = blockIdx.y * blockDim.y + threadIdx.y;
    if (x >= w || y >= h) return;
    const unsigned v = img[(size_t)y * w + x];
    if (lo) lo[(size_t)y * ls_lo + x] = (u8)(v & 0xFF);
    if (hi) hi[(size_t)y * ls_hi + x] = (u8)(v >> 8);
    if (aux) aux[(size_t)y * ls_aux + x] = it ? it[(size_t)y * w + x] : (u8)0;
}

__global__ void merge_rows_kernel(const u8* __restrict__ lo, int ls_lo, const u8* __restrict__ hi, int ls_hi,
                                  const u8* __restrict__ aux, int ls_aux, int w, int h, u16* __restrict__ img, u8* __restrict__ it)
{
    const int x = blockIdx.x * blockDim.x + threadIdx.x;
    const int y = blockIdx.y * blockDim.y + threadIdx.y;
    if (x >= w || y >= h) return;
    img[(size_t)y * w + x] = (u16)(lo[(size_t)y * ls_lo + x] | (hi[(size_t)y * ls_hi + x] << 8));
    if (it && aux) it[(size_t)y * w + x] = aux[(size_t)y * ls_aux + x];
}

int launch_split_planes(const u16* img, const u8* it, int w, int h, u8* aux_plane, u8* lo_plane, u8* hi_plane, int ls_aux,
                        int ls_lo, int ls_hi, cudaStream_t st)
{
    if (w <= 0 || h <= 0) return 0;
    dim3 block(32, 8);
    dim3 grid((unsigned)ceil_div(w, 32), (unsigned)ceil_div(h, 8));
    RIRB_LAUNCH(split_rows_kernel, grid, block, 0, st, img, it, w, h, lo_plane, ls_lo, hi_plane, ls_hi, aux_plane, ls_aux);
    return 0;
}

int launch_merge_planes(const u8* aux_plane, const u8* lo_plane, const u8* hi_plane, int ls_aux, int ls_lo, int ls_hi, int w, int h,
                        u16* img, u8* it, cudaStream_t st)
{
    if (w <= 0 || h <= 0) return 0;
    dim3 block(32, 8);
    dim3 grid((unsigned)ceil_div(w, 32), (unsigned)ceil_div(h, 8));
    RIRB_LAUNCH(merge_rows_kernel, grid, block, 0, st, lo_plane, ls_lo, hi_plane, ls_hi, aux_plane, ls_aux, w, h, img, it);
    return 0;
}

}  // namespace rirb
