// librir_b200/csrc/common.cuh -- shared host/device utilities of the sm_100a hot path.
//
// Conventions used by every kernel file:
//   * images are dense row-major [h][w]; a movie is nframes such frames back to back;
//   * every launch goes through RIRB_LAUNCH so that the library can report how many of its
//     own kernels ran (rirb_kernel_launch_count) and surfaces launch errors as status codes;
//   * kernels are launched on the calling thread's current stream (rirb_set_stream), which
//     defaults to the legacy default stream.
#pragma once

#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>

#include <atomic>
#include <memory>
#include <string>

#include "handles.h"

namespace rirb {

typedef unsigned short u16;
typedef unsigned char u8;

// ---- error / bookkeeping (defined in capi.cu) ------------------------------------------------
void set_error(const char* fmt, ...);
cudaStream_t current_stream();
extern std::atomic<long long> g_launches;
int sm_count();
int require_device();  // -1 (set_error) when there is no usable CUDA device: this library has no CPU fallback
// run-time switches (rirb_set_parameter; initial values from the environment): kernel variants for A/B runs
enum { OPT_TRANSLATE_TMA = 0, OPT_GAUSS_TMA = 1, OPT_LOADER_FUSED = 2, OPT_ECC_FUSED = 3, OPT_LOSSY_RUN = 4, OPT_TRANSLATE_ROWS = 5, OPT_ECC_QUEUE = 6, OPT_ZSTD_DECODER = 7, OPT_COUNT = 8 };
bool option_enabled(int which);
int option_value(int which);  // the switch's integer value (option_enabled: != 0)

#define RIRB_CUDA_OK(expr)                                                                    \
    do {                                                                                      \
        cudaError_t _e = (expr);                                                              \
        if (_e != cudaSuccess) {                                                              \
            ::rirb::set_error("%s failed: %s (%s:%d)", #expr, cudaGetErrorString(_e), __FILE__, __LINE__); \
            (void)cudaGetLastError(); /* do not leave it for the next launch check to find */ \
            return -1;                                                                        \
        }                                                                                     \
    } while (0)

// Launch + count + check.  Usage: RIRB_LAUNCH(kernel, grid, block, smem, stream, args...)
#define RIRB_LAUNCH(kern, grid, block, smem, stream, ...)                                     \
    do {                                                                                      \
        kern<<<(grid), (block), (smem), (stream)>>>(__VA_ARGS__);                             \
        ::rirb::g_launches.fetch_add(1, std::memory_order_relaxed);                           \
        cudaError_t _e = cudaGetLastError();                                                  \
        if (_e != cudaSuccess) {                                                              \
            ::rirb::set_error("launch of %s failed: %s", #kern, cudaGetErrorString(_e));     \
            return -1;                                                                        \
        }                                                                                     \
    } while (0)

// Opt a kernel into more than 48 KB of dynamic shared memory, once per device (the attribute belongs to the
// function in one context; a process may drive several GPUs).  Usage: RIRB_SMEM_ATTR(kernel, bytes).
#define RIRB_SMEM_ATTR(kern, bytes)                                                                        \
    do {                                                                                                   \
        static std::atomic<unsigned long long> _done{0};                                                   \
        int _dev = 0;                                                                                      \
        cudaGetDevice(&_dev);                                                                              \
        const unsigned long long _bit = 1ull << (_dev & 63);                                               \
        if (!(_done.load(std::memory_order_relaxed) & _bit)) {                                             \
            RIRB_CUDA_OK(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)(bytes))); \
            _done.fetch_or(_bit, std::memory_order_relaxed);                                               \
        }                                                                                                  \
    } while (0)

// A handle's buffers live in the memory of the device it was created on (T::device): entries that launch kernels refuse a
// handle from another device instead of faulting on its pointers.  nullptr (set_error) when unknown or elsewhere.
template <typename T> std::shared_ptr<T> find_handle_here(Table<T>& table, int id, const char* what)
{
    auto s = table.get(id);
    if (!s) {
        set_error("%s: unknown handle %d", what, id);
        return nullptr;
    }
    int dev = -1;
    if (cudaGetDevice(&dev) != cudaSuccess) cudaGetLastError();
    if (dev != s->device) {
        set_error("%s: handle %d belongs to CUDA device %d, the calling thread is on device %d", what, id, s->device, dev);
        return nullptr;
    }
    return s;
}

static inline bool aligned16(const void* p) { return (reinterpret_cast<uintptr_t>(p) & 15u) == 0; }
static inline long long ceil_div(long long a, long long b) { return (a + b - 1) / b; }

// ---- device helpers ----------------------------------------------------------------------------
#ifdef __CUDACC__

// Streaming accesses: every byte of a movie is touched once, so keep it out of L1
// (ld.global.nc.L1::no_allocate / st.global.L1::no_allocate -> LDG.E.NA / STG.E.NA).
__device__ __forceinline__ uint4 ld_stream(const uint4* p)
{
    uint4 r;
    asm volatile("ld.global.nc.L1::no_allocate.v4.u32 {%0,%1,%2,%3}, [%4];"
                 : "=r"(r.x), "=r"(r.y), "=r"(r.z), "=r"(r.w)
                 : "l"(p));
    return r;
}
__device__ __forceinline__ uint2 ld_stream(const uint2* p)
{
    uint2 r;
    asm volatile("ld.global.nc.L1::no_allocate.v2.u32 {%0,%1}, [%2];" : "=r"(r.x), "=r"(r.y) : "l"(p));
    return r;
}
__device__ __forceinline__ float4 ld_stream(const float4* p)
{
    float4 r;
    asm volatile("ld.global.nc.L1::no_allocate.v4.f32 {%0,%1,%2,%3}, [%4];"
                 : "=f"(r.x), "=f"(r.y), "=f"(r.z), "=f"(r.w)
                 : "l"(p));
    return r;
}
__device__ __forceinline__ void st_stream(uint4* p, const uint4& v)
{
    asm volatile("st.global.L1::no_allocate.v4.u32 [%0], {%1,%2,%3,%4};" ::"l"(p), "r"(v.x), "r"(v.y), "r"(v.z), "r"(v.w)
                 : "memory");
}
__device__ __forceinline__ void st_stream(uint2* p, const uint2& v)
{
    asm volatile("st.global.L1::no_allocate.v2.u32 [%0], {%1,%2};" ::"l"(p), "r"(v.x), "r"(v.y) : "memory");
}
__device__ __forceinline__ void st_stream(float4* p, const float4& v)
{
    asm volatile("st.global.L1::no_allocate.v4.f32 [%0], {%1,%2,%3,%4};" ::"l"(p), "f"(v.x), "f"(v.y), "f"(v.z), "f"(v.w)
                 : "memory");
}

// sm_100 has 256-bit per-thread global accesses (LDG.E.256 / STG.E.256).  32-byte alignment
// required.  evict_first: the line is not needed again (pure streams).
struct __align__(32) U32x8 {
    unsigned v[8];
};
__device__ __forceinline__ U32x8 ld_stream256(const void* p)
{
    U32x8 r;
    asm volatile("ld.global.nc.L1::no_allocate.L2::evict_first.v8.b32 {%0,%1,%2,%3,%4,%5,%6,%7}, [%8];"
                 : "=r"(r.v[0]), "=r"(r.v[1]), "=r"(r.v[2]), "=r"(r.v[3]), "=r"(r.v[4]), "=r"(r.v[5]), "=r"(r.v[6]),
                   "=r"(r.v[7])
                 : "l"(p));
    return r;
}
__device__ __forceinline__ void st_stream256(void* p, const U32x8& r)
{
    asm volatile("st.global.L1::no_allocate.v8.b32 [%0], {%1,%2,%3,%4,%5,%6,%7,%8};" ::"l"(p), "r"(r.v[0]), "r"(r.v[1]),
                 "r"(r.v[2]), "r"(r.v[3]), "r"(r.v[4]), "r"(r.v[5]), "r"(r.v[6]), "r"(r.v[7])
                 : "memory");
}
// same width, normal L2 eviction priority: for streams whose lines are touched again shortly after
// (bad-pixel fix-ups gather the neighbours of flagged pixels from the rows their CTA just streamed)
__device__ __forceinline__ U32x8 ld_stream256_keep(const void* p)
{
    U32x8 r;
    asm volatile("ld.global.nc.L1::no_allocate.v8.b32 {%0,%1,%2,%3,%4,%5,%6,%7}, [%8];"
                 : "=r"(r.v[0]), "=r"(r.v[1]), "=r"(r.v[2]), "=r"(r.v[3]), "=r"(r.v[4]), "=r"(r.v[5]), "=r"(r.v[6]),
                   "=r"(r.v[7])
                 : "l"(p));
    return r;
}
static inline bool aligned32(const void* p) { return (reinterpret_cast<uintptr_t>(p) & 31u) == 0; }

// per-halfword unsigned max of two packed u16 pairs
__device__ __forceinline__ unsigned vmaxu2(unsigned a, unsigned b) { return __vmaxu2(a, b); }

#endif  // __CUDACC__

}  // namespace rirb
