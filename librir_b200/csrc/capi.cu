// librir_b200/csrc/capi.cu -- the C ABI (include/librir_b200.h): argument checking, host<->device
// staging for host-pointer callers, the bad-pixel handle table, forwarding of the out-of-scope
// entries.  All compute happens in the kernels of this directory; there is no CPU path.
#include <dlfcn.h>
#include <math.h>
#include <stdarg.h>
#include <stdlib.h>
#include <string.h>

#include <map>
#include <memory>
#include <mutex>
#include <vector>

#include "../../include/librir_b200.h"
#include "common.cuh"
#include "kernels.h"

namespace rirb {

// ------------------------------------------------------------------------------------------------
// per-thread state: last error, stream, scratch buffers
// ------------------------------------------------------------------------------------------------
std::atomic<long long> g_launches{0};

struct ThreadState {
    char err[512] = {0};
    cudaStream_t stream = 0;
    // grow-only device scratch slots for host-pointer callers (never shared between threads)
    // slots 0-5: operands of the entry that is running; 6-7: bad_pixels_create, which other entries call
    // 8-11: launchers' own work space (kernels.h: scratch_buffer)
    static constexpr int SLOTS = 12;
    void* dev[SLOTS] = {};
    size_t cap[SLOTS] = {};
    int dev_of[SLOTS] = {};
    bool enqueued = false;  // something of this thread may still be running on `stream` (device-pointer calls do not synchronise)
    ThreadState()
    {
        for (int i = 0; i < SLOTS; ++i) dev_of[i] = -1;
    }
    // a thread that exits gives its device memory back (cudaFree of a UVA pointer works from any current device; at process
    // exit the runtime may already be gone: cudaErrorCudartUnloading is expected and ignored)
    ~ThreadState() { release(); }
    void release()
    {
        for (int i = 0; i < SLOTS; ++i) {
            if (dev[i]) (void)cudaFree(dev[i]);
            dev[i] = nullptr;
            cap[i] = 0;
            dev_of[i] = -1;
        }
        (void)cudaGetLastError();
    }
};
static thread_local ThreadState tls;

void set_error(const char* fmt, ...)
{
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(tls.err, sizeof(tls.err), fmt, ap);
    va_end(ap);
    if (getenv("LIBRIR_B200_VERBOSE")) fprintf(stderr, "[librir_b200] %s\n", tls.err);
}

cudaStream_t current_stream() { return tls.stream; }

// ---- run-time switches ---------------------------------------------------------------------------
static const char* const k_opt_names[OPT_COUNT] = {"translate_tma", "gauss_tma", "loader_fused", "ecc_fused", "lossy_run", "translate_rows", "ecc_queue", "zstd_decoder"};
static const char* const k_opt_env[OPT_COUNT] = {"RIRB_TRANSLATE_TMA", "RIRB_GAUSS_TMA", "RIRB_LOADER_FUSED", "RIRB_ECC_FUSED", "RIRB_LOSSY_RUN", "RIRB_TRANSLATE_ROWS", "RIRB_ECC_QUEUE", "RIRB_ZSTD_DECODER"};
static const int k_opt_default[OPT_COUNT] = {1, 1, 0, 1, 1, 1, 1, 1};
static std::atomic<int> g_opts[OPT_COUNT];
static std::once_flag g_opts_once;
static void init_options()
{
    for (int i = 0; i < OPT_COUNT; ++i) {
        const char* e = getenv(k_opt_env[i]);
        g_opts[i].store(e && *e ? atoi(e) : k_opt_default[i]);
    }
}
bool option_enabled(int which)
{
    std::call_once(g_opts_once, init_options);
    return which >= 0 && which < OPT_COUNT && g_opts[which].load() != 0;
}

int option_value(int which)
{
    std::call_once(g_opts_once, init_options);
    return which >= 0 && which < OPT_COUNT ? g_opts[which].load() : 0;
}

int sm_count()
{
    static int cached[64] = {0};
    int dev = 0;
    if (cudaGetDevice(&dev) != cudaSuccess || dev < 0 || dev >= 64) return 148;
    if (cached[dev] == 0) {
        int n = 0;
        if (cudaDeviceGetAttribute(&n, cudaDevAttrMultiProcessorCount, dev) != cudaSuccess || n <= 0) n = 148;
        cached[dev] = n;
    }
    return cached[dev];
}

// No device -> every compute entry fails loudly: this library has no CPU fallback.
static int require_device()
{
    static std::atomic<int> state{0};  // 0 unknown, 1 ok, -1 none
    int s = state.load();
    if (s == 0) {
        int n = 0;
        cudaError_t e = cudaGetDeviceCount(&n);
        s = (e == cudaSuccess && n > 0) ? 1 : -1;
        if (s < 0) cudaGetLastError();
        state.store(s);
    }
    if (s < 0) {
        set_error("no usable CUDA device: librir_b200 computes on the GPU only and has no CPU fallback");
        return -1;
    }
    return 0;
}

static bool is_device_ptr(const void* p) { return p && operand_on_device(p); }

static void* scratch(int slot, size_t bytes)
{
    int dev = 0;
    cudaGetDevice(&dev);
    tls.enqueued = true;  // whoever asks for scratch is about to enqueue work that uses it (see rirb_set_stream)
    if (tls.cap[slot] < bytes || tls.dev_of[slot] != dev) {
        if (tls.dev[slot]) cudaFree(tls.dev[slot]);  // also when the thread moved to another device: UVA pointers free from anywhere
        tls.dev[slot] = nullptr;
        tls.cap[slot] = 0;
        size_t want = bytes < (1u << 20) ? (1u << 20) : bytes + bytes / 4;
        if (cudaMalloc(&tls.dev[slot], want) != cudaSuccess) {
            cudaGetLastError();
            set_error("out of device memory for a %zu-byte staging buffer", want);
            return nullptr;
        }
        tls.cap[slot] = want;
        tls.dev_of[slot] = dev;
    }
    return tls.dev[slot];
}

void* scratch_buffer(int slot, size_t bytes) { return (slot >= 8 && slot < ThreadState::SLOTS) ? scratch(slot, bytes) : nullptr; }

// ---- pageable host buffers --------------------------------------------------------------------
// A device->host cudaMemcpyAsync into pageable memory is staged by the driver at ~5 GB/s for one
// 640x512 frame (measured: profiles/r1_percall.md).  Host-pointer callers are the reference's own
// one-frame-per-call seam, so the library keeps a small per-thread ring of pinned chunks and
// pipelines  DMA | memcpy(pinned -> host)  itself; pinned or registered caller buffers
// (cudaMemoryTypeHost) skip the ring and are written in place.
constexpr size_t PIN_CHUNK = 256u << 10;
constexpr int PIN_NB = 4;
constexpr size_t PIN_MAX_BYTES = 64u << 20;  // beyond this the driver's own pageable path is as good
struct PinRing {
    char* buf[PIN_NB] = {nullptr, nullptr, nullptr, nullptr};
    cudaEvent_t ev[PIN_NB] = {nullptr, nullptr, nullptr, nullptr};
    int state = 0;  // 0 not tried, 1 ready, -1 unavailable (fall back to plain copies)
    ~PinRing() { release(); }
    void release()
    {
        for (int i = 0; i < PIN_NB; ++i) {
            if (buf[i]) (void)cudaFreeHost(buf[i]);
            if (ev[i]) (void)cudaEventDestroy(ev[i]);
            buf[i] = nullptr;
            ev[i] = nullptr;
        }
        (void)cudaGetLastError();
        state = 0;
    }
};
// Events belong to the device that was current when they were created, so a thread that moves between devices
// (rirb_set_device) gets one ring per device.
constexpr int PIN_MAX_DEVICES = 16;
static thread_local PinRing pin_rings[PIN_MAX_DEVICES];
static thread_local PinRing pin_none;
#define pin (*pin_current())
static PinRing* pin_current()
{
    int dev = -1;
    if (cudaGetDevice(&dev) != cudaSuccess) cudaGetLastError();
    if (dev < 0 || dev >= PIN_MAX_DEVICES) {
        pin_none.state = -1;  // plain copies
        return &pin_none;
    }
    return &pin_rings[dev];
}

static bool pin_ready()
{
    if (pin.state == 0) {
        pin.state = 1;
        for (int i = 0; i < PIN_NB && pin.state == 1; ++i)
            if (cudaMallocHost((void**)&pin.buf[i], PIN_CHUNK) != cudaSuccess ||
                cudaEventCreateWithFlags(&pin.ev[i], cudaEventDisableTiming) != cudaSuccess) {
                cudaGetLastError();
                pin.state = -1;
            }
    }
    return pin.state == 1;
}

static bool is_pageable(const void* p) { return operand_memory_type(p) == cudaMemoryTypeUnregistered; }

// Uploads stay with the driver: its pageable host->device path already runs at the speed of one
// host memcpy (~10 GB/s here), the ring was no faster at 640x512 and 20 % slower at 1280x1024.
static cudaError_t copy_h2d(void* dev, const void* host, size_t bytes, cudaStream_t st)
{
    return cudaMemcpyAsync(dev, host, bytes, cudaMemcpyHostToDevice, st);
}

// Returns with the bytes in `host` (synchronous for pageable destinations).
static cudaError_t copy_d2h(void* host, const void* dev, size_t bytes, cudaStream_t st)
{
    if (bytes > PIN_MAX_BYTES || !is_pageable(host) || !pin_ready()) return cudaMemcpyAsync(host, dev, bytes, cudaMemcpyDeviceToHost, st);
    cudaError_t e = cudaSuccess;
    const size_t nchunks = (bytes + PIN_CHUNK - 1) / PIN_CHUNK;
    auto enqueue = [&](size_t k) -> cudaError_t {
        const size_t off = k * PIN_CHUNK;
        const size_t len = bytes - off < PIN_CHUNK ? bytes - off : PIN_CHUNK;
        const int i = (int)(k % PIN_NB);
        cudaError_t r = cudaMemcpyAsync(pin.buf[i], (const char*)dev + off, len, cudaMemcpyDeviceToHost, st);
        if (r == cudaSuccess) r = cudaEventRecord(pin.ev[i], st);
        return r;
    };
    for (size_t k = 0; k < nchunks && k < (size_t)PIN_NB && e == cudaSuccess; ++k) e = enqueue(k);
    for (size_t k = 0; k < nchunks && e == cudaSuccess; ++k) {
        const size_t off = k * PIN_CHUNK;
        const size_t len = bytes - off < PIN_CHUNK ? bytes - off : PIN_CHUNK;
        const int i = (int)(k % PIN_NB);
        if ((e = cudaEventSynchronize(pin.ev[i])) != cudaSuccess) break;
        memcpy((char*)host + off, pin.buf[i], len);
        if (k + PIN_NB < nchunks) e = enqueue(k + PIN_NB);
    }
    return e;
}

#undef pin

// Input operand: device pointer as is, host pointer uploaded into scratch slot `slot`.
static const void* stage_in(const void* p, size_t bytes, int slot, cudaStream_t st)
{
    if (is_device_ptr(p)) return p;
    void* d = scratch(slot, bytes);
    if (!d) return nullptr;
    if (copy_h2d(d, p, bytes, st) != cudaSuccess) {
        set_error("host->device copy failed: %s", cudaGetErrorString(cudaGetLastError()));
        return nullptr;
    }
    return d;
}

// Output operand: `preload` uploads the caller's current contents first (outputs that are only
// partially overwritten, e.g. translate's "noborder" strategy or padded planes).
struct StagedOut {
    void* dev = nullptr;
    void* host = nullptr;
    size_t bytes = 0;
};
static bool stage_out(StagedOut& o, void* p, size_t bytes, int slot, bool preload, cudaStream_t st)
{
    o.bytes = bytes;
    if (is_device_ptr(p)) {
        o.dev = p;
        o.host = nullptr;
        return true;
    }
    o.host = p;
    o.dev = scratch(slot, bytes);
    if (!o.dev) return false;
    if (preload && copy_h2d(o.dev, p, bytes, st) != cudaSuccess) {
        set_error("host->device copy failed: %s", cudaGetErrorString(cudaGetLastError()));
        return false;
    }
    return true;
}
// Copies staged outputs back and waits; device-pointer outputs return without synchronising.
static int finish_out(StagedOut* outs, int n, cudaStream_t st)
{
    bool any = false;
    for (int i = 0; i < n; ++i)
        if (outs[i].host && outs[i].bytes) {
            RIRB_CUDA_OK(copy_d2h(outs[i].host, outs[i].dev, outs[i].bytes, st));
            any = true;
        }
    if (any) RIRB_CUDA_OK(cudaStreamSynchronize(st));
    return 0;
}

static int strategy_code(const char* s)
{
    if (!s || !*s || strcmp(s, "noborder") == 0) return STRAT_NOBORDER;
    if (strcmp(s, "background") == 0) return STRAT_BACKGROUND;
    if (strcmp(s, "wrap") == 0) return STRAT_WRAP;
    if (strcmp(s, "nearest") == 0) return STRAT_NEAREST;
    return -1;
}

static size_t dtype_size(int type)
{
    switch (type) {
    case '?': case 'b': case 'B': return 1;
    case 'h': case 'H': return 2;
    case 'i': case 'I': case 'f': return 4;
    case 'l': case 'L': case 'd': return 8;
    default: return 0;
    }
}

// ------------------------------------------------------------------------------------------------
// bad-pixel handle table (the reference's set_void_ptr / get_void_ptr / rm_void_ptr, tools.cpp:40-85:
// process-global, mutex-guarded, lowest free positive slot)
// ------------------------------------------------------------------------------------------------
struct BadPixelState {
    int w = 0, h = 0, device = 0;
    int clamp_value = -1;         // m_median_value, BadPixels.cpp:22-31
    unsigned global_thr = 0;      // Filters.h:157-160
    u8* mask_dev = nullptr;       // bitmap, row stride (w+7)/8
    int* xy_dev = nullptr;        // raster-ordered list (x,y), device copy
    int* span_off_dev = nullptr;  // list offsets per BP_SPAN-pixel span (correction kernel)
    int* nbr_dev = nullptr;       // per list entry: which cells of the loader variant's shifted 3x3 window are flagged
    int* row_off_dev = nullptr;   // first list entry of each image row (h + 1 entries), fused reader kernel
    std::vector<int> xy;          // host copy
    ~BadPixelState()
    {
        if (mask_dev) cudaFree(mask_dev);
        if (xy_dev) cudaFree(xy_dev);
        if (span_off_dev) cudaFree(span_off_dev);
        if (nbr_dev) cudaFree(nbr_dev);
        if (row_off_dev) cudaFree(row_off_dev);
    }
};
static std::mutex g_handles_mutex;
static std::map<int, std::shared_ptr<BadPixelState>> g_handles;

static int register_handle(std::shared_ptr<BadPixelState> s)
{
    std::lock_guard<std::mutex> lock(g_handles_mutex);
    int id = 1;
    for (auto& kv : g_handles) {
        if (kv.first != id) break;
        ++id;
    }
    g_handles[id] = s;
    return id;
}
static std::shared_ptr<BadPixelState> find_handle(int id)
{
    std::lock_guard<std::mutex> lock(g_handles_mutex);
    auto it = g_handles.find(id);
    return it == g_handles.end() ? nullptr : it->second;
}

// A handle's tables live in the memory of the device it was created on: entries that launch kernels refuse a handle
// from another device instead of faulting on its pointers.
static std::shared_ptr<BadPixelState> find_handle_here(int id, const char* what)
{
    auto s = find_handle(id);
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

// ------------------------------------------------------------------------------------------------
// forwarding of out-of-scope entries to a reference build
// ------------------------------------------------------------------------------------------------
static void* forward_symbol(const char* name)
{
    static std::mutex m;
    static void* lib = nullptr;
    static bool tried = false;
    std::lock_guard<std::mutex> lock(m);
    if (!tried) {
        tried = true;
        const char* path = getenv("LIBRIR_B200_FORWARD_LIB");
        if (path && *path) lib = dlopen(path, RTLD_NOW | RTLD_LOCAL);
    }
    if (!lib) {
        set_error("%s is outside the GPU hot path; set LIBRIR_B200_FORWARD_LIB to a reference libsignal_processing.so", name);
        return nullptr;
    }
    void* f = dlsym(lib, name);
    if (!f) set_error("%s not found in LIBRIR_B200_FORWARD_LIB", name);
    return f;
}

}  // namespace rirb

using namespace rirb;

#define RIRB_REQUIRE_DEVICE()            \
    do {                                 \
        if (require_device() != 0) return -1; \
    } while (0)

// =================================================================================================
// runtime
// =================================================================================================
extern "C" {

int rirb_device_count(void)
{
    int n = 0;
    if (cudaGetDeviceCount(&n) != cudaSuccess) {
        cudaGetLastError();
        return 0;
    }
    return n;
}
int rirb_set_device(int device)
{
    RIRB_REQUIRE_DEVICE();
    RIRB_CUDA_OK(cudaSetDevice(device));
    return 0;
}
int rirb_set_stream(void* s)
{
    // The scratch slots belong to the thread, not to the stream, and device-pointer calls return without synchronising: work
    // enqueued on the old stream may still be using them when the next call arrives on the new one.  The new stream is made
    // to wait for the old one (an event, no host synchronisation); errors -- the old stream may be gone -- are ignored.
    const cudaStream_t next = (cudaStream_t)s;
    if (next != tls.stream && tls.enqueued) {
        cudaEvent_t ev = nullptr;
        if (cudaEventCreateWithFlags(&ev, cudaEventDisableTiming) == cudaSuccess) {
            if (cudaEventRecord(ev, tls.stream) == cudaSuccess) (void)cudaStreamWaitEvent(next, ev, 0);
            (void)cudaEventDestroy(ev);
        }
        (void)cudaGetLastError();
    }
    tls.stream = next;
    return 0;
}
int rirb_synchronize(void)
{
    RIRB_REQUIRE_DEVICE();
    RIRB_CUDA_OK(cudaStreamSynchronize(tls.stream));
    tls.enqueued = false;
    return 0;
}
int rirb_set_parameter(const char* key, const char* value)
{
    std::call_once(g_opts_once, init_options);
    if (key && value)
        for (int i = 0; i < OPT_COUNT; ++i)
            if (strcmp(key, k_opt_names[i]) == 0) {
                g_opts[i].store(atoi(value));  // 0 = off; switches with more than two settings take 1, 2, ...
                return 0;
            }
    set_error("set_parameter: unknown key '%s'", key ? key : "(null)");
    return -1;
}
const char* rirb_last_error(void) { return tls.err; }
long long rirb_kernel_launch_count(void) { return g_launches.load(); }
const char* rirb_version(void) { return "librir_b200 0.1 (sm_100a)"; }

// =================================================================================================
// translate
// =================================================================================================
int rirb_translate_batch(int type, const void* src, void* dst, int w, int h, long long nframes, const float* dx, const float* dy,
                         long long n_shifts, const void* background, const char* strategy)
{
    const size_t esize = dtype_size(type);
    const int strat = strategy_code(strategy);
    if (esize == 0 || strat < 0) {
        set_error("translate: unknown %s", esize == 0 ? "dtype code" : "strategy");
        return -1;
    }
    if (!src || !dst || !dx || !dy || !background || w <= 0 || h <= 0 || nframes < 0 || (n_shifts != 1 && n_shifts != nframes)) {
        set_error("translate: bad arguments");
        return -1;
    }
    if (nframes == 0) return 0;
    RIRB_REQUIRE_DEVICE();
    const size_t bytes = (size_t)w * h * esize * (size_t)nframes;
    const size_t sbytes = sizeof(float) * (size_t)n_shifts;
    if (refuse_overlap("translate", {{"src", src, bytes}, {"dx", dx, sbytes}, {"dy", dy, sbytes}}, {{"dst", dst, bytes}})) return -1;
    cudaStream_t st = tls.stream;
    const void* d_src = stage_in(src, bytes, 0, st);
    if (!d_src) return -1;
    StagedOut out;
    if (!stage_out(out, dst, bytes, 1, strat == STRAT_NOBORDER, st)) return -1;
    // background: one element, host or device
    unsigned long long bg = 0;
    if (is_device_ptr(background)) {
        RIRB_CUDA_OK(cudaMemcpyAsync(&bg, background, esize, cudaMemcpyDeviceToHost, st));
        RIRB_CUDA_OK(cudaStreamSynchronize(st));
    } else {
        memcpy(&bg, background, esize);
    }
    const float *d_dx = nullptr, *d_dy = nullptr;
    float dx0 = 0.f, dy0 = 0.f;
    if (n_shifts == 1 && !is_device_ptr(dx) && !is_device_ptr(dy)) {
        dx0 = dx[0];
        dy0 = dy[0];
    } else {
        d_dx = (const float*)stage_in(dx, sizeof(float) * (size_t)n_shifts, 2, st);
        d_dy = (const float*)stage_in(dy, sizeof(float) * (size_t)n_shifts, 3, st);
        if (!d_dx || !d_dy) return -1;
        if (n_shifts == 1 && nframes > 1) {  // broadcast a device-resident scalar shift
            float tmp[2];
            RIRB_CUDA_OK(cudaMemcpyAsync(&tmp[0], d_dx, sizeof(float), cudaMemcpyDeviceToHost, st));
            RIRB_CUDA_OK(cudaMemcpyAsync(&tmp[1], d_dy, sizeof(float), cudaMemcpyDeviceToHost, st));
            RIRB_CUDA_OK(cudaStreamSynchronize(st));
            dx0 = tmp[0];
            dy0 = tmp[1];
            d_dx = d_dy = nullptr;
        }
    }
    if (launch_translate(type, d_src, out.dev, w, h, nframes, d_dx, d_dy, dx0, dy0, strat, &bg, st) != 0) return -1;
    return finish_out(&out, 1, st);
}

int translate(int type, void* src, void* dst, int w, int h, float dx, float dy, void* background, const char* strategy)
{
    return rirb_translate_batch(type, src, dst, w, h, 1, &dx, &dy, 1, background, strategy);
}

// =================================================================================================
// gaussian
// =================================================================================================
static int gaussian_any(const void* src, bool src_u16, float* dst, int w, int h, long long nframes, float sigma)
{
    if (!src || !dst || w <= 0 || h <= 0 || nframes < 0) {
        set_error("gaussian_filter: bad arguments");
        return -1;
    }
    if (nframes == 0) return 0;
    GaussTaps taps;
    if (gaussian_taps_host(sigma, &taps) != 0) return -1;
    RIRB_REQUIRE_DEVICE();
    const size_t npx = (size_t)w * h * (size_t)nframes;
    if (refuse_overlap("gaussian_filter", {{"src", src, npx * (src_u16 ? 2 : 4)}}, {{"dst", dst, npx * 4}})) return -1;
    cudaStream_t st = tls.stream;
    const void* d_src = stage_in(src, npx * (src_u16 ? 2 : 4), 0, st);
    if (!d_src) return -1;
    StagedOut out;
    if (!stage_out(out, dst, npx * 4, 1, false, st)) return -1;
    int rc = src_u16 ? launch_gaussian_u16((const u16*)d_src, (float*)out.dev, w, h, nframes, taps, st)
                     : launch_gaussian_f32((const float*)d_src, (float*)out.dev, w, h, nframes, taps, st);
    if (rc != 0) return -1;
    return finish_out(&out, 1, st);
}

int rirb_gaussian_filter_batch(const float* src, float* dst, int w, int h, long long nframes, float sigma)
{
    return gaussian_any(src, false, dst, w, h, nframes, sigma);
}
int rirb_gaussian_filter_u16_batch(const unsigned short* src, float* dst, int w, int h, long long nframes, float sigma)
{
    return gaussian_any(src, true, dst, w, h, nframes, sigma);
}
int gaussian_filter(float* src, float* dst, int w, int h, float sigma)
{
    // the reference has no failure path here and Python ignores the result
    // (rir_signal_processing.py:103-111); we still report ours.
    return gaussian_any(src, false, dst, w, h, 1, sigma);
}

// =================================================================================================
// bad pixels
// =================================================================================================
int bad_pixels_create(unsigned short* first_image, int width, int height)
{
    if (!first_image || width <= 0 || height <= 0) {
        set_error("bad_pixels_create: bad arguments");
        return 0;
    }
    if (require_device() != 0) return 0;
    cudaStream_t st = tls.stream;
    const size_t n = (size_t)width * height;
    auto fail = [](const char* what) {
        set_error("bad_pixels_create: %s: %s", what, cudaGetErrorString(cudaGetLastError()));
        return 0;
    };
    const u16* d_img = (const u16*)stage_in(first_image, n * 2, 6, st);
    if (!d_img) return 0;
    // (i) frame histogram -> median (sorted[N/2]) and spread, as Filters.h:145-160 / BadPixels.cpp:19-31
    unsigned* d_hist = (unsigned*)scratch(7, 65536 * sizeof(unsigned));
    if (!d_hist) return 0;
    if (launch_hist_frame(d_img, n, d_hist, st) != 0) return 0;
    std::vector<unsigned> hist(65536);
    if (cudaMemcpyAsync(hist.data(), d_hist, 65536 * sizeof(unsigned), cudaMemcpyDeviceToHost, st) != cudaSuccess) return fail("D2H");
    if (cudaStreamSynchronize(st) != cudaSuccess) return fail("sync");
    int median = 0;
    {
        size_t cum = 0;
        const size_t rank = n / 2;  // 0-based index into the sorted frame
        for (int v = 0; v < 65536; ++v) {
            cum += hist[v];
            if (cum > rank) {
                median = v;
                break;
            }
        }
    }
    // Sum of int squares (the reference adds int products into a double, which stays exact below 2^53).  For
    // |d| >= 46341 -- a saturated 65535 pixel over an 8000-count background -- the reference's int product overflows:
    // undefined in C++, a wrap modulo 2^32 in every x86-64 build of it (checked against the compiled reference by the tests, 300 extreme frames).
    // Real movies contain such pixels, so the wrap is reproduced, as are the x86 float->integer conversions below.
    long long ssum = 0;
    for (int v = 0; v < 65536; ++v) {
        const int d = v - median;
        ssum += (long long)(int)((unsigned)d * (unsigned)d) * (long long)hist[v];
    }
    const double gstd = sqrt((double)ssum / (double)(int)n);  // NaN when the wrapped sum is negative
    const double std_factor = 5.0;
    const double cutd = gstd * std_factor;
    // (unsigned short)(double): cvttsd2si to a 32-bit int, low 16 bits kept; NaN / out of int range -> 0x80000000 -> 0
    const unsigned cut = (cutd > -2147483649.0 && cutd < 2147483648.0) ? ((unsigned)(int)cutd & 0xFFFFu) : 0u;
    const unsigned gthr = ((unsigned)median > cut) ? (unsigned)median - cut : 0u;
    const double twice = gstd * 2;
    const int clamp_value = (twice > -2147483649.0 && twice < 2147483648.0) ? median - (int)twice : -1;  // <= 0: no clamp

    auto state = std::make_shared<BadPixelState>();
    state->w = width;
    state->h = height;
    cudaGetDevice(&state->device);
    state->clamp_value = clamp_value;
    state->global_thr = gthr;
    const int mstride = (width + 7) / 8;
    const size_t mbytes = (size_t)mstride * height;
    if (cudaMalloc(&state->mask_dev, mbytes) != cudaSuccess) return fail("cudaMalloc(mask)");
    // (ii) per-pixel 5x5 test -> bitmap
    if (launch_bp_detect(d_img, width, height, std_factor, gthr, state->mask_dev, st) != 0) return 0;
    std::vector<u8> mask(mbytes);
    if (cudaMemcpyAsync(mask.data(), state->mask_dev, mbytes, cudaMemcpyDeviceToHost, st) != cudaSuccess) return fail("D2H(mask)");
    if (cudaStreamSynchronize(st) != cudaSuccess) return fail("sync");
    // raster-ordered list, the order the reference's Polygon has
    for (int y = 0; y < height; ++y)
        for (int xb = 0; xb < mstride; ++xb) {
            unsigned m = mask[(size_t)y * mstride + xb];
            while (m) {
                int b = __builtin_ctz(m);
                m &= m - 1;
                state->xy.push_back(xb * 8 + b);
                state->xy.push_back(y);
            }
        }
    // where each BP_SPAN-pixel span of the frame starts in the (raster-ordered, hence sorted) list
    const size_t nspans = (n + BP_SPAN - 1) / BP_SPAN;
    std::vector<int> span_off(nspans + 1, 0);
    {
        const size_t k = state->xy.size() / 2;
        size_t i = 0;
        for (size_t s = 0; s <= nspans; ++s) {
            const size_t first_px = s * (size_t)BP_SPAN;
            while (i < k && (size_t)state->xy[2 * i + 1] * width + state->xy[2 * i] < first_px) ++i;
            span_off[s] = (int)i;
        }
    }
    if (cudaMalloc(&state->span_off_dev, span_off.size() * sizeof(int)) != cudaSuccess) return fail("cudaMalloc(span offsets)");
    if (cudaMemcpyAsync(state->span_off_dev, span_off.data(), span_off.size() * sizeof(int), cudaMemcpyHostToDevice, st) != cudaSuccess)
        return fail("H2D(span offsets)");
    std::vector<int> nbr, row_off((size_t)height + 1, 0);
    {
        const size_t kk = state->xy.size() / 2;
        size_t i = 0;
        for (int y = 0; y <= height; ++y) {
            while (i < kk && state->xy[2 * i + 1] < y) ++i;
            row_off[y] = (int)i;
        }
        if (cudaMalloc(&state->row_off_dev, row_off.size() * sizeof(int)) != cudaSuccess) return fail("cudaMalloc(row offsets)");
        if (cudaMemcpyAsync(state->row_off_dev, row_off.data(), row_off.size() * sizeof(int), cudaMemcpyHostToDevice, st) != cudaSuccess)
            return fail("H2D(row offsets)");
    }
    if (!state->xy.empty()) {
        if (cudaMalloc(&state->xy_dev, state->xy.size() * sizeof(int)) != cudaSuccess) return fail("cudaMalloc(list)");
        if (cudaMemcpyAsync(state->xy_dev, state->xy.data(), state->xy.size() * sizeof(int), cudaMemcpyHostToDevice, st) !=
            cudaSuccess)
            return fail("H2D(list)");
        // IRFileLoader::removeBadPixels (IRFileLoader.cpp:754-790) skips the flagged cells of its window (shifted
        // inside the image): bit k of nbr[i] = cell (x0 + k/3, y0 + k%3) of entry i's window is flagged
        if (width >= 3 && height >= 3) {
            const size_t kk = state->xy.size() / 2;
            nbr.resize(kk);
            for (size_t i = 0; i < kk; ++i) {
                const int x = state->xy[2 * i], y = state->xy[2 * i + 1];
                const int x0 = x == 0 ? 0 : (x == width - 1 ? width - 3 : x - 1);
                const int y0 = y == 0 ? 0 : (y == height - 1 ? height - 3 : y - 1);
                int bits = 0;
                for (int c = 0; c < 9; ++c) {
                    const int xx = x0 + c / 3, yy = y0 + c % 3;
                    if (mask[(size_t)yy * mstride + (xx >> 3)] & (1u << (xx & 7))) bits |= 1 << c;
                }
                nbr[i] = bits;
            }
            if (cudaMalloc(&state->nbr_dev, kk * sizeof(int)) != cudaSuccess) return fail("cudaMalloc(window flags)");
            if (cudaMemcpyAsync(state->nbr_dev, nbr.data(), kk * sizeof(int), cudaMemcpyHostToDevice, st) != cudaSuccess)
                return fail("H2D(window flags)");
        }
    }
    if (cudaStreamSynchronize(st) != cudaSuccess) return fail("sync");
    return register_handle(state);
}

int rirb_bad_pixels_correct_batch(int handle, const unsigned short* in, unsigned short* out, long long nframes)
{
    auto s = find_handle_here(handle, "bad_pixels_correct");
    if (!s) return -1;
    if (!in || !out || nframes < 0) {
        set_error("bad_pixels_correct: bad arguments");
        return -1;
    }
    if (nframes == 0) return 0;
    RIRB_REQUIRE_DEVICE();
    cudaStream_t st = tls.stream;
    const size_t fpx = (size_t)s->w * s->h;
    const size_t bytes = fpx * 2 * (size_t)nframes;
    if (in != out && refuse_overlap("bad_pixels_correct", {{"in", in, bytes}}, {{"out", out, bytes}})) return -1;
    if (in == out) {  // sequential in-place meaning of the reference (BadPixels.cpp:41-59)
        StagedOut io;
        if (!stage_out(io, out, bytes, 0, true, st)) return -1;
        if (launch_bp_correct_inplace((u16*)io.dev, s->xy_dev, (int)(s->xy.size() / 2), s->w, s->h, s->clamp_value, nframes, fpx,
                                      st) != 0)
            return -1;
        return finish_out(&io, 1, st);
    }
    const u16* d_in = (const u16*)stage_in(in, bytes, 0, st);
    if (!d_in) return -1;
    StagedOut o;
    if (!stage_out(o, out, bytes, 1, false, st)) return -1;
    if (launch_bp_correct(d_in, (u16*)o.dev, s->xy_dev, s->span_off_dev, s->w, s->h, s->clamp_value, nframes, fpx, st) != 0) return -1;
    return finish_out(&o, 1, st);
}

// bad_pixels_correct + gaussian_filter of the corrected frames, reading the movie once (gaussian.cu, BpFuse):
// corrected[n][h][w] uint16 and smoothed[n][h][w] float32 are both produced.  Layouts the tiled kernel cannot take
// (w % 8 != 0, unaligned buffers, radius > 4) run the two kernels instead; results are the same either way.
int rirb_bad_pixels_correct_gaussian_batch(int handle, const unsigned short* in, unsigned short* corrected, float* smoothed,
                                           long long nframes, float sigma)
{
    auto s = find_handle_here(handle, "bad_pixels_correct_gaussian");
    if (!s) return -1;
    if (!in || !corrected || !smoothed || nframes < 0) {
        set_error("bad_pixels_correct_gaussian: bad arguments");
        return -1;
    }
    if (nframes == 0) return 0;
    GaussTaps taps;
    if (gaussian_taps_host(sigma, &taps) != 0) return -1;
    RIRB_REQUIRE_DEVICE();
    cudaStream_t st = tls.stream;
    const size_t fpx = (size_t)s->w * s->h;
    // in place is not supported here: the filter reads corrected pixels of neighbouring rows that the correction of other
    // blocks may not have written yet
    if (refuse_overlap("bad_pixels_correct_gaussian", {{"in", in, fpx * 2 * (size_t)nframes}},
                       {{"corrected", corrected, fpx * 2 * (size_t)nframes}, {"smoothed", smoothed, fpx * 4 * (size_t)nframes}}))
        return -1;
    const u16* d_in = (const u16*)stage_in(in, fpx * 2 * (size_t)nframes, 0, st);
    if (!d_in) return -1;
    StagedOut o[2];
    if (!stage_out(o[0], corrected, fpx * 2 * (size_t)nframes, 1, false, st)) return -1;
    if (!stage_out(o[1], smoothed, fpx * 4 * (size_t)nframes, 2, false, st)) return -1;
    const int rc = launch_gaussian_bp_u16(d_in, (u16*)o[0].dev, (float*)o[1].dev, s->w, s->h, nframes, taps, s->xy_dev, s->row_off_dev,
                                          s->clamp_value, st);
    if (rc < 0) return -1;
    if (rc == 1) {
        if (launch_bp_correct(d_in, (u16*)o[0].dev, s->xy_dev, s->span_off_dev, s->w, s->h, s->clamp_value, nframes, fpx, st) != 0 ||
            launch_gaussian_u16((const u16*)o[0].dev, (float*)o[1].dev, s->w, s->h, nframes, taps, st) != 0)
            return -1;
    }
    return finish_out(o, 2, st);
}

int bad_pixels_correct(int handle, unsigned short* in, unsigned short* out)
{
    return rirb_bad_pixels_correct_batch(handle, in, out, 1);
}

void bad_pixels_destroy(int handle)
{
    std::lock_guard<std::mutex> lock(g_handles_mutex);
    g_handles.erase(handle);
}

int rirb_bad_pixels_count(int handle)
{
    auto s = find_handle(handle);
    if (!s) {
        set_error("bad_pixels: unknown handle %d", handle);
        return -1;
    }
    return (int)(s->xy.size() / 2);
}

int rirb_bad_pixels_get(int handle, int* xy, int capacity, int* clamp_value)
{
    auto s = find_handle(handle);
    if (!s) {
        set_error("bad_pixels: unknown handle %d", handle);
        return -1;
    }
    const int k = (int)(s->xy.size() / 2);
    if (clamp_value) *clamp_value = s->clamp_value;
    if (xy) {
        if (capacity < k) return -2;  // "output too small" convention, signal_processing.h:52
        memcpy(xy, s->xy.data(), s->xy.size() * sizeof(int));
    }
    return k;
}

int rirb_loader_remove_bad_pixels(int handle, unsigned short* frames, long long nframes, size_t frame_stride)
{
    auto s = find_handle_here(handle, "remove_bad_pixels");
    if (!s) return -1;
    if (!frames || nframes < 0 || frame_stride < (size_t)s->w * s->h) {
        set_error("remove_bad_pixels: bad arguments");
        return -1;
    }
    if (nframes == 0) return 0;
    RIRB_REQUIRE_DEVICE();
    cudaStream_t st = tls.stream;
    StagedOut io;
    if (!stage_out(io, frames, frame_stride * 2 * (size_t)nframes, 0, true, st)) return -1;
    if (launch_loader_bp((u16*)io.dev, s->xy_dev, s->mask_dev, (int)(s->xy.size() / 2), s->w, s->h, nframes, frame_stride, st) != 0)
        return -1;
    return finish_out(&io, 1, st);
}

// =================================================================================================
// motion-correction variant
// =================================================================================================
int rirb_loader_remove_motion(const unsigned short* in, unsigned short* out, int w, int h, long long nframes, size_t frame_stride,
                              const double* shift_x, const double* shift_y)
{
    if (!in || !out || !shift_x || !shift_y || w <= 0 || h <= 0 || nframes < 0 || frame_stride < (size_t)w * h) {
        set_error("remove_motion: bad arguments");
        return -1;
    }
    if (nframes == 0) return 0;
    RIRB_REQUIRE_DEVICE();
    const size_t bytes = frame_stride * 2 * (size_t)nframes;
    if (in != out && refuse_overlap("remove_motion", {{"in", in, bytes}}, {{"out", out, bytes}})) return -1;
    cudaStream_t st = tls.stream;
    // shifts: doubles on the host (PointF), negated and narrowed to float as the reference's call does
    std::vector<double> sx((size_t)nframes), sy((size_t)nframes);
    if (is_device_ptr(shift_x) || is_device_ptr(shift_y)) {
        RIRB_CUDA_OK(cudaMemcpyAsync(sx.data(), shift_x, sizeof(double) * nframes, cudaMemcpyDefault, st));
        RIRB_CUDA_OK(cudaMemcpyAsync(sy.data(), shift_y, sizeof(double) * nframes, cudaMemcpyDefault, st));
        RIRB_CUDA_OK(cudaStreamSynchronize(st));
    } else {
        memcpy(sx.data(), shift_x, sizeof(double) * nframes);
        memcpy(sy.data(), shift_y, sizeof(double) * nframes);
    }
    std::vector<float> fx((size_t)nframes), fy((size_t)nframes);
    for (long long i = 0; i < nframes; ++i) {
        fx[i] = (float)(-sx[i]);
        fy[i] = (float)(-sy[i]);
    }
    const float* d_dx = (const float*)stage_in(fx.data(), sizeof(float) * nframes, 2, st);
    const float* d_dy = (const float*)stage_in(fy.data(), sizeof(float) * nframes, 3, st);
    if (!d_dx || !d_dy) return -1;
    const bool inplace = (in == out);
    const u16* d_in;
    StagedOut o;
    if (inplace) {
        // the reference translates into a temporary and copies back; keep a private copy of the input
        if (!stage_out(o, out, bytes, 1, true, st)) return -1;
        void* copy = scratch(0, bytes);
        if (!copy) return -1;
        RIRB_CUDA_OK(cudaMemcpyAsync(copy, o.dev, bytes, cudaMemcpyDeviceToDevice, st));
        d_in = (const u16*)copy;
    } else {
        d_in = (const u16*)stage_in(in, bytes, 0, st);
        if (!d_in) return -1;
        if (!stage_out(o, out, bytes, 1, false, st)) return -1;
        if (frame_stride > (size_t)w * h)  // pass the untouched tail rows through
            RIRB_CUDA_OK(cudaMemcpy2DAsync((u16*)o.dev + (size_t)w * h, frame_stride * 2, d_in + (size_t)w * h, frame_stride * 2,
                                           (frame_stride - (size_t)w * h) * 2, (size_t)nframes, cudaMemcpyDeviceToDevice, st));
    }
    if (launch_translate_u16(d_in, (u16*)o.dev, w, h, nframes, frame_stride, frame_stride, d_dx, d_dy, 0.f, 0.f, STRAT_NEAREST, 0u,
                             true, st) != 0)
        return -1;
    if (o.host) {
        RIRB_CUDA_OK(copy_d2h(o.host, o.dev, bytes, st));
    }
    // fx/fy are stack-owned host vectors read by an async copy: always wait before returning
    RIRB_CUDA_OK(cudaStreamSynchronize(st));
    return 0;
}

// =================================================================================================
// reader's post-decode chain
// =================================================================================================
int rirb_loader_read_movie(int handle, const unsigned char* lo, const unsigned char* hi, long long nframes, int w, int h, int min_T,
                           int min_T_height, const double* shift_x, const double* shift_y, int meta_rows, unsigned short* out)
{
    if (!lo || !hi || !out || w <= 0 || h <= 0 || nframes < 0 || meta_rows < 0 || meta_rows >= h || (!shift_x) != (!shift_y)) {
        set_error("loader_read_movie: bad arguments");
        return -1;
    }
    if (nframes == 0) return 0;
    const int hb = h - meta_rows;
    // an absent / zero MIN_T_HEIGHT means "every row but the metadata rows" (IRFileLoader::open, IRFileLoader.cpp:918-921)
    if (min_T_height == 0) min_T_height = hb;
    std::shared_ptr<BadPixelState> s;
    if (handle != 0) {
        s = find_handle_here(handle, "loader_read_movie");
        if (!s) return -1;
        if (s->w != w || s->h != hb) {
            set_error("loader_read_movie: the handle was created on a %dx%d image, expected %dx%d", s->w, s->h, w, hb);
            return -1;
        }
    }
    RIRB_REQUIRE_DEVICE();
    cudaStream_t st = tls.stream;
    const size_t fpx = (size_t)w * h;
    const size_t pbytes = fpx * (size_t)nframes;
    if (refuse_overlap("loader_read_movie", {{"lo", lo, pbytes}, {"hi", hi, pbytes}}, {{"out", out, pbytes * 2}})) return -1;
    const u8* d_lo = (const u8*)stage_in(lo, pbytes, 0, st);
    const u8* d_hi = (const u8*)stage_in(hi, pbytes, 1, st);
    if (!d_lo || !d_hi) return -1;
    StagedOut o;
    if (!stage_out(o, out, pbytes * 2, 2, false, st)) return -1;
    const bool motion = shift_x != nullptr;
    const int k = s ? (int)(s->xy.size() / 2) : 0;
    const bool fused_bp = s && k > 0 && w >= 3 && hb >= 3;
    if (!motion) {
        u16* merged = (u16*)o.dev;
        if (launch_loader_merge(d_lo, d_hi, merged, w, h, hb, nframes, fpx, min_T, min_T_height, fused_bp ? s->xy_dev : nullptr,
                                fused_bp ? s->span_off_dev : nullptr, fused_bp ? s->nbr_dev : nullptr, st) != 0)
            return -1;
        if (s && k > 0 && !fused_bp)  // degenerate sizes keep the reference's sequential loop (IRFileLoader.cpp:735-752)
            if (launch_loader_bp(merged, s->xy_dev, s->mask_dev, k, w, hb, nframes, fpx, st) != 0) return -1;
        return finish_out(&o, 1, st);
    }
    // shifts: translate(..., -x[pos], -y[pos], ...) with float arguments (IRFileLoader.cpp:621)
    std::vector<double> sx((size_t)nframes), sy((size_t)nframes);
    if (is_device_ptr(shift_x) || is_device_ptr(shift_y)) {
        RIRB_CUDA_OK(cudaMemcpyAsync(sx.data(), shift_x, sizeof(double) * nframes, cudaMemcpyDefault, st));
        RIRB_CUDA_OK(cudaMemcpyAsync(sy.data(), shift_y, sizeof(double) * nframes, cudaMemcpyDefault, st));
        RIRB_CUDA_OK(cudaStreamSynchronize(st));
    } else {
        memcpy(sx.data(), shift_x, sizeof(double) * nframes);
        memcpy(sy.data(), shift_y, sizeof(double) * nframes);
    }
    std::vector<float> fx((size_t)nframes), fy((size_t)nframes);
    for (long long i = 0; i < nframes; ++i) {
        fx[i] = (float)(-sx[i]);
        fy[i] = (float)(-sy[i]);
    }
    const float* d_dx = (const float*)stage_in(fx.data(), sizeof(float) * nframes, 4, st);
    const float* d_dy = (const float*)stage_in(fy.data(), sizeof(float) * nframes, 5, st);
    if (!d_dx || !d_dy) return -1;
    // one pass: planes -> merge -> += min_T -> medians -> motion translate (translate.cu, PLANES)
    const int rows_t = (min_T == 0 || min_T_height < 0) ? 0 : (min_T_height > h ? h : min_T_height);
    int rc = (s && k > 0 && !fused_bp)
                 ? 1
                 : launch_loader_fused(d_lo, d_hi, (u16*)o.dev, w, h, hb, nframes, min_T, rows_t, fused_bp ? s->xy_dev : nullptr,
                                       fused_bp ? s->nbr_dev : nullptr, fused_bp ? s->row_off_dev : nullptr,
                                       fused_bp ? s->mask_dev : nullptr, d_dx, d_dy, st);
    if (rc < 0) return -1;
    if (rc == 1) {  // layouts the fused kernel does not take: merge pass, then the motion pass through a scratch movie
        u16* merged = (u16*)scratch(3, pbytes * 2);
        if (!merged) return -1;
        if (launch_loader_merge(d_lo, d_hi, merged, w, h, hb, nframes, fpx, min_T, min_T_height, fused_bp ? s->xy_dev : nullptr,
                                fused_bp ? s->span_off_dev : nullptr, fused_bp ? s->nbr_dev : nullptr, st) != 0)
            return -1;
        if (s && k > 0 && !fused_bp)
            if (launch_loader_bp(merged, s->xy_dev, s->mask_dev, k, w, hb, nframes, fpx, st) != 0) return -1;
        if (meta_rows > 0)  // the metadata rows are not translated
            RIRB_CUDA_OK(cudaMemcpy2DAsync((u16*)o.dev + (size_t)w * hb, fpx * 2, merged + (size_t)w * hb, fpx * 2,
                                           (size_t)w * meta_rows * 2, (size_t)nframes, cudaMemcpyDeviceToDevice, st));
        if (launch_translate_u16(merged, (u16*)o.dev, w, hb, nframes, fpx, fpx, d_dx, d_dy, 0.f, 0.f, STRAT_NEAREST, 0u, true, st) != 0)
            return -1;
    }
    if (o.host) RIRB_CUDA_OK(copy_d2h(o.host, o.dev, o.bytes, st));
    RIRB_CUDA_OK(cudaStreamSynchronize(st));  // fx / fy are host vectors read by an async copy
    return 0;
}

// The same chain for frames that are uint16 already (decoded from the zstd movie file): += min_T -> removeBadPixels ->
// removeMotion, in place.
int rirb_loader_finish_frames(int handle, unsigned short* frames, long long nframes, int w, int h, int min_T, int min_T_height,
                              const double* shift_x, const double* shift_y, int meta_rows)
{
    if (!frames || w <= 0 || h <= 0 || nframes < 0 || meta_rows < 0 || meta_rows >= h || (!shift_x) != (!shift_y)) {
        set_error("loader_finish_frames: bad arguments");
        return -1;
    }
    if (nframes == 0) return 0;
    const int hb = h - meta_rows;
    if (min_T_height == 0) min_T_height = hb;  // IRFileLoader.cpp:918-921
    std::shared_ptr<BadPixelState> s;
    if (handle != 0) {
        s = find_handle_here(handle, "loader_finish_frames");
        if (!s) return -1;
        if (s->w != w || s->h != hb) {
            set_error("loader_finish_frames: the handle was created on a %dx%d image, expected %dx%d", s->w, s->h, w, hb);
            return -1;
        }
    }
    RIRB_REQUIRE_DEVICE();
    cudaStream_t st = tls.stream;
    const size_t fpx = (size_t)w * h;
    StagedOut io;
    if (!stage_out(io, frames, fpx * 2 * (size_t)nframes, 0, true, st)) return -1;
    u16* d = (u16*)io.dev;
    const int rows_t = (min_T == 0 || min_T_height < 0) ? 0 : (min_T_height > h ? h : min_T_height);
    if (launch_loader_add_min(d, w, rows_t, nframes, fpx, min_T, st) != 0) return -1;
    if (s && !s->xy.empty())
        if (launch_loader_bp(d, s->xy_dev, s->mask_dev, (int)(s->xy.size() / 2), w, hb, nframes, fpx, st) != 0) return -1;
    if (shift_x) {
        // the motion step is out of place: through a scratch copy, on device pointers (no further staging)
        u16* tmp = (u16*)scratch(4, fpx * 2 * (size_t)nframes);  // not 0-3: rirb_loader_remove_motion stages its shifts there
        if (!tmp) return -1;
        RIRB_CUDA_OK(cudaMemcpyAsync(tmp, d, fpx * 2 * (size_t)nframes, cudaMemcpyDeviceToDevice, st));
        if (rirb_loader_remove_motion(tmp, d, w, hb, nframes, fpx, shift_x, shift_y) != 0) return -1;
    }
    return finish_out(&io, 1, st);
}

// =================================================================================================
// pre-coder
// =================================================================================================
int rirb_split_yuv444(const unsigned short* img, const unsigned char* it, int w, int h, unsigned char* y_plane,
                      unsigned char* u_plane, unsigned char* v_plane, int ls_y, int ls_u, int ls_v)
{
    if (!img || !u_plane || !v_plane || w <= 0 || h <= 0 || ls_u < w || ls_v < w || (y_plane && ls_y < w)) {
        set_error("split_yuv444: bad arguments");
        return -1;
    }
    RIRB_REQUIRE_DEVICE();
    if (refuse_overlap("split_yuv444", {{"img", img, (size_t)w * h * 2}, {"it", it, (size_t)w * h}},
                       {{"y_plane", y_plane, (size_t)ls_y * h}, {"u_plane", u_plane, (size_t)ls_u * h}, {"v_plane", v_plane, (size_t)ls_v * h}}))
        return -1;
    cudaStream_t st = tls.stream;
    const u16* d_img = (const u16*)stage_in(img, (size_t)w * h * 2, 0, st);
    if (!d_img) return -1;
    const u8* d_it = nullptr;
    if (it) {
        d_it = (const u8*)stage_in(it, (size_t)w * h, 1, st);
        if (!d_it) return -1;
    }
    StagedOut o[3];
    // row padding must survive untouched: preload padded planes
    if (!stage_out(o[1], u_plane, (size_t)ls_u * h, 3, ls_u != w, st)) return -1;
    if (!stage_out(o[2], v_plane, (size_t)ls_v * h, 4, ls_v != w, st)) return -1;
    if (y_plane && !stage_out(o[0], y_plane, (size_t)ls_y * h, 2, ls_y != w, st)) return -1;
    if (launch_split_planes(d_img, d_it, w, h, (u8*)o[0].dev, (u8*)o[1].dev, (u8*)o[2].dev, ls_y, ls_u, ls_v, st) != 0) return -1;
    return finish_out(o, 3, st);
}

int rirb_merge_yuv444(const unsigned char* y_plane, const unsigned char* u_plane, const unsigned char* v_plane, int ls_y, int ls_u,
                      int ls_v, int w, int h, unsigned short* img, unsigned char* it)
{
    if (!img || !u_plane || !v_plane || w <= 0 || h <= 0 || ls_u < w || ls_v < w) {
        set_error("merge_yuv444: bad arguments");
        return -1;
    }
    RIRB_REQUIRE_DEVICE();
    if (refuse_overlap("merge_yuv444",
                       {{"y_plane", it ? y_plane : nullptr, (size_t)ls_y * h}, {"u_plane", u_plane, (size_t)ls_u * h}, {"v_plane", v_plane, (size_t)ls_v * h}},
                       {{"img", img, (size_t)w * h * 2}, {"it", y_plane ? it : nullptr, (size_t)w * h}}))
        return -1;
    cudaStream_t st = tls.stream;
    const u8* d_u = (const u8*)stage_in(u_plane, (size_t)ls_u * h, 0, st);
    const u8* d_v = (const u8*)stage_in(v_plane, (size_t)ls_v * h, 1, st);
    if (!d_u || !d_v) return -1;
    const u8* d_y = nullptr;
    if (y_plane && it) {
        d_y = (const u8*)stage_in(y_plane, (size_t)ls_y * h, 2, st);
        if (!d_y) return -1;
    }
    StagedOut o[2];
    if (!stage_out(o[0], img, (size_t)w * h * 2, 3, false, st)) return -1;
    if (it && d_y && !stage_out(o[1], it, (size_t)w * h, 4, false, st)) return -1;
    if (launch_merge_planes(d_y, d_u, d_v, ls_y, ls_u, ls_v, w, h, (u16*)o[0].dev, (u8*)o[1].dev, st) != 0) return -1;
    return finish_out(o, 2, st);
}

int rirb_split_yuv420(const unsigned short* img, const unsigned char* it, int w, int h, unsigned char* y_plane, int ls_y,
                      unsigned char* u_plane, int ls_u)
{
    if (!img || !y_plane || w <= 0 || h <= 0 || ls_y < w) {
        set_error("split_yuv420: bad arguments");
        return -1;
    }
    RIRB_REQUIRE_DEVICE();
    const bool with_it = it && u_plane;
    if (refuse_overlap("split_yuv420", {{"img", img, (size_t)w * h * 2}, {"it", with_it ? it : nullptr, (size_t)w * h}},
                       {{"y_plane", y_plane, (size_t)ls_y * 2 * h}, {"u_plane", with_it ? u_plane : nullptr, (size_t)ls_u * h}}))
        return -1;
    cudaStream_t st = tls.stream;
    const u16* d_img = (const u16*)stage_in(img, (size_t)w * h * 2, 0, st);
    if (!d_img) return -1;
    const u8* d_it = nullptr;
    if (with_it) {
        d_it = (const u8*)stage_in(it, (size_t)w * h, 1, st);
        if (!d_it) return -1;
    }
    StagedOut o[2];
    if (!stage_out(o[0], y_plane, (size_t)ls_y * 2 * h, 2, ls_y != w, st)) return -1;
    if (with_it && !stage_out(o[1], u_plane, (size_t)ls_u * h, 3, ls_u != w, st)) return -1;
    u8* d_y = (u8*)o[0].dev;
    if (launch_split_planes(d_img, d_it, w, h, with_it ? (u8*)o[1].dev : nullptr, d_y, d_y + (size_t)h * ls_y, ls_u, ls_y, ls_y,
                            st) != 0)
        return -1;
    return finish_out(o, 2, st);
}

int rirb_merge_yuv420(const unsigned char* y_plane, int ls_y, const unsigned char* u_plane, int ls_u, int w, int h,
                      unsigned short* img, unsigned char* it)
{
    if (!img || !y_plane || w <= 0 || h <= 0 || ls_y < w) {
        set_error("merge_yuv420: bad arguments");
        return -1;
    }
    RIRB_REQUIRE_DEVICE();
    const bool with_it = it && u_plane;
    if (refuse_overlap("merge_yuv420", {{"y_plane", y_plane, (size_t)ls_y * 2 * h}, {"u_plane", with_it ? u_plane : nullptr, (size_t)ls_u * h}},
                       {{"img", img, (size_t)w * h * 2}, {"it", with_it ? it : nullptr, (size_t)w * h}}))
        return -1;
    cudaStream_t st = tls.stream;
    const u8* d_yp = (const u8*)stage_in(y_plane, (size_t)ls_y * 2 * h, 0, st);
    if (!d_yp) return -1;
    const u8* d_up = nullptr;
    if (with_it) {
        d_up = (const u8*)stage_in(u_plane, (size_t)ls_u * h, 1, st);
        if (!d_up) return -1;
    }
    StagedOut o[2];
    if (!stage_out(o[0], img, (size_t)w * h * 2, 2, false, st)) return -1;
    if (with_it && !stage_out(o[1], it, (size_t)w * h, 3, false, st)) return -1;
    if (launch_merge_planes(d_up, d_yp, d_yp + (size_t)h * ls_y, ls_u, ls_y, ls_y, w, h, (u16*)o[0].dev, (u8*)o[1].dev, st) != 0)
        return -1;
    return finish_out(o, 2, st);
}

int rirb_precode_movie(const unsigned short* movie, long long nframes, int w, int h, int gop, int delta, long long first_frame,
                       unsigned char* lo, unsigned char* hi)
{
    if (!movie || !lo || !hi || w <= 0 || h <= 0 || nframes < 0 || gop < 1) {
        set_error("precode_movie: bad arguments");
        return -1;
    }
    if (nframes == 0) return 0;
    RIRB_REQUIRE_DEVICE();
    cudaStream_t st = tls.stream;
    const size_t n = (size_t)w * h * (size_t)nframes;
    if (refuse_overlap("precode_movie", {{"movie", movie, n * 2}}, {{"lo", lo, n}, {"hi", hi, n}})) return -1;
    const u16* d_mov = (const u16*)stage_in(movie, n * 2, 0, st);
    if (!d_mov) return -1;
    StagedOut o[2];
    if (!stage_out(o[0], lo, n, 1, false, st) || !stage_out(o[1], hi, n, 2, false, st)) return -1;
    if (launch_precode_movie(d_mov, nframes, w, h, gop, delta, first_frame, (u8*)o[0].dev, (u8*)o[1].dev, st) != 0) return -1;
    return finish_out(o, 2, st);
}

int rirb_precode_movie_stats(const unsigned short* movie, long long nframes, int w, int h, int gop, int delta, long long first_frame,
                             unsigned char* lo, unsigned char* hi, unsigned int* minmax, unsigned long long* hist, int accumulate)
{
    if (!movie || !lo || !hi || !minmax || !hist || w <= 0 || h <= 0 || nframes < 0 || gop < 1) {
        set_error("precode_movie_stats: bad arguments");
        return -1;
    }
    if (nframes == 0) return 0;
    RIRB_REQUIRE_DEVICE();
    cudaStream_t st = tls.stream;
    const size_t n = (size_t)w * h * (size_t)nframes;
    if (refuse_overlap("precode_movie_stats", {{"movie", movie, n * 2}},
                       {{"lo", lo, n}, {"hi", hi, n}, {"minmax", minmax, 2 * sizeof(unsigned)}, {"hist", hist, 65536 * sizeof(unsigned long long)}}))
        return -1;
    const u16* d_mov = (const u16*)stage_in(movie, n * 2, 0, st);
    if (!d_mov) return -1;
    StagedOut o[4];
    if (!stage_out(o[0], lo, n, 1, false, st) || !stage_out(o[1], hi, n, 2, false, st)) return -1;
    if (!stage_out(o[2], minmax, 2 * sizeof(unsigned), 3, accumulate != 0, st)) return -1;
    if (!stage_out(o[3], hist, 65536 * sizeof(unsigned long long), 4, accumulate != 0, st)) return -1;
    if (!accumulate && launch_stats_init((unsigned*)o[2].dev, (unsigned long long*)o[3].dev, st) != 0) return -1;
    const int rc = launch_precode_movie_stats(d_mov, nframes, w, h, gop, delta, first_frame, (u8*)o[0].dev, (u8*)o[1].dev,
                                              (unsigned*)o[2].dev, (unsigned long long*)o[3].dev, st);
    if (rc < 0) return -1;
    if (rc == 1) {  // layouts the fused kernel does not take: the two kernels
        if (launch_precode_movie(d_mov, nframes, w, h, gop, delta, first_frame, (u8*)o[0].dev, (u8*)o[1].dev, st) != 0) return -1;
        if (launch_movie_stats(d_mov, n, nullptr, (unsigned*)o[2].dev, (unsigned long long*)o[3].dev, st) != 0) return -1;
    }
    return finish_out(o, 4, st);
}

int rirb_decode_movie(const unsigned char* lo, const unsigned char* hi, long long nframes, int w, int h, int gop, int delta,
                      long long first_frame, unsigned short* movie)
{
    if (!movie || !lo || !hi || w <= 0 || h <= 0 || nframes < 0 || gop < 1) {
        set_error("decode_movie: bad arguments");
        return -1;
    }
    if (nframes == 0) return 0;
    RIRB_REQUIRE_DEVICE();
    cudaStream_t st = tls.stream;
    const size_t n = (size_t)w * h * (size_t)nframes;
    if (refuse_overlap("decode_movie", {{"lo", lo, n}, {"hi", hi, n}}, {{"movie", movie, n * 2}})) return -1;
    const u8* d_lo = (const u8*)stage_in(lo, n, 0, st);
    const u8* d_hi = (const u8*)stage_in(hi, n, 1, st);
    if (!d_lo || !d_hi) return -1;
    StagedOut o;
    if (!stage_out(o, movie, n * 2, 2, false, st)) return -1;
    if (launch_decode_movie(d_lo, d_hi, nframes, w, h, gop, delta, first_frame, (u16*)o.dev, st) != 0) return -1;
    return finish_out(&o, 1, st);
}

// host-side writer logic, no device involved: AddFrame's key-frame decision (h264.cpp:1050-1061)
int rirb_key_frames(long long nframes, int gop, unsigned char* key)
{
    if (!key || nframes < 0) {
        set_error("key_frames: bad arguments");
        return -1;
    }
    long long last = 0;
    for (long long n = 0; n < nframes; ++n) {
        const bool k = (n == 0) || (n - last >= gop);
        if (k) last = n;
        key[n] = k ? 1 : 0;
    }
    return 0;
}

// =================================================================================================
// lossy pre-conditioner (stateful, frames in time order)
// =================================================================================================
namespace {
struct LossyState {
    int w = 0, h = 0, stop_h = 0, low = 6, high = 2, ra = 32, subtract_min = 0, bp_enabled = 0, device = 0;
    int variant = 0;      // 0 = addImageLossyNoCamera (h264_add_image_lossy), 1 = addLoss (h264_add_loss)
    int quirk = 1;        // the compiled reference's overlapping memcpy of the spread window (lossy.cu, lossy_window_quirk)
    unsigned* hist_scratch = nullptr;  // lossy_back_kernel's per-frame histograms
    bool use_run = true;  // several frames per cooperative launch; cleared if the device cannot do it (or by "lossy_run" = 0)
    double std_factor = 5.0;
    long long frames = 0;
    int bp_handle = 0;
    char* buf = nullptr;  // one allocation: lastDL | refT | prevT | tmp | tmpT | sums | cvalue | ccount | ring | scalars | errors
    size_t o_lastDL = 0, o_refT = 0, o_prevT = 0, o_tmp = 0, o_tmpT = 0, o_sums = 0, o_cval = 0, o_ccnt = 0, o_ring = 0, o_scal = 0;
    int* errors_dev = nullptr;
    long long errors_cap = 0;
    u16* cur_batch = nullptr;  // bad-pixel-corrected copies of a run of frames (lossy_run_kernel), when that is enabled
    size_t cur_batch_frames = 0;
    ~LossyState()
    {
        if (cur_batch) cudaFree(cur_batch);
        if (hist_scratch) cudaFree(hist_scratch);
        if (buf) cudaFree(buf);
        if (errors_dev) cudaFree(errors_dev);
        if (bp_handle) bad_pixels_destroy(bp_handle);
    }
};
std::mutex g_lossy_mutex;
std::map<int, std::shared_ptr<LossyState>> g_lossy;
}  // namespace

int rirb_lossy_open(int w, int h, int stop_lossy_height, int low_error, int high_error, double std_factor, int running_average,
                    int subtract_min, int remove_bad_pixels)
{
    if (w <= 0 || h <= 0 || stop_lossy_height < 0 || stop_lossy_height > h || running_average < 0 || (long long)w * h > 0x7FFFFFFFLL) {
        set_error("lossy_open: bad arguments");
        return 0;
    }
    if (require_device() != 0) return 0;
    auto s = std::make_shared<LossyState>();
    s->w = w; s->h = h; s->stop_h = stop_lossy_height;
    s->low = low_error; s->high = high_error; s->std_factor = std_factor;
    s->ra = running_average > 64 ? 64 : running_average;  // setParameter clamps to 64 (h264.cpp:1774)
    s->subtract_min = subtract_min != 0; s->bp_enabled = remove_bad_pixels != 0;
    cudaGetDevice(&s->device);
    const size_t n = (size_t)w * h, ns = (size_t)w * stop_lossy_height;
    auto al = [](size_t v) { return (v + 255) & ~(size_t)255; };
    size_t off = 0;
    s->o_lastDL = off; off += al(n * 2);
    s->o_refT = off; off += al(n * 2);
    s->o_prevT = off; off += al(n * 2);
    s->o_tmp = off; off += al(n * 2);
    s->o_tmpT = off; off += al(n * 2);
    s->o_sums = off; off += al(ns * 4 + 4);
    s->o_cval = off; off += al(ns * 2 + 2);
    s->o_ccnt = off; off += al(ns * 2 + 2);
    s->o_ring = off; off += al(ns * 2 * (size_t)(s->ra > 0 ? s->ra : 1) + 2);
    s->o_scal = off; off += al(lossy_scalars_bytes());
    if (cudaMalloc(&s->buf, off) != cudaSuccess || cudaMemset(s->buf, 0, off) != cudaSuccess) {
        set_error("lossy_open: out of device memory (%zu bytes): %s", off, cudaGetErrorString(cudaGetLastError()));
        return 0;
    }
    std::lock_guard<std::mutex> lock(g_lossy_mutex);
    int id = 1;
    for (auto& kv : g_lossy) {
        if (kv.first != id) break;
        ++id;
    }
    g_lossy[id] = s;
    return id;
}

void rirb_lossy_close(int handle)
{
    std::lock_guard<std::mutex> lock(g_lossy_mutex);
    g_lossy.erase(handle);
}

int rirb_lossy_set_parameter(int handle, const char* key, const char* value)
{
    std::shared_ptr<LossyState> s;
    {
        std::lock_guard<std::mutex> lock(g_lossy_mutex);
        auto it = g_lossy.find(handle);
        if (it != g_lossy.end()) s = it->second;
    }
    if (!s || !key || !value) {
        set_error("lossy_set_parameter: unknown handle %d or NULL argument", handle);
        return -1;
    }
    const std::string k(key), v(value);
    if (k == "variant") {
        if (s->frames != 0) {
            set_error("lossy_set_parameter: the variant cannot change once frames were added");
            return -1;
        }
        if (v == "add_image_lossy" || v == "0") s->variant = 0;
        else if (v == "add_loss" || v == "1") s->variant = 1;
        else {
            set_error("lossy_set_parameter: variant must be add_image_lossy or add_loss");
            return -1;
        }
        return 0;
    }
    if (k == "memcpyQuirk") {
        s->quirk = atoi(value) != 0;
        return 0;
    }
    set_error("lossy_set_parameter: unknown key %s", key);
    return -1;
}

int rirb_lossy_get_min(int handle, int* min_value)
{
    std::shared_ptr<LossyState> s;
    {
        std::lock_guard<std::mutex> lock(g_lossy_mutex);
        auto it = g_lossy.find(handle);
        if (it != g_lossy.end()) s = it->second;
    }
    if (!s || !min_value) {
        set_error("lossy_get_min: unknown handle %d", handle);
        return -1;
    }
    *min_value = 0;
    if (!s->subtract_min || s->frames == 0) return 0;
    unsigned m = 0;  // LossyScalars starts with m_data->min
    RIRB_CUDA_OK(cudaMemcpyAsync(&m, s->buf + s->o_scal, sizeof(unsigned), cudaMemcpyDeviceToHost, tls.stream));
    RIRB_CUDA_OK(cudaStreamSynchronize(tls.stream));
    *min_value = (int)m;
    return 0;
}

int rirb_lossy_add_images(int handle, const unsigned short* frames, long long nframes, unsigned short* out, int* errors)
{
    std::shared_ptr<LossyState> s;
    {
        std::lock_guard<std::mutex> lock(g_lossy_mutex);
        auto it = g_lossy.find(handle);
        if (it != g_lossy.end()) s = it->second;
    }
    if (!s) {
        set_error("lossy_add_images: unknown handle %d", handle);
        return -1;
    }
    if (!frames || !out || nframes < 0) {
        set_error("lossy_add_images: bad arguments");
        return -1;
    }
    if (nframes == 0) return 0;
    RIRB_REQUIRE_DEVICE();
    {
        int dev = -1;
        if (cudaGetDevice(&dev) != cudaSuccess) cudaGetLastError();
        if (dev != s->device) {
            set_error("lossy_add_images: handle %d belongs to CUDA device %d, the calling thread is on device %d", handle, s->device, dev);
            return -1;
        }
    }
    cudaStream_t st = tls.stream;
    const int w = s->w, h = s->h, n = w * h, ns = w * s->stop_h;
    const size_t bytes = (size_t)n * 2 * (size_t)nframes;
    if (refuse_overlap("lossy_add_images", {{"frames", frames, bytes}}, {{"out", out, bytes}, {"errors", errors, sizeof(int) * 2 * (size_t)nframes}}))
        return -1;
    const u16* d_in = (const u16*)stage_in(frames, bytes, 0, st);
    if (!d_in) return -1;
    StagedOut o;
    if (!stage_out(o, out, bytes, 1, false, st)) return -1;
    if (s->errors_cap < nframes) {
        if (s->errors_dev) cudaFree(s->errors_dev);
        s->errors_dev = nullptr;
        s->errors_cap = 0;
        RIRB_CUDA_OK(cudaMalloc(&s->errors_dev, sizeof(int) * 2 * (size_t)nframes));
        s->errors_cap = nframes;
    }
    char* b = s->buf;
    u16 *lastDL = (u16*)(b + s->o_lastDL), *refT = (u16*)(b + s->o_refT), *prevT = (u16*)(b + s->o_prevT), *tmp = (u16*)(b + s->o_tmp),
        *tmpT = (u16*)(b + s->o_tmpT), *cval = (u16*)(b + s->o_cval), *ring = (u16*)(b + s->o_ring);
    unsigned* sums = (unsigned*)(b + s->o_sums);
    short* ccnt = (short*)(b + s->o_ccnt);
    void* scal = b + s->o_scal;
    long long f = 0;
    while (f < nframes) {
        const u16* img = d_in + (size_t)f * n;
        u16* dst = (u16*)o.dev + (size_t)f * n;
        if (s->frames >= 1 && s->use_run && option_enabled(OPT_LOSSY_RUN)) {
            // a run of non-initial frames in one cooperative launch (lossy_run_kernel)
            const long long m = std::min<long long>(nframes - f, lossy_max_run());
            if (!s->hist_scratch) {
                RIRB_CUDA_OK(cudaMalloc((void**)&s->hist_scratch, lossy_hist_scratch_bytes()));
                RIRB_CUDA_OK(cudaMemsetAsync(s->hist_scratch, 0, lossy_hist_scratch_bytes(), st));
            }
            const u16* cur = img;
            if (s->bp_enabled && ns > 0) {
                if (s->cur_batch_frames < (size_t)m) {
                    if (s->cur_batch) cudaFree(s->cur_batch);
                    s->cur_batch = nullptr;
                    s->cur_batch_frames = 0;
                    RIRB_CUDA_OK(cudaMalloc((void**)&s->cur_batch, (size_t)lossy_max_run() * n * 2));
                    s->cur_batch_frames = (size_t)lossy_max_run();
                }
                auto bp = find_handle(s->bp_handle);
                if (!bp) {
                    set_error("lossy_add_images: the bad-pixel handle of the first frame is gone");
                    return -1;
                }
                if (launch_bp_correct(img, s->cur_batch, bp->xy_dev, bp->span_off_dev, w, s->stop_h, bp->clamp_value, m, (size_t)n, st) != 0)
                    return -1;
                if (n > ns)
                    RIRB_CUDA_OK(cudaMemcpy2DAsync(s->cur_batch + ns, (size_t)n * 2, img + ns, (size_t)n * 2, (size_t)(n - ns) * 2, (size_t)m,
                                                   cudaMemcpyDeviceToDevice, st));
                cur = s->cur_batch;
            }
            const int rc = launch_lossy_run(img, cur, dst, lastDL, refT, prevT, sums, cval, ccnt, ring, n, ns, s->ra, s->subtract_min,
                                            s->frames, (int)m, s->low, s->high, s->std_factor, s->variant, s->quirk, scal,
                                            s->hist_scratch, s->errors_dev + 2 * f, st);
            if (rc < 0) return -1;
            if (rc == 0) {
                s->frames += m;
                f += m;
                continue;
            }
            s->use_run = false;  // no cooperative launch on this device: frame by frame from here on
        }
        const u16* cur = img;  // "tmp" of the reference
        if (s->bp_enabled && ns > 0) {  // bp.init on the first image's lossy rows, bp.correct on every image (:2259-2266)
            if (s->frames == 0 && s->bp_handle == 0) {
                s->bp_handle = bad_pixels_create((unsigned short*)img, w, s->stop_h);
                if (s->bp_handle == 0) return -1;
            }
            auto bp = find_handle(s->bp_handle);
            if (launch_bp_correct(img, tmp, bp->xy_dev, bp->span_off_dev, w, s->stop_h, bp->clamp_value, 1, (size_t)n, st) != 0) return -1;
            if (n > ns) RIRB_CUDA_OK(cudaMemcpyAsync(tmp + ns, img + ns, (size_t)(n - ns) * 2, cudaMemcpyDeviceToDevice, st));
            cur = tmp;
        }
        int rc;
        if (s->frames == 0)
            rc = launch_lossy_first(cur, dst, lastDL, refT, prevT, n, ns, s->subtract_min, scal, s->errors_dev + 2 * f, s->low, s->high, st);
        else
            rc = launch_lossy_frame(img, cur, tmpT, dst, lastDL, refT, prevT, sums, cval, ccnt, ring, n, ns, s->ra, s->subtract_min,
                                    s->frames, s->low, s->high, s->std_factor, s->variant, s->quirk, scal, s->errors_dev + 2 * f, st);
        if (rc != 0) return -1;
        ++s->frames;
        ++f;
    }
    if (errors) RIRB_CUDA_OK(cudaMemcpyAsync(errors, s->errors_dev, sizeof(int) * 2 * (size_t)nframes, cudaMemcpyDefault, st));
    if (o.host) RIRB_CUDA_OK(copy_d2h(o.host, o.dev, o.bytes, st));
    if (o.host || (errors && !is_device_ptr(errors))) RIRB_CUDA_OK(cudaStreamSynchronize(st));
    return 0;
}

// =================================================================================================
// the whole path on host buffers
// =================================================================================================
namespace {
constexpr int HP_SLOTS = 3;
struct HostPipeSlot {
    cudaStream_t stream = nullptr;
    void* buf = nullptr;   // in | corrected | registered | lo | hi | smoothed | dx | dy for `cap` frames
    size_t cap_bytes = 0;
};
struct HostPipe {
    HostPipeSlot slot[HP_SLOTS];
    int device = -1;
    ~HostPipe() { release(); }
    void release()
    {
        for (int k = 0; k < HP_SLOTS; ++k) {
            if (slot[k].buf) (void)cudaFree(slot[k].buf);
            if (slot[k].stream) (void)cudaStreamDestroy(slot[k].stream);
            slot[k] = HostPipeSlot();
        }
        (void)cudaGetLastError();
        device = -1;
    }
};
thread_local HostPipe g_host_pipe;
}  // namespace

int rirb_process_movie_host(int handle, const unsigned short* frames, long long nframes, int w, int h, float sigma, const float* dx,
                            const float* dy, const char* strategy, unsigned int background, int gop, int delta,
                            long long first_frame, unsigned char* lo, unsigned char* hi, float* smoothed)
{
    auto s = find_handle_here(handle, "process_movie_host");
    if (!s) return -1;
    const int strat = strategy_code(strategy);
    if (!frames || !dx || !dy || !lo || !hi || w != s->w || h != s->h || nframes < 0 || gop < 1 || strat < 0 ||
        (delta && first_frame % gop != 0)) {
        set_error("process_movie_host: bad arguments");
        return -1;
    }
    if (strat == STRAT_NOBORDER) {
        // untouched pixels keep whatever the destination held (the Python wrapper pre-fills it with the
        // image, rir_signal_processing.py:56-57); there is no caller-visible destination here
        set_error("process_movie_host: strategy \"noborder\" needs a caller-initialised destination; use rirb_translate_batch");
        return -1;
    }
    if (nframes == 0) return 0;
    GaussTaps taps;
    if (gaussian_taps_host(sigma, &taps) != 0) return -1;
    RIRB_REQUIRE_DEVICE();
    const size_t fpx = (size_t)w * h;
    // every operand is host memory read and written by copies on three streams at once: an output that overlaps an input
    // races with the upload of a later sub-chunk whatever the kind of memory, so refuse_overlap's device-only rule for
    // inputs does not apply
    {
        const size_t n = fpx * (size_t)nframes;
        const Operand ins[] = {{"frames", frames, n * 2}, {"dx", dx, 4 * (size_t)nframes}, {"dy", dy, 4 * (size_t)nframes}};
        const Operand outs[] = {{"lo", lo, n}, {"hi", hi, n}, {"smoothed", smoothed, n * 4}};
        for (const Operand& o : outs)
            for (const Operand& i : ins)
                if (bytes_overlap(o, i)) {
                    set_error("process_movie_host: %s and %s overlap", i.name, o.name);
                    return -1;
                }
        if (refuse_overlap("process_movie_host", {}, {outs[0], outs[1], outs[2]})) return -1;
    }
    // sub-chunk: whole GOPs, about 64 MB of input (RIRB_HOST_SUB_BYTES overrides the size: tests use it to make
    // small movies rotate through all the slots)
    long long sub_bytes = 64ll << 20;
    if (const char* e = getenv("RIRB_HOST_SUB_BYTES")) {
        const long long v = atoll(e);
        if (v > 0) sub_bytes = v;
    }
    long long sub = sub_bytes / (long long)(fpx * 2);
    sub = sub / gop * gop;
    if (sub < gop) sub = gop;
    // per-slot layout (every section 256-byte aligned)
    auto al = [](size_t v) { return (v + 255) & ~(size_t)255; };
    const size_t o_in = 0, o_cor = o_in + al(fpx * 2 * sub), o_reg = o_cor + al(fpx * 2 * sub), o_lo = o_reg + al(fpx * 2 * sub),
                 o_hi = o_lo + al(fpx * sub), o_sm = o_hi + al(fpx * sub), o_dx = o_sm + al(fpx * 4 * sub), o_dy = o_dx + al(4 * sub),
                 total = o_dy + al(4 * sub);
    HostPipe& hp = g_host_pipe;
    int dev = 0;
    RIRB_CUDA_OK(cudaGetDevice(&dev));
    for (int k = 0; k < HP_SLOTS; ++k) {
        HostPipeSlot& sl = hp.slot[k];
        if (hp.device != dev && sl.buf) {  // the thread moved to another device: drop the old buffers
            cudaFree(sl.buf);
            sl.buf = nullptr;
            sl.cap_bytes = 0;
            if (sl.stream) cudaStreamDestroy(sl.stream);
            sl.stream = nullptr;
        }
        if (!sl.stream) RIRB_CUDA_OK(cudaStreamCreateWithFlags(&sl.stream, cudaStreamNonBlocking));
        if (sl.cap_bytes < total) {
            if (sl.buf) cudaFree(sl.buf);
            sl.buf = nullptr;
            sl.cap_bytes = 0;
            RIRB_CUDA_OK(cudaMalloc(&sl.buf, total));
            sl.cap_bytes = total;
        }
    }
    hp.device = dev;
    // work already enqueued by this thread (e.g. bad_pixels_create) is complete before the slots start
    RIRB_CUDA_OK(cudaStreamSynchronize(tls.stream));
    int rc = 0;
    long long k = 0;
    for (long long a = 0; a < nframes && rc == 0; a += sub, ++k) {
        const long long m = (nframes - a < sub) ? nframes - a : sub;
        HostPipeSlot& sl = hp.slot[k % HP_SLOTS];
        cudaStream_t st = sl.stream;
        char* base = (char*)sl.buf;
        u16 *d_in = (u16*)(base + o_in), *d_cor = (u16*)(base + o_cor), *d_reg = (u16*)(base + o_reg);
        u8 *d_lo = (u8*)(base + o_lo), *d_hi = (u8*)(base + o_hi);
        float *d_sm = (float*)(base + o_sm), *d_dx = (float*)(base + o_dx), *d_dy = (float*)(base + o_dy);
        // no early return in here: copies already queued on the other slots' streams write into the caller's buffers, so the
        // streams are drained below whatever happens
        auto ok = [&](cudaError_t e, const char* what) {
            if (e == cudaSuccess) return true;
            set_error("process_movie_host: %s failed: %s", what, cudaGetErrorString(e));
            (void)cudaGetLastError();
            rc = -1;
            return false;
        };
        if (!ok(cudaMemcpyAsync(d_in, frames + a * fpx, fpx * 2 * m, cudaMemcpyDefault, st), "upload of the frames") ||
            !ok(cudaMemcpyAsync(d_dx, dx + a, 4 * m, cudaMemcpyDefault, st), "upload of the shifts") ||
            !ok(cudaMemcpyAsync(d_dy, dy + a, 4 * m, cudaMemcpyDefault, st), "upload of the shifts"))
            break;
        if (launch_bp_correct(d_in, d_cor, s->xy_dev, s->span_off_dev, w, h, s->clamp_value, m, fpx, st) != 0 ||
            launch_gaussian_u16(d_cor, d_sm, w, h, m, taps, st) != 0 ||
            launch_translate_u16(d_cor, d_reg, w, h, m, fpx, fpx, d_dx, d_dy, 0.f, 0.f, strat, background & 0xFFFFu, false, st) != 0 ||
            launch_precode_movie(d_reg, m, w, h, gop, delta, first_frame + a, d_lo, d_hi, st) != 0) {
            rc = -1;
            break;
        }
        if (!ok(cudaMemcpyAsync(lo + a * fpx, d_lo, fpx * m, cudaMemcpyDefault, st), "download of the low-byte planes") ||
            !ok(cudaMemcpyAsync(hi + a * fpx, d_hi, fpx * m, cudaMemcpyDefault, st), "download of the high-byte planes") ||
            (smoothed && !ok(cudaMemcpyAsync(smoothed + a * fpx, d_sm, fpx * 4 * m, cudaMemcpyDefault, st), "download of the smoothed frames")))
            break;
    }
    for (int q = 0; q < HP_SLOTS; ++q) {
        cudaError_t e = cudaStreamSynchronize(hp.slot[q].stream);
        if (e != cudaSuccess && rc == 0) {
            set_error("process_movie_host: %s", cudaGetErrorString(e));
            rc = -1;
        }
    }
    return rc;
}

void rirb_release_thread_resources(void)
{
    if (tls.stream) (void)cudaStreamSynchronize(tls.stream);
    g_host_pipe.release();
    for (int d = 0; d < PIN_MAX_DEVICES; ++d) pin_rings[d].release();
    tls.release();
}

// =================================================================================================
// statistics
// =================================================================================================
int rirb_movie_stats(const unsigned short* pixels, size_t n, unsigned int* minmax, unsigned long long* hist, int accumulate)
{
    if (!pixels || !minmax) {
        set_error("movie_stats: bad arguments");
        return -1;
    }
    RIRB_REQUIRE_DEVICE();
    if (refuse_overlap("movie_stats", {{"pixels", pixels, n * 2}},
                       {{"minmax", minmax, 2 * sizeof(unsigned)}, {"hist", hist, 65536 * sizeof(unsigned long long)}}))
        return -1;
    cudaStream_t st = tls.stream;
    const u16* d_p = (const u16*)stage_in(pixels, n * 2, 0, st);
    if (!d_p) return -1;
    StagedOut o[2];
    if (!stage_out(o[0], minmax, 2 * sizeof(unsigned), 1, accumulate != 0, st)) return -1;
    if (hist && !stage_out(o[1], hist, 65536 * sizeof(unsigned long long), 2, accumulate != 0, st)) return -1;
    if (!accumulate && launch_stats_init((unsigned*)o[0].dev, (unsigned long long*)o[1].dev, st) != 0) return -1;
    if (launch_movie_stats(d_p, n, nullptr, (unsigned*)o[0].dev, (unsigned long long*)o[1].dev, st) != 0) return -1;
    return finish_out(o, 2, st);
}

int rirb_hist_quantile(const unsigned long long* hist, long long count, float percent)
{
    if (!hist) {
        set_error("hist_quantile: bad arguments");
        return -1;
    }
    RIRB_REQUIRE_DEVICE();
    cudaStream_t st = tls.stream;
    const unsigned long long* d_h = (const unsigned long long*)stage_in(hist, 65536 * sizeof(unsigned long long), 0, st);
    int* d_out = (int*)scratch(5, sizeof(int));
    if (!d_h || !d_out) return -1;
    if (launch_hist_quantile(d_h, count, percent, 0, d_out, st) != 0) return -1;
    int r = 0;
    RIRB_CUDA_OK(cudaMemcpyAsync(&r, d_out, sizeof(int), cudaMemcpyDeviceToHost, st));
    RIRB_CUDA_OK(cudaStreamSynchronize(st));
    return r;
}

static int median_pixel_any(const unsigned short* pixels, const unsigned char* mask, int size, float percent)
{
    if (!pixels || size < 0) {
        set_error("find_median_pixel: bad arguments");
        return -1;
    }
    RIRB_REQUIRE_DEVICE();
    cudaStream_t st = tls.stream;
    const u16* d_p = (const u16*)stage_in(pixels, (size_t)size * 2, 0, st);
    if (!d_p && size) return -1;
    const u8* d_m = nullptr;
    if (mask) {
        d_m = (const u8*)stage_in(mask, (size_t)size, 1, st);
        if (!d_m && size) return -1;
    }
    unsigned long long* d_hist = (unsigned long long*)scratch(2, 65536 * sizeof(unsigned long long));
    unsigned* d_mm = (unsigned*)scratch(3, 2 * sizeof(unsigned));
    int* d_out = (int*)scratch(5, sizeof(int));
    if (!d_hist || !d_mm || !d_out) return -1;
    if (launch_stats_init(d_mm, d_hist, st) != 0) return -1;
    if (launch_movie_stats(d_p, (size_t)size, d_m, d_mm, d_hist, st) != 0) return -1;
    if (launch_hist_quantile(d_hist, mask ? -1 : (long long)size, percent, mask ? 1 : 0, d_out, st) != 0) return -1;
    int r = 0;
    RIRB_CUDA_OK(cudaMemcpyAsync(&r, d_out, sizeof(int), cudaMemcpyDeviceToHost, st));
    RIRB_CUDA_OK(cudaStreamSynchronize(st));
    return r;
}

int find_median_pixel(unsigned short* pixels, int size, float percent) { return median_pixel_any(pixels, nullptr, size, percent); }
int find_median_pixel_mask(unsigned short* pixels, unsigned char* mask, int size, float percent)
{
    if (!mask) {
        set_error("find_median_pixel_mask: NULL mask");
        return -1;
    }
    return median_pixel_any(pixels, mask, size, percent);
}

int rirb_get_background(const unsigned short* pixels, int size)
{
    if (!pixels || size <= 0) {
        set_error("get_background: bad arguments");
        return -1;
    }
    RIRB_REQUIRE_DEVICE();
    cudaStream_t st = tls.stream;
    const u16* d_p = (const u16*)stage_in(pixels, (size_t)size * 2, 0, st);
    unsigned long long* d_hist = (unsigned long long*)scratch(2, 65536 * sizeof(unsigned long long));
    unsigned* d_mm = (unsigned*)scratch(3, 2 * sizeof(unsigned));
    unsigned* d_out = (unsigned*)scratch(5, sizeof(unsigned));
    if (!d_p || !d_hist || !d_mm || !d_out) return -1;
    if (launch_stats_init(d_mm, d_hist, st) != 0) return -1;
    if (launch_movie_stats(d_p, (size_t)size, nullptr, d_mm, d_hist, st) != 0) return -1;
    if (launch_hist_mode4(d_hist, d_out, st) != 0) return -1;
    unsigned r = 0;
    RIRB_CUDA_OK(cudaMemcpyAsync(&r, d_out, sizeof(unsigned), cudaMemcpyDeviceToHost, st));
    RIRB_CUDA_OK(cudaStreamSynchronize(st));
    return (int)r;
}

// =================================================================================================
// forwarded entries (outside the hot path)
// =================================================================================================
int extract_times(double* time_vector, int vector_count, int* vector_sizes, int s, double* output, int* output_size)
{
    typedef int (*fn)(double*, int, int*, int, double*, int*);
    fn f = (fn)forward_symbol("extract_times");
    return f ? f(time_vector, vector_count, vector_sizes, s, output, output_size) : -1;
}
int resample_time_serie(double* sample_x, double* sample_y, int size, double* times, int times_size, int s, double padds,
                        double* output, int* output_size)
{
    typedef int (*fn)(double*, double*, int, double*, int, int, double, double*, int*);
    fn f = (fn)forward_symbol("resample_time_serie");
    return f ? f(sample_x, sample_y, size, times, times_size, s, padds, output, output_size) : -1;
}
int label_image(int type, void* src, int* dst, int w, int h, void* background, double* out_xy, int* out_area)
{
    typedef int (*fn)(int, void*, int*, int, int, void*, double*, int*);
    fn f = (fn)forward_symbol("label_image");
    return f ? f(type, src, dst, w, h, background, out_xy, out_area) : -1;
}
int keep_largest_area(int type, void* src, int* dst, int w, int h, void* background, int foreground)
{
    typedef int (*fn)(int, void*, int*, int, int, void*, int);
    fn f = (fn)forward_symbol("keep_largest_area");
    return f ? f(type, src, dst, w, h, background, foreground) : -1;
}
size_t hash_bytes(void* ptr, size_t len)
{
    typedef size_t (*fn)(void*, size_t);
    fn f = (fn)forward_symbol("hash_bytes");
    return f ? f(ptr, len) : 0;
}

}  // extern "C"
