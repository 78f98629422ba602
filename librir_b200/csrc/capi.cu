// librir_b200/csrc/capi.cu -- the C ABI (include/librir_b200.h): argument checking, host<->device
// staging for host-pointer callers, the bad-pixel handle table, forwarding of the out-of-scope
// entries.  All compute happens in the kernels of this directory; there is no CPU path.
#include <dlfcn.h>
#include <limits.h>
#include <math.h>
#include <stdarg.h>
#include <stdlib.h>
#include <string.h>

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
    // grow-only device work space (never shared between threads), used as a stack: an entry's Call takes slots from `top`
    // up -- for host operands, and for the work space its launchers ask for (scratch_buffer) -- and gives them back when
    // it returns, so an entry called inside another starts above its caller's slots.  The deepest call,
    // rirb_label_movie with every operand on the host, takes 9: five operands and four work buffers.
    static constexpr int SLOTS = 9;
    void* dev[SLOTS] = {};
    size_t cap[SLOTS] = {};
    int dev_of[SLOTS] = {};
    int top = 0;  // the first free slot
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
int require_device()
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

void* scratch_buffer(size_t bytes)
{
    if (tls.top == ThreadState::SLOTS) {
        set_error("out of staging slots: a call needs more than %d device buffers", ThreadState::SLOTS);
        return nullptr;
    }
    const int slot = tls.top++;
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

// ---- the operands of one entry call -----------------------------------------------------------------
// An entry names each array operand once, with its size; nullptr is an absent operand.  stage() refuses overlapping
// operands (refuse_overlap, on the memory kind looked up when the operand was named), then gives every host operand a
// device copy in the thread's work space: inputs, and outputs that are only partly written (preload: translate's
// "noborder", padded planes, frames corrected in place, accumulated statistics), go up first.  Device and managed
// operands are used in place.  finish() copies host outputs back and waits for them; a call whose operands are all on
// the device returns without synchronising.  The slots the call took, its launchers' included, go back when it ends.
struct Staged : Operand {
    void* dev = nullptr;  // what the kernels get: p itself, or its copy in the work space
    bool load = true;     // host input, preloaded host output: stage() uploads it
    bool staged = true;   // false: only the overlap rule applies, the entry reads or writes the operand itself
};
class Call {
  public:
    explicit Call(const char* what) : what_(what), base_(tls.top) {}
    ~Call() { tls.top = base_; }
    Call(const Call&) = delete;
    Call& operator=(const Call&) = delete;
    Staged& in(const char* name, const void* p, size_t bytes) { return add(ins_, nin_, name, p, bytes, true); }
    Staged& out(const char* name, void* p, size_t bytes, bool preload = false) { return add(outs_, nout_, name, p, bytes, preload); }
    int stage()
    {
        if (nin_ > MAX || nout_ > MAX) {
            set_error("%s: more than %d inputs or outputs", what_, MAX);
            return -1;
        }
        if (refuse_overlap(what_, ins_, ins_ + nin_, outs_, outs_ + nout_)) return -1;
        for (int i = 0; i < nin_ + nout_; ++i) {
            Staged& o = i < nin_ ? ins_[i] : outs_[i - nin_];
            if (!o.p || o.on_device || !o.staged) {
                o.dev = o.on_device ? (void*)o.p : nullptr;
                continue;
            }
            if (!(o.dev = scratch_buffer(o.bytes))) return -1;
            if (o.load && copy_h2d(o.dev, o.p, o.bytes, st_) != cudaSuccess) {
                set_error("host->device copy failed: %s", cudaGetErrorString(cudaGetLastError()));
                return -1;
            }
        }
        return 0;
    }
    // sync: wait for the stream even when every output is on the device (the entry's own host buffers are being read)
    int finish(bool sync = false)
    {
        for (int i = 0; i < nout_; ++i) {
            const Staged& o = outs_[i];
            if (o.p && !o.on_device && o.staged && o.bytes) {
                RIRB_CUDA_OK(copy_d2h((void*)o.p, o.dev, o.bytes, st_));
                sync = true;
            }
        }
        if (sync) RIRB_CUDA_OK(cudaStreamSynchronize(st_));
        return 0;
    }

  private:
    static constexpr int MAX = 4;
    Staged& add(Staged* list, int& n, const char* name, const void* p, size_t bytes, bool load)
    {
        Staged& o = list[n < MAX ? n : MAX - 1];  // stage() refuses a call that names too many
        ++n;
        o.name = name;
        o.p = p;
        o.bytes = bytes;
        o.on_device = is_device_ptr(p);
        o.load = load;
        return o;
    }
    const char* what_;
    const int base_;
    const cudaStream_t st_ = tls.stream;
    Staged ins_[MAX], outs_[MAX];
    int nin_ = 0, nout_ = 0;
};

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
// bad-pixel handle table (the reference's set_void_ptr / get_void_ptr / rm_void_ptr, tools.cpp:40-85: process-global,
// handles.h's Table)
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
static Table<BadPixelState> g_bad_pixels;

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
    Call c("translate");
    auto& in = c.in("src", src, bytes);
    auto& ddx = c.in("dx", dx, sbytes);
    auto& ddy = c.in("dy", dy, sbytes);
    auto& out = c.out("dst", dst, bytes, strat == STRAT_NOBORDER);
    const bool host_scalar = n_shifts == 1 && !ddx.on_device && !ddy.on_device;  // read here, not uploaded
    ddx.staged = ddy.staged = !host_scalar;
    if (c.stage() != 0) return -1;
    cudaStream_t st = tls.stream;
    // background: one element, host or device
    unsigned long long bg = 0;
    if (is_device_ptr(background)) {
        RIRB_CUDA_OK(cudaMemcpyAsync(&bg, background, esize, cudaMemcpyDeviceToHost, st));
        RIRB_CUDA_OK(cudaStreamSynchronize(st));
    } else {
        memcpy(&bg, background, esize);
    }
    const float *d_dx = (const float*)ddx.dev, *d_dy = (const float*)ddy.dev;
    float dx0 = 0.f, dy0 = 0.f;
    if (host_scalar) {
        dx0 = dx[0];
        dy0 = dy[0];
    } else {
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
    if (launch_translate(type, in.dev, out.dev, w, h, nframes, d_dx, d_dy, dx0, dy0, strat, &bg, st) != 0) return -1;
    return c.finish();
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
    Call c("gaussian_filter");
    auto& in = c.in("src", src, npx * (src_u16 ? 2 : 4));
    auto& out = c.out("dst", dst, npx * 4);
    if (c.stage() != 0) return -1;
    cudaStream_t st = tls.stream;
    int rc = src_u16 ? launch_gaussian_u16((const u16*)in.dev, (float*)out.dev, w, h, nframes, taps, st)
                     : launch_gaussian_f32((const float*)in.dev, (float*)out.dev, w, h, nframes, taps, st);
    if (rc != 0) return -1;
    return c.finish();
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
    Call c("bad_pixels_create");
    auto& img = c.in("first_image", first_image, n * 2);
    if (c.stage() != 0) return 0;
    const u16* d_img = (const u16*)img.dev;
    // (i) frame histogram -> median (sorted[N/2]) and spread, as Filters.h:145-160 / BadPixels.cpp:19-31
    unsigned* d_hist = (unsigned*)scratch_buffer(sizeof(unsigned) * 65536);
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
    return g_bad_pixels.add(state);
}

int rirb_bad_pixels_correct_batch(int handle, const unsigned short* in, unsigned short* out, long long nframes)
{
    auto s = find_handle_here(g_bad_pixels, handle, "bad_pixels_correct");
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
    Call c("bad_pixels_correct");
    if (in == out) {  // sequential in-place meaning of the reference (BadPixels.cpp:41-59)
        auto& io = c.out("out", out, bytes, true);
        if (c.stage() != 0) return -1;
        if (launch_bp_correct_inplace((u16*)io.dev, s->xy_dev, (int)(s->xy.size() / 2), s->w, s->h, s->clamp_value, nframes, fpx,
                                      st) != 0)
            return -1;
        return c.finish();
    }
    auto& i = c.in("in", in, bytes);
    auto& o = c.out("out", out, bytes);
    if (c.stage() != 0) return -1;
    if (launch_bp_correct((const u16*)i.dev, (u16*)o.dev, s->xy_dev, s->span_off_dev, s->w, s->h, s->clamp_value, nframes, fpx, st) != 0)
        return -1;
    return c.finish();
}

// bad_pixels_correct + gaussian_filter of the corrected frames, reading the movie once (gaussian.cu, BpFuse):
// corrected[n][h][w] uint16 and smoothed[n][h][w] float32 are both produced.  Layouts the tiled kernel cannot take
// (w % 8 != 0, unaligned buffers, radius > 4) run the two kernels instead; results are the same either way.
int rirb_bad_pixels_correct_gaussian_batch(int handle, const unsigned short* in, unsigned short* corrected, float* smoothed,
                                           long long nframes, float sigma)
{
    auto s = find_handle_here(g_bad_pixels, handle, "bad_pixels_correct_gaussian");
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
    Call c("bad_pixels_correct_gaussian");
    auto& i = c.in("in", in, fpx * 2 * (size_t)nframes);
    auto& cor = c.out("corrected", corrected, fpx * 2 * (size_t)nframes);
    auto& sm = c.out("smoothed", smoothed, fpx * 4 * (size_t)nframes);
    if (c.stage() != 0) return -1;
    const u16* d_in = (const u16*)i.dev;
    const int rc = launch_gaussian_bp_u16(d_in, (u16*)cor.dev, (float*)sm.dev, s->w, s->h, nframes, taps, s->xy_dev, s->row_off_dev,
                                          s->clamp_value, st);
    if (rc < 0) return -1;
    if (rc == 1) {
        if (launch_bp_correct(d_in, (u16*)cor.dev, s->xy_dev, s->span_off_dev, s->w, s->h, s->clamp_value, nframes, fpx, st) != 0 ||
            launch_gaussian_u16((const u16*)cor.dev, (float*)sm.dev, s->w, s->h, nframes, taps, st) != 0)
            return -1;
    }
    return c.finish();
}

int bad_pixels_correct(int handle, unsigned short* in, unsigned short* out)
{
    return rirb_bad_pixels_correct_batch(handle, in, out, 1);
}

void bad_pixels_destroy(int handle) { g_bad_pixels.remove(handle); }

int rirb_bad_pixels_count(int handle)
{
    auto s = g_bad_pixels.get(handle);
    if (!s) {
        set_error("bad_pixels: unknown handle %d", handle);
        return -1;
    }
    return (int)(s->xy.size() / 2);
}

int rirb_bad_pixels_get(int handle, int* xy, int capacity, int* clamp_value)
{
    auto s = g_bad_pixels.get(handle);
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
    auto s = find_handle_here(g_bad_pixels, handle, "remove_bad_pixels");
    if (!s) return -1;
    if (!frames || nframes < 0 || frame_stride < (size_t)s->w * s->h) {
        set_error("remove_bad_pixels: bad arguments");
        return -1;
    }
    if (nframes == 0) return 0;
    RIRB_REQUIRE_DEVICE();
    cudaStream_t st = tls.stream;
    Call c("remove_bad_pixels");
    auto& io = c.out("frames", frames, frame_stride * 2 * (size_t)nframes, true);
    if (c.stage() != 0) return -1;
    if (launch_loader_bp((u16*)io.dev, s->xy_dev, s->mask_dev, (int)(s->xy.size() / 2), s->w, s->h, nframes, frame_stride, st) != 0)
        return -1;
    return c.finish();
}

// =================================================================================================
// motion-correction variant
// =================================================================================================
// The reader's shifts, translate(..., -x[pos], -y[pos], ...) with float arguments (IRFileLoader.cpp:621): doubles on the
// host or the device -> f = (float)-x then (float)-y.  The entries stage f as their first input: a small pageable upload
// queued behind the frames' waits for them (6 us more per one-frame call, B200 at 1000 W).  An asynchronous copy reads f,
// so the entry waits for its stream before f goes away.
static int narrow_shifts(const double* x, const double* y, long long n, std::vector<float>& f, cudaStream_t st)
{
    std::vector<double> v(2 * (size_t)n);
    if (is_device_ptr(x) || is_device_ptr(y)) {
        RIRB_CUDA_OK(cudaMemcpyAsync(v.data(), x, sizeof(double) * n, cudaMemcpyDefault, st));
        RIRB_CUDA_OK(cudaMemcpyAsync(v.data() + n, y, sizeof(double) * n, cudaMemcpyDefault, st));
        RIRB_CUDA_OK(cudaStreamSynchronize(st));
    } else {
        memcpy(v.data(), x, sizeof(double) * n);
        memcpy(v.data() + n, y, sizeof(double) * n);
    }
    f.resize(v.size());
    for (size_t i = 0; i < v.size(); ++i) f[i] = (float)(-v[i]);
    return 0;
}

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
    cudaStream_t st = tls.stream;
    const bool inplace = (in == out);
    std::vector<float> f;
    if (narrow_shifts(shift_x, shift_y, nframes, f, st) != 0) return -1;
    Call c("remove_motion");
    auto& sh = c.in("shifts", f.data(), sizeof(float) * f.size());
    auto& i = c.in("in", inplace ? nullptr : in, bytes);
    auto& o = c.out("out", out, bytes, inplace);
    if (c.stage() != 0) return -1;
    const float* d_dx = (const float*)sh.dev;
    const u16* d_in = (const u16*)i.dev;
    if (inplace) {
        // the reference translates into a temporary and copies back; keep a private copy of the input
        void* copy = scratch_buffer(bytes);
        if (!copy) return -1;
        RIRB_CUDA_OK(cudaMemcpyAsync(copy, o.dev, bytes, cudaMemcpyDeviceToDevice, st));
        d_in = (const u16*)copy;
    } else if (frame_stride > (size_t)w * h) {  // pass the untouched tail rows through
        RIRB_CUDA_OK(cudaMemcpy2DAsync((u16*)o.dev + (size_t)w * h, frame_stride * 2, d_in + (size_t)w * h, frame_stride * 2,
                                       (frame_stride - (size_t)w * h) * 2, (size_t)nframes, cudaMemcpyDeviceToDevice, st));
    }
    if (launch_translate_u16(d_in, (u16*)o.dev, w, h, nframes, frame_stride, frame_stride, d_dx, d_dx + nframes, 0.f, 0.f,
                             STRAT_NEAREST, 0u, true, st) != 0)
        return -1;
    return c.finish(true);  // f is read by an asynchronous copy
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
        s = find_handle_here(g_bad_pixels, handle, "loader_read_movie");
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
    const bool motion = shift_x != nullptr;
    std::vector<float> f;
    if (motion && narrow_shifts(shift_x, shift_y, nframes, f, st) != 0) return -1;
    Call c("loader_read_movie");
    auto& sh = c.in("shifts", motion ? f.data() : nullptr, sizeof(float) * f.size());
    auto& l = c.in("lo", lo, pbytes);
    auto& hh = c.in("hi", hi, pbytes);
    auto& o = c.out("out", out, pbytes * 2);
    if (c.stage() != 0) return -1;
    const u8 *d_lo = (const u8*)l.dev, *d_hi = (const u8*)hh.dev;
    const int k = s ? (int)(s->xy.size() / 2) : 0;
    const bool fused_bp = s && k > 0 && w >= 3 && hb >= 3;
    if (!motion) {
        u16* merged = (u16*)o.dev;
        if (launch_loader_merge(d_lo, d_hi, merged, w, h, hb, nframes, fpx, min_T, min_T_height, fused_bp ? s->xy_dev : nullptr,
                                fused_bp ? s->span_off_dev : nullptr, fused_bp ? s->nbr_dev : nullptr, st) != 0)
            return -1;
        if (s && k > 0 && !fused_bp)  // degenerate sizes keep the reference's sequential loop (IRFileLoader.cpp:735-752)
            if (launch_loader_bp(merged, s->xy_dev, s->mask_dev, k, w, hb, nframes, fpx, st) != 0) return -1;
        return c.finish();
    }
    const float *d_dx = (const float*)sh.dev, *d_dy = d_dx + nframes;
    // one pass: planes -> merge -> += min_T -> medians -> motion translate (translate.cu, PLANES)
    const int rows_t = (min_T == 0 || min_T_height < 0) ? 0 : (min_T_height > h ? h : min_T_height);
    int rc = (s && k > 0 && !fused_bp)
                 ? 1
                 : launch_loader_fused(d_lo, d_hi, (u16*)o.dev, w, h, hb, nframes, min_T, rows_t, fused_bp ? s->xy_dev : nullptr,
                                       fused_bp ? s->nbr_dev : nullptr, fused_bp ? s->row_off_dev : nullptr,
                                       fused_bp ? s->mask_dev : nullptr, d_dx, d_dy, st);
    if (rc < 0) return -1;
    if (rc == 1) {  // layouts the fused kernel does not take: merge pass, then the motion pass through a scratch movie
        u16* merged = (u16*)scratch_buffer(pbytes * 2);
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
    return c.finish(true);  // f is read by an asynchronous copy
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
        s = find_handle_here(g_bad_pixels, handle, "loader_finish_frames");
        if (!s) return -1;
        if (s->w != w || s->h != hb) {
            set_error("loader_finish_frames: the handle was created on a %dx%d image, expected %dx%d", s->w, s->h, w, hb);
            return -1;
        }
    }
    RIRB_REQUIRE_DEVICE();
    cudaStream_t st = tls.stream;
    const size_t fpx = (size_t)w * h;
    Call c("loader_finish_frames");
    auto& io = c.out("frames", frames, fpx * 2 * (size_t)nframes, true);
    if (c.stage() != 0) return -1;
    u16* d = (u16*)io.dev;
    const int rows_t = (min_T == 0 || min_T_height < 0) ? 0 : (min_T_height > h ? h : min_T_height);
    if (launch_loader_add_min(d, w, rows_t, nframes, fpx, min_T, st) != 0) return -1;
    if (s && !s->xy.empty())
        if (launch_loader_bp(d, s->xy_dev, s->mask_dev, (int)(s->xy.size() / 2), w, hb, nframes, fpx, st) != 0) return -1;
    if (shift_x) {
        // the motion step is out of place: through a scratch copy, on device pointers (no further staging)
        u16* tmp = (u16*)scratch_buffer(fpx * 2 * (size_t)nframes);
        if (!tmp) return -1;
        RIRB_CUDA_OK(cudaMemcpyAsync(tmp, d, fpx * 2 * (size_t)nframes, cudaMemcpyDeviceToDevice, st));
        if (rirb_loader_remove_motion(tmp, d, w, hb, nframes, fpx, shift_x, shift_y) != 0) return -1;
    }
    return c.finish();
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
    cudaStream_t st = tls.stream;
    Call c("split_yuv444");
    auto& im = c.in("img", img, (size_t)w * h * 2);
    auto& t = c.in("it", it, (size_t)w * h);
    // row padding must survive untouched: preload padded planes
    auto& y = c.out("y_plane", y_plane, (size_t)ls_y * h, ls_y != w);
    auto& u = c.out("u_plane", u_plane, (size_t)ls_u * h, ls_u != w);
    auto& v = c.out("v_plane", v_plane, (size_t)ls_v * h, ls_v != w);
    if (c.stage() != 0) return -1;
    if (launch_split_planes((const u16*)im.dev, (const u8*)t.dev, w, h, (u8*)y.dev, (u8*)u.dev, (u8*)v.dev, ls_y, ls_u, ls_v, st) != 0)
        return -1;
    return c.finish();
}

int rirb_merge_yuv444(const unsigned char* y_plane, const unsigned char* u_plane, const unsigned char* v_plane, int ls_y, int ls_u,
                      int ls_v, int w, int h, unsigned short* img, unsigned char* it)
{
    if (!img || !u_plane || !v_plane || w <= 0 || h <= 0 || ls_u < w || ls_v < w) {
        set_error("merge_yuv444: bad arguments");
        return -1;
    }
    RIRB_REQUIRE_DEVICE();
    cudaStream_t st = tls.stream;
    const bool with_y = y_plane && it;
    Call c("merge_yuv444");
    auto& y = c.in("y_plane", with_y ? y_plane : nullptr, (size_t)ls_y * h);
    auto& u = c.in("u_plane", u_plane, (size_t)ls_u * h);
    auto& v = c.in("v_plane", v_plane, (size_t)ls_v * h);
    auto& im = c.out("img", img, (size_t)w * h * 2);
    auto& t = c.out("it", with_y ? it : nullptr, (size_t)w * h);
    if (c.stage() != 0) return -1;
    if (launch_merge_planes((const u8*)y.dev, (const u8*)u.dev, (const u8*)v.dev, ls_y, ls_u, ls_v, w, h, (u16*)im.dev, (u8*)t.dev, st) != 0)
        return -1;
    return c.finish();
}

int rirb_split_yuv420(const unsigned short* img, const unsigned char* it, int w, int h, unsigned char* y_plane, int ls_y,
                      unsigned char* u_plane, int ls_u)
{
    if (!img || !y_plane || w <= 0 || h <= 0 || ls_y < w) {
        set_error("split_yuv420: bad arguments");
        return -1;
    }
    RIRB_REQUIRE_DEVICE();
    cudaStream_t st = tls.stream;
    const bool with_it = it && u_plane;
    Call c("split_yuv420");
    auto& im = c.in("img", img, (size_t)w * h * 2);
    auto& t = c.in("it", with_it ? it : nullptr, (size_t)w * h);
    auto& y = c.out("y_plane", y_plane, (size_t)ls_y * 2 * h, ls_y != w);
    auto& u = c.out("u_plane", with_it ? u_plane : nullptr, (size_t)ls_u * h, ls_u != w);
    if (c.stage() != 0) return -1;
    u8* d_y = (u8*)y.dev;
    if (launch_split_planes((const u16*)im.dev, (const u8*)t.dev, w, h, (u8*)u.dev, d_y, d_y + (size_t)h * ls_y, ls_u, ls_y, ls_y, st) != 0)
        return -1;
    return c.finish();
}

int rirb_merge_yuv420(const unsigned char* y_plane, int ls_y, const unsigned char* u_plane, int ls_u, int w, int h,
                      unsigned short* img, unsigned char* it)
{
    if (!img || !y_plane || w <= 0 || h <= 0 || ls_y < w) {
        set_error("merge_yuv420: bad arguments");
        return -1;
    }
    RIRB_REQUIRE_DEVICE();
    cudaStream_t st = tls.stream;
    const bool with_it = it && u_plane;
    Call c("merge_yuv420");
    auto& y = c.in("y_plane", y_plane, (size_t)ls_y * 2 * h);
    auto& u = c.in("u_plane", with_it ? u_plane : nullptr, (size_t)ls_u * h);
    auto& im = c.out("img", img, (size_t)w * h * 2);
    auto& t = c.out("it", with_it ? it : nullptr, (size_t)w * h);
    if (c.stage() != 0) return -1;
    const u8* d_yp = (const u8*)y.dev;
    if (launch_merge_planes((const u8*)u.dev, d_yp, d_yp + (size_t)h * ls_y, ls_u, ls_y, ls_y, w, h, (u16*)im.dev, (u8*)t.dev, st) != 0)
        return -1;
    return c.finish();
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
    Call c("precode_movie");
    auto& m = c.in("movie", movie, n * 2);
    auto& l = c.out("lo", lo, n);
    auto& hh = c.out("hi", hi, n);
    if (c.stage() != 0) return -1;
    if (launch_precode_movie((const u16*)m.dev, nframes, w, h, gop, delta, first_frame, (u8*)l.dev, (u8*)hh.dev, st) != 0) return -1;
    return c.finish();
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
    Call c("precode_movie_stats");
    auto& m = c.in("movie", movie, n * 2);
    auto& l = c.out("lo", lo, n);
    auto& hh = c.out("hi", hi, n);
    auto& mm = c.out("minmax", minmax, 2 * sizeof(unsigned), accumulate != 0);
    auto& hs = c.out("hist", hist, 65536 * sizeof(unsigned long long), accumulate != 0);
    if (c.stage() != 0) return -1;
    const u16* d_mov = (const u16*)m.dev;
    u8 *d_lo = (u8*)l.dev, *d_hi = (u8*)hh.dev;
    unsigned* d_mm = (unsigned*)mm.dev;
    unsigned long long* d_hist = (unsigned long long*)hs.dev;
    if (!accumulate && launch_stats_init(d_mm, d_hist, st) != 0) return -1;
    const int rc = launch_precode_movie_stats(d_mov, nframes, w, h, gop, delta, first_frame, d_lo, d_hi, d_mm, d_hist, st);
    if (rc < 0) return -1;
    if (rc == 1) {  // layouts the fused kernel does not take: the two kernels
        if (launch_precode_movie(d_mov, nframes, w, h, gop, delta, first_frame, d_lo, d_hi, st) != 0) return -1;
        if (launch_movie_stats(d_mov, n, nullptr, d_mm, d_hist, st) != 0) return -1;
    }
    return c.finish();
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
    Call c("decode_movie");
    auto& l = c.in("lo", lo, n);
    auto& hh = c.in("hi", hi, n);
    auto& m = c.out("movie", movie, n * 2);
    if (c.stage() != 0) return -1;
    if (launch_decode_movie((const u8*)l.dev, (const u8*)hh.dev, nframes, w, h, gop, delta, first_frame, (u16*)m.dev, st) != 0) return -1;
    return c.finish();
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
Table<LossyState> g_lossy;
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
    return g_lossy.add(s);
}

void rirb_lossy_close(int handle) { g_lossy.remove(handle); }

int rirb_lossy_set_parameter(int handle, const char* key, const char* value)
{
    auto s = g_lossy.get(handle);
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
    auto s = g_lossy.get(handle);
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
    auto s = find_handle_here(g_lossy, handle, "lossy_add_images");
    if (!s) return -1;
    if (!frames || !out || nframes < 0) {
        set_error("lossy_add_images: bad arguments");
        return -1;
    }
    if (nframes == 0) return 0;
    RIRB_REQUIRE_DEVICE();
    cudaStream_t st = tls.stream;
    const int w = s->w, h = s->h, n = w * h, ns = w * s->stop_h;
    const size_t bytes = (size_t)n * 2 * (size_t)nframes;
    Call c("lossy_add_images");
    auto& i = c.in("frames", frames, bytes);
    auto& o = c.out("out", out, bytes);
    auto& e = c.out("errors", errors, sizeof(int) * 2 * (size_t)nframes);
    e.staged = false;  // copied from the state's own buffer at the end, in any memory
    if (c.stage() != 0) return -1;
    const u16* d_in = (const u16*)i.dev;
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
                auto bp = g_bad_pixels.get(s->bp_handle);
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
            auto bp = g_bad_pixels.get(s->bp_handle);
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
    return c.finish(errors && !e.on_device);
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
    auto s = find_handle_here(g_bad_pixels, handle, "process_movie_host");
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
        Call scope("process_movie_host");  // gives back the order buffer launch_translate_u16 may take, sub-chunk by sub-chunk
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
    cudaStream_t st = tls.stream;
    Call c("movie_stats");
    auto& px = c.in("pixels", pixels, n * 2);
    auto& mm = c.out("minmax", minmax, 2 * sizeof(unsigned), accumulate != 0);
    auto& hs = c.out("hist", hist, 65536 * sizeof(unsigned long long), accumulate != 0);
    if (c.stage() != 0) return -1;
    unsigned* d_mm = (unsigned*)mm.dev;
    unsigned long long* d_hist = (unsigned long long*)hs.dev;
    if (!accumulate && launch_stats_init(d_mm, d_hist, st) != 0) return -1;
    if (launch_movie_stats((const u16*)px.dev, n, nullptr, d_mm, d_hist, st) != 0) return -1;
    return c.finish();
}

int rirb_hist_quantile(const unsigned long long* hist, long long count, float percent)
{
    if (!hist) {
        set_error("hist_quantile: bad arguments");
        return -1;
    }
    RIRB_REQUIRE_DEVICE();
    cudaStream_t st = tls.stream;
    Call c("hist_quantile");
    auto& hs = c.in("hist", hist, 65536 * sizeof(unsigned long long));
    if (c.stage() != 0) return -1;
    int* d_out = (int*)scratch_buffer(sizeof(int));
    if (!d_out) return -1;
    if (launch_hist_quantile((const unsigned long long*)hs.dev, count, percent, 0, d_out, st) != 0) return -1;
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
    Call c("find_median_pixel");
    auto& px = c.in("pixels", pixels, (size_t)size * 2);
    auto& m = c.in("mask", mask, (size_t)size);
    if (c.stage() != 0) return -1;
    unsigned long long* d_hist = (unsigned long long*)scratch_buffer(sizeof(unsigned long long) * 65536);
    unsigned* d_mm = (unsigned*)scratch_buffer(sizeof(unsigned) * 2);
    int* d_out = (int*)scratch_buffer(sizeof(int));
    if (!d_hist || !d_mm || !d_out) return -1;
    if (launch_stats_init(d_mm, d_hist, st) != 0) return -1;
    if (launch_movie_stats((const u16*)px.dev, (size_t)size, (const u8*)m.dev, d_mm, d_hist, st) != 0) return -1;
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
    Call c("get_background");
    auto& px = c.in("pixels", pixels, (size_t)size * 2);
    if (c.stage() != 0) return -1;
    unsigned long long* d_hist = (unsigned long long*)scratch_buffer(sizeof(unsigned long long) * 65536);
    unsigned* d_mm = (unsigned*)scratch_buffer(sizeof(unsigned) * 2);
    unsigned* d_out = (unsigned*)scratch_buffer(sizeof(unsigned));
    if (!d_hist || !d_mm || !d_out) return -1;
    if (launch_stats_init(d_mm, d_hist, st) != 0) return -1;
    if (launch_movie_stats((const u16*)px.dev, (size_t)size, nullptr, d_mm, d_hist, st) != 0) return -1;
    if (launch_hist_mode4(d_hist, d_out, st) != 0) return -1;
    unsigned r = 0;
    RIRB_CUDA_OK(cudaMemcpyAsync(&r, d_out, sizeof(unsigned), cudaMemcpyDeviceToHost, st));
    RIRB_CUDA_OK(cudaStreamSynchronize(st));
    return (int)r;
}

// =================================================================================================
// connected components (label.cu)
// =================================================================================================
int rirb_label_batch(const unsigned short* frames, int w, int h, long long nframes, const unsigned short* thresholds,
                     long long n_thresholds, int connectivity, int* labels, int* counts, long long* stats, int max_components)
{
    if (connectivity != 4 && connectivity != 8) {
        set_error("label_batch: connectivity must be 4 or 8, not %d", connectivity);
        return -1;
    }
    if (!frames || !thresholds || !labels || !counts || w <= 0 || h <= 0 || (long long)w * h > INT_MAX || nframes < 0 ||
        (n_thresholds != 1 && n_thresholds != nframes) || (stats && max_components < 0)) {
        set_error("label_batch: bad arguments");
        return -1;
    }
    if (nframes == 0) return 0;
    RIRB_REQUIRE_DEVICE();
    const int cap = stats ? max_components : 0;
    const size_t npx = (size_t)w * h * (size_t)nframes;
    const size_t sbytes = (size_t)nframes * cap * 10 * sizeof(long long);
    cudaStream_t st = tls.stream;
    Call c("label_batch");
    auto& fr = c.in("frames", frames, npx * 2);
    auto& th = c.in("thresholds", thresholds, 2 * (size_t)n_thresholds);
    auto& lb = c.out("labels", labels, npx * 4);
    auto& ct = c.out("counts", counts, 4 * (size_t)nframes);
    // rows past K_t keep what the caller had in them: a host stats array goes up first
    auto& sts = c.out("stats", sbytes ? stats : nullptr, sbytes, true);
    if (c.stage() != 0) return -1;
    if (launch_label((const u16*)fr.dev, w, h, nframes, (const u16*)th.dev, n_thresholds > 1, connectivity, (int*)lb.dev, (int*)ct.dev,
                     (long long*)sts.dev, cap, st) != 0)
        return -1;
    return c.finish();
}

int rirb_label_movie(const unsigned short* frames, int w, int h, long long nframes, const unsigned short* thresholds,
                     long long n_thresholds, int connectivity, int* labels, int* count, long long* stats, int max_events)
{
    if (connectivity != 6 && connectivity != 18 && connectivity != 26) {
        set_error("label_movie: connectivity must be 6, 18 or 26, not %d", connectivity);
        return -1;
    }
    if (!frames || !thresholds || !labels || !count || w <= 0 || h <= 0 || (long long)w * h > INT_MAX || nframes < 0 ||
        (n_thresholds != 1 && n_thresholds != nframes) || max_events < 0) {
        set_error("label_movie: bad arguments");
        return -1;
    }
    if (nframes > 0 && (double)w * h * (double)nframes >= 281474976710656.0) {  // 2^48: the argmax column's packing
        set_error("label_movie: %lld frames of %d x %d are 2^48 voxels or more", nframes, w, h);
        return -1;
    }
    if (nframes == 0) {
        if (!is_device_ptr(count)) {
            *count = 0;
            return 0;
        }
        RIRB_REQUIRE_DEVICE();
        RIRB_CUDA_OK(cudaMemsetAsync(count, 0, sizeof(int), tls.stream));
        return 0;
    }
    RIRB_REQUIRE_DEVICE();
    const int cap = stats ? max_events : 0;
    const size_t npx = (size_t)w * h * (size_t)nframes;
    const size_t sbytes = (size_t)cap * 13 * sizeof(long long);
    cudaStream_t st = tls.stream;
    Call c("label_movie");
    auto& fr = c.in("frames", frames, npx * 2);
    auto& th = c.in("thresholds", thresholds, 2 * (size_t)n_thresholds);
    auto& lb = c.out("labels", labels, npx * 4);
    auto& ct = c.out("count", count, sizeof(int));
    // rows past K keep what the caller had in them: a host stats array goes up first
    auto& sts = c.out("stats", sbytes ? stats : nullptr, sbytes, true);
    if (c.stage() != 0) return -1;
    if (launch_label_movie((const u16*)fr.dev, w, h, nframes, (const u16*)th.dev, n_thresholds > 1, connectivity, (int*)lb.dev,
                           (int*)ct.dev, (long long*)sts.dev, cap, st) != 0)
        return -1;
    return c.finish();
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
