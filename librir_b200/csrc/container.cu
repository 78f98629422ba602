// librir_b200/csrc/container.cu -- the on-disk formats either side of the path (SURVEY.md 8f-3).
//
// Host code (the zstd kernels are zcoder.cu / zdecoder.cu): what the per-frame path reads from and writes to when it runs inside
// librir's own file tooling.
//   attribute trailer   rir::FileAttributes, FileAttributes.cpp:51-165 (strings, maps), :250-372
//                       (open / openReadOnly), :454-514 (writeIfDirty); C interface tools.cpp:87-350
//   zstd movie file     ZFile.cpp:18-46 (two 128-byte headers), :483-542 (record = i64 timestamp,
//                       u32 compressed size, zstd frame of the raw uint16 image), :410-452 (close:
//                       sample count patched into the header, image positions stored as the global
//                       attribute "positions" of the trailer), :124-253 (open for reading)
//
// Layout of a file, all integers little-endian:
//   [128 B header: version=1, triggers=1, compression=1]
//   [128 B trigger: 11 x u64 = date, rate, samples, samples_pre_trigger, type=1, nb_channels=1,
//                   data_type=0, data_format=3, data_repetition=1, data_size_x, data_size_y]
//   samples x [i64 timestamp][u32 csize][csize bytes: ZSTD frame of w*h uint16]
//   trailer:  map(global) , samples x map(frame) , samples x i64 timestamp , u64 samples ,
//             u64 trailer_bytes , "H264ATTRIBUTES"
//   map    = u64 count, then count x (string key, string value) in key order
//   string = u64 n, n bytes; values of >= 1000 bytes that zstd shrinks are stored as
//            u64 (8 + csize) | 1<<63, u64 raw size, zstd bytes
// Methods 2 and 3 -- which the reference documents ("blosc + ZSTD", video_io.h:298-305, ZFile.cpp:77) but never
// implemented (ZFile.cpp:492-499 compresses only when compression == 1) -- are defined HERE as the north star's
// pre-coder in front of the same zstd stage: the payload of a record is the ZSTD frame of [low-byte plane | high-byte
// plane] (w*h bytes each) of the image (method 2) or of its temporal residual (method 3: key frame every GOP frames,
// otherwise (frame[t] - frame[t-1]) mod 2^16; the GOP is stored in trigger word 12 and as the global attribute "GOP").
// The split / delta and their inverses run on the GPU (rirb_precode_movie / rirb_decode_movie), whole GOPs per launch.
// The entropy stage is host zstd by default.  What this file adds over the reference is that a run of frames is compressed /
// decompressed by a pool of host threads while the records keep their order, that frames may be handed over as device
// pointers (downloaded / uploaded in one copy per call), and that a writer may switch to the device coder (zcoder.cu,
// rirb_z_set_coder): the payloads are then encoded in HBM and one copy per pass brings back the packed records.
// A method-1 read into device memory of records without LZ sequences (the device coder's) goes the other way through
// the device decoder (zdecoder.cu): a pass's records are one span of the file, read into pinned memory, uploaded in one
// copy and decoded in HBM; a record it refuses (checksum, dictionary, ...) or finds malformed is decoded by host zstd
// instead.  Records with sequences stay on the host pool, which decodes them faster (DESIGN.md 7 f-3, r4), and so does
// method 1 into host memory, so a host-only caller never initialises CUDA.  The "zstd_decoder" switch: 2 sends every
// read that ends on the device (methods 2/3 too) through the device decoder, 0 none; both for A/B runs.
#include <dlfcn.h>
#include <stdint.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>
#include <sys/stat.h>
#include <unistd.h>

#include <algorithm>
#include <atomic>
#include <chrono>
#include <map>
#include <memory>
#include <mutex>
#include <string>
#include <thread>
#include <vector>

#include "../../include/librir_b200.h"
#include "common.cuh"
#include "handles.h"
#include "kernels.h"

namespace rirb {

// ---- zstd, resolved at run time (the image ships libzstd.so.1 without headers) ----------------
struct Zstd {
    size_t (*compressBound)(size_t) = nullptr;
    size_t (*compress)(void*, size_t, const void*, size_t, int) = nullptr;
    size_t (*decompress)(void*, size_t, const void*, size_t) = nullptr;
    unsigned (*isError)(size_t) = nullptr;
    // reusable contexts: ZSTD_compress / ZSTD_decompress build and free one per call (megabytes of tables per frame);
    // the bytes produced are the same
    void* (*createCCtx)() = nullptr;
    size_t (*freeCCtx)(void*) = nullptr;
    size_t (*compressCCtx)(void*, void*, size_t, const void*, size_t, int) = nullptr;
    void* (*createDCtx)() = nullptr;
    size_t (*freeDCtx)(void*) = nullptr;
    size_t (*decompressDCtx)(void*, void*, size_t, const void*, size_t) = nullptr;
    bool ok = false;
    bool ctx = false;
};
static const Zstd& zstd()
{
    static const Zstd z = [] {
        Zstd r;
        void* h = nullptr;
        const char* env = getenv("LIBRIR_B200_ZSTD_LIB");
        const char* names[] = {env, "libzstd.so.1", "libzstd.so"};
        for (const char* n : names)
            if (n && *n && (h = dlopen(n, RTLD_NOW | RTLD_LOCAL))) break;
        if (!h) return r;
        r.compressBound = (size_t(*)(size_t))dlsym(h, "ZSTD_compressBound");
        r.compress = (size_t(*)(void*, size_t, const void*, size_t, int))dlsym(h, "ZSTD_compress");
        r.decompress = (size_t(*)(void*, size_t, const void*, size_t))dlsym(h, "ZSTD_decompress");
        r.isError = (unsigned (*)(size_t))dlsym(h, "ZSTD_isError");
        r.ok = r.compressBound && r.compress && r.decompress && r.isError;
        r.createCCtx = (void* (*)())dlsym(h, "ZSTD_createCCtx");
        r.freeCCtx = (size_t(*)(void*))dlsym(h, "ZSTD_freeCCtx");
        r.compressCCtx = (size_t(*)(void*, void*, size_t, const void*, size_t, int))dlsym(h, "ZSTD_compressCCtx");
        r.createDCtx = (void* (*)())dlsym(h, "ZSTD_createDCtx");
        r.freeDCtx = (size_t(*)(void*))dlsym(h, "ZSTD_freeDCtx");
        r.decompressDCtx = (size_t(*)(void*, void*, size_t, const void*, size_t))dlsym(h, "ZSTD_decompressDCtx");
        r.ctx = r.createCCtx && r.freeCCtx && r.compressCCtx && r.createDCtx && r.freeDCtx && r.decompressDCtx;
        return r;
    }();
    return z;
}
static bool need_zstd()
{
    if (zstd().ok) return true;
    set_error("libzstd.so.1 not found (set LIBRIR_B200_ZSTD_LIB)");
    return false;
}

// ------------------------------------------------------------------------------------------------
// attribute trailer
// ------------------------------------------------------------------------------------------------
static const char k_magic[] = "H264ATTRIBUTES";
constexpr size_t k_magic_len = 14;
constexpr size_t k_min_compress = 1000;  // MIN_SIZE_FOR_COMRPESSION, FileAttributes.cpp:26
constexpr uint64_t k_cflag = 1ull << 63;

typedef std::map<std::string, std::string> AttrMap;

struct Trailer {
    AttrMap global;
    std::vector<AttrMap> frames;
    std::vector<int64_t> times;
};

static void put_u64(std::string& s, uint64_t v) { s.append(reinterpret_cast<const char*>(&v), 8); }

static void put_string(std::string& s, const std::string& v)
{
    if (v.size() >= k_min_compress && zstd().ok) {  // FileAttributes.cpp:61-85: level 0, kept only if smaller
        std::vector<char> buf(zstd().compressBound(v.size()));
        const size_t c = zstd().compress(buf.data(), buf.size(), v.data(), v.size(), 0);
        if (!zstd().isError(c) && c < v.size()) {
            put_u64(s, (uint64_t)(c + 8) | k_cflag);
            put_u64(s, (uint64_t)v.size());
            s.append(buf.data(), c);
            return;
        }
    }
    put_u64(s, (uint64_t)v.size());
    s.append(v);
}
static void put_map(std::string& s, const AttrMap& m)
{
    put_u64(s, (uint64_t)m.size());
    for (const auto& kv : m) {
        put_string(s, kv.first);
        put_string(s, kv.second);
    }
}
static std::string serialize(const Trailer& t)
{
    std::string s;
    put_map(s, t.global);
    for (const auto& m : t.frames) put_map(s, m);
    for (int64_t ts : t.times) put_u64(s, (uint64_t)ts);
    put_u64(s, (uint64_t)t.times.size());
    put_u64(s, (uint64_t)(s.size() + 8 + k_magic_len));  // the whole trailer, this field and the magic included
    s.append(k_magic, k_magic_len);
    return s;
}

// Bounds-checked reader over the trailer bytes (the reference trusts the file; a damaged one must
// fail here, not read out of bounds).
struct Cursor {
    const char* p;
    const char* end;
    bool ok = true;
    uint64_t u64()
    {
        if (!ok || end - p < 8) {
            ok = false;
            return 0;
        }
        uint64_t v;
        memcpy(&v, p, 8);
        p += 8;
        return v;
    }
    std::string str()
    {
        uint64_t n = u64();
        const bool comp = (n & k_cflag) != 0;
        n &= ~k_cflag;
        if (!ok || (uint64_t)(end - p) < n) {
            ok = false;
            return std::string();
        }
        if (!comp) {
            std::string r(p, p + n);
            p += n;
            return r;
        }
        if (n < 8) {
            ok = false;
            return std::string();
        }
        uint64_t raw;
        memcpy(&raw, p, 8);
        std::string r;
        if (raw > (1ull << 32) || !zstd().ok) {
            ok = false;
            return r;
        }
        r.resize(raw);
        const size_t got = zstd().decompress(&r[0], raw, p + 8, n - 8);
        if (zstd().isError(got) || got != raw) r.clear();  // FileAttributes.cpp:131-136: an empty value, not a failure
        p += n;
        return r;
    }
    AttrMap map()
    {
        AttrMap m;
        const uint64_t n = u64();
        for (uint64_t i = 0; ok && i < n; ++i) {
            std::string k = str();
            std::string v = str();
            if (ok) m[k] = v;
        }
        return m;
    }
};

// tail = the last `size` bytes of a file; returns the trailer size found there, 0 if there is none, -1 if damaged
static long long parse_trailer(const char* data, size_t size, Trailer& t)
{
    if (size < 16 + k_magic_len) return 0;
    const char* e = data + size;
    if (memcmp(e - k_magic_len, k_magic, k_magic_len) != 0) return 0;
    uint64_t count, tsize;
    memcpy(&count, e - k_magic_len - 16, 8);
    memcpy(&tsize, e - k_magic_len - 8, 8);
    if (tsize < 16 + k_magic_len + 8 || tsize > size || count > (tsize / 8)) return -1;
    Cursor c{e - tsize, e - k_magic_len - 16};
    t.global = c.map();
    t.frames.assign(count, AttrMap());
    for (uint64_t i = 0; c.ok && i < count; ++i) t.frames[i] = c.map();
    t.times.assign(count, 0);
    for (uint64_t i = 0; c.ok && i < count; ++i) t.times[i] = (int64_t)c.u64();
    return c.ok ? (long long)tsize : -1;
}

static long long file_bytes(const char* name)
{
    struct stat st;
    return stat(name, &st) == 0 ? (long long)st.st_size : -1;
}

struct AttrsFile {
    std::string filename;  // empty: opened from memory, never written
    Trailer t;
    size_t table_size = 0;       // 0 = the in-memory table differs from the file's (FileAttributes.cpp:456)
    size_t file_table_size = 0;  // bytes of the trailer currently at the end of the file
    std::mutex mu;
};

// FileAttributes::open, FileAttributes.cpp:316-372 -- including its habit of creating (truncating) a file
// that is shorter than a trailer.
static bool attrs_open(AttrsFile& a, const char* filename)
{
    a.filename = filename;
    const long long fsize = file_bytes(filename);
    if (fsize >= (long long)(16 + k_magic_len)) {
        FILE* f = fopen(filename, "rb");
        if (!f) return false;
        char tail[16 + k_magic_len];
        fseek(f, (long)(fsize - (long long)sizeof(tail)), SEEK_SET);
        if (fread(tail, 1, sizeof(tail), f) != sizeof(tail)) {
            fclose(f);
            return false;
        }
        if (memcmp(tail + 16, k_magic, k_magic_len) == 0) {
            uint64_t tsize;
            memcpy(&tsize, tail + 8, 8);
            if (tsize > (uint64_t)fsize) {
                fclose(f);
                return false;
            }
            std::vector<char> buf(tsize);
            fseek(f, (long)(fsize - (long long)tsize), SEEK_SET);
            const bool got = fread(buf.data(), 1, tsize, f) == tsize;
            fclose(f);
            if (!got || parse_trailer(buf.data(), buf.size(), a.t) <= 0) return false;
            a.table_size = a.file_table_size = tsize;
            return true;
        }
        fclose(f);
        return true;  // no trailer yet: one is appended when the handle is closed
    }
    FILE* f = fopen(filename, "wb");
    if (!f) return false;
    fclose(f);
    return true;
}

// FileAttributes::writeIfDirty, FileAttributes.cpp:454-514: the trailer replaces the one at the end of the file.
static void attrs_write_if_dirty(AttrsFile& a)
{
    if (a.table_size != 0 || a.filename.empty()) return;
    const std::string s = serialize(a.t);
    a.table_size = s.size();
    const long long fsize = file_bytes(a.filename.c_str());
    if (fsize < 0 || (size_t)fsize < a.file_table_size) {
        a.table_size = 0;
        return;
    }
    const long long at = fsize - (long long)a.file_table_size;
    if (a.table_size < a.file_table_size && truncate(a.filename.c_str(), at + (long long)a.table_size) != 0) {
        a.table_size = 0;
        return;
    }
    FILE* f = fopen(a.filename.c_str(), "r+b");
    if (!f) {
        a.table_size = 0;
        return;
    }
    fseek(f, (long)at, SEEK_SET);
    const bool ok = fwrite(s.data(), 1, s.size(), f) == s.size();
    fclose(f);
    if (!ok) {
        a.table_size = 0;
        return;
    }
    a.file_table_size = a.table_size;
}

static Table<AttrsFile> g_attrs;

static int copy_out(const std::string& s, char* dst, int* len)
{
    if (!len) return -1;
    if (*len < (int)s.size()) {
        *len = (int)s.size();
        return -2;
    }
    *len = (int)s.size();
    if (dst && !s.empty()) memcpy(dst, s.data(), s.size());
    return 0;
}
static int nth(const AttrMap& m, int pos, bool value, char* dst, int* len)
{
    if (pos < 0 || pos >= (int)m.size()) return -1;
    auto it = m.begin();
    std::advance(it, pos);
    return copy_out(value ? it->second : it->first, dst, len);
}
static AttrMap unpack_map(const char* keys, const int* key_lens, const char* values, const int* value_lens, int count)
{
    AttrMap m;
    for (int i = 0; i < count; ++i) {
        std::string k(keys, keys + key_lens[i]);
        std::string v(values, values + value_lens[i]);
        keys += key_lens[i];
        values += value_lens[i];
        m.insert(std::make_pair(k, v));  // first occurrence of a key wins (tools.cpp:318)
    }
    return m;
}

// ------------------------------------------------------------------------------------------------
// zstd movie file
// ------------------------------------------------------------------------------------------------
struct ZHeader {  // BIN_HEADER + BIN_TRIGGER, ZFile.cpp:18-46
    unsigned char head[128];
    uint64_t trig[16];
};
static_assert(sizeof(ZHeader) == 256, "two 128-byte blocks");
enum { T_DATE, T_RATE, T_SAMPLES, T_PRE, T_TYPE, T_CHANNELS, T_DTYPE, T_FORMAT, T_REPETITION, T_SIZE_X, T_SIZE_Y, T_SPARE, T_GOP };

static int pool_size(int threads, long long jobs)
{
    int n = threads > 0 ? threads : (int)std::thread::hardware_concurrency();
    if (n < 1) n = 1;
    if (n > 64) n = 64;
    if ((long long)n > jobs) n = (int)jobs;
    return n < 1 ? 1 : n;
}
// fn(job, worker): jobs are handed out one by one, `worker` < pool size names the calling thread
template <typename F> static void parallel_for(long long jobs, int nworkers, F&& fn)
{
    if (nworkers <= 1 || jobs <= 1) {
        for (long long i = 0; i < jobs; ++i) fn(i, 0);
        return;
    }
    std::atomic<long long> next{0};
    std::vector<std::thread> pool;
    for (int t = 0; t < nworkers && t < jobs; ++t)
        pool.emplace_back([&, t] {
            for (long long i = next.fetch_add(1); i < jobs; i = next.fetch_add(1)) fn(i, t);
        });
    for (auto& th : pool) th.join();
}

// One zstd context per worker, for the duration of a call.
struct Contexts {
    std::vector<void*> c;
    bool compress;
    Contexts(int n, bool comp) : c((size_t)n, nullptr), compress(comp) {}
    ~Contexts()
    {
        for (void* p : c)
            if (p) (compress ? zstd().freeCCtx : zstd().freeDCtx)(p);
    }
    void* get(int worker)
    {
        if (!zstd().ctx) return nullptr;
        if (!c[worker]) c[worker] = compress ? zstd().createCCtx() : zstd().createDCtx();
        return c[worker];
    }
};
static size_t z_compress(void* cctx, void* dst, size_t cap, const void* src, size_t n, int level)
{
    return cctx ? zstd().compressCCtx(cctx, dst, cap, src, n, level) : zstd().compress(dst, cap, src, n, level);
}
static size_t z_decompress(void* dctx, void* dst, size_t cap, const void* src, size_t n)
{
    return dctx ? zstd().decompressDCtx(dctx, dst, cap, src, n) : zstd().decompress(dst, cap, src, n);
}

// A grow-only buffer in device memory or pinned host memory.
struct ZBuf {
    bool pinned;
    char* p = nullptr;
    size_t bytes = 0;
    explicit ZBuf(bool pin) : pinned(pin) {}
    // false + set_error when memory runs out
    bool grow(size_t need)
    {
        if (bytes >= need) return true;
        release();
        if ((pinned ? cudaMallocHost((void**)&p, need) : cudaMalloc((void**)&p, need)) != cudaSuccess) {
            cudaGetLastError();
            p = nullptr;
            set_error("zstd movie file: out of %s memory (%zu bytes)", pinned ? "pinned host" : "device", need);
            return false;
        }
        bytes = need;
        return true;
    }
    void release()
    {
        if (p) (void)(pinned ? cudaFreeHost(p) : cudaFree(p));
        p = nullptr;
        bytes = 0;
    }
};

// Every work buffer of an open file, all on one device: the pinned planes of methods 2 / 3 ([frame][lo plane | hi plane]), the
// device frames | lo planes | hi planes of a pass, the device coder's or decoder's scratch, and a pass's records on the device
// and their pinned copy.
struct ZBuffers {
    ZBuf host_planes{true}, frames{false}, scratch{false}, records{false}, host_records{true};
    int device = -1;
    bool empty() const { return !host_planes.p && !frames.p && !scratch.p && !records.p && !host_records.p; }
    void release()
    {
        for (ZBuf* b : {&host_planes, &frames, &scratch, &records, &host_records}) b->release();
        (void)cudaGetLastError();
        device = -1;
    }
};

// Pinning and unpinning cost 10-800 ms a time on the measured host (a VM), more than reading a 400-frame file, so a closed file
// PARKS its buffers here and the next file of the process that needs buffers on that device takes them over.  One set is kept,
// the newer: files opened one after another then hand on one set that has grown to what each of them needed, and of two files
// open at once the one closed last is the likelier to resemble the next.  The older set is freed.
static std::mutex g_parked_mu;
static ZBuffers g_parked;
static void z_park(ZBuffers& b)
{
    if (b.empty()) return;
    {
        std::lock_guard<std::mutex> lock(g_parked_mu);
        std::swap(b, g_parked);
    }
    b.release();
}

struct ZMovie {
    bool writing = false;
    std::string filename;
    FILE* f = nullptr;
    ZHeader hdr;
    int w = 0, h = 0, clevel = 0, method = 1;
    std::vector<int64_t> times, positions;
    std::vector<uint32_t> sizes;  // reading: compressed size of each record
    long long pos = 0;            // writing: bytes so far
    // kept between calls so that one-frame-per-call writers / readers do not rebuild them every frame
    std::vector<std::unique_ptr<char[]>> slots;  // compressed records of the batch in flight (compressBound each)
    std::unique_ptr<Contexts> ctx;
    std::unique_ptr<char[]> raw;  // reading: the record bytes of the batch in flight
    size_t raw_cap = 0;
    // methods 2 / 3 (byte planes, + temporal delta): the pre-coder runs on the GPU in whole GOPs
    int gop = 50;
    std::vector<u16> pending;            // writing: frames that do not fill a GOP yet (host)
    std::vector<int64_t> pending_times;
    ZBuffers buf;                        // use through buffers()
    size_t dev_frames = 0;               // the frames | lo planes | hi planes layout of buf.frames is for this many frames
    long long cache_first = -1, cache_count = 0;  // reading: decoded frames [cache_first, +cache_count) still in buf.frames
    std::mutex mu;
    // writing with the device coder (coder 1)
    int coder = 0;
    bool lz = false;  // the device coder with LZ matches (rirb_z_set_lz): rirb_zstd_encode_batch_lz's frames
    ~ZMovie()
    {
        if (f) fclose(f);
        z_park(buf);
    }
    // the work buffers on the current device: a change of device frees them and takes over a set parked on the new one
    ZBuffers& buffers()
    {
        int dev = 0;
        cudaGetDevice(&dev);
        if (buf.device != dev) {
            buf.release();
            cache_first = -1;
            std::lock_guard<std::mutex> lock(g_parked_mu);
            if (g_parked.device == dev) std::swap(buf, g_parked);
            buf.device = dev;
        }
        return buf;
    }
    // frames and planes for m frames; false + set_error when memory runs out
    bool reserve(size_t m)
    {
        const size_t npx = (size_t)w * h;
        ZBuffers& b = buffers();
        dev_frames = std::max(dev_frames, m);  // the layout only grows
        return b.frames.grow(dev_frames * npx * 4) && b.host_planes.grow(dev_frames * npx * 2);
    }
    char* host_planes() const { return buf.host_planes.p; }
    u16* dev_movie() const { return (u16*)buf.frames.p; }
    u8* dev_lo() const { return (u8*)buf.frames.p + dev_frames * (size_t)w * h * 2; }
    u8* dev_hi() const { return dev_lo() + dev_frames * (size_t)w * h; }
};
static Table<ZMovie> g_zfiles;

// Two pinned staging buffers for frames that live in HBM: batch b+1 moves while batch b is (de)compressed.
struct PinnedPair {
    char* buf[2] = {nullptr, nullptr};
    cudaEvent_t ev[2] = {nullptr, nullptr};
    bool init(size_t bytes)
    {
        for (int i = 0; i < 2; ++i)
            if (cudaMallocHost((void**)&buf[i], bytes) != cudaSuccess || cudaEventCreateWithFlags(&ev[i], cudaEventDisableTiming) != cudaSuccess) {
                cudaGetLastError();
                return false;
            }
        return true;
    }
    ~PinnedPair()
    {
        for (int i = 0; i < 2; ++i) {
            if (buf[i]) cudaFreeHost(buf[i]);
            if (ev[i]) cudaEventDestroy(ev[i]);
        }
    }
};

// Host-only callers must not pay for CUDA: initialising the driver alone costs ~0.7 s on a B200 host (measured,
// scripts/probes/zstd_write_probe.py).  A pointer can only be device memory if the driver is already loaded AND
// initialised AND some device's primary context is active; driver entry points answer NOT_INITIALIZED instead of
// initialising, so asking is free.
static bool any_context_active()
{
    void* h = dlopen("libcuda.so.1", RTLD_NOW | RTLD_NOLOAD);
    if (!h) return false;
    typedef int (*count_fn)(int*);
    typedef int (*state_fn)(int, unsigned*, int*);
    const count_fn count = (count_fn)dlsym(h, "cuDeviceGetCount");
    const state_fn state = (state_fn)dlsym(h, "cuDevicePrimaryCtxGetState");
    bool active = false;
    int n = 0;
    if (count && state && count(&n) == 0)
        for (int d = 0; d < n && !active; ++d) {
            unsigned flags = 0;
            int on = 0;
            active = state(d, &flags, &on) == 0 && on != 0;
        }
    dlclose(h);
    return active;
}
static bool device_pointer(const void* p)
{
    if (!any_context_active()) return false;
    cudaPointerAttributes a;
    if (cudaPointerGetAttributes(&a, p) != cudaSuccess) {
        cudaGetLastError();
        return false;
    }
    return a.type == cudaMemoryTypeDevice || a.type == cudaMemoryTypeManaged;
}

// all n bytes at file offset `at` (one pread / pwrite may move fewer); false on an error or the end of the file
static bool pread_all(int fd, void* p, size_t n, long long at)
{
    for (size_t done = 0; done < n;) {
        const ssize_t r = pread(fd, (char*)p + done, n - done, (off_t)(at + (long long)done));
        if (r <= 0) return false;
        done += (size_t)r;
    }
    return true;
}
static bool pwrite_all(int fd, const void* p, size_t n, long long at)
{
    for (size_t done = 0; done < n;) {
        const ssize_t r = pwrite(fd, (const char*)p + done, n - done, (off_t)(at + (long long)done));
        if (r <= 0) return false;
        done += (size_t)r;
    }
    return true;
}

// frames in one pass of the GPU paths: about 64 MB of pixels, in whole GOPs of `gop` frames
static long long z_pass_frames(const ZMovie* z, long long gop)
{
    const long long chunk = std::max<long long>(1, (64ll << 20) / ((long long)z->w * z->h * 2));
    return std::max(gop, chunk / gop * gop);
}

// m frames' planes from dev_lo / dev_hi into `planes`, per frame [lo | hi], so that a record's payload is one contiguous run
static cudaError_t interleave_planes(const ZMovie* z, void* planes, long long m, cudaMemcpyKind kind, cudaStream_t st)
{
    const size_t npx = (size_t)z->w * z->h;
    const cudaError_t e = cudaMemcpy2DAsync(planes, 2 * npx, z->dev_lo(), npx, npx, (size_t)m, kind, st);
    return e == cudaSuccess ? cudaMemcpy2DAsync((char*)planes + npx, 2 * npx, z->dev_hi(), npx, npx, (size_t)m, kind, st) : e;
}
// the other way: per frame [lo | hi] at `planes` apart into dev_lo / dev_hi
static cudaError_t split_planes(const ZMovie* z, const void* planes, long long m, cudaMemcpyKind kind, cudaStream_t st)
{
    const size_t npx = (size_t)z->w * z->h;
    const cudaError_t e = cudaMemcpy2DAsync(z->dev_lo(), npx, planes, 2 * npx, npx, (size_t)m, kind, st);
    return e == cudaSuccess ? cudaMemcpy2DAsync(z->dev_hi(), npx, (const char*)planes + npx, 2 * npx, npx, (size_t)m, kind, st) : e;
}

static int z_unreadable(const ZMovie* z)
{
    set_error("z_read_images: a record cannot be read or does not decompress to a %d x %d image", z->w, z->h);
    return -1;
}

}  // namespace rirb

using namespace rirb;

// ================================================================================================
// C ABI: attribute trailer
// ================================================================================================
extern "C" {

int rirb_attrs_open_file(const char* filename)
{
    if (!filename) return 0;
    auto a = std::make_shared<AttrsFile>();
    if (!attrs_open(*a, filename)) {
        set_error("attrs_open_file: cannot open '%s' or its attribute trailer is damaged", filename);
        return 0;
    }
    return g_attrs.add(a);
}

int rirb_attrs_open_from_memory(const void* ptr, long long size)
{
    if (!ptr || size <= 0) return 0;
    auto a = std::make_shared<AttrsFile>();
    const long long tsize = parse_trailer((const char*)ptr, (size_t)size, a->t);
    if (tsize <= 0) {  // FileAttributes::openReadOnly fails when there is no trailer (FileAttributes.cpp:268-272)
        set_error("attrs_open_from_memory: no attribute trailer");
        return 0;
    }
    a->table_size = a->file_table_size = (size_t)tsize;
    return g_attrs.add(a);
}

void rirb_attrs_close(int handle)
{
    auto a = g_attrs.get(handle);
    if (!a) return;
    {
        std::lock_guard<std::mutex> lock(a->mu);
        attrs_write_if_dirty(*a);
    }
    g_attrs.remove(handle);
}

// The reference's attrs_discard calls FileAttributes::close(), which WRITES (tools.cpp:124-131); a drop-in
// has to do the same.  rirb_attrs_abandon below is the entry that really throws the changes away.
void rirb_attrs_discard(int handle) { rirb_attrs_close(handle); }

void rirb_attrs_abandon(int handle) { g_attrs.remove(handle); }

int rirb_attrs_flush(int handle)
{
    auto a = g_attrs.get(handle);
    if (!a) return -1;
    std::lock_guard<std::mutex> lock(a->mu);
    attrs_write_if_dirty(*a);
    return 0;
}

int rirb_attrs_image_count(int handle)
{
    auto a = g_attrs.get(handle);
    return a ? (int)a->t.times.size() : -1;
}

int rirb_attrs_global_attribute_count(int handle)
{
    auto a = g_attrs.get(handle);
    return a ? (int)a->t.global.size() : -1;
}
int rirb_attrs_global_attribute_name(int handle, int pos, char* name, int* len)
{
    auto a = g_attrs.get(handle);
    return a ? nth(a->t.global, pos, false, name, len) : -1;
}
int rirb_attrs_global_attribute_value(int handle, int pos, char* value, int* len)
{
    auto a = g_attrs.get(handle);
    return a ? nth(a->t.global, pos, true, value, len) : -1;
}
int rirb_attrs_frame_attribute_count(int handle, int frame)
{
    auto a = g_attrs.get(handle);
    if (!a || frame < 0 || frame >= (int)a->t.frames.size()) return -1;
    return (int)a->t.frames[frame].size();
}
int rirb_attrs_frame_attribute_name(int handle, int frame, int pos, char* name, int* len)
{
    auto a = g_attrs.get(handle);
    if (!a || frame < 0 || frame >= (int)a->t.frames.size()) return -1;
    return nth(a->t.frames[frame], pos, false, name, len);
}
int rirb_attrs_frame_attribute_value(int handle, int frame, int pos, char* value, int* len)
{
    auto a = g_attrs.get(handle);
    if (!a || frame < 0 || frame >= (int)a->t.frames.size()) return -1;
    return nth(a->t.frames[frame], pos, true, value, len);
}
int rirb_attrs_frame_timestamp(int handle, int frame, long long* time)
{
    auto a = g_attrs.get(handle);
    if (!a || !time || frame < 0 || frame >= (int)a->t.times.size()) return -1;
    *time = a->t.times[frame];
    return 0;
}
int rirb_attrs_timestamps(int handle, long long* times)
{
    auto a = g_attrs.get(handle);
    if (!a || !times) return -1;
    for (size_t i = 0; i < a->t.times.size(); ++i) times[i] = a->t.times[i];
    return 0;
}
int rirb_attrs_set_times(int handle, const long long* times, int size)
{
    auto a = g_attrs.get(handle);
    if (!a || size < 0 || (size > 0 && !times)) return -1;
    std::lock_guard<std::mutex> lock(a->mu);
    a->t.times.resize(size);   // earlier frame attributes are kept up to the new size (FileAttributes.cpp:408-413)
    a->t.frames.resize(size);
    for (int i = 0; i < size; ++i) a->t.times[i] = times[i];
    a->table_size = 0;
    return 0;
}
int rirb_attrs_set_time(int handle, int pos, long long time)
{
    auto a = g_attrs.get(handle);
    if (!a || pos < 0 || pos >= (int)a->t.times.size()) return -1;
    std::lock_guard<std::mutex> lock(a->mu);
    a->t.times[pos] = time;
    a->table_size = 0;
    return 0;
}
int rirb_attrs_set_frame_attributes(int handle, int pos, const char* keys, const int* key_lens, const char* values,
                                    const int* value_lens, int count)
{
    auto a = g_attrs.get(handle);
    if (!a || pos < 0 || pos >= (int)a->t.frames.size() || count < 0) return -1;
    std::lock_guard<std::mutex> lock(a->mu);
    a->t.frames[pos] = unpack_map(keys, key_lens, values, value_lens, count);
    a->table_size = 0;
    return 0;
}
int rirb_attrs_set_global_attributes(int handle, const char* keys, const int* key_lens, const char* values, const int* value_lens,
                                     int count)
{
    auto a = g_attrs.get(handle);
    if (!a || count < 0) return -1;
    std::lock_guard<std::mutex> lock(a->mu);
    a->t.global = unpack_map(keys, key_lens, values, value_lens, count);
    a->table_size = 0;
    return 0;
}

// ================================================================================================
// C ABI: zstd movie file
// ================================================================================================
int rirb_z_open_file_write(const char* filename, int width, int height, int rate, int method, int clevel)
{
    return rirb_z_open_file_write_gop(filename, width, height, rate, method, clevel, 50);
}

int rirb_z_open_file_write_gop(const char* filename, int width, int height, int rate, int method, int clevel, int gop)
{
    if (!filename || width <= 0 || height <= 0 || gop < 1 || gop > 65535) {
        set_error("z_open_file_write: bad arguments");
        return 0;
    }
    if (method < 1 || method > 3) {
        set_error("z_open_file_write: method must be 1 (zstd), 2 (byte planes + zstd) or 3 (temporal delta + byte planes + zstd)");
        return 0;
    }
    if (!need_zstd()) return 0;
    if (method != 1 && rirb_device_count() <= 0) {  // the pre-coder is a CUDA kernel and there is no CPU fallback
        set_error("z_open_file_write: methods 2 and 3 need a CUDA device (no CPU implementation)");
        return 0;
    }
    auto z = std::make_shared<ZMovie>();
    z->f = fopen(filename, "wb");
    if (!z->f) {
        set_error("z_open_file_write: cannot create '%s'", filename);
        return 0;
    }
    z->writing = true;
    z->filename = filename;
    z->w = width;
    z->h = height;
    z->clevel = clevel;
    z->method = method;
    memset(&z->hdr, 0, sizeof(z->hdr));
    z->hdr.head[0] = 1;                      // version
    z->hdr.head[1] = 1;                      // triggers
    z->hdr.head[2] = (unsigned char)method;  // compression
    z->hdr.trig[T_RATE] = (uint64_t)rate;
    z->hdr.trig[T_TYPE] = 1;
    z->hdr.trig[T_CHANNELS] = 1;
    z->hdr.trig[T_FORMAT] = 3;
    z->hdr.trig[T_REPETITION] = 1;
    z->hdr.trig[T_SIZE_X] = (uint64_t)width;
    z->hdr.trig[T_SIZE_Y] = (uint64_t)height;
    z->gop = gop;
    if (method == 3) z->hdr.trig[T_GOP] = (uint64_t)gop;
    if (fwrite(&z->hdr, 1, sizeof(z->hdr), z->f) != sizeof(z->hdr) || fflush(z->f) != 0) {  // records go through pwrite
        set_error("z_open_file_write: write failed");
        return 0;
    }
    z->pos = sizeof(z->hdr);
    return g_zfiles.add(z);
}

// Appends m records (i64 timestamp, u32 size, payload) at z->pos and adds them to the index.  Record i is 12 + sizes[i] bytes at
// rec[i], its payload from rec[i] + 12 on; the heads are written here.  Records that follow one another in memory go out in one
// pwrite (the device coder's packed pass), the others one each, `workers` at a time.
static int z_append_records(ZMovie* z, char* const* rec, const size_t* sizes, const long long* timestamps, long long m, int workers)
{
    std::vector<long long> at((size_t)m + 1, z->pos);  // where each record goes, then the end
    std::vector<long long> runs;                        // the first record of each run that is contiguous in memory, then m
    for (long long i = 0; i < m; ++i) {
        const int64_t ts = timestamps[i];
        const uint32_t c32 = (uint32_t)sizes[i];
        memcpy(rec[i], &ts, 8);
        memcpy(rec[i] + 8, &c32, 4);
        at[i + 1] = at[i] + 12 + (long long)sizes[i];
        if (i == 0 || rec[i] != rec[i - 1] + 12 + sizes[i - 1]) runs.push_back(i);
    }
    runs.push_back(m);
    const int fd = fileno(z->f);
    std::atomic<bool> failed{false};
    parallel_for((long long)runs.size() - 1, workers, [&](long long r, int) {
        const long long i = runs[r], j = runs[r + 1];
        if (!pwrite_all(fd, rec[i], (size_t)(at[j] - at[i]), at[i])) failed = true;
    });
    if (failed) {
        set_error("z_write_images: write failed");
        return -1;
    }
    z->times.insert(z->times.end(), timestamps, timestamps + m);
    z->positions.insert(z->positions.end(), at.begin(), at.end() - 1);
    z->pos = at[m];
    return 0;
}

// m payloads of bytes_each bytes on the DEVICE -> device coder -> records packed back to back -> host -> file
static int z_encode_records(ZMovie* z, const u8* src, long long m, long long bytes_each, long long segment, const long long* timestamps)
{
    cudaStream_t st = current_stream();
    const size_t records = (size_t)m * (size_t)(12 + zcoder_frame_bound(bytes_each, segment));
    const size_t head = ((size_t)(m + 1) * 8 + 63) & ~(size_t)63;  // pinned: the record offsets, then the records
    ZBuffers& b = z->buffers();
    const bool lz = z->lz;
    const size_t scratch = lz ? zcoder_lz_scratch_bytes(m, bytes_each, segment) : zcoder_scratch_bytes(m, bytes_each, segment);
    if (!b.scratch.grow(scratch) || !b.records.grow(records) || !b.host_records.grow(head + records)) return -1;
    long long* dev_off = nullptr;
    if ((lz ? launch_zstd_encode_lz : launch_zstd_encode)(src, m, bytes_each, segment, (u8*)b.records.p, 0, 12, nullptr, &dev_off,
                                                          b.scratch.p, st) != 0)
        return -1;
    long long* off = (long long*)b.host_records.p;
    char* rec = b.host_records.p + head;
    RIRB_CUDA_OK(cudaMemcpyAsync(off, dev_off, (size_t)(m + 1) * 8, cudaMemcpyDeviceToHost, st));
    RIRB_CUDA_OK(cudaStreamSynchronize(st));
    RIRB_CUDA_OK(cudaMemcpyAsync(rec, b.records.p, (size_t)off[m], cudaMemcpyDeviceToHost, st));
    RIRB_CUDA_OK(cudaStreamSynchronize(st));
    std::vector<char*> recs((size_t)m);
    std::vector<size_t> sizes((size_t)m);
    for (long long i = 0; i < m; ++i) {
        recs[i] = rec + off[i];
        sizes[i] = (size_t)(off[i + 1] - off[i] - 12);
    }
    return z_append_records(z, recs.data(), sizes.data(), timestamps, m, 1);
}

// method 1 with the device coder: device frames are encoded where they are, host frames go up in passes of ~64 MB
static int z_write_records_device(ZMovie* z, const void* frames, long long nframes, const long long* timestamps)
{
    const size_t fbytes = (size_t)z->w * z->h * 2;
    const long long chunk = z_pass_frames(z, 1);
    const bool on_device = device_pointer(frames);
    cudaStream_t st = current_stream();
    for (long long done = 0; done < nframes;) {
        const long long m = std::min(chunk, nframes - done);
        const u8* src = (const u8*)frames + (size_t)done * fbytes;
        if (!on_device) {
            if (!z->reserve((size_t)chunk)) return -1;
            RIRB_CUDA_OK(cudaMemcpyAsync(z->dev_movie(), src, (size_t)m * fbytes, cudaMemcpyHostToDevice, st));
            src = (const u8*)z->dev_movie();
        }
        if (z_encode_records(z, src, m, (long long)fbytes, 0, timestamps + done) != 0) return -1;
        done += m;
    }
    return 0;
}

// `nframes` payloads of w*h*2 bytes each, back to back at `frames` (host or device) -> zstd -> records
static int z_write_records(ZMovie* z, const void* frames, long long nframes, const long long* timestamps, int threads)
{
    if (z->coder == 1) return z_write_records_device(z, frames, nframes, timestamps);
    const size_t fbytes = (size_t)z->w * z->h * 2;
    const size_t bound = zstd().compressBound(fbytes);
    const int workers = pool_size(threads, nframes);
    // batches of a few frames per worker: the compressed records of one batch wait in memory (buffers reused
    // from batch to batch, so they stay warm), then go to the file in order
    const long long batch = std::min<long long>(nframes, std::max<long long>(2LL * workers, 8));
    auto& out = z->slots;
    while ((long long)out.size() < batch) out.emplace_back(new char[bound + 12]);
    std::vector<char*> rec((size_t)batch);
    for (long long i = 0; i < batch; ++i) rec[i] = out[i].get();
    std::vector<size_t> csize((size_t)batch);
    if (!z->ctx || (int)z->ctx->c.size() < workers) z->ctx.reset(new Contexts(workers, true));
    Contexts& ctx = *z->ctx;
    const bool on_device = device_pointer(frames);
    PinnedPair pin;
    cudaStream_t st = current_stream();
    auto fetch = [&](long long b0, int slot) -> cudaError_t {  // device frames of the batch at b0 -> pinned slot
        const long long m = std::min(batch, nframes - b0);
        cudaError_t e = cudaMemcpyAsync(pin.buf[slot], (const char*)frames + (size_t)b0 * fbytes, fbytes * m, cudaMemcpyDeviceToHost, st);
        return e == cudaSuccess ? cudaEventRecord(pin.ev[slot], st) : e;
    };
    if (on_device) {
        if (!pin.init(fbytes * batch)) {
            set_error("z_write_images: cannot allocate pinned staging buffers");
            return -1;
        }
        RIRB_CUDA_OK(fetch(0, 0));
    }
    int slot = 0;
    for (long long b0 = 0; b0 < nframes; b0 += batch, slot ^= 1) {
        const long long m = std::min(batch, nframes - b0);
        const char* src = (const char*)frames + (size_t)b0 * fbytes;
        if (on_device) {
            if (b0 + batch < nframes) RIRB_CUDA_OK(fetch(b0 + batch, slot ^ 1));
            RIRB_CUDA_OK(cudaEventSynchronize(pin.ev[slot]));
            src = pin.buf[slot];
        }
        std::atomic<bool> failed{false};
        parallel_for(m, workers, [&](long long i, int t) {
            const size_t c = z_compress(ctx.get(t), rec[i] + 12, bound, src + (size_t)i * fbytes, fbytes, z->clevel);
            if (zstd().isError(c)) failed = true;
            csize[i] = c;
        });
        if (failed) {
            set_error("z_write_images: zstd failed");
            return -1;
        }
        if (z_append_records(z, rec.data(), csize.data(), timestamps + b0, m, workers) != 0) return -1;
    }
    return 0;
}

// RIRB_Z_TRACE=1: wall-clock milliseconds of the phases of a methods-2/3 pass on stderr (diagnostics; off by default)
static bool z_trace()
{
    static const bool on = [] { const char* e = getenv("RIRB_Z_TRACE"); return e && *e == '1'; }();
    return on;
}
struct ZPhase {
    std::chrono::steady_clock::time_point t0 = std::chrono::steady_clock::now();
    void mark(const char* what, long long frames)
    {
        if (!z_trace()) return;
        const auto t1 = std::chrono::steady_clock::now();
        fprintf(stderr, "[rirb z] %-28s %6lld frames %9.3f ms\n", what, frames, std::chrono::duration<double, std::milli>(t1 - t0).count());
        t0 = t1;
    }
};

// m frames on the DEVICE, the first of them a key frame (frame number `first`): pre-coder -> pinned planes -> zstd -> records
static int z_flush_gops(ZMovie* z, const u16* dev_frames, long long m, long long first, const long long* timestamps, int threads)
{
    cudaStream_t st = current_stream();
    ZPhase ph;
    if (rirb_precode_movie(dev_frames, m, z->w, z->h, z->gop, z->method == 3, first, z->dev_lo(), z->dev_hi()) != 0) return -1;
    if (z->coder == 1) {
        // into the frames' part of the device buffer (the pre-coder has read them by now, in stream order)
        u8* planes = (u8*)z->dev_movie();
        RIRB_CUDA_OK(interleave_planes(z, planes, m, cudaMemcpyDeviceToDevice, st));
        const int rc = z_encode_records(z, planes, m, 2 * (long long)z->w * z->h, (long long)z->w * z->h, timestamps);
        ph.mark("write: pre-code + device zstd", m);
        return rc;
    }
    RIRB_CUDA_OK(interleave_planes(z, z->host_planes(), m, cudaMemcpyDeviceToHost, st));
    RIRB_CUDA_OK(cudaStreamSynchronize(st));
    ph.mark("write: pre-code + download", m);
    const int rc = z_write_records(z, z->host_planes(), m, timestamps, threads);
    ph.mark("write: zstd + records", m);
    return rc;
}

// the frames of an unfinished GOP (it starts on a key frame, so it stands on its own)
static int z_flush_pending(ZMovie* z, int threads)
{
    const long long m = (long long)z->pending_times.size();
    if (m == 0) return 0;
    const size_t npx = (size_t)z->w * z->h;
    if (!z->reserve((size_t)m)) return -1;
    RIRB_CUDA_OK(cudaMemcpyAsync(z->dev_movie(), z->pending.data(), (size_t)m * npx * 2, cudaMemcpyHostToDevice, current_stream()));
    const int rc = z_flush_gops(z, z->dev_movie(), m, (long long)z->times.size(), (const long long*)z->pending_times.data(), threads);
    z->pending.clear();
    z->pending_times.clear();
    return rc;
}

// n frames (host or device) onto the pending GOP (host); device frames on the caller's stream, so that the copy sees the work
// queued there
static cudaError_t z_pend(ZMovie* z, const u16* frames, long long n, const long long* timestamps, bool on_device, cudaStream_t st)
{
    const size_t npx = (size_t)z->w * z->h, have = z->pending_times.size();
    z->pending.resize((have + (size_t)n) * npx);
    cudaError_t e = cudaSuccess;
    if (!on_device)
        memcpy(z->pending.data() + have * npx, frames, (size_t)n * npx * 2);
    else if ((e = cudaMemcpyAsync(z->pending.data() + have * npx, frames, (size_t)n * npx * 2, cudaMemcpyDeviceToHost, st)) == cudaSuccess)
        e = cudaStreamSynchronize(st);
    if (e == cudaSuccess) z->pending_times.insert(z->pending_times.end(), timestamps, timestamps + n);
    return e;
}

// methods 2 / 3.  Whole GOPs go through the GPU pre-coder as they come; what does not fill a GOP waits in z->pending
// (host) for the next call or for the close.
static int z_write_precoded(ZMovie* z, const unsigned short* frames, long long nframes, const long long* timestamps, int threads)
{
    const size_t npx = (size_t)z->w * z->h;
    const long long gop = z->method == 3 ? z->gop : 1;
    const long long chunk = z_pass_frames(z, gop);
    const bool on_device = device_pointer(frames);
    cudaStream_t st = current_stream();
    long long done = 0;
    // 1. top up a GOP that is already waiting
    if (!z->pending_times.empty()) {
        done = std::min(nframes, gop - (long long)z->pending_times.size());
        RIRB_CUDA_OK(z_pend(z, frames, done, timestamps, on_device, st));
        if ((long long)z->pending_times.size() == gop && (!z->reserve((size_t)chunk) || z_flush_pending(z, threads) != 0)) return -1;
    }
    // 2. whole GOPs straight from the caller's buffer
    while (nframes - done >= gop) {
        const long long m = std::min(chunk, (nframes - done) / gop * gop);
        if (!z->reserve((size_t)chunk)) return -1;
        const u16* src = frames + (size_t)done * npx;
        if (!on_device) {
            RIRB_CUDA_OK(cudaMemcpyAsync(z->dev_movie(), src, (size_t)m * npx * 2, cudaMemcpyHostToDevice, st));
            src = z->dev_movie();
        }
        if (z_flush_gops(z, src, m, (long long)z->times.size(), timestamps + done, threads) != 0) return -1;
        done += m;
    }
    // 3. the rest waits
    if (done < nframes) RIRB_CUDA_OK(z_pend(z, frames + (size_t)done * npx, nframes - done, timestamps + done, on_device, st));
    return 0;
}

// frames[nframes][h][w] host or device; timestamps host.  Records are appended in order; the frames
// are compressed `threads` at a time (0: all host cores).
int rirb_z_write_images(int handle, const unsigned short* frames, long long nframes, const long long* timestamps, int threads)
{
    auto z = g_zfiles.get(handle);
    if (!z || !z->writing || !frames || nframes < 0 || (nframes > 0 && !timestamps)) {
        set_error("z_write_images: bad handle or arguments");
        return -1;
    }
    if (nframes == 0) return 0;
    std::lock_guard<std::mutex> lock(z->mu);
    return z->method == 1 ? z_write_records(z.get(), frames, nframes, timestamps, threads)
                          : z_write_precoded(z.get(), frames, nframes, timestamps, threads);
}

int rirb_z_set_coder(int handle, int coder)
{
    auto z = g_zfiles.get(handle);
    if (!z || !z->writing) {
        set_error("z_set_coder: not a handle open for writing");
        return -1;
    }
    if (coder != 0 && coder != 1) {
        set_error("z_set_coder: coder must be 0 (host zstd) or 1 (device coder), not %d", coder);
        return -1;
    }
    if (coder == 1 && rirb_device_count() <= 0) {
        set_error("z_set_coder: the device coder needs a CUDA device (no CPU fallback)");
        return -1;
    }
    std::lock_guard<std::mutex> lock(z->mu);
    z->coder = coder;
    return 0;
}

int rirb_z_set_lz(int handle, int on)
{
    auto z = g_zfiles.get(handle);
    if (!z || !z->writing) {
        set_error("z_set_lz: not a handle open for writing");
        return -1;
    }
    if (on != 0 && on != 1) {
        set_error("z_set_lz: on must be 0 or 1, not %d", on);
        return -1;
    }
    if (on && rirb_device_count() <= 0) {
        set_error("z_set_lz: the device coder needs a CUDA device (no CPU fallback)");
        return -1;
    }
    std::lock_guard<std::mutex> lock(z->mu);
    z->lz = on != 0;
    return 0;
}

int rirb_z_write_image(int handle, const unsigned short* img, long long timestamp)
{
    return rirb_z_write_images(handle, img, 1, &timestamp, 1);
}

// Returns the size of the image data (headers + records), like z_close_file; the trailer follows it.
long long rirb_z_close_file(int handle)
{
    auto z = g_zfiles.get(handle);
    if (!z) return 0;
    long long res = 0;
    if (z->writing) {
        std::lock_guard<std::mutex> lock(z->mu);
        if (z->method != 1 && z_flush_pending(z.get(), 0) != 0) set_error("z_close_file: the last frames could not be written");
        z->hdr.trig[T_SAMPLES] = (uint64_t)z->times.size();
        if (pwrite(fileno(z->f), z->hdr.trig, 128, 128) != 128) set_error("z_close_file: cannot update the sample count");
        fclose(z->f);
        z->f = nullptr;
        res = z->pos;
        // timestamps + record positions go into the attribute trailer (ZFile.cpp:431-447)
        AttrsFile a;
        a.filename = z->filename;
        a.t.times = z->times;
        a.t.frames.assign(z->times.size(), AttrMap());
        a.t.global["positions"] = std::string((const char*)z->positions.data(), z->positions.size() * 8);
        if (z->method == 3) a.t.global["GOP"] = std::to_string(z->gop);
        attrs_write_if_dirty(a);
    }
    g_zfiles.remove(handle);
    return res;
}

int rirb_z_open_file_read(const char* filename)
{
    if (!filename || !need_zstd()) return 0;
    auto z = std::make_shared<ZMovie>();
    z->f = fopen(filename, "rb");
    if (!z->f) {
        set_error("z_open_file_read: cannot open '%s'", filename);
        return 0;
    }
    z->filename = filename;
    const long long fsize = file_bytes(filename);
    if (fread(&z->hdr, 1, sizeof(z->hdr), z->f) != sizeof(z->hdr)) {
        set_error("z_open_file_read: '%s' is shorter than its headers", filename);
        return 0;
    }
    const unsigned comp = z->hdr.head[2];
    const uint64_t sx = z->hdr.trig[T_SIZE_X], sy = z->hdr.trig[T_SIZE_Y], rate = z->hdr.trig[T_RATE];
    // ZFile.cpp:143-152: same validity window as the reference
    if (z->hdr.head[0] != 1 || z->hdr.head[1] != 1 || comp < 1 || comp > 3 || sx == 0 || sx >= 3000 || sy == 0 || sy >= 3000 ||
        rate == 0 || rate >= 1000) {
        set_error("z_open_file_read: '%s' is not a zstd movie file", filename);
        return 0;
    }
    if (comp != 1 && rirb_device_count() <= 0) {
        set_error("z_open_file_read: compression methods 2 and 3 are decoded on the GPU, and there is no CUDA device");
        return 0;
    }
    z->w = (int)sx;
    z->h = (int)sy;
    z->method = (int)comp;
    z->gop = comp == 3 ? (int)z->hdr.trig[T_GOP] : 1;
    if (comp == 3 && (z->gop < 1 || z->gop > 65535)) {
        set_error("z_open_file_read: '%s' claims method 3 without a GOP length", filename);
        return 0;
    }
    // The trailer, when present, bounds the record area and carries the record positions and timestamps
    // (ZFile.cpp:163-190); without it, or if it does not add up, the records are walked (:192-249).
    long long end = fsize;
    bool indexed = false;
    {
        char tail[16 + k_magic_len];
        if (fsize >= (long long)(256 + sizeof(tail))) {
            fseek(z->f, (long)(fsize - (long long)sizeof(tail)), SEEK_SET);
            if (fread(tail, 1, sizeof(tail), z->f) == sizeof(tail) && memcmp(tail + 16, k_magic, k_magic_len) == 0) {
                uint64_t tsize;
                memcpy(&tsize, tail + 8, 8);
                if (tsize <= (uint64_t)(fsize - 256)) {
                    end = fsize - (long long)tsize;
                    std::vector<char> buf(tsize);
                    Trailer t;
                    fseek(z->f, (long)end, SEEK_SET);
                    if (fread(buf.data(), 1, tsize, z->f) == tsize && parse_trailer(buf.data(), buf.size(), t) > 0) {
                        auto it = t.global.find("positions");
                        const size_t n = t.times.size();
                        if (it != t.global.end() && it->second.size() == n * 8) {
                            std::vector<int64_t> posv(n);
                            memcpy(posv.data(), it->second.data(), n * 8);
                            bool ok = true;
                            for (size_t i = 0; ok && i < n; ++i) {
                                const long long next = i + 1 < n ? posv[i + 1] : end;
                                ok = posv[i] >= 256 && next - posv[i] >= 12 && next <= end;
                            }
                            if (ok) {
                                z->times = t.times;
                                z->positions = posv;
                                z->sizes.resize(n);
                                for (size_t i = 0; i < n; ++i) z->sizes[i] = (uint32_t)((i + 1 < n ? posv[i + 1] : end) - posv[i] - 12);
                                indexed = true;
                            }
                        }
                    }
                }
            }
        }
    }
    long long p = 256;
    while (!indexed && p + 12 <= end) {
        int64_t ts;
        uint32_t c;
        fseek(z->f, (long)p, SEEK_SET);
        if (fread(&ts, 8, 1, z->f) != 1 || fread(&c, 4, 1, z->f) != 1) break;
        if (p + 12 + (long long)c > end) break;
        z->times.push_back(ts);
        z->positions.push_back(p);
        z->sizes.push_back(c);
        p += 12 + (long long)c;
    }
    return g_zfiles.add(z);
}

int rirb_z_image_count(int handle)
{
    auto z = g_zfiles.get(handle);
    return z ? (int)z->times.size() : -1;
}
int rirb_z_method(int handle)
{
    auto z = g_zfiles.get(handle);
    return z ? z->method : -1;
}
int rirb_z_image_size(int handle, int* width, int* height)
{
    auto z = g_zfiles.get(handle);
    if (!z) return -1;
    if (width) *width = z->w;
    if (height) *height = z->h;
    return 0;
}
int rirb_z_get_timestamps(int handle, long long* times)
{
    auto z = g_zfiles.get(handle);
    if (!z || !times) return -1;
    for (size_t i = 0; i < z->times.size(); ++i) times[i] = z->times[i];
    return 0;
}

// records [pos, pos + count) -> decompressed payloads (w*h*2 bytes each) back to back at `out`; to_pinned_planes: `out` is
// the pinned planes (host memory, whatever cudaPointerGetAttributes says about pinned buffers)
static int z_read_records(ZMovie* z, int pos, int count, void* out, int threads, bool to_pinned_planes)
{
    const size_t fbytes = (size_t)z->w * z->h * 2;
    const int workers = pool_size(threads, count);
    const int batch = std::min(count, std::max(2 * workers, 8));
    const bool to_device = !to_pinned_planes && device_pointer(out);
    PinnedPair pin;
    cudaStream_t st = current_stream();
    if (to_device && !pin.init(fbytes * batch)) {
        set_error("z_read_images: cannot allocate pinned staging buffers");
        return -1;
    }
    if (!z->ctx || (int)z->ctx->c.size() < workers) z->ctx.reset(new Contexts(workers, false));
    Contexts& ctx = *z->ctx;
    auto& raw = z->raw;
    size_t& raw_cap = z->raw_cap;
    const int fd = fileno(z->f);
    int slot = 0;
    bool used[2] = {false, false};
    for (int b0 = 0; b0 < count; b0 += batch, slot ^= 1) {
        const int m = std::min(batch, count - b0);
        // every worker reads its own record (pread) into its place in the batch buffer and decompresses it
        const long long a = z->positions[pos + b0];
        const long long b = z->positions[pos + b0 + m - 1] + 12 + (long long)z->sizes[pos + b0 + m - 1];
        if ((size_t)(b - a) > raw_cap) {
            raw_cap = (size_t)(b - a) + (size_t)(b - a) / 4;
            raw.reset(new char[raw_cap]);
        }
        char* dst = (char*)out + (size_t)b0 * fbytes;
        if (to_device) {
            if (used[slot]) RIRB_CUDA_OK(cudaEventSynchronize(pin.ev[slot]));  // its previous upload has left the buffer
            dst = pin.buf[slot];
        }
        std::atomic<bool> failed{false};
        parallel_for(m, workers, [&](long long i, int t) {
            const long long at = z->positions[pos + b0 + i] + 12;
            const size_t len = z->sizes[pos + b0 + i];
            char* rec = raw.get() + (at - a);
            if (!pread_all(fd, rec, len, at)) {
                failed = true;
                return;
            }
            const size_t got = z_decompress(ctx.get(t), dst + (size_t)i * fbytes, fbytes, rec, len);
            if (zstd().isError(got) || got != fbytes) failed = true;
        });
        if (failed) return z_unreadable(z);
        if (to_device) {
            RIRB_CUDA_OK(cudaMemcpyAsync((char*)out + (size_t)b0 * fbytes, dst, fbytes * m, cudaMemcpyHostToDevice, st));
            RIRB_CUDA_OK(cudaEventRecord(pin.ev[slot], st));
            used[slot] = true;
        }
    }
    if (to_device) RIRB_CUDA_OK(cudaStreamSynchronize(st));
    return 0;
}

// Records [pos, pos + count) -> their payloads (w*h*2 bytes each) back to back at `out` in DEVICE memory, decoded by the
// device decoder: per pass of ~64 MB of payloads, the records' span of the file is read into pinned memory (by the host
// pool when it is large), goes up in one copy with its offset / size table, and is decoded in place.  A record the decoder
// refuses or finds malformed is decoded by host libzstd from the bytes already read; if that fails too, the read fails.
static int z_read_records_device(ZMovie* z, int pos, int count, u8* out, int threads)
{
    const size_t fbytes = (size_t)z->w * z->h * 2;
    const long long chunk = z_pass_frames(z, 1);
    cudaStream_t st = current_stream();
    ZBuffers& b = z->buffers();
    const int fd = fileno(z->f);
    long long fallbacks = 0;
    for (long long p0 = pos; p0 < (long long)pos + count;) {
        const long long m = std::min<long long>(chunk, (long long)pos + count - p0);
        ZPhase ph;
        const long long a = z->positions[p0];
        const size_t span = (size_t)(z->positions[p0 + m - 1] + 12 + (long long)z->sizes[p0 + m - 1] - a);
        const size_t table = ((span + 63) & ~(size_t)63);  // pinned: the span, then offsets | statuses | sizes
        const size_t bytes = table + (size_t)m * (8 + 8 + 4);
        if (!b.scratch.grow(zdecoder_scratch_bytes(m, (long long)fbytes)) || !b.records.grow(bytes) || !b.host_records.grow(bytes))
            return -1;
        char* h = b.host_records.p;
        long long* off = (long long*)(h + table);
        long long* status = off + m;
        unsigned* len = (unsigned*)(status + m);
        for (long long i = 0; i < m; ++i) {
            off[i] = z->positions[p0 + i] + 12 - a;  // past the record's timestamp and size
            len[i] = z->sizes[p0 + i];
        }
        const size_t piece = 4u << 20;
        const long long npieces = (long long)((span + piece - 1) / piece);
        std::atomic<bool> failed{false};
        parallel_for(npieces, pool_size(threads, npieces), [&](long long k, int) {
            const size_t lo = (size_t)k * piece;
            if (!pread_all(fd, h + lo, std::min(piece, span - lo), a + (long long)lo)) failed = true;
        });
        if (failed) return z_unreadable(z);
        ph.mark("read: pread span", m);
        const u8* d = (const u8*)b.records.p;
        long long* dstatus = (long long*)(b.records.p + ((char*)status - h));
        u8* to = out + (size_t)(p0 - pos) * fbytes;
        RIRB_CUDA_OK(cudaMemcpyAsync(b.records.p, h, bytes, cudaMemcpyHostToDevice, st));
        if (launch_zstd_decode(d, (const long long*)(d + table), (const unsigned*)(d + ((char*)len - h)), m, to, (long long)fbytes,
                               (long long)fbytes, dstatus, b.scratch.p, st) != 0)
            return -1;
        RIRB_CUDA_OK(cudaMemcpyAsync(status, dstatus, (size_t)m * 8, cudaMemcpyDeviceToHost, st));
        RIRB_CUDA_OK(cudaStreamSynchronize(st));
        ph.mark("read: upload + device zstd", m);
        std::vector<long long> redo;
        for (long long i = 0; i < m; ++i) {
            if (status[i] == -1 || status[i] == -2)
                redo.push_back(i);
            else if (status[i] != (long long)fbytes)
                return z_unreadable(z);
        }
        if (!redo.empty()) {
            const int workers = pool_size(threads, (long long)redo.size());
            if (!z->ctx || (int)z->ctx->c.size() < workers) z->ctx.reset(new Contexts(workers, false));
            std::vector<char> host((size_t)redo.size() * fbytes);
            parallel_for((long long)redo.size(), workers, [&](long long j, int t) {
                const long long i = redo[j];
                const size_t got = z_decompress(z->ctx->get(t), host.data() + (size_t)j * fbytes, fbytes, h + off[i], len[i]);
                if (zstd().isError(got) || got != fbytes) failed = true;
            });
            if (failed) return z_unreadable(z);
            for (size_t j = 0; j < redo.size(); ++j)
                RIRB_CUDA_OK(cudaMemcpyAsync(to + (size_t)redo[j] * fbytes, host.data() + j * fbytes, fbytes, cudaMemcpyHostToDevice, st));
            RIRB_CUDA_OK(cudaStreamSynchronize(st));
            fallbacks += (long long)redo.size();
            ph.mark("read: host zstd fallback", (long long)redo.size());
        }
        p0 += m;
    }
    if (z_trace() && fallbacks) fprintf(stderr, "[rirb z] %-28s %6lld frames\n", "read: records on host zstd", fallbacks);
    return 0;
}

// methods 2 / 3: records -> planes (host zstd, or the device decoder) -> device -> merge (+ undo the temporal delta from the GOP's
// key frame on).  The decoded frames of the last pass stay on the device: a reader that asks for one frame at a time decodes a
// GOP once.
static int z_read_precoded(ZMovie* z, int pos, int count, unsigned short* out, int threads, bool device_decoder)
{
    const size_t npx = (size_t)z->w * z->h;
    const long long gop = z->method == 3 ? z->gop : 1;
    const long long chunk = z_pass_frames(z, gop);
    cudaStream_t st = current_stream();
    const bool to_device = device_pointer(out);
    long long p = pos;
    const long long end = (long long)pos + count;
    bool in_flight = false;  // the stream may still be reading the pinned planes / device frames for the previous chunk
    while (p < end) {
        if (!(z->cache_first >= 0 && p >= z->cache_first && p < z->cache_first + z->cache_count)) {
            const long long k0 = p - p % gop;                                            // the GOP's key frame
            const long long m = std::min<long long>(chunk, (long long)z->times.size() - k0);
            ZPhase ph;
            if (in_flight) RIRB_CUDA_OK(cudaStreamSynchronize(st));  // before the host threads overwrite the pinned planes
            in_flight = false;
            ph.mark("read: wait for previous pass", m);
            if (!z->reserve((size_t)chunk)) return -1;
            ph.mark("read: reserve", m);
            z->cache_first = -1;
            if (device_decoder) {
                // [frame][lo | hi] into the frames' part of the device buffer, then apart into the two plane buffers
                u8* planes = (u8*)z->dev_movie();
                if (z_read_records_device(z, (int)k0, (int)m, planes, threads) != 0) return -1;
                RIRB_CUDA_OK(split_planes(z, planes, m, cudaMemcpyDeviceToDevice, st));
            } else {
                if (z_read_records(z, (int)k0, (int)m, z->host_planes(), threads, true) != 0) return -1;
                ph.mark("read: records + zstd", m);
                RIRB_CUDA_OK(split_planes(z, z->host_planes(), m, cudaMemcpyHostToDevice, st));
            }
            if (rirb_decode_movie(z->dev_lo(), z->dev_hi(), m, z->w, z->h, z->gop, z->method == 3, k0, z->dev_movie()) != 0) return -1;
            z->cache_first = k0;
            z->cache_count = m;
        }
        const long long n = std::min(end, z->cache_first + z->cache_count) - p;
        const u16* from = z->dev_movie() + (size_t)(p - z->cache_first) * npx;
        u16* to = out + (size_t)(p - pos) * npx;
        if (to_device) {
            RIRB_CUDA_OK(cudaMemcpyAsync(to, from, (size_t)n * npx * 2, cudaMemcpyDeviceToDevice, st));
            in_flight = true;
        } else if (n >= 4) {
            // a run of frames for a host caller: down into the pinned buffer (the planes in it are consumed by now, it holds
            // exactly a chunk of frames), then into the caller's pageable memory by the host pool -- the driver's own pageable
            // download is one thread faulting the destination in page by page (0.3 GB/s measured on a fresh numpy array)
            const char* hp = z->host_planes();
            RIRB_CUDA_OK(cudaMemcpyAsync(z->host_planes(), from, (size_t)n * npx * 2, cudaMemcpyDeviceToHost, st));
            RIRB_CUDA_OK(cudaStreamSynchronize(st));
            parallel_for(n, pool_size(threads, (int)n), [&](long long i, int) { memcpy(to + (size_t)i * npx, hp + (size_t)i * npx * 2, npx * 2); });
        } else {
            RIRB_CUDA_OK(cudaMemcpyAsync(to, from, (size_t)n * npx * 2, cudaMemcpyDeviceToHost, st));
            RIRB_CUDA_OK(cudaStreamSynchronize(st));
        }
        p += n;
    }
    RIRB_CUDA_OK(cudaStreamSynchronize(st));
    return 0;
}

// Which decoder a read takes.  The "zstd_decoder" switch: 0 host zstd, 2 the device decoder for every read that ends on the
// device (methods 2 / 3 always do), 1 (the default) the device decoder only for a method-1 read into device memory whose first
// record is a frame without LZ sequences -- what the device coder writes.  The device decoder runs the sequences of a frame
// on one warp, which is slower than the host pool (DESIGN.md 7 f-3, r4); frames without sequences it decodes faster.
static bool z_use_device_decoder(ZMovie* z, int pos, const void* out)
{
    const int mode = option_value(OPT_ZSTD_DECODER);
    if (z->method != 1) return mode == 2;
    if (mode == 0 || !device_pointer(out)) return false;
    if (mode == 2) return true;
    std::vector<u8> f(z->sizes[pos]);
    return pread_all(fileno(z->f), f.data(), f.size(), z->positions[pos] + 12) &&
           zdecoder_frame_plain(f.data(), (long long)f.size(), (long long)z->w * z->h * 2);
}

// frames [pos, pos + count) -> out[count][h][w] (host or device), timestamps (host, may be NULL)
int rirb_z_read_images(int handle, int pos, int count, unsigned short* out, long long* timestamps, int threads)
{
    auto z = g_zfiles.get(handle);
    if (!z || z->writing || !out || pos < 0 || count < 0 || (size_t)pos + (size_t)count > z->times.size()) {
        set_error("z_read_images: bad handle or range");
        return -1;
    }
    if (count == 0) return 0;
    std::lock_guard<std::mutex> lock(z->mu);
    const bool device_decoder = z_use_device_decoder(z.get(), pos, out);
    const int rc = z->method != 1 ? z_read_precoded(z.get(), pos, count, out, threads, device_decoder)
                   : device_decoder ? z_read_records_device(z.get(), pos, count, (u8*)out, threads)
                                    : z_read_records(z.get(), pos, count, out, threads, false);
    if (rc == 0 && timestamps)
        for (int i = 0; i < count; ++i) timestamps[i] = z->times[pos + i];
    return rc;
}

int rirb_z_read_image(int handle, int pos, unsigned short* img, long long* timestamp)
{
    return rirb_z_read_images(handle, pos, 1, img, timestamp, 1);
}

}  // extern "C"
