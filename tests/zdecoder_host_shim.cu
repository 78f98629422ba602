// tests/zdecoder_host_shim.cu -- the device zstd decoder's per-frame bodies (librir_b200/csrc/zdecoder.cu) compiled for the
// host: scan, literals and sequences of one frame in the order the three kernels run them, with one "lane" (ZD_WIDTH 1).
// tests/test_zdecoder_fuzz.py builds it into a shared library and drives it from Python; the symbols zdecoder.cu takes
// from capi.cu are defined here, so the library stands alone and needs no device.
#include "../librir_b200/csrc/zdecoder.cu"

#include <cstdarg>
#include <cstdio>

namespace rirb {
static char g_err[512];
std::atomic<long long> g_launches{0};
void set_error(const char* fmt, ...)
{
    va_list a;
    va_start(a, fmt);
    vsnprintf(g_err, sizeof g_err, fmt, a);
    va_end(a);
}
cudaStream_t current_stream() { return 0; }
}  // namespace rirb

extern "C" RIRB_API int rirb_device_count(void) { return 0; }

// One frame f[0, size) into dst[0, cap) with cap bytes of literal scratch; returns what zd_frames_kernel writes to the
// frame's status: the content size, -1 (malformed) or -2 (refused).
extern "C" RIRB_API long long zd_host_decode(const unsigned char* f, long long size, unsigned char* dst, long long cap,
                                             unsigned char* lit_scratch)
{
    using namespace rirb;
    ZdFrame fr;
    zd_scan_frame(f, size, cap, fr);
    if (fr.err) return fr.err;
    ZdHufSmem hs;
    zd_literals_frame(f, size, fr, dst, lit_scratch, 0, 1, hs);
    if (fr.err) return fr.err;
    ZdSeqSmem ss;
    return zd_decode_frame(f, size, fr, dst, cap, lit_scratch, ss);
}
