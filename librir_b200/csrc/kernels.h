// librir_b200/csrc/kernels.h -- internal launch API between the kernel files and capi.cu.
// Every function enqueues on `st`, returns 0 on success or -1 after set_error(); pointers are
// DEVICE pointers unless named *_host.
#pragma once
#include <cuda_runtime.h>
#include <stddef.h>

#include <initializer_list>

namespace rirb {

typedef unsigned short u16;
typedef unsigned char u8;

enum { STRAT_NOBORDER = 0, STRAT_BACKGROUND = 1, STRAT_WRAP = 2, STRAT_NEAREST = 3 };

// bad_pixels.cu
int launch_hist_frame(const u16* img, size_t n, unsigned* hist65536, cudaStream_t st);
int launch_bp_detect(const u16* img, int w, int h, double std_factor, unsigned gthr, u8* mask, cudaStream_t st);
// Correction CTAs own flat spans of BP_SPAN pixels; span_off[s] .. span_off[s+1] is the slice of the
// raster-ordered (x,y) list that falls into span s (ceil(w*h / BP_SPAN) + 1 entries, built at create).
constexpr int BP_SPAN = 16384;
int launch_bp_correct(const u16* in, u16* out, const int* xy_dev, const int* span_off_dev, int w, int h, int clamp_value,
                      long long nframes, size_t frame_stride, cudaStream_t st);
int launch_bp_correct_inplace(u16* img, const int* xy_dev, int count, int w, int h, int clamp_value, long long nframes,
                              size_t frame_stride, cudaStream_t st);
int launch_loader_bp(u16* img, const int* xy_dev, const u8* mask, int count, int w, int h, long long nframes,
                     size_t frame_stride, cudaStream_t st);

// loader.cu
int launch_loader_merge(const u8* lo, const u8* hi, u16* out, int w, int h, int hb, long long nframes, size_t frame_stride,
                        int min_t, int min_t_height, const int* xy_dev, const int* span_off_dev, const int* nbr_dev,
                        cudaStream_t st);

// translate.cu: the reader's chain fused into the motion translate; returns 1 if the layout cannot take it
int launch_loader_add_min(u16* frames, int w, int t_rows, long long nframes, size_t frame_stride, int min_t, cudaStream_t st);
int launch_loader_fused(const u8* lo, const u8* hi, u16* out, int w, int h_full, int hb, long long nframes, int min_t, int t_rows,
                        const int* xy_dev, const int* nbr_dev, const int* row_off_dev, const u8* mask_dev, const float* dxs,
                        const float* dys, cudaStream_t st);

// translate.cu
int launch_translate(int type, const void* src, void* dst, int w, int h, long long nframes, const float* dxs, const float* dys,
                     float dx0, float dy0, int strategy, const void* background_host, cudaStream_t st);
int launch_translate_u16(const u16* src, u16* dst, int w, int h, long long nframes, size_t src_stride, size_t dst_stride,
                         const float* dxs, const float* dys, float dx0, float dy0, int strategy, unsigned background, bool motion,
                         cudaStream_t st);

// gaussian.cu
constexpr int GAUSS_MAX_RADIUS = 64;
struct GaussTaps {
    int radius;
    float k[2 * GAUSS_MAX_RADIUS + 1];  // 1-D taps, k[d + radius]
};
// Host: taps the way the reference builds its 2-D kernel (signal_processing.cpp:79-99), reduced
// to 1-D by row sums.  Returns -1 if the radius exceeds GAUSS_MAX_RADIUS.
int gaussian_taps_host(float sigma, GaussTaps* taps);
int launch_gaussian_f32(const float* src, float* dst, int w, int h, long long nframes, const GaussTaps& taps, cudaStream_t st);
int launch_gaussian_u16(const u16* src, float* dst, int w, int h, long long nframes, const GaussTaps& taps, cudaStream_t st);
// a w x h region of larger frames (strides in pixels) -> dense dst; 1 when the layout is not taken (see gaussian.cu)
int launch_gaussian_u16_region(const u16* src, size_t src_row, size_t src_frame, float* dst, int w, int h, long long nframes,
                               const GaussTaps& taps, cudaStream_t st);
int launch_gaussian_f32_region(const float* src, size_t src_row, size_t src_frame, float* dst, int w, int h, long long nframes,
                               const GaussTaps& taps, cudaStream_t st);
// correction + filter in one pass (gaussian.cu, BpFuse); 1: layout not eligible, run the two kernels
int launch_gaussian_bp_u16(const u16* raw, u16* corrected, float* dst, int w, int h, long long nframes, const GaussTaps& taps,
                           const int* xy_dev, const int* row_off_dev, int clamp_value, cudaStream_t st);

// capi.cu: grow-only per-thread device work space for launchers, slots 8..11 (nullptr + set_error when out of memory)
void* scratch_buffer(int slot, size_t bytes);

// The operand checks of the entries, defined here so that every source file that has an entry carries them (the host
// build of zdecoder.cu in the tests included).  A kernel that writes bytes it (or another kernel of the same call) also
// reads races, so refuse_overlap fails (-1, set_error naming both operands) when an output shares a byte with an input --
// both device or managed memory; host operands are staged into separate buffers -- or with another output, in any
// memory.  Inputs may share bytes: they are only read.
void set_error(const char* fmt, ...);
struct Operand {
    const char* name;
    const void* p;
    size_t bytes;
};
inline bool bytes_overlap(const Operand& a, const Operand& b)
{
    const size_t x = (size_t)a.p, y = (size_t)b.p;
    return a.p && b.p && a.bytes && b.bytes && x < y + b.bytes && y < x + a.bytes;
}
// cudaMemoryTypeUnregistered (pageable host memory) when the runtime does not know the pointer
inline cudaMemoryType operand_memory_type(const void* p)
{
    cudaPointerAttributes a;
    if (cudaPointerGetAttributes(&a, p) != cudaSuccess) {
        cudaGetLastError();
        return cudaMemoryTypeUnregistered;
    }
    return a.type;
}
inline bool operand_on_device(const void* p)
{
    const cudaMemoryType t = operand_memory_type(p);
    return t == cudaMemoryTypeDevice || t == cudaMemoryTypeManaged;
}
inline int refuse_overlap(const char* what, std::initializer_list<Operand> ins, std::initializer_list<Operand> outs)
{
    for (auto o = outs.begin(); o != outs.end(); ++o) {
        for (const Operand& i : ins)
            if (bytes_overlap(*o, i) && operand_on_device(o->p) && operand_on_device(i.p)) {
                set_error("%s: %s and %s overlap in device memory", what, i.name, o->name);
                return -1;
            }
        for (auto q = outs.begin(); q != o; ++q)
            if (bytes_overlap(*o, *q)) {
                set_error("%s: the outputs %s and %s overlap", what, q->name, o->name);
                return -1;
            }
    }
    return 0;
}
// -1 (set_error naming the operand) unless every non-null pointer is device, managed or page-locked host memory: what a
// kernel may dereference directly
inline int refuse_pageable(const char* what, std::initializer_list<Operand> ops)
{
    for (const Operand& o : ops)
        if (o.p && operand_memory_type(o.p) == cudaMemoryTypeUnregistered) {
            set_error("%s: %s is pageable host memory; pass device, managed or pinned memory", what, o.name);
            return -1;
        }
    return 0;
}

// precode.cu
int launch_split_planes(const u16* img, const u8* it, int w, int h, u8* y_plane, u8* u_plane, u8* v_plane, int ls_y, int ls_u,
                        int ls_v, cudaStream_t st);
int launch_merge_planes(const u8* y_plane, const u8* u_plane, const u8* v_plane, int ls_y, int ls_u, int ls_v, int w, int h,
                        u16* img, u8* it, cudaStream_t st);
int launch_precode_movie(const u16* mov, long long nframes, int w, int h, int gop, int delta, long long first_frame, u8* lo,
                         u8* hi, cudaStream_t st);
int launch_precode_movie_stats(const u16* mov, long long nframes, int w, int h, int gop, int delta, long long first_frame, u8* lo,
                               u8* hi, unsigned* minmax, unsigned long long* hist, cudaStream_t st);
int launch_decode_movie(const u8* lo, const u8* hi, long long nframes, int w, int h, int gop, int delta, long long first_frame,
                        u16* mov, cudaStream_t st);

// zcoder.cu: n payloads of bytes_each bytes at src -> one zstd frame each (blocks cut at multiples of `segment` bytes, 0 = none).
// dst_stride > 0: frame i at dst + i * dst_stride.  dst_stride == 0: records packed back to back, frame i at
// foff[i] + rec_head with foff[n] = the total; rec_head bytes before each frame are left for the caller.  sizes (may be null):
// frame bytes.  *frame_offsets (may be null) receives the device array foff (inside scratch).
size_t zcoder_scratch_bytes(long long n, long long bytes_each, long long segment);
long long zcoder_frame_bound(long long bytes_each, long long segment);  // the largest frame: raw blocks plus headers
int launch_zstd_encode(const u8* src, long long n, long long bytes_each, long long segment, u8* dst, long long dst_stride,
                       int rec_head, long long* sizes, long long** frame_offsets, void* scratch, cudaStream_t st);
// coder 2 (rirb_zstd_encode_batch_lz): the same arguments, coder 1's frame with an LZ form wherever it is smaller; its scratch
// (zcoder_lz_scratch_bytes) holds coder 1's and a candidate sort of at most 512 blocks at a time (about 1.6 GB)
size_t zcoder_lz_scratch_bytes(long long n, long long bytes_each, long long segment);
int launch_zstd_encode_lz(const u8* src, long long n, long long bytes_each, long long segment, u8* dst, long long dst_stride,
                          int rec_head, long long* sizes, long long** frame_offsets, void* scratch, cudaStream_t st);
// zdecoder.cu: n zstd frames (frame i at src + offsets[i], sizes[i] bytes) -> content at dst + i * dst_stride, at most cap
// bytes; status[i] = bytes, -1 malformed, -2 refused (rirb_zstd_decode_batch).  scratch: zdecoder_scratch_bytes(n, cap).
size_t zdecoder_scratch_bytes(long long n, long long cap);
// Host: 1 when the frame at f (host memory) is one the decoder takes, with content of at most cap bytes and no LZ sequences.
int zdecoder_frame_plain(const u8* f, long long size, long long cap);
int launch_zstd_decode(const u8* src, const long long* offsets, const unsigned* sizes, long long n, u8* dst, long long dst_stride,
                       long long cap, long long* status, void* scratch, cudaStream_t st);

// lossy.cu (H264_Saver::addImageLossyNoCamera, h264.cpp:2253-2424)
size_t lossy_scalars_bytes();
int launch_lossy_first(const u16* tmp, u16* out, u16* lastDL, u16* refT, u16* prevT, int n, int ns, int subtract_min, void* scalars,
                       int* errors_out_dev, int low0, int high0, cudaStream_t st);
// a run of consecutive non-initial frames: backgrounds of all of them in one launch, then ONE cooperative launch with one
// grid barrier per frame (lossy.cu, lossy_run_kernel); 1: not available.  variant 0 = addImageLossyNoCamera, 1 = addLoss;
// quirk: the compiled reference's overlapping memcpy (lossy_window_quirk)
int launch_lossy_run(const u16* img, const u16* cur, u16* out, u16* lastDL, u16* refT, u16* prevT, unsigned* sums, u16* cvalue,
                     short* ccount, u16* ring, int n, int ns, int ra, int subtract_min, long long frame_index, int m, int low0,
                     int high0, double std_factor, int variant, int quirk, void* scalars, unsigned* hist_scratch, int* errors_out_dev,
                     cudaStream_t st);
size_t lossy_hist_scratch_bytes();
int lossy_max_run();
int launch_lossy_frame(const u16* img, const u16* tmp, u16* tmpT, u16* out, u16* lastDL, u16* refT, u16* prevT, unsigned* sums,
                       u16* cvalue, short* ccount, u16* ring, int n, int ns, int ra, int subtract_min, long long frame_index,
                       int low0, int high0, double std_factor, int variant, int quirk, void* scalars, int* errors_out_dev,
                       cudaStream_t st);

// stats.cu
// minmax[0] = min, minmax[1] = max (unsigned, device); hist = 65536 x u64 (device) or nullptr.
// Accumulates INTO the outputs: callers zero hist / seed minmax with {65535, 0} first
// (launch_stats_init) so that several chunks of one movie can be reduced in place.
int launch_stats_init(unsigned* minmax, unsigned long long* hist, cudaStream_t st);
int launch_movie_stats(const u16* mov, size_t n, const u8* mask, unsigned* minmax, unsigned long long* hist, cudaStream_t st);

int launch_hist_quantile(const unsigned long long* hist, long long count, float percent, int masked_rule, int* out,
                         cudaStream_t st);
int launch_hist_mode4(const unsigned long long* hist, unsigned* out, cudaStream_t st);

}  // namespace rirb
