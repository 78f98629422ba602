/*
 * include/librir_b200.h -- C ABI of libsignal_processing_b200.so
 *
 * A B200-native (sm_100a CUDA) implementation of librir's per-frame hot path, behind the
 * reference's own C interface.  Part 1 re-declares, with identical names, argument order and
 * status codes, the entry points of the reference's signal_processing library that the path
 * touches -- the library can therefore be dropped into librir/libs/ in place of
 * libsignal_processing.so and is picked up by librir/low_level/misc.py:98-136 unchanged.
 * Part 2 holds additive entry points (prefix rirb_) that make the speed reachable: batches of
 * frames in one launch, device-resident buffers, the writer's pre-coder, movie statistics.
 *
 * Conventions (same as the reference, SURVEY.md 8b):
 *   - images are dense row-major [h][w]; WIDTH IS PASSED BEFORE HEIGHT;
 *   - the caller owns every buffer; nothing is retained after a call returns
 *     (bad_pixels_create copies what it needs);
 *   - status: 0 success, -1 failure (rirb_last_error() / the reference's get_last_log_error
 *     convention), create-functions return a handle > 0 or 0 on failure;
 *   - no exception crosses the boundary; every entry is re-entrant.
 * Pointers may be HOST pointers (pageable or pinned: the call stages them through the GPU and
 * returns when the result is in the caller's buffer) or DEVICE pointers (detected with
 * cudaPointerGetAttributes: zero copies, the work is enqueued on the calling thread's stream
 * set with rirb_set_stream and the call returns without synchronising).
 * There is NO CPU implementation behind any compute entry: without a CUDA device they fail (-1).
 */
#ifndef LIBRIR_B200_H
#define LIBRIR_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define RIRB_API __attribute__((visibility("default")))

/* ===================== Part 1: the reference's interface (signal_processing.h) ============ */

/* replaces translate, signal_processing.h:29 / signal_processing.cpp:44-73
 * (rir::translate<T,T>, Filters.h:249-326).  type = numpy char code '?bBhHiIlLfd';
 * strategy = NULL / "" / "noborder" / "background" / "wrap" / "nearest";
 * -1 for an unknown type or strategy. */
RIRB_API int translate(int type, void* src, void* dst, int w, int h, float dx, float dy, void* background,
                       const char* strategy);

/* replaces gaussian_filter, signal_processing.h:33 / signal_processing.cpp:101-148. */
RIRB_API int gaussian_filter(float* src, float* dst, int w, int h, float sigma);

/* replace find_median_pixel(_mask), signal_processing.h:39,44 / Filters.cpp:56-101. */
RIRB_API int find_median_pixel(unsigned short* pixels, int size, float percent);
RIRB_API int find_median_pixel_mask(unsigned short* pixels, unsigned char* mask, int size, float percent);

/* replace bad_pixels_create / _correct / _destroy, signal_processing.h:77,81,85 /
 * signal_processing.cpp:199-222 (BadPixels.cpp:13-66, Filters.h:135-193). */
RIRB_API int bad_pixels_create(unsigned short* first_image, int width, int height);
RIRB_API int bad_pixels_correct(int handle, unsigned short* in, unsigned short* out);
RIRB_API void bad_pixels_destroy(int handle);

/* Out of the hot path (1-D time series, connected components, hashing): forwarded verbatim to
 * the reference build named by $LIBRIR_B200_FORWARD_LIB (a libsignal_processing.so of the
 * reference), -1 when it is not set.  signal_processing.h:55,71,90,92,94. */
RIRB_API int extract_times(double* time_vector, int vector_count, int* vector_sizes, int s, double* output,
                           int* output_size);
RIRB_API int resample_time_serie(double* sample_x, double* sample_y, int size, double* times, int times_size, int s,
                                 double padds, double* output, int* output_size);
RIRB_API int label_image(int type, void* src, int* dst, int w, int h, void* background, double* out_xy, int* out_area);
RIRB_API int keep_largest_area(int type, void* src, int* dst, int w, int h, void* background, int foreground);
RIRB_API size_t hash_bytes(void* ptr, size_t len);

/* ===================== Part 2: additive entry points ====================================== */

/* ---- runtime ---- */
RIRB_API int rirb_device_count(void);                 /* 0 when no CUDA device is usable */
RIRB_API int rirb_set_device(int device);             /* cudaSetDevice for the calling thread */
/* (changing the stream makes the new one wait, on the device, for what this thread enqueued on the old one: the thread's
 * scratch buffers are shared by its calls) */
RIRB_API int rirb_set_stream(void* cuda_stream);      /* stream for the calling thread (NULL = default) */
RIRB_API int rirb_synchronize(void);                  /* wait for the calling thread's stream */
RIRB_API const char* rirb_last_error(void);           /* calling thread's last error text */
/* The calling thread's staging buffers (device scratch, pinned ring, the three streams + buffers of
 * rirb_process_movie_host) are grow-only while the thread lives and are freed when it exits; this frees them now. */
RIRB_API void rirb_release_thread_resources(void);
RIRB_API long long rirb_kernel_launch_count(void);    /* kernels launched by this library so far */
RIRB_API const char* rirb_version(void);
/* string key/value switches, the reference's *_set_parameter convention (h264.cpp:1709-1781); process-wide.
 * "translate_tma" / "gauss_tma" (default 1): TMA-tiled kernels vs the register-only ones;
 * "loader_fused" (default 0): rirb_loader_read_movie as one fused pass instead of merge pass + motion pass.
 * "ecc_fused" (default 1): rirb_ecc_compute as ONE cooperative launch (grid barriers between the phases and the
 *   iterations) instead of one launch per iteration.
 * "lossy_run" (default 1): rirb_lossy_add_images walks a run of frames in ONE cooperative launch (one grid barrier
 *   per frame) instead of three launches per frame.
 * "translate_rows" (default 1): the second-generation tiled translate kernel (0: the first one, for A/B runs).
 * "ecc_queue" (default 1): rirb_ecc_track solves runs of up to 16 device-resident frames in ONE cooperative launch (the
 *   warm start stays on the device, a frame that fails or triggers the replacement of the reference image ends the
 *   run) instead of one launch + copy back + synchronisation per frame.
 * "zstd_decoder" (default 1): a method-1 zstd movie file read into device memory whose first record has no LZ sequences
 *   (what the device coder writes) uploads the records and decodes them with rirb_zstd_decode_batch; 2: every read that
 *   ends on the device does (methods 2/3 too); 0: host libzstd for every read.  2 and 0 are for A/B runs.
 * Initial values can also come from RIRB_TRANSLATE_TMA / RIRB_GAUSS_TMA / RIRB_LOADER_FUSED / RIRB_ECC_FUSED /
 * RIRB_LOSSY_RUN / RIRB_TRANSLATE_ROWS / RIRB_ECC_QUEUE / RIRB_ZSTD_DECODER.  -1: unknown key. */
RIRB_API int rirb_set_parameter(const char* key, const char* value);

/* ---- batches of frames (nframes dense frames back to back) ---- */
/* Operands may be host (pageable, pinned or registered), managed or device memory.  Host operands are staged through
 * separate device buffers; device and managed operands go to the kernels as they are, so an output that shares a byte
 * with an input of the same call in device or managed memory is refused (-1), except where an entry documents in-place
 * use and the two pointers are equal.  Outputs that overlap each other are refused in any memory. */

/* translate on nframes frames; n_shifts == 1: one (dx[0],dy[0]) for all frames, n_shifts ==
 * nframes: per-frame shifts (registration).  dx/dy: host or device arrays of float. */
RIRB_API int rirb_translate_batch(int type, const void* src, void* dst, int w, int h, long long nframes, const float* dx,
                                  const float* dy, long long n_shifts, const void* background, const char* strategy);

RIRB_API int rirb_gaussian_filter_batch(const float* src, float* dst, int w, int h, long long nframes, float sigma);
/* fused uint16 -> float32 variant (what rir_signal_processing.py:100 does on the host first) */
RIRB_API int rirb_gaussian_filter_u16_batch(const unsigned short* src, float* dst, int w, int h, long long nframes,
                                            float sigma);

RIRB_API int rirb_bad_pixels_correct_batch(int handle, const unsigned short* in, unsigned short* out, long long nframes);
/* bad_pixels_correct + gaussian_filter of the corrected frames in ONE pass over the movie: corrected[n][h][w] (uint16) and
 * smoothed[n][h][w] (float32) are both written, the raw frames are read once (8 B/px instead of 4 + 6).  Same results as
 * the two calls; layouts the tiled kernel cannot take fall back to them internally. */
RIRB_API int rirb_bad_pixels_correct_gaussian_batch(int handle, const unsigned short* in, unsigned short* corrected, float* smoothed,
                                                    long long nframes, float sigma);
/* introspection of a handle: number of flagged pixels; raster-ordered (x,y) list; clamp level */
RIRB_API int rirb_bad_pixels_count(int handle);
RIRB_API int rirb_bad_pixels_get(int handle, int* xy, int capacity, int* clamp_value);

/* ---- in-library variants used by the reference's file loader ---- */

/* IRFileLoader::removeBadPixels, IRFileLoader.cpp:722-802: in place, on the handle's w x h
 * region of each frame (create the handle on the first frame cropped to height-3, as
 * setBadPixelsEnabled :693-716 does); frames are frame_stride pixels apart. */
RIRB_API int rirb_loader_remove_bad_pixels(int handle, unsigned short* frames, long long nframes, size_t frame_stride);
/* removeMotionGeneric, IRFileLoader.cpp:617-627: rows [0,h) of each frame are translated by
 * (-shift_x[t], -shift_y[t]) (uint16 -> float, nearest border, float -> uint16 truncation);
 * the remaining rows up to frame_stride are copied.  in == out allowed. */
RIRB_API int rirb_loader_remove_motion(const unsigned short* in, unsigned short* out, int w, int h, long long nframes,
                                       size_t frame_stride, const double* shift_x, const double* shift_y);

/* IRFileLoader::readImage's post-decode chain for a run of frames (IRFileLoader.cpp:1168-1247, the
 * calibration == 0 branch), from the decoder's byte planes to corrected, registered uint16 frames:
 *   v = lo | hi << 8                          VideoGrabber::toArray, h264.cpp:3016-3051
 *   v += min_T on rows [0, min_T_height)      IRFileLoader.cpp:1174-1179 (min_T == 0: skipped; min_T_height == 0:
 *                                             h - meta_rows, the default the reference applies at open, :918-921)
 *   removeBadPixels on rows [0, h-meta_rows)  IRFileLoader.cpp:722-802 (handle == 0: skipped; else a handle
 *                                             created on the first frame cropped to h-meta_rows rows)
 *   removeMotion on rows [0, h-meta_rows)     IRFileLoader.cpp:617-627 (shift_x/shift_y NULL: skipped)
 * lo, hi: dense planes [nframes][h][w]; out: [nframes][h][w].  Merge, min_T and the bad-pixel medians are
 * one streaming pass (2 B/px read, 2 B/px written), the motion step a second one. */
RIRB_API int rirb_loader_read_movie(int handle, const unsigned char* lo, const unsigned char* hi, long long nframes, int w, int h,
                                    int min_T, int min_T_height, const double* shift_x, const double* shift_y, int meta_rows,
                                    unsigned short* out);

/* readImage's chain for frames that are uint16 already (e.g. decoded from the zstd movie file, rirb_z_read_images):
 * += min_T on rows [0, min_T_height) -> removeBadPixels -> removeMotion, IN PLACE on frames[nframes][h][w] (host or device);
 * handle / shifts / meta_rows as in rirb_loader_read_movie. */
RIRB_API int rirb_loader_finish_frames(int handle, unsigned short* frames, long long nframes, int w, int h, int min_T, int min_T_height,
                                       const double* shift_x, const double* shift_y, int meta_rows);

/* ---- lossless-writer pre-coder (H264Capture::AddFrame, h264.cpp:1066-1103; inverse
 *      VideoGrabber::toArray, h264.cpp:3016-3051) ---- */

/* YUV444P: Y = it[] or 0, U = low bytes, V = high bytes; planes [h][linesize]. it may be NULL. */
RIRB_API int rirb_split_yuv444(const unsigned short* img, const unsigned char* it, int w, int h, unsigned char* y_plane,
                               unsigned char* u_plane, unsigned char* v_plane, int ls_y, int ls_u, int ls_v);
RIRB_API int rirb_merge_yuv444(const unsigned char* y_plane, const unsigned char* u_plane, const unsigned char* v_plane,
                               int ls_y, int ls_u, int ls_v, int w, int h, unsigned short* img, unsigned char* it);
/* YUV420P: luma plane of 2h rows (rows [0,h) low bytes, [h,2h) high bytes); u_plane (h rows)
 * receives it[] when both are non-NULL. */
RIRB_API int rirb_split_yuv420(const unsigned short* img, const unsigned char* it, int w, int h, unsigned char* y_plane,
                               int ls_y, unsigned char* u_plane, int ls_u);
RIRB_API int rirb_merge_yuv420(const unsigned char* y_plane, int ls_y, const unsigned char* u_plane, int ls_u, int w, int h,
                               unsigned short* img, unsigned char* it);
/* Whole movie, dense planes lo[t][h][w], hi[t][h][w].  delta = 0: the reference's split.
 * delta = 1: non-key frames hold (frame[t]-frame[t-1]) mod 2^16; key frames follow the AddFrame
 * rule for a writer whose frame counter is first_frame + t (key iff counter % gop == 0);
 * first_frame must be a multiple of gop (shards start on key frames). */
RIRB_API int rirb_precode_movie(const unsigned short* movie, long long nframes, int w, int h, int gop, int delta,
                                long long first_frame, unsigned char* lo, unsigned char* hi);
/* rirb_precode_movie and rirb_movie_stats of the same frames in ONE pass over them (the pre-coder is purely
 * bandwidth-bound, the histogram rides along): minmax / hist / accumulate as in rirb_movie_stats. */
RIRB_API int rirb_precode_movie_stats(const unsigned short* movie, long long nframes, int w, int h, int gop, int delta,
                                      long long first_frame, unsigned char* lo, unsigned char* hi, unsigned int* minmax,
                                      unsigned long long* hist, int accumulate);
RIRB_API int rirb_decode_movie(const unsigned char* lo, const unsigned char* hi, long long nframes, int w, int h, int gop,
                               int delta, long long first_frame, unsigned short* movie);
/* key[t] = 1 iff frame t of a writer starting at frame 0 is a key frame (h264.cpp:1050-1061) */
RIRB_API int rirb_key_frames(long long nframes, int gop, unsigned char* key);

/* ---- lossy "bounded-error" pre-conditioner of the H.264 saver (H264_Saver::addImageLossyNoCamera,
 *      h264.cpp:2253-2424; the frames it produces are what addImageLossLess then encodes; and H264_Saver::addLoss,
 *      :2426-2607, see rirb_lossy_set_parameter) ----
 * open: image size, stop_lossy_height (rows [0, stop) are lossy, the rest is copied), lowValueError /
 * highValueError (reference defaults 6 / 2), stdFactor (5), runningAverage (32, <= 64, 0 = off), subtractMin,
 * removeBadPixels -- the saver's string parameters (h264.cpp:1709-1781).  Returns a handle > 0, 0 on failure.
 * add_images: nframes frames IN TIME ORDER (the state carries over between calls); out receives the
 * pre-conditioned frames, errors (2 ints per frame, host or device, may be NULL) the per-frame
 * BackgroundError / ForegroundError attributes.  Inputs must be in temperature already (the camera
 * calibration of the "WithCamera" variant is outside this library). */
RIRB_API int rirb_lossy_open(int w, int h, int stop_lossy_height, int low_error, int high_error, double std_factor,
                             int running_average, int subtract_min, int remove_bad_pixels);
RIRB_API int rirb_lossy_add_images(int handle, const unsigned short* frames, long long nframes, unsigned short* out, int* errors);
/* string switches of a handle, before the first frame:
 *   "variant" = "add_image_lossy" (default; addImageLossyNoCamera, behind h264_add_image_lossy) | "add_loss"
 *               (H264_Saver::addLoss, h264.cpp:2426-2607, behind h264_add_loss: the bounds only tighten when the
 *               spread is above its running mean, no integration-time test);
 *   "memcpyQuirk" = "1" (default) | "0": the reference shifts its window of 40 spreads with an overlapping memcpy
 *               (h264.cpp:2347, undefined behaviour); 1 reproduces what the reference does as compiled with its
 *               stock flags (g++ -O3, x86-64: one .second value is smeared, oracle/oracle.c), 0 the intended memmove. */
RIRB_API int rirb_lossy_set_parameter(int handle, const char* key, const char* value);
RIRB_API void rirb_lossy_close(int handle);
/* the minimum the first image fixed (the saver's MIN_T global attribute, h264.cpp:2277-2296); 0 without subtractMin */
RIRB_API int rirb_lossy_get_min(int handle, int* min_value);

/* ---- the whole per-frame path on HOST buffers, one call (the end-to-end drop-in) ----
 * frames[nframes][h][w] (host) -> bad_pixels_correct (handle) -> gaussian_filter (sigma; result kept on
 * the device unless `smoothed` is non-NULL) -> translate by the per-frame shifts dx[t], dy[t] (host floats,
 * `strategy`, `background`) -> rirb_precode_movie (gop, delta, first_frame) -> lo/hi[nframes][h][w] (host).
 * The movie is cut into sub-chunks of whole GOPs that rotate over three CUDA streams, so the upload of
 * one, the kernels of another and the download of a third overlap; pinned (page-locked) buffers make
 * the copies asynchronous, pageable ones work but serialise.  Returns when lo/hi (and smoothed) are
 * complete.  With delta != 0, first_frame must be a multiple of gop.  Any operand may also be device or managed memory.
 * An output that overlaps an input or another output is refused (-1), whatever the kind of memory. */
RIRB_API int rirb_process_movie_host(int handle, const unsigned short* frames, long long nframes, int w, int h, float sigma,
                                     const float* dx, const float* dy, const char* strategy, unsigned int background, int gop,
                                     int delta, long long first_frame, unsigned char* lo, unsigned char* hi, float* smoothed);

/* ---- statistics (the quantities the multi-GPU path all-reduces) ---- */

/* minmax[2] = {min, max}; hist = 65,536 x uint64 or NULL.  accumulate != 0: fold into the
 * existing contents (several chunks / later NCCL all-reduce); else outputs are initialised. */
RIRB_API int rirb_movie_stats(const unsigned short* pixels, size_t n, unsigned int* minmax, unsigned long long* hist,
                              int accumulate);
/* find_median_pixel's rule on an (all-reduced) histogram holding `count` pixels */
RIRB_API int rirb_hist_quantile(const unsigned long long* hist, long long count, float percent);
/* get_background (h264.cpp:1955-1991) of one image */
RIRB_API int rirb_get_background(const unsigned short* pixels, int size);

/* ===================== Part 3: the file formats either side of the path (host code) ========
 * SURVEY.md 8f-3.  No kernels here: the entropy stage is zstd on the host by design.  What is added
 * over the reference: a run of frames is (de)compressed by a pool of host threads with the records
 * kept in order, and frame buffers may be device pointers. */

/* ---- attribute trailer: replaces attrs_*, tools.h:96-179 / tools.cpp:87-350 (rir::FileAttributes,
 *      FileAttributes.cpp).  Same arguments and status codes: handle > 0 or 0; getters return 0, -1 on a bad
 *      handle / index, -2 with *len set when the buffer is too small; changes are written when the handle is
 *      closed or flushed.  Like the reference, open_file creates a missing (or < 30-byte) file, a file
 *      without a trailer gets one on close, and attrs_discard WRITES (tools.cpp:124-131 calls close());
 *      rirb_attrs_abandon is the entry that drops the changes. */
RIRB_API int rirb_attrs_open_file(const char* filename);
RIRB_API int rirb_attrs_open_from_memory(const void* ptr, long long size);
RIRB_API void rirb_attrs_close(int handle);
RIRB_API void rirb_attrs_discard(int handle);
RIRB_API void rirb_attrs_abandon(int handle);
RIRB_API int rirb_attrs_flush(int handle);
RIRB_API int rirb_attrs_image_count(int handle);
RIRB_API int rirb_attrs_global_attribute_count(int handle);
RIRB_API int rirb_attrs_global_attribute_name(int handle, int pos, char* name, int* len);
RIRB_API int rirb_attrs_global_attribute_value(int handle, int pos, char* value, int* len);
RIRB_API int rirb_attrs_frame_attribute_count(int handle, int frame);
RIRB_API int rirb_attrs_frame_attribute_name(int handle, int frame, int pos, char* name, int* len);
RIRB_API int rirb_attrs_frame_attribute_value(int handle, int frame, int pos, char* value, int* len);
RIRB_API int rirb_attrs_frame_timestamp(int handle, int frame, long long* time);
RIRB_API int rirb_attrs_timestamps(int handle, long long* times);
RIRB_API int rirb_attrs_set_times(int handle, const long long* times, int size);
RIRB_API int rirb_attrs_set_time(int handle, int pos, long long time);
RIRB_API int rirb_attrs_set_frame_attributes(int handle, int pos, const char* keys, const int* key_lens, const char* values,
                                             const int* value_lens, int count);
RIRB_API int rirb_attrs_set_global_attributes(int handle, const char* keys, const int* key_lens, const char* values,
                                              const int* value_lens, int count);

/* ---- zstd movie file: replaces z_open_file_write / z_write_image / z_close_file / z_open_file_read /
 *      z_image_count / z_image_size / z_read_image / z_get_timestamps, ZFile.h:16-52 / ZFile.cpp (the
 *      BIN_FILE_Z_COMPRESSED branch of IRFileLoader, IRFileLoader.cpp:331-370,540-541).  Files are
 *      byte-compatible both ways with the reference's.  Handles are ints (the reference hands out pointers).
 *      method 1 = zstd of the raw image (the only one ZFile.cpp implements; byte-identical files).  Methods 2 and 3,
 *      which the reference documents (video_io.h:298-305) but never implemented, are defined here as the path's
 *      pre-coder in front of the same zstd stage: record payload = zstd([low-byte plane | high-byte plane]) of the image
 *      (2) or of its temporal residual with a key frame every GOP frames (3); split / delta and their inverses run on
 *      the GPU in whole GOPs (frames that do not fill a GOP wait for the next call or the close).  The *_images entries take
 *      frames[n][h][w] as host or device pointers and use `threads` host threads (0 = all cores). */
RIRB_API int rirb_z_open_file_write(const char* filename, int width, int height, int rate, int method, int clevel);
/* the same with the GOP length of method 3 (rirb_z_open_file_write uses 50, the saver's default) */
RIRB_API int rirb_z_open_file_write_gop(const char* filename, int width, int height, int rate, int method, int clevel, int gop);
RIRB_API int rirb_z_write_image(int handle, const unsigned short* img, long long timestamp);
RIRB_API int rirb_z_write_images(int handle, const unsigned short* frames, long long nframes, const long long* timestamps,
                                 int threads);
RIRB_API long long rirb_z_close_file(int handle);
RIRB_API int rirb_z_open_file_read(const char* filename);
RIRB_API int rirb_z_image_count(int handle);
RIRB_API int rirb_z_method(int handle); /* 1: zstd of the raw image (the reference's files), 2 / 3: pre-coded (this repo) */
RIRB_API int rirb_z_image_size(int handle, int* width, int* height);
RIRB_API int rirb_z_get_timestamps(int handle, long long* times);
RIRB_API int rirb_z_read_image(int handle, int pos, unsigned short* img, long long* timestamp);
RIRB_API int rirb_z_read_images(int handle, int pos, int count, unsigned short* out, long long* timestamps, int threads);
/* Entropy coder of the records written after the call: 0 = host zstd at the file's clevel (the default), 1 = the device
 * coder (rirb_zstd_encode_batch; clevel is ignored).  Every record is a standalone zstd frame, so a file may mix them.
 * Returns -1 for an unknown coder, a read handle, or coder 1 without a CUDA device (no CPU fallback). */
RIRB_API int rirb_z_set_coder(int handle, int coder);
/* LZ matches in the device coder ("coder 2"): on = 1 makes the records the device coder writes after the call
 * rirb_zstd_encode_batch_lz's frames, 0 (the default) rirb_zstd_encode_batch's.  It applies while rirb_z_set_coder selects
 * the device coder (1), for methods 1, 2 and 3.  Returns -1 for a value other than 0 / 1, a read handle, or on = 1 without
 * a CUDA device. */
RIRB_API int rirb_z_set_lz(int handle, int on);

/* Device zstd coder: n payloads of bytes_each bytes back to back at src -> one zstd frame each (RFC 8878: Huffman-coded
 * literals, no sequences; RLE / raw blocks where they are smaller), frame i at dst + i * dst_stride, its size in sizes[i].
 * Blocks are at most 128 KiB and never cross a multiple of `segment` bytes (0 = no segments; methods 2/3 pass w*h so that
 * each byte plane gets its own tables).  src, dst and sizes are DEVICE pointers; the call is asynchronous on the current
 * stream.  dst_stride must be at least 9 + 3 * blocks + bytes_each (the frame when every block is raw). */
RIRB_API int rirb_zstd_encode_batch(const unsigned char* src, long long n, long long bytes_each, long long segment,
                                    unsigned char* dst, long long dst_stride, long long* sizes);

/* Device zstd coder with LZ matches ("coder 2"): the same arguments and contract as rirb_zstd_encode_batch.  Each block is
 * coder 1's block, or an LZ form when that is smaller: a greedy parse of matches of at least 8 bytes inside the block
 * (the latest earlier position with the same 8 bytes), literals coded as coder 1 codes a block, sequences with the
 * predefined or RLE FSE tables.  A frame where no block takes the LZ form is byte for byte coder 1's frame.  It needs
 * about 30 bytes of device memory per input byte while it runs. */
RIRB_API int rirb_zstd_encode_batch_lz(const unsigned char* src, long long n, long long bytes_each, long long segment,
                                       unsigned char* dst, long long dst_stride, long long* sizes);

/* Device zstd decoder: n zstd frames, frame i at src + offsets[i] (sizes[i] bytes) -> its content at dst + i * dst_stride,
 * at most dst_capacity bytes.  status[i] = bytes written, -1 = malformed frame, -2 = a frame this decoder does not take
 * (dictionary ID, content checksum, skippable frame, bytes after the frame's last block).  All pointers are DEVICE
 * pointers; asynchronous on the current stream.  Returns -1 (and sets the last error) for bad arguments or no device. */
RIRB_API int rirb_zstd_decode_batch(const unsigned char* src, const long long* offsets, const unsigned* sizes, long long n,
                                    unsigned char* dst, long long dst_stride, long long dst_capacity, long long* status);

/* ===================== Part 4: the registration front end (SURVEY.md 8f-4) ==================
 * MaskedRegistratorECC.compute, librir/registration/masked_registration_ecc.py:105-191: quantile clamp,
 * min/max normalisation and cv2.findTransformECC(template, image, warp, MOTION_TRANSLATION,
 * (COUNT|EPS, iterations, eps), mask, gaussFiltSize = 1) -- OpenCV 4.13's iteration, including warpAffine's
 * fixed-point (1/32 pixel) coordinates -- on float windows that stay in device memory.  A handle owns one
 * w x h problem: the reference window, the current window, the optional mask and all scratch.
 * set_image: which = 0 reference / 1 current; img = first pixel of the window inside a float image whose rows
 *            are `stride` floats apart (host or device pointer).
 * set_mask : which = 0 the mask findTransformECC gets, 1 the mask of the quantile thresholds (w x h bytes, host or
 *            device, NULL = none).  Two masks because the reference's wrapper hands find_median_pixel a non-contiguous
 *            view of a full-size uint8 mask uncompacted (rir_signal_processing.py:134-136); the Python mirror reproduces it.
 * quantile : find_median_pixel(window.astype(uint16), percent[, mask 1]) of the reference (0) or current (1) window.
 * compute  : thresh = the clamp of :147-151 (+inf / NaN: none); shift[2] = {tx, ty} warm start in, result out
 *            (warp_matrix[0,2], warp_matrix[1,2]); returns 0, or 1 ("NaN encountered.") / 2 ("The algorithm
 *            stopped before its convergence...") where cv2 raises cv2.error, -1 on a bad call.
 * reset_reference: reference = translate(current, dx, dy), the rule of :182-185. */
RIRB_API int rirb_ecc_open(int width, int height);
RIRB_API void rirb_ecc_close(int handle);
RIRB_API int rirb_ecc_set_mask(int handle, int which, const unsigned char* mask);
RIRB_API int rirb_ecc_set_image(int handle, int which, const float* img, int stride);
RIRB_API int rirb_ecc_reset_reference(int handle, float dx, float dy);
RIRB_API int rirb_ecc_quantile(int handle, int which, float percent, int use_mask);
RIRB_API int rirb_ecc_compute(int handle, float thresh, int use_mask, int max_iterations, double eps, float* shift, double* rho,
                              int* iterations);
/* The class's whole tracking loop without leaving the library (start :89-103, compute :105-191,
 * manage_computation_and_tries :229-260).  track_config: sigma / median of the constructor; fixed_ref != 0 keeps the
 * reference window set with rirb_ecc_set_image(handle, 0, ...) for good; clears the history.
 * track: frames[nframes][full_h][full_w], type 'H' (uint16) or 'f' (float32), host or device, in time order; window origin
 *   (x0, y0).  The first frame the handle sees is start() (0, 0, confidence 1), the others compute(): Gaussian, window,
 *   quantile clamp, normalisation, ECC with the previous shift as warm start, and the confidence rule that replaces the
 *   reference (confidence < min - 2 std of the first 21).  max_try = 0: an ECC failure stops the call and is returned
 *   (1 / 2, *processed = frames done); max_try > 0: the manage rule (median lowered by 0.01 per attempt, then the previous
 *   estimate repeated; a median < 1 returns to 1 after a success).  x / y / conf (and iters, may be NULL): nframes entries.
 * track_state: current median, confidence threshold (NaN until it exists), warm start, frames seen. */
RIRB_API int rirb_ecc_track_config(int handle, float sigma, double median, int fixed_ref);
RIRB_API int rirb_ecc_track_set_median(int handle, double median); /* the class's public attribute; keeps the history */
RIRB_API int rirb_ecc_track(int handle, int type, const void* frames, long long nframes, int full_w, int full_h, int x0, int y0,
                            int use_mask, int max_try, double* x, double* y, double* conf, int* iters, long long* processed);
RIRB_API int rirb_ecc_track_state(int handle, double* median, double* conf_thresh, float* start, long long* count);

#ifdef __cplusplus
}
#endif
#endif /* LIBRIR_B200_H */
