/*
 * include/librir_b200_video_io.h -- C ABI of libvideo_io_b200.so
 *
 * The video_io side of the drop-in boundary: the entry points of the reference's video_io library that the per-frame path
 * touches, with identical names, argument orders and status codes (video_io.h, video_io.cpp), so that the file can be
 * dropped into librir/libs/ in place of libvideo_io.so (librir/low_level/misc.py:98-136 globs "*video_io*.so") and the
 * reference's unmodified Python (librir/video_io/rir_video_io.py, IRSaver) drives it.
 *
 * What is behind them: the hot path's kernels (libsignal_processing_b200.so, which this library links), not ffmpeg.  The
 * bitstream codecs of the reference (libx264 / kvazaar through ffmpeg 7.1) are out of scope; movies are stored in the
 * reference's zstd movie file (ZFile.cpp) with compression method 3 = temporal delta + byte planes + zstd, the method
 * video_io.h:298-305 documents and the reference never implemented: GPU pre-coder -> host zstd -> records, plus the
 * reference's attribute trailer.  There is NO CPU implementation: without a CUDA device h264_open_file returns 0.
 * Entry points of video_io.h that are not listed here (HCC tooling, the file-reader callbacks, float-image loads) are not
 * exported.
 */
#ifndef LIBRIR_B200_VIDEO_IO_H
#define LIBRIR_B200_VIDEO_IO_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define RIRB_VIO_API __attribute__((visibility("default")))
#define RIRB_UNSPECIFIED_CHAR_LENGTH 200 /* UNSPECIFIED_CHAR_LENGTH, tools.h: size of the caller's filename buffer */

/* ---- saver: replaces video_io.h:222-280 / video_io.cpp:659-843 (H264_Saver, h264.cpp:1668-2617) ----
 * h264_open_file returns a handle > 0 (0 on failure) and removes an existing file; the container is created by the first
 * image.  h264_set_parameter takes the saver's keys (h264.cpp:1709-1781): lowValueError, highValueError, compressionLevel
 * (0..8, mapped onto zstd levels 1..12), codec ("h264" / "h265": accepted, the frames go to the zstd container with the
 * pre-coder in front; "zstd1" / "zstd2" / "zstd3" pick the container method), GOP, threads (host zstd threads, 0 = all),
 * slices (ignored), stdFactor, inputCamera (must stay 0: the camera calibration is outside this library), removeBadPixels,
 * subtractMin, subtractLocalMin (ignored), runningAverage, and this library's entropyCoder ("host": host zstd at
 * compressionLevel, the default; "gpu": the device coder, Huffman-literal zstd frames that any zstd decoder reads; "gpu-lz":
 * the device coder with LZ matches in the blocks where they make the frame smaller; the device coders need a CUDA device,
 * and the value applies to the images added after the call); -1 for an unknown key or value.
 * h264_add_image_lossy = addImageLossyNoCamera (h264.cpp:2253-2424) in front of the lossless stage, with the
 * BackgroundError / ForegroundError frame attributes and the MIN_T / MIN_T_HEIGHT / Global*Error global ones;
 * h264_add_loss = addLoss (:2426-2607), in place on the caller's image, nothing is stored;
 * h264_get_low/high_errors: -2 and *size = required count when the buffer is too small. */
RIRB_VIO_API int h264_open_file(const char* filename, int width, int height, int lossy_height);
RIRB_VIO_API void h264_close_file(int file);
RIRB_VIO_API int h264_set_parameter(int file, const char* param, const char* value);
RIRB_VIO_API int h264_set_global_attributes(int file, int attribute_count, char* keys, int* key_lens, char* values, int* value_lens);
RIRB_VIO_API int h264_add_image_lossless(int file, unsigned short* img, int64_t timestamps_ns, int attribute_count, char* keys,
                                         int* key_lens, char* values, int* value_lens);
RIRB_VIO_API int h264_add_image_lossy(int file, unsigned short* img_DL, int64_t timestamps_ns, int attribute_count, char* keys,
                                      int* key_lens, char* values, int* value_lens);
RIRB_VIO_API int h264_add_loss(int file, unsigned short* img);
RIRB_VIO_API int h264_get_low_errors(int file, unsigned short* errors, int* size);
RIRB_VIO_API int h264_get_high_errors(int file, unsigned short* errors, int* size);
RIRB_VIO_API void set_ffmpeg_log_enabled(int enable); /* video_io.h:215; nothing to switch here */

/* ---- the zstd writer trio, video_io.h:298-314 (declared by the reference, defined nowhere in it): method 1 = zstd of the
 *      raw image (files byte-identical to ZFile.cpp's), 2 = byte planes + zstd, 3 = temporal delta + byte planes + zstd ---- */
RIRB_VIO_API int open_video_write(const char* filename, int width, int height, int rate, int method, int clevel);
RIRB_VIO_API int image_write(int writter, unsigned short* img, int64_t time);
RIRB_VIO_API int64_t close_video(int writter);

/* ---- reader: replaces video_io.h:30-209 / video_io.cpp:16-644 for zstd movie files (methods 1-3; *file_format = 4,
 *      FILE_FORMAT_ZSTD_COMPRESSED).  load_image (calibration 0 only) is IRFileLoader::readImage's chain
 *      (IRFileLoader.cpp:1168-1247): decode -> += MIN_T on the first MIN_T_HEIGHT rows -> removeBadPixels -> removeMotion,
 *      the last three on the GPU; enable_bad_pixels detects on readImage(0) without its last 3 rows (:693-716);
 *      load_motion_correction_file reads the 4-column .regfile (:822-847).  get_attribute* refer to the image read last;
 *      -2 with the required sizes written back when a buffer is too small. ---- */
RIRB_VIO_API int open_camera_file(const char* filename, int* file_format);
RIRB_VIO_API int video_file_format(const char* filename);
RIRB_VIO_API int close_camera(int camera);
RIRB_VIO_API int get_image_count(int camera);
RIRB_VIO_API int get_image_time(int camera, int pos, int64_t* time);
RIRB_VIO_API int get_image_size(int camera, int* width, int* height);
RIRB_VIO_API int get_filename(int camera, char* filename);
RIRB_VIO_API int supported_calibrations(int camera, int* count);
RIRB_VIO_API int calibration_name(int camera, int calibration, char* name);
RIRB_VIO_API int load_image(int camera, int pos, int calibration, unsigned short* pixels);
RIRB_VIO_API int enable_bad_pixels(int cam, int enable);
RIRB_VIO_API int bad_pixels_enabled(int cam);
RIRB_VIO_API int load_motion_correction_file(int cam, const char* filename);
RIRB_VIO_API int enable_motion_correction(int cam, int enable);
RIRB_VIO_API int motion_correction_enabled(int cam);
RIRB_VIO_API int get_attribute_count(int camera);
RIRB_VIO_API int get_attribute(int camera, int index, char* key, int* key_len, char* value, int* value_len);
RIRB_VIO_API int get_global_attribute_count(int camera);
RIRB_VIO_API int get_global_attribute(int camera, int index, char* key, int* key_len, char* value, int* value_len);

/* ---- raw movies and the entries of the calibration objects.  open_camera_file also opens the reference's raw files: PCR (a
 *      1024-byte header, IRFileLoader.h:43-61, then frames; *file_format = 1, or 3 for the encapsulated form) -- what
 *      IRMovie.from_numpy_array writes before it converts -- and uncompressed WEST acquisition files (*file_format = 2), with
 *      the reference's timestamp search and conversions (IRFileLoader.cpp:256-283, 404-466); open_camera_from_memory (video_io.cpp:110-145) goes through a
 *      temporary file; correct_PCR_file as video_io.cpp:911-930.  The movies this library opens carry no camera calibration:
 *      emissivities are loader state (IRVideoLoader.h:47-95), calibration_files / support_emissivity / calibrate_* /
 *      get_table* answer -1 and flip_camera_calibration -2, the reference's answers for such a movie. ---- */
RIRB_VIO_API int open_camera_from_memory(void* ptr, int64_t size, int* file_format);
RIRB_VIO_API int correct_PCR_file(const char* filename, int width, int height, int freq);
RIRB_VIO_API int flip_camera_calibration(int camera, int flip_rl, int flip_ud);
RIRB_VIO_API int set_global_emissivity(int cam, float emi);
RIRB_VIO_API int set_emissivity(int cam, float* emi, int size);
RIRB_VIO_API int get_emissivity(int cam, float* emi, int size);
RIRB_VIO_API int support_emissivity(int cam);
RIRB_VIO_API int camera_saturate(int cam);
RIRB_VIO_API int calibration_files(int cam, char* dst, int* dstSize);
RIRB_VIO_API int calibrate_inplace(int cam, unsigned short* img, int size, int calibration);
RIRB_VIO_API int calibrate_image(int cam, unsigned short* img, float* out, int size, int calib);
RIRB_VIO_API int calibrate_image_inplace(int cam, unsigned short* img, int size, int calib);
RIRB_VIO_API int get_table_names(int cam, char* dst, int* dst_size);
RIRB_VIO_API int get_table(int cam, const char* name, float* dst, int* dst_size);

/* additive: text of the calling thread's last failure in this library */
RIRB_VIO_API const char* rirb_video_io_last_error(void);

#ifdef __cplusplus
}
#endif
#endif /* LIBRIR_B200_VIDEO_IO_H */
