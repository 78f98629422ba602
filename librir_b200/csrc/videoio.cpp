// librir_b200/csrc/videoio.cpp -- libvideo_io_b200.so: the video_io side of the drop-in boundary (include/librir_b200_video_io.h).
//
// Host code over the C ABI of libsignal_processing_b200.so (the CUDA kernels live there; this file contains no device code and
// no CPU implementation of any of them).  It gives the reference's own entry points
//   * the saver:   h264_open_file / h264_set_parameter / h264_set_global_attributes / h264_add_image_lossless /
//                  h264_add_image_lossy / h264_add_loss / h264_get_low_errors / h264_get_high_errors / h264_close_file
//                  (video_io.h:222-280, video_io.cpp:659-843) and the declared-but-never-defined zstd writer trio
//                  open_video_write / image_write / close_video (video_io.h:298-314);
//   * the reader:  open_camera_file / video_file_format / close_camera / get_image_count / get_image_time / get_image_size /
//                  get_filename / supported_calibrations / calibration_name / load_image / enable_bad_pixels /
//                  bad_pixels_enabled / load_motion_correction_file / enable_motion_correction / motion_correction_enabled /
//                  get_attribute_count / get_attribute / get_global_attribute_count / get_global_attribute
//                  (video_io.h:30-209, video_io.cpp:16-644)
// the names, argument orders and status codes the reference's Python (librir/video_io/rir_video_io.py) binds.
//
// What is behind them is the hot path, not ffmpeg: the bitstream stage of the reference (libx264 / kvazaar through ffmpeg 7.1)
// is out of scope, so a movie is stored in the reference's OTHER container, the zstd movie file (ZFile.cpp), with the
// compression method the reference documents for it but never implemented -- 3 = temporal delta + byte planes + zstd
// (video_io.h:298-305) -- i.e. GPU pre-coder (rirb_precode_movie) -> host zstd -> records, plus the reference's attribute
// trailer (timestamps, per-frame and global attributes, "GOP", "MIN_T" ...).  The lossy saver runs the bounded-error
// pre-conditioner on the GPU (rirb_lossy_*) in front of it.  Files written with method 1 are byte-identical to the reference's
// and readable by it; the reader below opens methods 1-3 and applies IRFileLoader::readImage's chain on the GPU
// (+= MIN_T, bad pixels, motion correction).
#include <stdint.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>

#include <fstream>
#include <map>
#include <memory>
#include <mutex>
#include <sstream>
#include <string>
#include <vector>

#include "../../include/librir_b200.h"
#include "../../include/librir_b200_video_io.h"
#include "handles.h"

namespace {

typedef std::map<std::string, std::string> AttrMap;

using rirb::Table;

thread_local std::string g_last_error;
void fail(const std::string& what)
{
    g_last_error = what;
    if (getenv("LIBRIR_B200_VERBOSE")) fprintf(stderr, "[librir_b200 video_io] %s\n", what.c_str());
}

AttrMap unpack(int count, const char* keys, const int* key_lens, const char* values, const int* value_lens)
{
    AttrMap m;
    for (int i = 0; i < count; ++i) {
        m[std::string(keys, keys + key_lens[i])] = std::string(values, values + value_lens[i]);
        keys += key_lens[i];
        values += value_lens[i];
    }
    return m;
}

// the (keys, key_lens, values, value_lens) convention of the attrs_* interface
struct Packed {
    std::string keys, values;
    std::vector<int> klens, vlens;
    explicit Packed(const AttrMap& m)
    {
        for (const auto& kv : m) {
            keys += kv.first;
            values += kv.second;
            klens.push_back((int)kv.first.size());
            vlens.push_back((int)kv.second.size());
        }
    }
    int count() const { return (int)klens.size(); }
};

std::string attr_string(int (*get)(int, int, char*, int*), int handle, int pos)
{
    int len = 0;
    std::string out;
    if (get(handle, pos, nullptr, &len) != -2 && len == 0) return out;  // -2: too small, len = required size
    out.resize((size_t)len);
    if (len > 0 && get(handle, pos, &out[0], &len) != 0) out.clear();
    return out;
}
std::string frame_attr_string(int (*get)(int, int, int, char*, int*), int handle, int frame, int pos)
{
    int len = 0;
    std::string out;
    if (get(handle, frame, pos, nullptr, &len) != -2 && len == 0) return out;
    out.resize((size_t)len);
    if (len > 0 && get(handle, frame, pos, &out[0], &len) != 0) out.clear();
    return out;
}

// ---------------------------------------------------------------------------------------------------------------------
// saver
// ---------------------------------------------------------------------------------------------------------------------
// the saver's coder 0 / 1 / 2 on a container handle: the device coder (1) with LZ matches off / on
static int set_coder(int zfile, int coder)
{
    if (rirb_z_set_coder(zfile, coder == 0 ? 0 : 1) != 0) return -1;
    return coder == 0 ? 0 : rirb_z_set_lz(zfile, coder == 2 ? 1 : 0);
}

struct Saver {
    std::string filename;
    int w = 0, h = 0, lossy_height = 0;
    // H264_Saver's parameters (h264.cpp:1709-1781) and their defaults (PrivateData(), :1663-1665)
    int clevel = 0, low_error = 6, high_error = 2, gop = 50, threads = 0, slices = 1, running_average = 32;
    int input_camera = 0, remove_bad_pixels = 0, subtract_min = 0, subtract_local_min = 0;
    double std_factor = 5.0;
    std::string codec = "h264";
    int method = 3;  // container method: 3 = delta + byte planes + zstd; "codec" = "zstd1" / "zstd2" / "zstd3" selects it
    int coder = 0;   // entropy coder of the records: 0 = host zstd, 1 / 2 = the device coder without / with LZ matches
                     // ("entropyCoder" = "host" / "gpu" / "gpu-lz")
    AttrMap global;
    // open state
    int zfile = 0;        // rirb_z_* handle, 0 until the first image
    int lossy = 0;        // rirb_lossy_* handle
    int lossy_variant = -1;  // 0 add_image_lossy, 1 add_loss
    std::vector<AttrMap> frame_attrs;
    std::vector<unsigned short> low_errors, high_errors;
    std::vector<unsigned short> scratch;
    unsigned short min_T = 0;
    bool have_min = false;
    std::mutex mu;

    bool open_container()
    {
        if (zfile) return true;
        // zstd levels: the saver's compressionLevel 0..8 picks an x264 preset (ultrafast..veryslow, h264.cpp:464-494); the same
        // scale is used for zstd (0 = its fast default, 3; 8 = 19)
        static const int level_of[9] = {1, 2, 3, 4, 5, 6, 8, 10, 12};  // beyond 12 zstd costs 5-10x more per frame for a few per cent on byte planes
        const int lv = level_of[clevel < 0 ? 0 : (clevel > 8 ? 8 : clevel)];
        zfile = rirb_z_open_file_write_gop(filename.c_str(), w, h, 50, method, lv, gop);  // 50: the fps h264_* hands H264_Saver::open
        if (!zfile) fail(std::string("cannot create the movie file: ") + rirb_last_error());
        else if (coder != 0 && set_coder(zfile, coder) != 0) fail(std::string("entropyCoder: ") + rirb_last_error());
        return zfile != 0;
    }
    bool open_lossy(int variant)
    {
        if (lossy) {
            if (variant != lossy_variant) {
                fail("h264_add_image_lossy and h264_add_loss cannot be mixed on one file");
                return false;
            }
            return true;
        }
        if (input_camera) {
            fail("inputCamera = 1 needs the camera calibration, which is outside this library: feed temperatures (inputCamera = 0)");
            return false;
        }
        lossy = rirb_lossy_open(w, h, lossy_height, low_error, high_error, std_factor, running_average, subtract_min, remove_bad_pixels);
        if (!lossy) {
            fail(std::string("cannot set up the lossy pre-conditioner: ") + rirb_last_error());
            return false;
        }
        rirb_lossy_set_parameter(lossy, "variant", variant ? "add_loss" : "add_image_lossy");
        lossy_variant = variant;
        return true;
    }
    // one frame through the pre-conditioner; out = what the lossless stage then stores
    bool precondition(const unsigned short* img, unsigned short* out)
    {
        int err[2] = {0, 0};
        if (rirb_lossy_add_images(lossy, img, 1, out, err) != 0) {
            fail(std::string("lossy pre-conditioner: ") + rirb_last_error());
            return false;
        }
        low_errors.push_back((unsigned short)err[0]);
        high_errors.push_back((unsigned short)err[1]);
        if (subtract_min && !have_min) {  // the first image fixes MIN_T: the minimum of its (corrected) lossy rows, h264.cpp:2277-2296
            int m = 0;
            if (rirb_lossy_get_min(lossy, &m) != 0) {
                fail(std::string("lossy pre-conditioner: ") + rirb_last_error());
                return false;
            }
            min_T = (unsigned short)m;
            have_min = true;
        }
        return true;
    }
};
Table<Saver> g_savers;

// ---------------------------------------------------------------------------------------------------------------------
// reader
// ---------------------------------------------------------------------------------------------------------------------
// The raw movie files of the reference's reader (IRFileLoader.h:43-61): a 1024-byte PCR header (int32 Version, NbImages, X, Y,
// Band, Bits, Interlaced, Frequency, ImagesPerBuffer, TransfertSize, GrabSizeX, GrabSizeY), optionally behind 133 bytes of
// envelope, then frames of TransfertSize bytes.  What IRMovie.from_numpy_array writes before it converts to a compressed movie.
struct PcrHeader {
    int32_t version, nb_images, x, y, band, bits, interlaced, frequency, images_per_buffer, transfer_size, grab_x, grab_y;
};
#define FILE_FORMAT_PCR 1
#define FILE_FORMAT_WEST 2
#define FILE_FORMAT_ZSTD_COMPRESSED 4 /* video_io.h:17-23 */
#define FILE_FORMAT_PCR_ENCAPSULATED 3

struct Camera {
    std::string filename;
    int format = FILE_FORMAT_ZSTD_COMPRESSED;
    FILE* raw = nullptr;  // PCR files: frames at raw_start + pos * raw_transfer
    long long raw_start = 0, raw_transfer = 0;
    int zfile = 0;
    int w = 0, h = 0, count = 0;
    std::vector<long long> times;
    AttrMap global;
    std::vector<AttrMap> frame_attrs;
    int min_T = 0, min_T_height = 0;
    bool bp_enabled = false, motion_enabled = false;
    int bp_handle = 0;
    std::vector<double> shift_x, shift_y;
    std::vector<float> inv_emissivity;  // IRVideoLoader::m_invEmissivities: state only, no calibration uses it here
    std::string temp_file;              // open_camera_from_memory: the bytes live in a temporary file, removed on close
    int last_pos = -1;
    std::mutex mu;
    ~Camera()
    {
        if (zfile) rirb_z_close_file(zfile);
        if (raw) fclose(raw);
        if (bp_handle) bad_pixels_destroy(bp_handle);
        if (!temp_file.empty()) remove(temp_file.c_str());
    }
    bool read_raw(int pos, unsigned short* pixels)
    {
        // bin_read_image's last branch, IRFileLoader.cpp:547-557
        const size_t bytes = (size_t)w * h * 2;
        if (fseeko(raw, (off_t)(raw_start + raw_transfer * pos), SEEK_SET) != 0) return false;
        return fread(pixels, 1, bytes, raw) == bytes;
    }
    // IRFileLoader::readImage, calibration 0 (IRFileLoader.cpp:1168-1247): decode -> += MIN_T -> removeBadPixels -> removeMotion
    bool read(int pos, unsigned short* pixels, bool with_bad_pixels)
    {
        if (pos < 0 || pos >= count) return false;
        if (raw ? !read_raw(pos, pixels) : rirb_z_read_image(zfile, pos, pixels, nullptr) != 0) return false;
        const bool bp = with_bad_pixels && bp_enabled && bp_handle != 0;
        const bool mo = motion_enabled && !shift_x.empty();
        if (min_T == 0 && !bp && !mo) return true;
        return rirb_loader_finish_frames(bp ? bp_handle : 0, pixels, 1, w, h, min_T, min_T_height, mo ? &shift_x[pos] : nullptr,
                                         mo ? &shift_y[pos] : nullptr, h > 3 ? 3 : 0) == 0;
    }
};
Table<Camera> g_cameras;

// IRFileLoader::findFileType's PCR tests (IRFileLoader.cpp:124-181) and bin_open_file's raw branch (:404-431): frame count from
// the file size, timestamps from the last 8 bytes of every frame when they increase strictly (findTimes, :256-283), else
// i / Frequency.
static bool open_raw(Camera& c)
{
    FILE* f = fopen(c.filename.c_str(), "rb");
    if (!f) return false;
    char buf[2000];
    memset(buf, 0, sizeof(buf));
    if (fread(buf, 1, sizeof(buf), f) < sizeof(PcrHeader)) {
        fclose(f);
        return false;
    }
    PcrHeader hd, enc;
    memcpy(&hd, buf, sizeof(hd));
    memcpy(&enc, buf + 128 + 5, sizeof(enc));
    auto plausible = [](const PcrHeader& p, int lim) {
        return p.bits == 16 && llabs((long long)p.transfer_size - (long long)p.x * p.y * 2) < 2000 && p.x > 0 && p.y > 0 && p.x < lim && p.y < lim;
    };
    if (hd.bits == 16 && hd.x == 640 && hd.y == 512 && hd.frequency == 50) {  // "IR lab videos": the transfer size is forced
        hd.transfer_size = hd.x * hd.y * 2;
        c.raw_start = 1024;
    } else if (plausible(hd, 2000)) {
        c.raw_start = 1024;
    } else if (plausible(enc, 1000)) {
        hd = enc;
        c.raw_start = 1024 + 128 + 5;
        c.format = FILE_FORMAT_PCR_ENCAPSULATED;
    } else if ((unsigned char)buf[0] < 10 && buf[2] == 0 && buf[1] == 1) {
        // uncompressed WEST acquisition file (:183-207): BIN_HEADER {version, triggers, compression} in 128 bytes, then one
        // BIN_TRIGGER of int64 {date, rate, samples, ..., data_size_x, data_size_y} in 128 bytes, then the frames
        int64_t trig[11];
        memcpy(trig, buf + 128, sizeof(trig));
        const int64_t rate = trig[1], sxz = trig[9], syz = trig[10];
        if (!(sxz > 0 && sxz < 1000 && syz > 0 && syz < 1000 && rate > 0 && rate < 1000)) {
            fclose(f);
            return false;
        }
        memset(&hd, 0, sizeof(hd));
        hd.x = (int)sxz;
        hd.y = (int)syz;
        hd.transfer_size = hd.x * hd.y * 2;
        hd.frequency = (int)rate;
        hd.bits = 16;
        c.raw_start = 256;
        c.format = FILE_FORMAT_WEST;
    } else {
        fclose(f);
        return false;
    }
    if (c.format != FILE_FORMAT_PCR_ENCAPSULATED && c.format != FILE_FORMAT_WEST) c.format = FILE_FORMAT_PCR;
    fseeko(f, 0, SEEK_END);
    const long long size = (long long)ftello(f);
    c.raw_transfer = hd.transfer_size;
    c.w = hd.x;
    c.h = hd.y;
    c.count = c.raw_transfer > 0 ? (int)((size - c.raw_start) / c.raw_transfer) : 0;
    if (c.count <= 0 || c.raw_transfer < (long long)c.w * c.h * 2) {
        fclose(f);
        return false;
    }
    c.times.resize((size_t)c.count);
    bool has_times = true;
    for (int i = 0; i < c.count && has_times; ++i) {
        long long t = 0;
        has_times = fseeko(f, (off_t)(c.raw_start + c.raw_transfer * (long long)(i + 1) - 8), SEEK_SET) == 0 && fread(&t, 1, 8, f) == 8;
        c.times[(size_t)i] = t;
        if (i > 0 && c.times[(size_t)i] <= c.times[(size_t)i - 1]) has_times = false;
    }
    if (!has_times) {
        const double sampling = 1000000000.0 / (double)(hd.frequency > 0 ? hd.frequency : 50);
        for (int i = 0; i < c.count; ++i) c.times[(size_t)i] = (long long)(i * sampling);
    } else {  // :433-452: origin-relative ms -> ns; other values that are not ns already -> ns relative to the first image
        const long long t0 = c.times[0];
        if (t0 > 28000 && t0 < 32000) {
            for (auto& t : c.times) t *= 1000000LL;
        } else if (!(c.times.front() < -1000000000LL || c.times.back() > 1000000000LL)) {
            for (auto& t : c.times) t = (t - t0) * 1000000LL;
        }
    }
    if (c.times.front() > 28000000000LL && c.times.front() < 32000000000LL)  // :458-466
        for (auto& t : c.times) t -= 32000000000LL;
    c.raw = f;
    c.min_T_height = c.h - 3;
    return true;
}

std::shared_ptr<Camera> open_camera(const char* filename)
{
    if (!filename) return nullptr;
    auto c = std::make_shared<Camera>();
    c->filename = filename;
    for (auto& ch : c->filename)
        if (ch == '\\') ch = '/';
    c->zfile = rirb_z_open_file_read(filename);
    if (!c->zfile) {
        const std::string zerr = rirb_last_error();
        if (!open_raw(*c)) {
            fail(std::string("Unable to open camera file ") + filename + ": " + zerr);
            return nullptr;
        }
        return c;
    }
    c->count = rirb_z_image_count(c->zfile);
    rirb_z_image_size(c->zfile, &c->w, &c->h);
    c->times.resize((size_t)(c->count > 0 ? c->count : 0));
    if (c->count > 0) rirb_z_get_timestamps(c->zfile, c->times.data());
    if (c->count > 0 && rirb_z_method(c->zfile) == 1) {
        // The reference's own zstd movie files are WEST acquisition files with times in ms: bin_open_file_from_file_reader,
        // IRFileLoader.cpp:354-372 -- origin-relative ms (first value 28,000-32,000) become ns minus 10 ms, other values that
        // are not ns already become ns relative to the first image.  (Methods 2 / 3 are written by this library's saver, which
        // stands in for the mp4 writer: ns, as given.)
        const long long t0 = c->times[0];
        if (t0 > 28000 && t0 < 32000) {
            for (auto& t : c->times) t = t * 1000000LL - 10000000LL;
        } else if (!(c->times.front() < -1000000000LL || c->times.back() > 1000000000LL)) {
            for (auto& t : c->times) t = (t - t0) * 1000000LL;
        }
    }
    // "timestamps starting at -2 s for WEST videos" (:458-466, every file type)
    if (c->count > 0 && c->times.front() > 28000000000LL && c->times.front() < 32000000000LL)
        for (auto& t : c->times) t -= 32000000000LL;
    // the attribute trailer: global + per-frame attributes
    const int a = rirb_attrs_open_file(filename);
    if (a) {
        const int ng = rirb_attrs_global_attribute_count(a);
        for (int i = 0; i < ng; ++i) {
            const std::string k = attr_string(rirb_attrs_global_attribute_name, a, i);
            if (k == "positions") continue;  // the container's own index, not a user attribute
            c->global[k] = attr_string(rirb_attrs_global_attribute_value, a, i);
        }
        if (rirb_attrs_image_count(a) == c->count) {
            c->frame_attrs.resize((size_t)c->count);
            for (int f = 0; f < c->count; ++f) {
                const int nf = rirb_attrs_frame_attribute_count(a, f);
                for (int i = 0; i < nf; ++i)
                    c->frame_attrs[f][frame_attr_string(rirb_attrs_frame_attribute_name, a, f, i)] =
                        frame_attr_string(rirb_attrs_frame_attribute_value, a, f, i);
            }
        }
        rirb_attrs_abandon(a);  // read only: nothing is written back
    }
    // IRFileLoader::open, IRFileLoader.cpp:904-921
    auto it = c->global.find("MIN_T");
    if (it != c->global.end()) c->min_T = atoi(it->second.c_str());
    it = c->global.find("MIN_T_HEIGHT");
    if (it != c->global.end()) c->min_T_height = atoi(it->second.c_str());
    if (c->min_T_height == 0) c->min_T_height = c->h - 3;
    return c;
}

int copy_attr(const AttrMap& m, int index, char* key, int* key_len, char* value, int* value_len, bool global)
{
    if (index < 0 || index >= (int)m.size() || !key_len || !value_len) return -1;
    auto it = m.begin();
    std::advance(it, index);
    const int s1 = (int)it->first.size(), s2 = (int)it->second.size();
    const int oldk = *key_len, oldv = *value_len;
    // video_io.cpp:571-591 (frame attributes) and :624-642 (global ones, which want room for a terminating zero)
    if ((global ? s1 + 1 : s1) > oldk || s2 > oldv) {
        *key_len = global ? s1 + 1 : s1;
        *value_len = s2;
        return -2;
    }
    *key_len = s1;
    *value_len = s2;
    memcpy(key, it->first.data(), (size_t)s1);
    memcpy(value, it->second.data(), (size_t)s2);
    if (global || oldk > s1) key[s1] = 0;
    if (oldv > s2) value[s2] = 0;
    return 0;
}

}  // namespace

extern "C" {

const char* rirb_video_io_last_error(void) { return g_last_error.c_str(); }
void set_ffmpeg_log_enabled(int) {}  // no ffmpeg behind this library

// =====================================================================================================================
// saver
// =====================================================================================================================
int h264_open_file(const char* filename, int width, int height, int lossy_height)
{
    if (!filename || width <= 0 || height <= 0 || lossy_height < 0 || lossy_height > height) {
        fail("h264_open_file: bad arguments");
        return 0;
    }
    if (rirb_device_count() <= 0) {
        fail("h264_open_file: no CUDA device (this library has no CPU implementation)");
        return 0;
    }
    auto s = std::make_shared<Saver>();
    s->filename = filename;
    s->w = width;
    s->h = height;
    s->lossy_height = lossy_height;
    if (FILE* f = fopen(filename, "rb")) {  // video_io.cpp:668-676: an existing file is removed first
        fclose(f);
        if (remove(filename) != 0) {
            fail("h264_open_file: cannot remove output file");
            return 0;
        }
    }
    return g_savers.add(s);
}

int h264_set_parameter(int file, const char* param, const char* value)
{
    auto s = g_savers.get(file);
    if (!s || !param || !value) {
        fail("h264_set_parameter: NULL identifier");
        return -1;
    }
    std::lock_guard<std::mutex> lock(s->mu);
    const std::string k(param);
    if (k == "lowValueError") s->low_error = atoi(value);
    else if (k == "highValueError") s->high_error = atoi(value);
    else if (k == "compressionLevel") s->clevel = atoi(value);
    else if (k == "codec") {
        s->codec = value;
        // "h264" / "h265" name bitstream codecs this library does not contain: the frames go to the zstd container with the
        // pre-coder in front (method 3); "zstd1" .. "zstd3" pick the container method explicitly
        if (s->codec == "zstd1") s->method = 1;
        else if (s->codec == "zstd2") s->method = 2;
        else s->method = 3;
    } else if (k == "GOP") s->gop = atoi(value) > 0 ? atoi(value) : 50;
    else if (k == "threads") s->threads = atoi(value);
    else if (k == "slices") s->slices = atoi(value);
    else if (k == "stdFactor") s->std_factor = atof(value);
    else if (k == "inputCamera") s->input_camera = atoi(value);
    else if (k == "removeBadPixels") s->remove_bad_pixels = atoi(value) != 0;
    else if (k == "subtractMin") s->subtract_min = atoi(value) != 0;
    else if (k == "subtractLocalMin") s->subtract_local_min = atoi(value) != 0;
    else if (k == "runningAverage") s->running_average = atoi(value) > 64 ? 64 : atoi(value);
    else if (k == "entropyCoder") {
        // "host": zstd on the host threads at compressionLevel (the default); "gpu": the device coder, Huffman-coded zstd frames
        // that any zstd decoder reads (compressionLevel does not apply); "gpu-lz": the device coder with LZ matches in the
        // blocks where they make the frame smaller.  Applies to the images added after the call.
        const std::string v(value);
        if (v != "host" && v != "gpu" && v != "gpu-lz") return -1;
        const int c = v == "gpu" ? 1 : v == "gpu-lz" ? 2 : 0;
        if (c != 0 && rirb_device_count() <= 0) {
            fail("h264_set_parameter: entropyCoder " + v + " needs a CUDA device (no CPU fallback)");
            return -1;
        }
        if (s->zfile && set_coder(s->zfile, c) != 0) {
            fail(std::string("h264_set_parameter: ") + rirb_last_error());
            return -1;
        }
        s->coder = c;
    } else {
        return -1;  // H264_Saver::setParameter returns false for an unknown key (h264.cpp:1780)
    }
    return 0;
}

int h264_set_global_attributes(int file, int attribute_count, char* keys, int* key_lens, char* values, int* value_lens)
{
    auto s = g_savers.get(file);
    if (!s) {
        fail("h264_set_global_attributes: NULL identifier");
        return -1;
    }
    std::lock_guard<std::mutex> lock(s->mu);
    s->global = unpack(attribute_count, keys, key_lens, values, value_lens);
    return 0;
}

static int add_frame(Saver& s, const unsigned short* stored, int64_t ts, const AttrMap& attrs)
{
    if (!s.open_container()) return -1;
    long long t = ts;
    if (rirb_z_write_images(s.zfile, stored, 1, &t, s.threads) != 0) {
        fail(std::string("cannot write the image: ") + rirb_last_error());
        return -1;
    }
    s.frame_attrs.push_back(attrs);
    return 0;
}

int h264_add_image_lossless(int file, unsigned short* img, int64_t timestamps_ns, int attribute_count, char* keys, int* key_lens,
                            char* values, int* value_lens)
{
    auto s = g_savers.get(file);
    if (!s || !img) {
        fail("h264_add_image_lossless: NULL identifier");
        return -1;
    }
    std::lock_guard<std::mutex> lock(s->mu);
    return add_frame(*s, img, timestamps_ns, unpack(attribute_count, keys, key_lens, values, value_lens));
}

int h264_add_image_lossy(int file, unsigned short* img_DL, int64_t timestamps_ns, int attribute_count, char* keys, int* key_lens,
                         char* values, int* value_lens)
{
    auto s = g_savers.get(file);
    if (!s || !img_DL) {
        fail("h264_add_image_lossy: NULL identifier");
        return -1;
    }
    std::lock_guard<std::mutex> lock(s->mu);
    if (!s->open_lossy(0)) return -1;
    s->scratch.resize((size_t)s->w * s->h);
    const bool first = s->low_errors.empty();
    if (!s->precondition(img_DL, s->scratch.data())) return -1;
    AttrMap attrs = unpack(attribute_count, keys, key_lens, values, value_lens);
    if (first) {  // h264.cpp:2293-2299
        if (s->subtract_min) {
            s->global["MIN_T"] = std::to_string((int)s->min_T);
            s->global["MIN_T_HEIGHT"] = std::to_string(s->lossy_height);
        }
        s->global["GlobalBackgroundError"] = std::to_string(s->low_error);
        s->global["GlobalForegroundError"] = std::to_string(s->high_error);
    } else {  // :2378-2380
        attrs["BackgroundError"] = std::to_string((int)s->low_errors.back());
        attrs["ForegroundError"] = std::to_string((int)s->high_errors.back());
    }
    return add_frame(*s, s->scratch.data(), timestamps_ns, attrs);
}

int h264_add_loss(int file, unsigned short* img)
{
    auto s = g_savers.get(file);
    if (!s || !img) {
        fail("h264_add_loss: NULL identifier");
        return -1;
    }
    std::lock_guard<std::mutex> lock(s->mu);
    if (!s->open_lossy(1)) return -1;
    s->scratch.resize((size_t)s->w * s->h);
    if (!s->precondition(img, s->scratch.data())) return -1;
    // addLoss hands back the lossy rows only (h264.cpp:2604); the caller's other rows stay as they were
    memcpy(img, s->scratch.data(), (size_t)s->w * s->lossy_height * 2);
    return 0;
}

static int copy_errors(const std::vector<unsigned short>& v, unsigned short* errors, int* size)
{
    if (!size) return -1;
    if (*size < (int)v.size()) {  // video_io.cpp:817-821
        *size = (int)v.size();
        return -2;
    }
    *size = (int)v.size();
    if (errors && !v.empty()) memcpy(errors, v.data(), v.size() * sizeof(unsigned short));
    return 0;
}
int h264_get_low_errors(int file, unsigned short* errors, int* size)
{
    auto s = g_savers.get(file);
    if (!s) {
        fail("h264_get_low_erros: NULL identifier");
        return -1;
    }
    std::lock_guard<std::mutex> lock(s->mu);
    return copy_errors(s->low_errors, errors, size);
}
int h264_get_high_errors(int file, unsigned short* errors, int* size)
{
    auto s = g_savers.get(file);
    if (!s) {
        fail("h264_get_high_erros: NULL identifier");
        return -1;
    }
    std::lock_guard<std::mutex> lock(s->mu);
    return copy_errors(s->high_errors, errors, size);
}

void h264_close_file(int file)
{
    auto s = g_savers.get(file);
    if (!s) {
        fail("h264_close_file: NULL identifier");
        return;
    }
    {
        std::lock_guard<std::mutex> lock(s->mu);
        if (s->zfile) {
            rirb_z_close_file(s->zfile);  // flushes the last GOP, writes timestamps + record positions into the trailer
            s->zfile = 0;
            // the saver's own trailer entries (H264_Saver::close, h264.cpp:1883-1912) next to the container's
            const int a = rirb_attrs_open_file(s->filename.c_str());
            if (a) {
                AttrMap g = s->global;
                const int ng = rirb_attrs_global_attribute_count(a);
                for (int i = 0; i < ng; ++i) {  // keep what the container stored ("positions", "GOP")
                    const std::string k = attr_string(rirb_attrs_global_attribute_name, a, i);
                    if (!g.count(k)) g[k] = attr_string(rirb_attrs_global_attribute_value, a, i);
                }
                g["GOP"] = std::to_string(s->gop);
                const Packed pg(g);
                rirb_attrs_set_global_attributes(a, pg.keys.data(), pg.klens.data(), pg.values.data(), pg.vlens.data(), pg.count());
                const int n = rirb_attrs_image_count(a);
                for (int f = 0; f < n && f < (int)s->frame_attrs.size(); ++f) {
                    if (s->frame_attrs[f].empty()) continue;
                    const Packed pf(s->frame_attrs[f]);
                    rirb_attrs_set_frame_attributes(a, f, pf.keys.data(), pf.klens.data(), pf.values.data(), pf.vlens.data(), pf.count());
                }
                rirb_attrs_close(a);
            }
        }
        if (s->lossy) rirb_lossy_close(s->lossy);
        s->lossy = 0;
    }
    g_savers.remove(file);
}

// ---- the zstd writer trio of video_io.h:298-314 (declared by the reference, defined nowhere in it) ----
int open_video_write(const char* filename, int width, int height, int rate, int method, int clevel)
{
    if (method != 1 && rirb_device_count() <= 0) {
        fail("open_video_write: methods 2 and 3 need a CUDA device");
        return 0;
    }
    const int z = rirb_z_open_file_write(filename, width, height, rate, method, clevel);
    if (!z) fail(std::string("open_video_write: ") + rirb_last_error());
    return z;
}
int image_write(int writter, unsigned short* img, int64_t time)
{
    long long t = time;
    return rirb_z_write_images(writter, img, 1, &t, 1);
}
int64_t close_video(int writter) { return rirb_z_close_file(writter); }

// =====================================================================================================================
// reader
// =====================================================================================================================

int open_camera_file(const char* filename, int* file_format)
{
    if (file_format) *file_format = 0;
    auto c = open_camera(filename);
    if (!c) return 0;
    if (file_format) *file_format = c->format;
    return g_cameras.add(c);
}
int video_file_format(const char* filename)
{
    auto c = open_camera(filename);
    return c ? c->format : -1;
}
int close_camera(int cam)
{
    if (!g_cameras.get(cam)) {
        fail("close_camera: NULL camera");
        return -1;
    }
    g_cameras.remove(cam);
    return 0;
}
int get_image_count(int cam)
{
    auto c = g_cameras.get(cam);
    if (!c) {
        fail("get_image_count: NULL camera");
        return -1;
    }
    return c->count;
}
int get_image_time(int cam, int pos, int64_t* time)
{
    auto c = g_cameras.get(cam);
    if (!c || !time) {
        fail("get_image_time: NULL camera");
        return -1;
    }
    if (pos < 0 || pos >= c->count) {
        fail("get_image_time: position out of range");
        return -1;
    }
    *time = c->times[(size_t)pos];
    return 0;
}
int get_image_size(int cam, int* width, int* height)
{
    auto c = g_cameras.get(cam);
    if (!c || !width || !height) {
        fail("get_image_size: NULL camera");
        return -1;
    }
    *width = c->w;
    *height = c->h;
    return 0;
}
int get_filename(int cam, char* filename)
{
    auto c = g_cameras.get(cam);
    if (!c || !filename) {
        fail("get_filename: NULL camera");
        return -1;
    }
    std::string f = c->filename;
    if (f.size() > RIRB_UNSPECIFIED_CHAR_LENGTH - 1) f = f.substr(0, RIRB_UNSPECIFIED_CHAR_LENGTH - 1);
    memset(filename, 0, RIRB_UNSPECIFIED_CHAR_LENGTH);
    memcpy(filename, f.data(), f.size());
    return 0;
}
int supported_calibrations(int cam, int* count)
{
    auto c = g_cameras.get(cam);
    if (!c || !count) {
        fail("support_calibration: NULL camera");
        return -1;
    }
    *count = 1;  // IRFileLoader::supportedCalibration without a calibration: "Digital Level" only (IRFileLoader.cpp:994-1003)
    return 0;
}
int calibration_name(int cam, int calibration, char* name)
{
    auto c = g_cameras.get(cam);
    if (!c || !name) {
        fail("support_calibration: NULL camera");
        return -1;
    }
    if (calibration != 0) {
        fail("calibration_name: calibration index out of range");
        return -1;
    }
    memcpy(name, "Digital Level", 13);
    return 0;
}
int load_image(int cam, int pos, int calibration, unsigned short* pixels)
{
    auto c = g_cameras.get(cam);
    if (!c || !pixels) {
        fail("load_image: NULL camera");
        return -1;
    }
    if (calibration != 0) {  // IRFileLoader::readImage without a calibration object returns false for calibration 1 (:1217-1218)
        fail("load_image: no calibration is attached to this file");
        return -1;
    }
    std::lock_guard<std::mutex> lock(c->mu);
    if (!c->read(pos, pixels, true)) return -1;
    c->last_pos = pos;
    return 0;
}
int enable_bad_pixels(int cam, int enable)
{
    auto c = g_cameras.get(cam);
    if (!c) {
        fail("enable_bad_pixels: NULL camera");
        return -1;
    }
    std::lock_guard<std::mutex> lock(c->mu);
    if (enable && !c->bp_handle && c->count > 0 && c->h > 3) {
        // setBadPixelsEnabled, IRFileLoader.cpp:693-716: detection on readImage(0) -- MIN_T added, motion applied if it is on,
        // bad pixels still off -- without its last 3 rows
        std::vector<unsigned short> first((size_t)c->w * c->h);
        if (!c->read(0, first.data(), false)) return -1;
        c->bp_handle = bad_pixels_create(first.data(), c->w, c->h - 3);
        if (c->bp_handle <= 0) {
            c->bp_handle = 0;
            fail(std::string("enable_bad_pixels: ") + rirb_last_error());
            return -1;
        }
    }
    c->bp_enabled = enable != 0;
    return 0;
}
int bad_pixels_enabled(int cam)
{
    auto c = g_cameras.get(cam);
    return c && c->bp_enabled ? 1 : 0;
}
int load_motion_correction_file(int cam, const char* filename)
{
    auto c = g_cameras.get(cam);
    if (!c || !filename) {
        fail("load_motion_correction_file: NULL camera");
        return -1;
    }
    // IRFileLoader::loadTranslationFile, IRFileLoader.cpp:822-847: one header line, then rows of 4 float columns
    std::ifstream in(filename);
    if (!in) {
        fail("unable to load file");
        return -1;
    }
    std::string line;
    std::getline(in, line);
    std::vector<double> sx, sy;
    while (std::getline(in, line)) {
        std::istringstream ls(line);
        float v[4];
        int n = 0;
        while (n < 4 && (ls >> v[n])) ++n;
        if (n == 0) continue;
        if (n != 4) {
            fail("error while loading motion correction file: 4 columns expected");
            return -1;
        }
        sx.push_back((double)v[1]);  // the reference parses floats (Array2D<float>)
        sy.push_back((double)v[2]);
    }
    if ((int)sx.size() != c->count) {
        fail("wrong number of images in motion correction file");
        return -1;
    }
    std::lock_guard<std::mutex> lock(c->mu);
    c->shift_x.swap(sx);
    c->shift_y.swap(sy);
    return 0;
}
int enable_motion_correction(int cam, int enable)
{
    auto c = g_cameras.get(cam);
    if (!c) {
        fail("enable_motion_correction: NULL camera");
        return -1;
    }
    c->motion_enabled = enable != 0;
    return 0;
}
int motion_correction_enabled(int cam)
{
    auto c = g_cameras.get(cam);
    return c && c->motion_enabled ? 1 : 0;
}
// ---- entries that belong to the camera CALIBRATION objects (video_io.cpp:259-360, 393-438, 464-493, 845-931).  The movies
//      this library opens carry none, so they answer what the reference answers for such a movie: emissivities are loader
//      state (IRVideoLoader.h:47-95), everything that needs a calibration says so. ----
int open_camera_from_memory(void* ptr, int64_t size, int* file_format)
{
    // video_io.cpp:110-145 reads the movie out of the caller's buffer; here the bytes go through a temporary file
    if (file_format) *file_format = 0;
    if (!ptr || size <= 0) {
        fail("open_camera_from_memory: empty buffer");
        return 0;
    }
    char name[] = "/tmp/rirb_movie_XXXXXX";
    const int fd = mkstemp(name);
    if (fd < 0) {
        fail("open_camera_from_memory: cannot create a temporary file");
        return 0;
    }
    FILE* f = fdopen(fd, "wb");
    const bool ok = f && fwrite(ptr, 1, (size_t)size, f) == (size_t)size;
    if (f) fclose(f);
    auto c = ok ? open_camera(name) : nullptr;
    if (!c) {
        remove(name);
        return 0;
    }
    c->temp_file = name;
    if (file_format) *file_format = c->format;
    return g_cameras.add(c);
}
int flip_camera_calibration(int camera, int, int) { return g_cameras.get(camera) ? -2 : -1; }  // -2: no calibration attached
int set_global_emissivity(int cam, float emi)
{
    auto c = g_cameras.get(cam);
    if (emi < 0.f || emi > 1.f || !c) {
        fail(c ? "set_emissivity: wrong emissivity value" : "set_global_emissivity: NULL camera");
        return -1;
    }
    c->inv_emissivity.assign((size_t)c->w * c->h, 1.f / emi);
    return 0;
}
int set_emissivity(int cam, float* emi, int size)
{
    auto c = g_cameras.get(cam);
    if (!c || !emi || size <= 0) {
        fail(c ? "set_emissivity: wrong vector size" : "set_emissivity: NULL camera");
        return -1;
    }
    c->inv_emissivity.assign((size_t)c->w * c->h, 1.f);
    const size_t n = std::min((size_t)size, c->inv_emissivity.size());
    for (size_t i = 0; i < n; ++i) c->inv_emissivity[i] = 1.f / emi[i];
    return 0;
}
int get_emissivity(int cam, float* emi, int size)
{
    auto c = g_cameras.get(cam);
    if (!c || !emi) {
        fail("get_emissivity: NULL camera");
        return -1;
    }
    const int s = std::min(size, (int)c->inv_emissivity.size());
    for (int i = 0; i < s; ++i) emi[i] = 1.f / c->inv_emissivity[(size_t)i];
    if (s == 0) *emi = 1;
    return s;
}
int support_emissivity(int cam)
{
    (void)cam;
    fail("support_emissivity: NULL camera");  // the reference's message when the loader has no calibration
    return -1;
}
int camera_saturate(int cam) { return g_cameras.get(cam) ? 0 : -1; }
int calibration_files(int, char*, int*) { return -1; }
// IRFileLoader::calibrate / calibrateInplace, IRFileLoader.cpp:1060-1097: calibration 0 (digital levels) succeeds and touches
// nothing; calibration 1 needs the calibration object
int calibrate_inplace(int cam, unsigned short*, int, int calibration) { return (g_cameras.get(cam) && calibration == 0) ? 0 : -1; }
int calibrate_image(int cam, unsigned short*, float*, int, int calib) { return (g_cameras.get(cam) && calib == 0) ? 0 : -1; }
int calibrate_image_inplace(int cam, unsigned short*, int, int calib) { return (g_cameras.get(cam) && calib == 0) ? 0 : -1; }
int get_table_names(int, char*, int*) { return -1; }
int get_table(int, const char*, float*, int*) { return -1; }
// video_io.cpp:911-930: only a file the reader canNOT open is touched; it gets a PCR header for the given geometry
int correct_PCR_file(const char* filename, int width, int height, int freq)
{
    if (!filename || open_camera(filename)) return -1;
    FILE* f = fopen(filename, "r+b");
    if (!f) return -1;
    PcrHeader h;
    memset(&h, 0, sizeof(h));
    if (fread(&h, 1, sizeof(h), f) != sizeof(h)) memset(&h, 0, sizeof(h));
    h.x = h.grab_x = width;
    h.y = h.grab_y = height;
    h.bits = 16;
    h.version = 0;
    h.transfer_size = width * height * 2;
    h.frequency = freq;
    fseeko(f, 0, SEEK_SET);
    fwrite(&h, 1, sizeof(h), f);
    fclose(f);
    return 0;
}

int get_attribute_count(int cam)
{
    auto c = g_cameras.get(cam);
    if (!c) {
        fail("get_attribute_count: NULL camera");
        return -1;
    }
    std::lock_guard<std::mutex> lock(c->mu);
    const int pos = c->last_pos < 0 ? 0 : c->last_pos;  // attributes of the image read last (H264_Loader::extractAttributes)
    return pos < (int)c->frame_attrs.size() ? (int)c->frame_attrs[(size_t)pos].size() : 0;
}
int get_attribute(int cam, int index, char* key, int* key_len, char* value, int* value_len)
{
    auto c = g_cameras.get(cam);
    if (!c) {
        fail("get_attribute: NULL camera");
        return -1;
    }
    std::lock_guard<std::mutex> lock(c->mu);
    const int pos = c->last_pos < 0 ? 0 : c->last_pos;
    if (pos >= (int)c->frame_attrs.size()) return -1;
    return copy_attr(c->frame_attrs[(size_t)pos], index, key, key_len, value, value_len, false);
}
int get_global_attribute_count(int cam)
{
    auto c = g_cameras.get(cam);
    if (!c) {
        fail("get_global_attribute_count: NULL camera");
        return -1;
    }
    return (int)c->global.size();
}
int get_global_attribute(int cam, int index, char* key, int* key_len, char* value, int* value_len)
{
    auto c = g_cameras.get(cam);
    if (!c) {
        fail("get_global_attribute: NULL camera");
        return -1;
    }
    return copy_attr(c->global, index, key, key_len, value, value_len, true);
}

}  // extern "C"
