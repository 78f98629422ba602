/*
 * oracle/oracle.c -- TEST INFRASTRUCTURE, NOT PRODUCT CODE.
 *
 * A plain-C, single-threaded CPU restatement of the librir (v6.1.2) algorithms on the
 * per-frame hot path (SURVEY.md section 8a).  It exists so that the CUDA path can be
 * checked against something that runs on the GPU box, where /root/reference is absent.
 * Only tests/, __graft_entry__.smoke() and bench.py's cpu_baseline / --impl reference legs
 * may load it; librir_b200 itself never does (no CPU fallback exists in the product).
 *
 * Pinning: every function here is compared, on seeded inputs, against the reference's own
 * sources compiled by oracle/build_ref.sh (oracle/_ref/libs/libsignal_processing.so) in
 * tests/test_oracle_vs_ref.py, and against the golden vectors that build produced
 * (tests/golden/, generator tests/golden/make_golden.py).  The byte-plane split/merge
 * (video_io) cannot be compiled here (needs ffmpeg/x264); it is pinned by the reference
 * code it restates (h264.cpp:1066-1103, 3016-3051) and by the round-trip identity the
 * reference's tests assert (tests/python/test_IRMovie.py:46-49).  The temporal delta stage
 * has no counterpart in the reference: PARITY UNPINNED, defined by this repo (DESIGN.md).
 *
 * Compile: gcc -O2 -ffp-contract=off -fPIC -shared oracle.c -lm   (no -march, no
 * -ffast-math: the reference's stock build has no FMA contraction, SURVEY.md 8c).
 */
#include <math.h>
#include <stdint.h>
#include <stdlib.h>
#include <string.h>

#define ORC_API __attribute__((visibility("default")))

typedef unsigned short u16;

/* ------------------------------------------------------------------------------------ */
/* helpers                                                                              */
/* ------------------------------------------------------------------------------------ */

static int cmp_u16(const void *a, const void *b)
{
    u16 x = *(const u16 *)a, y = *(const u16 *)b;
    return (x > y) - (x < y);
}

/* k-th smallest (0-based) of n<=25 values; any exact selection equals std::nth_element /
 * std::sort element k. */
static u16 kth_smallest(u16 *v, int n, int k)
{
    for (int i = 1; i < n; ++i) {
        u16 key = v[i];
        int j = i - 1;
        while (j >= 0 && v[j] > key) {
            v[j + 1] = v[j];
            --j;
        }
        v[j + 1] = key;
    }
    return v[k];
}

/* Frame median (upper median, sorted[N/2]) and the spread around it as the reference
 * computes them: Filters.h:145-156 and BadPixels.cpp:19-30.  The squared difference is an
 * int product there: for |p - median| >= 46341 -- a saturated pixel at 65535 over an 8000-count
 * background is enough -- it overflows, which is undefined in C++ and wraps modulo 2^32 in the
 * reference as every x86-64 compiler builds it (checked against oracle/_ref).  Real movies have such
 * pixels, so the wrap is part of the behaviour to reproduce; it is written out with unsigned
 * arithmetic here so that this file itself has no undefined behaviour. */
/* (unsigned short)(double) as x86-64 evaluates it (cvttsd2si to a 32-bit int, low 16 bits kept; NaN and
 * values beyond int range give the "integer indefinite" 0x80000000, whose low half is 0): defined for the
 * in-range values real frames produce, and spelled out for the rest instead of left undefined. */
static u16 orc_trunc_u16(double v)
{
    if (!(v > -2147483649.0 && v < 2147483648.0))
        return 0;
    return (u16)(unsigned)(int)v;
}
/* median - (int)(2 * std) with the same conversion rule; a NaN spread (negative wrapped sum) makes the
 * reference's result negative in practice, i.e. "no clamp". */
static int orc_clamp_value(int median, double gstd)
{
    double v = gstd * 2;
    if (!(v > -2147483649.0 && v < 2147483648.0))
        return -1;
    return median - (int)v;
}
/* The lossy pre-conditioner's two constructs of the same class (h264.cpp:1993-2036 and :2367-2368 / :2559-2563), as
 * g++ -O3 builds them for x86-64 (pinned by tests/test_lossy_extremes.py, which compiles the reference's statements):
 * `diff * diff` on int wraps modulo 2^32 for |diff| >= 46341, and `lowError -= (int)round(x)` converts with cvttsd2si --
 * the "integer indefinite" INT_MIN for NaN (an empty background / foreground split) and for values beyond int range --
 * and then subtracts modulo 2^32. */
static int orc_wrapped_square(int diff)
{
    return (int)(uint32_t)((unsigned)diff * (unsigned)diff);
}
static int orc_round_to_int(double x)
{
    double r = round(x);
    if (!(r >= -2147483648.0 && r <= 2147483647.0))
        return INT32_MIN;
    return (int)r;
}
static int orc_wrapping_sub(int a, int b)
{
    return (int)((unsigned)a - (unsigned)b);
}

static void frame_median_std(const u16 *img, size_t n, int *median, double *std_out)
{
    u16 *tmp = (u16 *)malloc(n * sizeof(u16));
    memcpy(tmp, img, n * sizeof(u16));
    qsort(tmp, n, sizeof(u16), cmp_u16);
    int m = tmp[n / 2];
    double sum = 0;
    for (size_t i = 0; i < n; ++i) {
        int d = (int)tmp[i] - m;
        sum += (double)(int)((unsigned)d * (unsigned)d);
    }
    free(tmp);
    sum /= (double)(int)n;
    *median = m;
    *std_out = sqrt(sum);
}

/* ------------------------------------------------------------------------------------ */
/* a-1  bad-pixel detection    Filters.h:135-193, BadPixels.cpp:13-32                    */
/* ------------------------------------------------------------------------------------ */

/* Writes up to cap (x,y) pairs in raster order into xy[2*i], xy[2*i+1]; returns the number
 * of bad pixels found (may exceed cap: call again with a larger buffer).  *global_thr gets
 * the "p < median - 5*std" threshold (Filters.h:157-160). */
ORC_API int orc_bad_pixels_detect(const u16 *img, int w, int h, double std_factor,
                                  int *xy, int cap, int *global_thr)
{
    size_t n = (size_t)w * (size_t)h;
    int median;
    double gstd;
    frame_median_std(img, n, &median, &gstd);
    u16 cut = orc_trunc_u16(gstd * std_factor); /* (T)(double): truncation, Filters.h:157 */
    u16 gthr = ((u16)median > cut) ? (u16)(median - cut) : 0;
    if (global_thr)
        *global_thr = gthr;

    int count = 0;
    u16 win[25];
    for (long y = 0; y < h; ++y)
        for (long x = 0; x < w; ++x) {
            int m = 0;
            for (long yy = y - 2; yy <= y + 2; ++yy)
                for (long xx = x - 2; xx <= x + 2; ++xx)
                    if (xx >= 0 && yy >= 0 && xx < w && yy < h)
                        win[m++] = img[xx + yy * w];
            kth_smallest(win, m, 0); /* full insertion sort */
            long med = win[m / 2];
            double sum2 = 0;
            long c = 0;
            for (long i = m / 5; i < m * 4 / 5; ++i, ++c) {
                long d = (long)win[i] - med;
                sum2 += (double)(d * d);
            }
            sum2 /= (double)c;
            double sd = sqrt(sum2);
            double lower = (double)med - std_factor * sd;
            double upper = (double)med + std_factor * sd;
            u16 p = img[x + y * w];
            if ((double)p < lower || (double)p > upper || p < gthr) {
                if (count < cap && xy) {
                    xy[2 * count] = (int)x;
                    xy[2 * count + 1] = (int)y;
                }
                ++count;
            }
        }
    return count;
}

/* Clamp level "median - (int)(2*std)" kept by BadPixels::init (BadPixels.cpp:19-31). */
ORC_API int orc_bad_pixels_clamp_value(const u16 *img, int w, int h)
{
    int median;
    double gstd;
    frame_median_std(img, (size_t)w * (size_t)h, &median, &gstd);
    return orc_clamp_value(median, gstd);
}

/* ------------------------------------------------------------------------------------ */
/* a-2  bad-pixel correction   BadPixels.cpp:34-66, Filters.cpp:43-49                    */
/* ------------------------------------------------------------------------------------ */

ORC_API void orc_bad_pixels_correct(const u16 *in, u16 *out, int w, int h, const int *xy,
                                    int count, int clamp_value)
{
    size_t n = (size_t)w * (size_t)h;
    if (in != out)
        memcpy(out, in, n * sizeof(u16));
    for (int i = 0; i < count; ++i) {
        int x = xy[2 * i], y = xy[2 * i + 1];
        u16 v[9];
        int c = 0;
        for (int xx = x - 1; xx <= x + 1; ++xx)     /* column-major gather, from `in` */
            for (int yy = y - 1; yy <= y + 1; ++yy)
                if (xx >= 0 && yy >= 0 && xx < w && yy < h)
                    v[c++] = in[xx + yy * w];
        out[x + y * w] = kth_smallest(v, c, c / 2);
    }
    if (clamp_value > 0) {
        u16 lo = (u16)clamp_value;
        for (size_t i = 0; i < n; ++i)
            if (out[i] < lo)
                out[i] = lo;
    }
}

/* ------------------------------------------------------------------------------------ */
/* a-3  loader variant         IRFileLoader.cpp:722-802                                  */
/* ------------------------------------------------------------------------------------ */

/* In place on rows [0,h) (callers pass height-3).  3x3 window shifted inside the image,
 * cells flagged bad are skipped, no clamp.  When every cell of the window is bad the
 * reference reads a stale stack slot (undefined); this restatement leaves the pixel as is. */
ORC_API void orc_loader_remove_bad_pixels(u16 *img, int w, int h, const int *xy, int count)
{
    if (w < 3 || h < 3) {
        for (int i = 0; i < count; ++i) { /* sequential, in place: IRFileLoader.cpp:735-752 */
            int x = xy[2 * i], y = xy[2 * i + 1];
            u16 v[9];
            int c = 0;
            for (int xx = x - 1; xx <= x + 1; ++xx)
                for (int yy = y - 1; yy <= y + 1; ++yy)
                    if (xx >= 0 && yy >= 0 && xx < w && yy < h)
                        v[c++] = img[xx + yy * w];
            if (c)
                img[x + y * w] = kth_smallest(v, c, c / 2);
        }
        return;
    }
    unsigned char *bad = (unsigned char *)calloc((size_t)w * (size_t)h, 1);
    for (int i = 0; i < count; ++i)
        bad[xy[2 * i] + xy[2 * i + 1] * w] = 1;
    for (int i = 0; i < count; ++i) {
        int x = xy[2 * i], y = xy[2 * i + 1];
        int x0 = x - 1, y0 = y - 1;
        if (x == 0) x0 = 0; else if (x == w - 1) x0 = w - 3;
        if (y == 0) y0 = 0; else if (y == h - 1) y0 = h - 3;
        u16 v[9];
        int c = 0;
        for (int xx = x0; xx <= x0 + 2; ++xx)
            for (int yy = y0; yy <= y0 + 2; ++yy)
                if (!bad[xx + yy * w])
                    v[c++] = img[xx + yy * w];
        if (c)
            img[x + y * w] = kth_smallest(v, c, c / 2);
    }
    free(bad);
}

/* ------------------------------------------------------------------------------------ */
/* a-4  gaussian filter        signal_processing.cpp:79-148                              */
/* ------------------------------------------------------------------------------------ */

ORC_API int orc_gaussian_radius(float sigma)
{
    int r = (int)(sigma * 2);
    return r < 1 ? 1 : r;
}

/* (2r+1)^2 float taps, index [dx+r + (dy+r)*kw]; signal_processing.cpp:79-99 */
ORC_API void orc_gaussian_kernel(float sigma, int r, float *k)
{
    float s = 2.0f * sigma * sigma;
    float sum = 0.0f;
    int kw = 2 * r + 1;
    for (int x = -r; x <= r; ++x)
        for (int y = -r; y <= r; ++y) {
            float rho = (float)sqrt((double)(x * x + y * y));
            float e = expf(-(rho * rho) / s);             /* std::exp(float) */
            float t = (float)((double)e / (3.14159265358979323846 * (double)s));
            k[x + r + (y + r) * kw] = t;
            sum += t;
        }
    for (int i = 0; i < kw * kw; ++i)
        k[i] /= sum;
}

ORC_API int orc_gaussian_filter(const float *src, float *dst, int w, int h, float sigma)
{
    int r = orc_gaussian_radius(sigma);
    int kw = 2 * r + 1;
    float *k = (float *)malloc(sizeof(float) * (size_t)kw * (size_t)kw);
    orc_gaussian_kernel(sigma, r, k);
    for (int y = 0; y < h; ++y)
        for (int x = 0; x < w; ++x) {
            int interior = x >= r && x < w - r && y >= r && y < h - r;
            float acc = 0, ksum = 0;
            for (int dx = -r; dx <= r; ++dx)
                for (int dy = -r; dy <= r; ++dy) {
                    int xx = x + dx, yy = y + dy;
                    if (interior || (xx >= 0 && xx < w && yy >= 0 && yy < h)) {
                        float t = k[dx + r + (dy + r) * kw];
                        ksum += t;
                        acc += t * src[xx + yy * w];
                    }
                }
            dst[x + y * w] = interior ? acc : acc / ksum;
        }
    free(k);
    return 0;
}

/* ------------------------------------------------------------------------------------ */
/* a-5  translate              Filters.h:249-326, signal_processing.cpp:14-73            */
/* ------------------------------------------------------------------------------------ */

enum { ORC_NOBORDER = 0, ORC_BACKGROUND = 1, ORC_WRAP = 2, ORC_NEAREST = 3 };

/* (size_t)float as x86-64 evaluates it for the value range seen here: truncate toward zero
 * as a signed 64-bit integer, then reinterpret (SURVEY.md appendix A.4). */
static inline uint64_t f2size(float v) { return (uint64_t)(int64_t)v; }
static inline uint64_t wrap_idx(uint64_t v, uint64_t n) { return (v + n) % n; }

/* One generic body; T = storage type, U = destination type, TODBL converts a pixel to the
 * double it is promoted to in the blend, CAST is detail::cast<U> (Filters.h:232-235). */
#define ORC_FLAT(i) ((i) < w * h ? (i) : w * h - 1)
#define ORC_DEFINE_TRANSLATE(NAME, T, U, CAST)                                                 \
    static void NAME(const T *src, U *dst, U background, size_t w, size_t h, float dx,        \
                     float dy, int strategy)                                                   \
    {                                                                                          \
        for (size_t y = 0; y < h; ++y)                                                         \
            for (size_t x = 0; x < w; ++x) {                                                   \
                float px = (float)x - dx;                                                      \
                float py = (float)y - dy;                                                      \
                size_t l, rt, t, b;                                                            \
                double u, v;                                                                   \
                if (px < 0 || px >= (float)w || py < 0 || py >= (float)h) {                    \
                    if (strategy == ORC_NOBORDER)                                              \
                        continue;                                                              \
                    if (strategy == ORC_BACKGROUND) {                                          \
                        dst[x + y * w] = background;                                           \
                        continue;                                                              \
                    }                                                                          \
                    if (strategy == ORC_NEAREST) {                                             \
                        size_t sx = px < 0 ? 0 : (px >= (float)w ? w - 1 : (size_t)px);        \
                        size_t sy = py < 0 ? 0 : (py >= (float)h ? h - 1 : (size_t)py);        \
                        dst[x + y * w] = (U)src[sx + sy * w];                                  \
                        continue;                                                              \
                    }                                                                          \
                    l = wrap_idx(f2size(px), w);                                               \
                    rt = wrap_idx(f2size(px + 1), w);                                          \
                    t = wrap_idx(f2size(py), h);                                               \
                    b = wrap_idx(f2size(py + 1), h);                                           \
                    u = (double)fabsf(px - (float)(int)px);                                    \
                    v = (double)fabsf(py - (float)(int)py);                                    \
                } else {                                                                       \
                    l = (size_t)px;                                                            \
                    rt = (size_t)(px + 1);                                                     \
                    if (rt == w) rt = l;                                                       \
                    t = (size_t)py;                                                            \
                    b = (size_t)(py + 1);                                                      \
                    if (b == h) b = t;                                                         \
                    u = (double)(px - (float)l);                                               \
                    v = (double)((float)b - py);                                               \
                }                                                                              \
                /* px (py) within half a float ulp below w (h): px + 1 rounds up to w + 1, the clamp above does   \
                 * not fire and the reference reads into the next row -- or past the buffer on the last row(s),  \
                 * which is undefined; there this restatement (and the CUDA path) reads the last pixel. */         \
                double p1 = (double)src[ORC_FLAT(b * w + l)], p2 = (double)src[ORC_FLAT(t * w + l)];               \
                double p3 = (double)src[ORC_FLAT(b * w + rt)], p4 = (double)src[ORC_FLAT(t * w + rt)];             \
                double val = (p1 * (1 - v) + p2 * v) * (1 - u) + (p3 * (1 - v) + p4 * v) * u;  \
                dst[x + y * w] = CAST(val);                                                    \
            }                                                                                  \
    }

#define CAST_BOOL(v) ((unsigned char)((v) != 0))
ORC_DEFINE_TRANSLATE(tr_bool, unsigned char, unsigned char, CAST_BOOL)
ORC_DEFINE_TRANSLATE(tr_i8, signed char, signed char, (signed char))
ORC_DEFINE_TRANSLATE(tr_u8, unsigned char, unsigned char, (unsigned char))
ORC_DEFINE_TRANSLATE(tr_i16, short, short, (short))
ORC_DEFINE_TRANSLATE(tr_u16, u16, u16, (u16))
ORC_DEFINE_TRANSLATE(tr_i32, int, int, (int))
ORC_DEFINE_TRANSLATE(tr_u32, unsigned int, unsigned int, (unsigned int))
ORC_DEFINE_TRANSLATE(tr_i64, long long, long long, (long long))
ORC_DEFINE_TRANSLATE(tr_u64, unsigned long long, unsigned long long, (unsigned long long))
ORC_DEFINE_TRANSLATE(tr_f32, float, float, (float))
ORC_DEFINE_TRANSLATE(tr_f64, double, double, (double))
ORC_DEFINE_TRANSLATE(tr_u16_f32, u16, float, (float))

static int strategy_code(const char *s)
{
    if (!s || !*s || strcmp(s, "noborder") == 0) return ORC_NOBORDER;
    if (strcmp(s, "background") == 0) return ORC_BACKGROUND;
    if (strcmp(s, "wrap") == 0) return ORC_WRAP;
    if (strcmp(s, "nearest") == 0) return ORC_NEAREST;
    return -1;
}

/* Same signature and return codes as the C facade (signal_processing.cpp:44-73). */
ORC_API int orc_translate(int type, const void *src, void *dst, int w, int h, float dx, float dy,
                          const void *background, const char *strategy)
{
    int st = strategy_code(strategy);
    size_t W = (size_t)w, H = (size_t)h;
#define ORC_CASE(CH, FN, T)                                                                    \
    case CH:                                                                                   \
        if (st < 0) return -1;                                                                 \
        FN((const T *)src, (T *)dst, *(const T *)background, W, H, dx, dy, st);                \
        return 0;
    switch (type) {
        ORC_CASE('?', tr_bool, unsigned char)
        ORC_CASE('b', tr_i8, signed char)
        ORC_CASE('B', tr_u8, unsigned char)
        ORC_CASE('h', tr_i16, short)
        ORC_CASE('H', tr_u16, u16)
        ORC_CASE('i', tr_i32, int)
        ORC_CASE('I', tr_u32, unsigned int)
        ORC_CASE('l', tr_i64, long long)
        ORC_CASE('L', tr_u64, unsigned long long)
        ORC_CASE('f', tr_f32, float)
        ORC_CASE('d', tr_f64, double)
    default:
        return -1;
    }
}

/* ------------------------------------------------------------------------------------ */
/* a-6  motion-correction variant   IRFileLoader.cpp:617-627                             */
/* ------------------------------------------------------------------------------------ */

/* In place on rows [0,h) (callers pass height-3): u16 -> float translate by
 * (-shift_x, -shift_y), nearest border, then float -> u16 truncation. */
ORC_API void orc_loader_remove_motion(u16 *img, int w, int h, double shift_x, double shift_y)
{
    size_t n = (size_t)w * (size_t)h;
    float *tmp = (float *)malloc(n * sizeof(float));
    tr_u16_f32(img, tmp, 0.f, (size_t)w, (size_t)h, (float)(-shift_x), (float)(-shift_y), ORC_NEAREST);
    for (size_t i = 0; i < n; ++i)
        img[i] = (u16)tmp[i];
    free(tmp);
}

/* ------------------------------------------------------------------------------------ */
/* a-7  lossless-writer pre-coder   h264.cpp:1050-1103 (split), 3016-3051 (merge)        */
/* ------------------------------------------------------------------------------------ */

/* YUV444P layout: Y = 0 (or the 8-bit integration-time image), U = low bytes, V = high
 * bytes, each plane [h][linesize]; padding bytes of a row are left untouched. */
ORC_API void orc_split_444(const u16 *img, const unsigned char *it, int w, int h,
                           unsigned char *y_plane, unsigned char *u_plane, unsigned char *v_plane,
                           int ls_y, int ls_u, int ls_v)
{
    for (int r = 0; r < h; ++r)
        for (int i = 0; i < w; ++i) {
            u16 p = img[i + r * w];
            u_plane[i + (size_t)r * ls_u] = (unsigned char)(p & 0xFF);
            v_plane[i + (size_t)r * ls_v] = (unsigned char)(p >> 8);
            y_plane[i + (size_t)r * ls_y] = it ? it[i + r * w] : 0;
        }
}

ORC_API void orc_merge_444(const unsigned char *y_plane, const unsigned char *u_plane,
                           const unsigned char *v_plane, int ls_y, int ls_u, int ls_v, int w,
                           int h, u16 *img, unsigned char *it)
{
    for (int r = 0; r < h; ++r)
        for (int i = 0; i < w; ++i) {
            img[i + r * w] = (u16)(u_plane[i + (size_t)r * ls_u] | (v_plane[i + (size_t)r * ls_v] << 8));
            if (it)
                it[i + r * w] = y_plane[i + (size_t)r * ls_y];
        }
}

/* YUV420P layout (kvazaar/vp8 path): luma plane of 2h rows, rows [0,h) = low bytes, rows
 * [h,2h) = high bytes: a type-size-2 byte shuffle of the frame (h264.cpp:1089-1102). */
ORC_API void orc_split_420(const u16 *img, int w, int h, unsigned char *y_plane, int ls_y)
{
    for (int r = 0; r < h; ++r)
        for (int i = 0; i < w; ++i) {
            u16 p = img[i + r * w];
            y_plane[i + (size_t)r * ls_y] = (unsigned char)(p & 0xFF);
            y_plane[i + (size_t)(h + r) * ls_y] = (unsigned char)(p >> 8);
        }
}

ORC_API void orc_merge_420(const unsigned char *y_plane, int ls_y, int w, int h, u16 *img)
{
    for (int r = 0; r < h; ++r)
        for (int i = 0; i < w; ++i)
            img[i + r * w] = (u16)(y_plane[i + (size_t)r * ls_y] | (y_plane[i + (size_t)(h + r) * ls_y] << 8));
}

/* Key-frame rule of AddFrame (h264.cpp:1050-1061): frame n is a key frame iff n == 0 or
 * n - last_key >= gop.  Fills key[0..nframes) with 0/1 for a writer that starts at n = 0. */
ORC_API void orc_key_frames(int nframes, int gop, unsigned char *key)
{
    int last = 0;
    for (int n = 0; n < nframes; ++n) {
        int k = (n == 0) || (n - last >= gop);
        if (k)
            last = n;
        key[n] = (unsigned char)k;
    }
}

/* Movie-level pre-coder, dense planes: lo[t][h][w], hi[t][h][w].  delta == 0 is exactly the
 * reference's split.  delta != 0 (THIS REPO'S DEFINITION, parity unpinned): a non-key frame
 * is replaced by (frame[t] - frame[t-1]) mod 2^16 before the split; key frames (rule above)
 * are stored raw. */
ORC_API void orc_precode_movie(const u16 *mov, int nframes, int w, int h, int gop, int delta,
                               unsigned char *lo, unsigned char *hi)
{
    size_t n = (size_t)w * (size_t)h;
    unsigned char *key = (unsigned char *)malloc((size_t)nframes + 1);
    orc_key_frames(nframes, gop, key);
    for (int t = 0; t < nframes; ++t) {
        const u16 *cur = mov + (size_t)t * n;
        const u16 *prev = cur - n;
        int use_delta = delta && !key[t];
        for (size_t i = 0; i < n; ++i) {
            u16 p = use_delta ? (u16)(cur[i] - prev[i]) : cur[i];
            lo[(size_t)t * n + i] = (unsigned char)(p & 0xFF);
            hi[(size_t)t * n + i] = (unsigned char)(p >> 8);
        }
    }
    free(key);
}

ORC_API void orc_decode_movie(const unsigned char *lo, const unsigned char *hi, int nframes, int w,
                              int h, int gop, int delta, u16 *mov)
{
    size_t n = (size_t)w * (size_t)h;
    unsigned char *key = (unsigned char *)malloc((size_t)nframes + 1);
    orc_key_frames(nframes, gop, key);
    for (int t = 0; t < nframes; ++t) {
        u16 *cur = mov + (size_t)t * n;
        const u16 *prev = cur - n;
        int use_delta = delta && !key[t];
        for (size_t i = 0; i < n; ++i) {
            u16 p = (u16)(lo[(size_t)t * n + i] | (hi[(size_t)t * n + i] << 8));
            cur[i] = use_delta ? (u16)(p + prev[i]) : p;
        }
    }
    free(key);
}

/* ------------------------------------------------------------------------------------ */
/* a-8  statistics    Filters.cpp:56-101, h264.cpp:1955-1991, 2093-2097                  */
/* ------------------------------------------------------------------------------------ */

/* 65,535 bins in the reference (value 65535 is out of bounds there); inputs must stay
 * below 65535.  s = round(size*percent) is evaluated in float (size_t * float). */
ORC_API int orc_find_median_pixel(const u16 *p, int size, float percent)
{
    size_t *hist = (size_t *)calloc(65536, sizeof(size_t));
    size_t n = (size_t)size;
    for (size_t i = 0; i < n; ++i)
        hist[p[i]]++;
    size_t s = (size_t)roundf((float)n * percent);
    size_t c = 0;
    int res = 0;
    for (int i = 0; i < 65535; ++i) {
        c += hist[i];
        if (c >= s) {
            res = i;
            break;
        }
    }
    free(hist);
    return res;
}

ORC_API int orc_find_median_pixel_mask(const u16 *p, const unsigned char *mask, int size, float percent)
{
    size_t *hist = (size_t *)calloc(65536, sizeof(size_t));
    size_t n = (size_t)size, cnt = 0;
    for (size_t i = 0; i < n; ++i)
        if (mask[i]) {
            hist[p[i]]++;
            ++cnt;
        }
    size_t s = (size_t)(int)roundf((float)cnt * percent);
    size_t c = 0;
    int res = 0;
    for (int i = 0; i < 65535; ++i) {
        c += hist[i];
        if (c >= s) {
            res = i;
            break;
        }
    }
    free(hist);
    return res;
}

/* Mode of the 16,384-bin histogram of p>>2, first maximum wins -> (bin<<2)+1. */
ORC_API unsigned orc_get_background(const u16 *p, int size)
{
    unsigned *hist = (unsigned *)calloc(16384, sizeof(unsigned));
    for (int i = 0; i < size; ++i)
        hist[p[i] >> 2]++;
    unsigned best = hist[0], idx = 0;
    for (unsigned i = 1; i < 16384; ++i)
        if (hist[i] > best) {
            best = hist[i];
            idx = i;
        }
    free(hist);
    return (idx << 2) + 1;
}

/* Movie statistics that the multi-GPU path all-reduces: min, max, 65,536-bin histogram. */
ORC_API void orc_movie_stats(const u16 *p, size_t n, unsigned *minv, unsigned *maxv,
                             unsigned long long *hist65536)
{
    unsigned lo = 65535, hi = 0;
    if (hist65536)
        memset(hist65536, 0, 65536 * sizeof(unsigned long long));
    for (size_t i = 0; i < n; ++i) {
        unsigned v = p[i];
        if (v < lo) lo = v;
        if (v > hi) hi = v;
        if (hist65536)
            hist65536[v]++;
    }
    *minv = lo;
    *maxv = hi;
}

/* Quantile from an (all-reduced) histogram, same rule as orc_find_median_pixel. */
ORC_API int orc_quantile_from_hist(const unsigned long long *hist65536, unsigned long long total, float percent)
{
    size_t s = (size_t)roundf((float)(size_t)total * percent);
    size_t c = 0;
    for (int i = 0; i < 65535; ++i) {
        c += (size_t)hist65536[i];
        if (c >= s)
            return i;
    }
    return 0;
}

/* ------------------------------------------------------------------------------------ */
/* f-2  lossy "bounded-error" pre-conditioner of the H.264 saver                         */
/*      H264_Saver::addImageLossyNoCamera  h264.cpp:2253-2424                           */
/*      RunningAverage2 h264.cpp:1526-1615, get_background :1955-1991, stdDev :1993-2036 */
/*      and H264_Saver::addLoss :2426-2607 (variant 1).                                   */
/*      PINNED BY EXECUTION (round 2): oracle/build_ref.sh builds the reference's video_io */
/*      against oracle/libav_stub.c; tests/test_oracle_vs_refvio.py and the goldens made   */
/*      by tests/golden/make_vio_golden.py compare frame by frame.                         */
/* ------------------------------------------------------------------------------------ */
typedef struct {
    int w, h, stop_h;           /* stop_h = stop_lossy_height: rows [0, stop_h) are lossy */
    int low_error, high_error;  /* lowValueError (6) / highValueError (2), PrivateData() :1663 */
    double std_factor;          /* 5 */
    int running_average;        /* 32; 0 = off */
    int subtract_min;
    int bp_enabled;
    int variant;                /* 0 = addImageLossyNoCamera (h264.cpp:2253-2424), 1 = addLoss (:2426-2607) */
    int memcpy_quirk;           /* 1 (default) = the compiled reference's overlapping-memcpy outcome, see orc_lossy_add_image */
    int exact_squares;          /* 0 (default) = the reference's wrapping int product; 1 = exact squares (what it does not do) */
    int saturating_round;       /* 0 (default) = x86's conversion; 1 = a saturating one with NaN -> 0 (what it does not do) */
    /* state */
    long frames;                /* m_data->attributes.size() */
    unsigned short minv;
    u16 *lastDL, *refT, *prevT, *tmp, *tmpT;
    int *bp_xy; int bp_count; int bp_clamp;
    double first_std[2]; int have_first;
    double stds[40][2]; int nstds;
    /* RunningAverage2 */
    u16 *ring; int ring_len;    /* images: ring[k*len + i], oldest first (kept compact, like the vector) */
    unsigned *sums; u16 *cvalue; short *ccount;
} orc_lossy;

ORC_API orc_lossy *orc_lossy_open(int w, int h, int stop_h, int low_error, int high_error, double std_factor, int running_average,
                                  int subtract_min, int bp_enabled)
{
    orc_lossy *s = (orc_lossy *)calloc(1, sizeof(orc_lossy));
    size_t n = (size_t)w * (size_t)h, ns = (size_t)w * (size_t)stop_h;
    s->w = w; s->h = h; s->stop_h = stop_h;
    s->low_error = low_error; s->high_error = high_error; s->std_factor = std_factor;
    if (running_average > 64) running_average = 64; /* setParameter :1774 */
    s->running_average = running_average; s->subtract_min = subtract_min; s->bp_enabled = bp_enabled;
    s->lastDL = (u16 *)calloc(n, 2); s->refT = (u16 *)calloc(n, 2); s->prevT = (u16 *)calloc(n, 2);
    s->tmp = (u16 *)calloc(n, 2); s->tmpT = (u16 *)calloc(n, 2);
    s->ring = (u16 *)calloc(ns * (size_t)(running_average > 0 ? running_average : 1), 2);
    s->sums = (unsigned *)calloc(ns ? ns : 1, 4); s->cvalue = (u16 *)calloc(ns ? ns : 1, 2); s->ccount = (short *)calloc(ns ? ns : 1, 2);
    s->bp_xy = (int *)malloc(sizeof(int) * 2 * (ns ? ns : 1));
    s->memcpy_quirk = 1;
    return s;
}
/* variant: 0 = h264_add_image_lossy's path, 1 = h264_add_loss's; memcpy_quirk: see orc_lossy_add_image */
ORC_API void orc_lossy_configure(orc_lossy *s, int variant, int memcpy_quirk)
{
    s->variant = variant;
    s->memcpy_quirk = memcpy_quirk;
}
/* Counterfactual arithmetic, for tests that show the reference's own makes a difference (like memcpy_quirk = 0):
 * exact_squares = 1 adds exact squares in stdDev, saturating_round = 1 converts with saturation and NaN -> 0 in the
 * bound update. */
ORC_API void orc_lossy_counterfactual(orc_lossy *s, int exact_squares, int saturating_round)
{
    s->exact_squares = exact_squares;
    s->saturating_round = saturating_round;
}
/* MIN_T of a subtractMin state: the minimum of the first frame's lossy rows (0 before the first frame or without subtractMin) */
ORC_API int orc_lossy_get_min(const orc_lossy *s)
{
    return (s->subtract_min && s->frames > 0) ? (int)s->minv : 0;
}
ORC_API void orc_lossy_close(orc_lossy *s)
{
    if (!s) return;
    free(s->lastDL); free(s->refT); free(s->prevT); free(s->tmp); free(s->tmpT); free(s->ring);
    free(s->sums); free(s->cvalue); free(s->ccount); free(s->bp_xy); free(s);
}

static double lossy_square(int diff, int exact)
{
    return exact ? (double)diff * (double)diff : (double)orc_wrapped_square(diff);
}

/* stdDev, h264.cpp:1993-2036: (first, second) = (background, foreground) spreads of |img - prev|.  Each int square is
 * added into the double sums in pixel order, like the reference (orc_wrapped_square: the product wraps for
 * |diff| >= 46341).  An empty side gives 0 / 0 = NaN. */
static void lossy_std_dev(const u16 *prev, const u16 *img, int n, const u16 *img_dl, const unsigned *back, int exact,
                          double out[2])
{
    if (!back || !img_dl) {
        double sum_diff2 = 0, sum_diff = 0;
        for (int i = 0; i < n; ++i) {
            int diff = abs((int)img[i] - (int)prev[i]);
            sum_diff2 += lossy_square(diff, exact);
            sum_diff += diff;
        }
        double res = sqrt((sum_diff * sum_diff - sum_diff2)) / n;
        out[0] = out[1] = res;
    } else {
        double sum_diff2 = 0, sum_diff = 0, b_sum_diff2 = 0, b_sum_diff = 0;
        int b_sum = 0, sum = 0;
        for (int i = 0; i < n; ++i) {
            int diff = abs((int)img[i] - (int)prev[i]);
            if (img_dl[i] > *back) { sum_diff2 += lossy_square(diff, exact); sum_diff += diff; sum++; }
            else { b_sum_diff2 += lossy_square(diff, exact); b_sum_diff += diff; b_sum++; }
        }
        out[0] = sqrt((b_sum_diff * b_sum_diff - b_sum_diff2)) / b_sum;
        out[1] = sqrt((sum_diff * sum_diff - sum_diff2)) / sum;
    }
}
/* stdDev as the tests call it: img_dl == NULL is the un-split form */
ORC_API void orc_lossy_std_dev(const u16 *prev, const u16 *img, int n, const u16 *img_dl, unsigned back, double out[2])
{
    lossy_std_dev(prev, img, n, img_dl, img_dl ? &back : NULL, 0, out);
}

static int lossy_round(double x, int saturating)
{
    if (!saturating)
        return orc_round_to_int(x);
    double r = round(x);
    return r != r ? 0 : r >= 2147483647.0 ? INT32_MAX : r <= -2147483648.0 ? INT32_MIN : (int)r;
}

/* The bound update of a frame (:2367-2376 in addImageLossyNoCamera, :2559-2567 in addLoss): errors = {low, high} in,
 * the frame's {BackgroundError, ForegroundError} out. */
static void lossy_bounds(int variant, int saturating, double sd0, double sd1, double mean0, double mean1, double std_factor,
                         int errors[2])
{
    int lowError = errors[0], highError = errors[1];
    double diff_high, diff_low;
    if (variant == 0) { /* :2367-2368 */
        diff_high = fabs(sd1 - mean1);
        diff_low = fabs(sd0 - mean0);
    } else { /* addLoss :2559-2563: only a spread ABOVE the running mean tightens the bound */
        diff_high = sd1 < mean1 ? 0 : sd1 - mean1;
        diff_low = sd0 < mean0 ? 0 : sd0 - mean0;
    }
    highError = orc_wrapping_sub(highError, lossy_round(diff_high * std_factor, saturating));
    lowError = orc_wrapping_sub(lowError, lossy_round(diff_low * std_factor, saturating));
    if (highError < 0) highError = 0;
    if (lowError < highError) lowError = highError;
    errors[0] = lowError; errors[1] = highError;
}
ORC_API void orc_lossy_bounds(int variant, double sd0, double sd1, double mean0, double mean1, double std_factor, int errors[2])
{
    lossy_bounds(variant, 0, sd0, sd1, mean0, mean1, std_factor, errors);
}

/* One frame in, one frame out (what addImageLossLess then receives).  errors[0] = BackgroundError
 * (lowError), errors[1] = ForegroundError (highError) of this frame. */
ORC_API void orc_lossy_add_image(orc_lossy *s, const u16 *img, u16 *out, int *errors)
{
    const int w = s->w, h = s->h;
    const int n = w * h, ns = w * s->stop_h;
    /* :2259-2271 bad pixels on the lossy rows, copy of the rest */
    if (s->bp_enabled) {
        if (s->frames == 0) {
            int thr;
            s->bp_count = orc_bad_pixels_detect(img, w, s->stop_h, 5.0, s->bp_xy, ns, &thr);
            s->bp_clamp = orc_bad_pixels_clamp_value(img, w, s->stop_h);
        }
        orc_bad_pixels_correct(img, s->tmp, w, s->stop_h, s->bp_xy, s->bp_count, s->bp_clamp);
        memcpy(s->tmp + ns, img + ns, (size_t)(n - ns) * 2);
    } else {
        memcpy(s->tmp, img, (size_t)n * 2);
    }
    if (s->frames == 0) { /* :2273-2311 first image */
        memcpy(s->lastDL, s->tmp, (size_t)n * 2);
        if (s->subtract_min) {
            s->minv = 65535;
            for (int i = 0; i < ns; ++i) if (s->tmp[i] < s->minv) s->minv = s->tmp[i];
            for (int i = 0; i < ns; ++i) s->tmp[i] = (s->tmp[i] < s->minv) ? 0 : (u16)(s->tmp[i] - s->minv);
        }
        errors[0] = s->low_error; errors[1] = s->high_error;
        memcpy(out, s->tmp, (size_t)n * 2);
        memcpy(s->refT, s->tmp, (size_t)ns * 2);
        memcpy(s->prevT, s->tmp, (size_t)ns * 2);
        s->frames++;
        return;
    }
    memcpy(s->tmpT, s->tmp, (size_t)n * 2); /* :2314 */
    if (s->subtract_min)
        for (int i = 0; i < ns; ++i) s->tmpT[i] = (s->tmpT[i] < s->minv) ? 0 : (u16)(s->tmpT[i] - s->minv);
    unsigned background = orc_get_background(s->tmp, ns); /* :2331 */
    double sd[2];
    const int running_average_frames = 40;
    if (s->nstds < running_average_frames) lossy_std_dev(s->prevT, s->tmpT, ns, NULL, NULL, s->exact_squares, sd);
    else lossy_std_dev(s->prevT, s->tmpT, ns, img, &background, s->exact_squares, sd);
    if (!s->have_first) { s->first_std[0] = sd[0]; s->first_std[1] = sd[1]; s->have_first = 1; }
    if (s->nstds < running_average_frames) { s->stds[s->nstds][0] = sd[0]; s->stds[s->nstds][1] = sd[1]; s->nstds++; }
    else {
        /* :2347 shifts the window with memcpy(data, data + 1, 39 pairs) -- OVERLAPPING, i.e. undefined behaviour.  What the
         * reference does as compiled with its stock flags (g++ 13 -O3, x86-64; oracle/_ref, pinned by execution): the
         * expansion copies the LAST 8 bytes first (pair 39's .second over pair 38's) and then the rest front to back, so
         * after the shift pairs 37 and 38 both carry old pair 39's .second and old pair 38's .second is lost; every
         * .first is shifted correctly.  memcpy_quirk == 0 gives the intended memmove. */
        double last_second = s->stds[39][1];
        memmove(&s->stds[0], &s->stds[1], sizeof(double) * 2 * (running_average_frames - 1));
        if (s->memcpy_quirk) s->stds[37][1] = last_second;
        s->stds[39][0] = sd[0]; s->stds[39][1] = sd[1];
    }
    double mean0 = s->first_std[0], mean1 = s->first_std[1]; /* :2353-2365 */
    for (int i = 0; i < s->nstds; ++i) { mean0 += s->stds[i][0]; mean1 += s->stds[i][1]; }
    mean0 /= (s->nstds + 1); mean1 /= (s->nstds + 1);
    errors[0] = s->low_error; errors[1] = s->high_error;
    lossy_bounds(s->variant, s->saturating_round, sd[0], sd[1], mean0, mean1, s->std_factor, errors);
    const int lowError = errors[0], highError = errors[1];
    /* RunningAverage2::addImage :1560-1594 */
    const int ra = s->running_average;
    if (ra > 0) {
        for (int i = 0; i < ns; ++i) {
            s->sums[i] += s->tmpT[i];
            if (s->ring_len == ra) {
                if (s->ccount[i]) { --s->ccount[i]; s->sums[i] -= s->cvalue[i]; }
                else if (s->ring_len > 0) s->sums[i] -= s->ring[i];
            }
        }
        if (s->ring_len < ra) { memcpy(s->ring + (size_t)s->ring_len * ns, s->tmpT, (size_t)ns * 2); s->ring_len++; }
        else { memmove(s->ring, s->ring + ns, (size_t)(ra - 1) * ns * 2); memcpy(s->ring + (size_t)(ra - 1) * ns, s->tmpT, (size_t)ns * 2); }
    }
    for (int i = 0; i < ns; ++i) { /* :2397-2413 */
        int diff = abs((int)s->tmpT[i] - (int)s->refT[i]);
        int max_error = s->tmp[i] > background ? highError : lowError;
        /* addLoss (:2584) has no integration-time test */
        if (diff <= max_error && (s->variant == 1 || (s->lastDL[i] >> 13) == (s->tmp[i] >> 13))) {
            s->tmpT[i] = ra > 0 ? (u16)(s->sums[i] / (unsigned long)s->ring_len) : s->refT[i];
        } else {
            s->refT[i] = s->tmpT[i];
            if (ra > 0) { s->cvalue[i] = s->tmpT[i]; s->ccount[i] = (short)s->ring_len; s->sums[i] = (unsigned)s->tmpT[i] * (unsigned)s->ring_len; }
        }
    }
    memcpy(s->prevT, s->tmpT, (size_t)ns * 2);
    memcpy(s->lastDL, s->tmp, (size_t)n * 2);
    memcpy(s->tmpT + ns, s->tmp + ns, (size_t)(n - ns) * 2);
    memcpy(out, s->tmpT, (size_t)n * 2);
    s->frames++;
}
