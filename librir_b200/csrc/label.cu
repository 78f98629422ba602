// librir_b200/csrc/label.cu -- connected components of thresholded frames with per-component statistics
// (rirb_label_batch), and events of the whole (t, y, x) volume built on them (rirb_label_movie, second half of the file).
//
// Contract: a pixel is foreground iff frame > threshold; labels are 0 for background and 1..K in raster order of each
// component's first pixel (scipy.ndimage.label's numbering); statistics are integer sums, extrema and the raster-first
// argmax, so the result does not depend on the order of the atomics.
//
// Algorithm: block-based union-find (Playne & Hawick 2018; Allegretti, Bolelli & Grana 2019) with the labels buffer
// as the parent array.  Parents are frame-local linear indices and a union links the larger root under the smaller
// (atomicMin), so every parent is smaller than its child and the root of a component is its raster-first pixel.
//   1. local:  each CTA labels a 32 x 32 tile in shared memory and writes, per foreground pixel, the index of its
//              tile-local root; a bit mask per 32-pixel row segment marks the tile-local roots.
//   2. merge:  the top row and left column of each tile are joined to the neighbouring tiles in global memory.  Only
//              tile-local roots change parent here (path halving starts one hop away from the border pixel).
//   3. roots:  every tile-local root is pointed straight at its component's root (read-only finds, then one store);
//              the masks keep the global roots.
//   4. scan:   per frame, an exclusive scan of the root counts of the row segments (raster order) gives each root's
//              label = 1 + roots before its segment + roots before it in the segment; counts[t]; stats rows reset.
//   5. final:  each CTA reads its tile's parents (pixel -> tile-local root -> root), writes the labels in place and
//              folds the statistics of the tile per tile-local component in shared memory before one set of global
//              atomics per component and tile.  A sixth kernel splits the packed (max value, argmax) column.
// Traffic: 2 B/px read + 4 B/px written (1), 4 B/px read + 2 B/px read + 4 B/px written (5); the border, root and
// scan passes touch 1/32 of that.
#include <limits.h>

#include <cub/device/device_scan.cuh>

#include "common.cuh"
#include "kernels.h"

namespace rirb {

constexpr int LB_TW = 32;  // tile width: one warp per tile row, one mask word per row segment
constexpr int LB_TH = 32;
constexpr int LB_BY = 8;  // CTA of 32 x 8 threads, four tile rows each
constexpr int LB_TPX = LB_TW * LB_TH;

// ---- union-find in shared memory (tile-local indices) ---------------------------------------------------------
__device__ __forceinline__ int find_s(const volatile int* s, int x)
{
    int p;
    while ((p = s[x]) != x) x = p;
    return x;
}
__device__ void union_s(int* s, int a, int b)
{
    for (;;) {
        a = find_s(s, a);
        b = find_s(s, b);
        if (a == b) return;
        if (a < b) {
            const int t = a;
            a = b;
            b = t;
        }
        const int old = atomicMin(s + a, b);
        if (old == a) return;
        a = old;  // a was linked meanwhile: join its new parent instead
    }
}

// ---- union-find in global memory (L2 loads: other CTAs change the parents) --------------------------------------
// T = int: frame-local pixel indices (rirb_label_batch); T = long long: movie-wide component ids (rirb_label_movie).
// Root of x with path halving.  The 2-D passes pass a tile-local root, so every parent it rewrites is one.
template <typename T>
__device__ T find_g(T* L, T x)
{
    T p = __ldcg(L + x);
    while (p != x) {
        const T gp = __ldcg(L + p);
        if (gp == p) return p;
        __stcg(L + x, gp);
        x = gp;
        p = __ldcg(L + x);
    }
    return x;
}
template <typename T>
__device__ void union_g(T* L, T a, T b)
{
    for (;;) {
        a = find_g(L, a);
        b = find_g(L, b);
        if (a == b) return;
        if (a < b) {
            const T t = a;
            a = b;
            b = t;
        }
        const T old = atomicMin(L + a, b);
        if (old == a) return;
        a = old;
    }
}

// Root of x without writes: the roots pass points each tile-local root at its component root, and a path-halving store
// from another thread landing after that would leave the tile-local root on an intermediate node.
template <typename T>
__device__ __forceinline__ T root_of(const T* L, T x)
{
    T p;
    while ((p = __ldcg(L + x)) != x) x = p;
    return x;
}

struct LabelGeom {
    int w, h, tiles_x, tiles;  // tiles per frame
    size_t npx, segs;          // pixels and 32-pixel row segments per frame (segs = h * tiles_x)
};

static LabelGeom label_geom(int w, int h)
{
    LabelGeom g;
    g.w = w;
    g.h = h;
    g.tiles_x = (int)ceil_div(w, LB_TW);
    g.tiles = g.tiles_x * (int)ceil_div(h, LB_TH);
    g.npx = (size_t)w * h;
    g.segs = (size_t)h * g.tiles_x;
    return g;
}

// ---- 1. tile-local labelling -----------------------------------------------------------------------------------
template <int CONN>
__global__ void __launch_bounds__(LB_TW* LB_BY)
label_local_kernel(const u16* __restrict__ frames, const u16* __restrict__ thr, int per_frame_thr, LabelGeom g,
                   int* __restrict__ L, unsigned* __restrict__ roots)
{
    __shared__ int s[LB_TPX];
    const long long t = blockIdx.x / g.tiles;
    const int tile = (int)(blockIdx.x - t * g.tiles);
    const int tcol = tile % g.tiles_x;
    const int tx0 = tcol * LB_TW, ty0 = (tile / g.tiles_x) * LB_TH;
    const u16* f = frames + t * g.npx;
    L += t * g.npx;
    roots += t * g.segs;
    const unsigned th = thr[per_frame_thr ? t : 0];
    const int lx = threadIdx.x, x = tx0 + lx;
    for (int ly = threadIdx.y; ly < LB_TH; ly += LB_BY) {
        const int y = ty0 + ly;
        const bool fg = x < g.w && y < g.h && f[(size_t)y * g.w + x] > th;
        s[ly * LB_TW + lx] = fg ? ly * LB_TW + lx : -1;
    }
    __syncthreads();
    for (int ly = threadIdx.y; ly < LB_TH; ly += LB_BY) {
        const int i = ly * LB_TW + lx;
        if (s[i] < 0) continue;  // a foreground entry stays >= 0 whatever the unions do
        if (lx > 0 && s[i - 1] >= 0) union_s(s, i, i - 1);
        if (ly > 0) {
            if (s[i - LB_TW] >= 0) union_s(s, i, i - LB_TW);
            if (CONN == 8) {
                if (lx > 0 && s[i - LB_TW - 1] >= 0) union_s(s, i, i - LB_TW - 1);
                if (lx < LB_TW - 1 && s[i - LB_TW + 1] >= 0) union_s(s, i, i - LB_TW + 1);
            }
        }
    }
    __syncthreads();
    for (int ly = threadIdx.y; ly < LB_TH; ly += LB_BY) {
        const int i = ly * LB_TW + lx, y = ty0 + ly;
        const int r = s[i] < 0 ? -1 : find_s(s, i);
        const unsigned is_root = __ballot_sync(0xFFFFFFFFu, r == i);
        if (y < g.h) {
            if (x < g.w) L[(size_t)y * g.w + x] = r < 0 ? -1 : (ty0 + r / LB_TW) * g.w + tx0 + r % LB_TW;
            if (lx == 0) roots[(size_t)y * g.tiles_x + tcol] = is_root;
        }
    }
}

// ---- 2. merges across tile borders -----------------------------------------------------------------------------
// 64 threads per tile: 0..31 join the top row to the row above, 32..63 the left column to the column on the left.
template <int CONN>
__global__ void __launch_bounds__(LB_TW + LB_TH) label_merge_kernel(LabelGeom g, int* __restrict__ L)
{
    const long long t = blockIdx.x / g.tiles;
    const int tile = (int)(blockIdx.x - t * g.tiles);
    const int tx0 = (tile % g.tiles_x) * LB_TW, ty0 = (tile / g.tiles_x) * LB_TH;
    L += t * g.npx;
    int x, y, nx, ny;  // pixel, and the neighbour across the border for d = 0
    if (threadIdx.x < LB_TW) {
        x = tx0 + threadIdx.x;
        y = ty0;
        nx = x;
        ny = y - 1;
        if (ty0 == 0 || x >= g.w) return;
    } else {
        x = tx0;
        y = ty0 + threadIdx.x - LB_TW;
        nx = x - 1;
        ny = y;
        if (tx0 == 0 || y >= g.h) return;
    }
    const int q = y * g.w + x;
    const int a = __ldcg(L + q);  // tile-local root of q (or, for a root, what it has been joined to)
    if (a < 0) return;
    const bool top = threadIdx.x < LB_TW;
    for (int d = (CONN == 8 ? -1 : 0); d <= (CONN == 8 ? 1 : 0); ++d) {
        const int mx = top ? nx + d : nx, my = top ? ny : ny + d;
        if (mx < 0 || mx >= g.w || my < 0 || my >= g.h) continue;
        const int b = __ldcg(L + my * g.w + mx);
        if (b >= 0) union_g(L, a, b);
    }
}

// ---- 3. tile-local roots -> component roots --------------------------------------------------------------------
__global__ void __launch_bounds__(256) label_roots_kernel(LabelGeom g, long long nseg, int* __restrict__ L, unsigned* __restrict__ roots)
{
    for (long long c = (long long)blockIdx.x * blockDim.x + threadIdx.x; c < nseg; c += (long long)gridDim.x * blockDim.x) {
        unsigned m = roots[c];
        if (!m) continue;
        const long long t = c / (long long)g.segs;
        const int k = (int)(c - t * (long long)g.segs);
        const int y = k / g.tiles_x, x0 = (k - y * g.tiles_x) * LB_TW;
        int* Lf = L + t * g.npx;
        unsigned keep = 0;
        while (m) {
            const int b = __ffs(m) - 1;
            m &= m - 1;
            const int p = y * g.w + x0 + b;
            const int r = root_of(Lf, p);
            if (r == p)
                keep |= 1u << b;
            else
                __stcg(Lf + p, r);
        }
        roots[c] = keep;
    }
}

// ---- 4. per-frame scan of the root counts ----------------------------------------------------------------------
constexpr int LB_SCAN_THREADS = 1024;
constexpr int LB_SCAN_ITEMS = 4;

__global__ void __launch_bounds__(LB_SCAN_THREADS)
label_scan_kernel(LabelGeom g, const unsigned* __restrict__ roots, int* __restrict__ off, int* __restrict__ counts,
                  long long* __restrict__ stats, int cap)
{
    __shared__ int warp_sum[LB_SCAN_THREADS / 32];
    __shared__ int carry_sh;
    const long long t = blockIdx.x;
    roots += t * g.segs;
    off += t * g.segs;
    const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
    int carry = 0;
    for (size_t base = 0; base < g.segs; base += (size_t)LB_SCAN_THREADS * LB_SCAN_ITEMS) {
        const size_t i0 = base + (size_t)threadIdx.x * LB_SCAN_ITEMS;
        int v[LB_SCAN_ITEMS], sum = 0;
#pragma unroll
        for (int k = 0; k < LB_SCAN_ITEMS; ++k) {
            v[k] = i0 + k < g.segs ? __popc(roots[i0 + k]) : 0;
            sum += v[k];
        }
        int incl = sum;
#pragma unroll
        for (int d = 1; d < 32; d <<= 1) {
            const int n = __shfl_up_sync(0xFFFFFFFFu, incl, d);
            if (lane >= d) incl += n;
        }
        if (lane == 31) warp_sum[wid] = incl;
        __syncthreads();
        if (wid == 0) {
            int ws = warp_sum[lane], wi = ws;
#pragma unroll
            for (int d = 1; d < 32; d <<= 1) {
                const int n = __shfl_up_sync(0xFFFFFFFFu, wi, d);
                if (lane >= d) wi += n;
            }
            warp_sum[lane] = wi - ws;
            if (lane == 31) carry_sh = wi;
        }
        __syncthreads();
        int run = carry + warp_sum[wid] + incl - sum;
#pragma unroll
        for (int k = 0; k < LB_SCAN_ITEMS; ++k) {
            if (i0 + k < g.segs) off[i0 + k] = run;
            run += v[k];
        }
        carry += carry_sh;
        __syncthreads();  // warp_sum / carry_sh are rewritten by the next round
    }
    if (threadIdx.x == 0) counts[t] = carry;
    if (stats) {
        const int rows = carry < cap ? carry : cap;
        long long* st = stats + t * cap * 10;
        for (int k = threadIdx.x; k < rows; k += LB_SCAN_THREADS) {
            long long* r = st + (size_t)k * 10;
            r[0] = 0;
            r[1] = r[2] = LLONG_MAX;
            r[3] = r[4] = -1;
            r[5] = r[6] = r[7] = r[8] = r[9] = 0;
        }
    }
}

// ---- 5. labels in place + statistics ---------------------------------------------------------------------------
// Shared accumulators per tile-local component (indexed by a tile pixel, see below), tile-relative coordinates so that
// 32-bit sums cannot overflow: area, sum x, sum y, sum value, min x, min y, max x, max y, (value << 10 | 1023 - i).
enum { A_AREA, A_SX, A_SY, A_SV, A_XMIN, A_YMIN, A_XMAX, A_YMAX, A_KEY, A_COUNT };

template <bool STATS>
__global__ void __launch_bounds__(LB_TW* LB_BY)
label_final_kernel(const u16* __restrict__ frames, LabelGeom g, int* __restrict__ L, const unsigned* __restrict__ roots,
                   const int* __restrict__ off, long long* __restrict__ stats, int cap)
{
    __shared__ int s[LB_TPX];
    __shared__ unsigned acc[STATS ? A_COUNT : 1][STATS ? LB_TPX : 1];
    __shared__ int lab[STATS ? LB_TPX : 1];
    const long long t = blockIdx.x / g.tiles;
    const int tile = (int)(blockIdx.x - t * g.tiles);
    const int tx0 = (tile % g.tiles_x) * LB_TW, ty0 = (tile / g.tiles_x) * LB_TH;
    const u16* f = frames + t * g.npx;
    L += t * g.npx;
    roots += t * g.segs;
    off += t * g.segs;
    const int lx = threadIdx.x, x = tx0 + lx;
    for (int ly = threadIdx.y; ly < LB_TH; ly += LB_BY) {
        const int y = ty0 + ly, i = ly * LB_TW + lx;
        s[i] = (x < g.w && y < g.h) ? L[(size_t)y * g.w + x] : -1;
        if (STATS) {
#pragma unroll
            for (int a = 0; a < A_COUNT; ++a) acc[a][i] = (a == A_XMIN || a == A_YMIN) ? 0xFFFFFFFFu : 0u;
        }
    }
    __syncthreads();  // every parent of the tile is read before any label overwrites one
    for (int ly = threadIdx.y; ly < LB_TH; ly += LB_BY) {
        const int y = ty0 + ly, i = ly * LB_TW + lx;
        const int v = s[i];
        int label = 0;
        if (v >= 0) {
            // v is the tile-local root of this pixel (then its own parent is the component root), or, for a tile-local
            // root, the component root itself.  Either way `key` names one tile-local piece of one component.
            const int vy = (unsigned)v / (unsigned)g.w, vx = v - vy * g.w;
            int key = i, r = v;
            if ((unsigned)(vx - tx0) < (unsigned)LB_TW && (unsigned)(vy - ty0) < (unsigned)LB_TH) {
                key = (vy - ty0) * LB_TW + (vx - tx0);
                r = s[key];
            }
            const int ry = (unsigned)r / (unsigned)g.w, rx = r - ry * g.w;
            const size_t seg = (size_t)ry * g.tiles_x + (rx >> 5);
            label = 1 + off[seg] + __popc(roots[seg] & ((1u << (rx & 31)) - 1u));
            if (STATS) {
                const unsigned val = f[(size_t)y * g.w + x];
                lab[key] = label;
                atomicAdd(&acc[A_AREA][key], 1u);
                atomicAdd(&acc[A_SX][key], (unsigned)lx);
                atomicAdd(&acc[A_SY][key], (unsigned)ly);
                atomicAdd(&acc[A_SV][key], val);
                atomicMin(&acc[A_XMIN][key], (unsigned)lx);
                atomicMin(&acc[A_YMIN][key], (unsigned)ly);
                atomicMax(&acc[A_XMAX][key], (unsigned)lx);
                atomicMax(&acc[A_YMAX][key], (unsigned)ly);
                atomicMax(&acc[A_KEY][key], val << 10 | (unsigned)(LB_TPX - 1 - i));
            }
        }
        if (x < g.w && y < g.h) L[(size_t)y * g.w + x] = label;
    }
    if (!STATS) return;
    __syncthreads();
    for (int k = threadIdx.y * LB_TW + threadIdx.x; k < LB_TPX; k += LB_TW * LB_BY) {
        const unsigned area = acc[A_AREA][k];
        if (area == 0 || lab[k] > cap) continue;
        long long* r = stats + ((size_t)t * cap + lab[k] - 1) * 10;
        atomicAdd((unsigned long long*)r + 0, (unsigned long long)area);
        atomicMin(r + 1, (long long)(tx0 + (int)acc[A_XMIN][k]));
        atomicMin(r + 2, (long long)(ty0 + (int)acc[A_YMIN][k]));
        atomicMax(r + 3, (long long)(tx0 + (int)acc[A_XMAX][k]));
        atomicMax(r + 4, (long long)(ty0 + (int)acc[A_YMAX][k]));
        atomicAdd((unsigned long long*)r + 5, (unsigned long long)acc[A_SX][k] + (unsigned long long)area * tx0);
        atomicAdd((unsigned long long*)r + 6, (unsigned long long)acc[A_SY][k] + (unsigned long long)area * ty0);
        atomicAdd((unsigned long long*)r + 7, (unsigned long long)acc[A_SV][k]);
        const unsigned key = acc[A_KEY][k];
        const int li = LB_TPX - 1 - (int)(key & (LB_TPX - 1));
        const unsigned at = (unsigned)((ty0 + li / LB_TW) * g.w + tx0 + li % LB_TW);
        // column 8 holds (max value << 32 | ~argmax) until label_stats_split_kernel: the max wins, then the first pixel
        atomicMax((unsigned long long*)r + 8, (unsigned long long)(key >> 10) << 32 | (0xFFFFFFFFu - at));
    }
}

// ---- 6. the packed (max value, argmax) column -> columns 8 and 9 -------------------------------------------------
__global__ void __launch_bounds__(256) label_stats_split_kernel(long long* __restrict__ stats, const int* __restrict__ counts,
                                                                long long nrows, int cap)
{
    for (long long r = (long long)blockIdx.x * blockDim.x + threadIdx.x; r < nrows; r += (long long)gridDim.x * blockDim.x) {
        if (r % cap >= counts[r / cap]) continue;
        long long* row = stats + r * 10;
        const unsigned long long key = (unsigned long long)row[8];
        row[8] = (long long)(key >> 32);
        row[9] = (long long)(0xFFFFFFFFu - (unsigned)(key & 0xFFFFFFFFu));
    }
}

int launch_label(const u16* frames, int w, int h, long long nframes, const u16* thr, int per_frame_thr, int connectivity,
                 int* labels, int* counts, long long* stats, int cap, cudaStream_t st)
{
    const LabelGeom g = label_geom(w, h);
    if (cap <= 0) stats = nullptr;
    // frames per round: a 1-D grid of tiles, and at most 256 MB of segment masks + offsets
    long long per = INT_MAX / g.tiles;
    const long long by_scratch = (long long)((256u << 20) / (8 * g.segs));
    if (per > by_scratch) per = by_scratch > 0 ? by_scratch : 1;
    if (per > nframes) per = nframes;
    unsigned* roots = (unsigned*)scratch_buffer((size_t)per * g.segs * 2 * sizeof(unsigned));
    if (!roots) return -1;
    int* off = (int*)(roots + (size_t)per * g.segs);
    const dim3 tile_block(LB_TW, LB_BY);
    for (long long f0 = 0; f0 < nframes; f0 += per) {
        const long long m = nframes - f0 < per ? nframes - f0 : per;
        const u16* fr = frames + f0 * g.npx;
        const u16* th = thr + (per_frame_thr ? f0 : 0);
        int* Lf = labels + f0 * g.npx;
        long long* sf = stats ? stats + f0 * cap * 10 : nullptr;
        const unsigned grid = (unsigned)(m * g.tiles);
        const long long nseg = m * (long long)g.segs;
        const unsigned rgrid = (unsigned)(ceil_div(nseg, 256) < 8LL * sm_count() ? ceil_div(nseg, 256) : 8LL * sm_count());
        if (connectivity == 8) {
            RIRB_LAUNCH(label_local_kernel<8>, grid, tile_block, 0, st, fr, th, per_frame_thr, g, Lf, roots);
            RIRB_LAUNCH(label_merge_kernel<8>, grid, LB_TW + LB_TH, 0, st, g, Lf);
        } else {
            RIRB_LAUNCH(label_local_kernel<4>, grid, tile_block, 0, st, fr, th, per_frame_thr, g, Lf, roots);
            RIRB_LAUNCH(label_merge_kernel<4>, grid, LB_TW + LB_TH, 0, st, g, Lf);
        }
        RIRB_LAUNCH(label_roots_kernel, rgrid, 256, 0, st, g, nseg, Lf, roots);
        RIRB_LAUNCH(label_scan_kernel, (unsigned)m, LB_SCAN_THREADS, 0, st, g, roots, off, counts + f0, sf, cap);
        if (sf) {
            RIRB_LAUNCH(label_final_kernel<true>, grid, tile_block, 0, st, fr, g, Lf, roots, off, sf, cap);
            const long long nrows = m * cap;
            const unsigned sgrid = (unsigned)(ceil_div(nrows, 256) < 8LL * sm_count() ? ceil_div(nrows, 256) : 8LL * sm_count());
            RIRB_LAUNCH(label_stats_split_kernel, sgrid, 256, 0, st, sf, counts + f0, nrows, cap);
        } else {
            RIRB_LAUNCH(label_final_kernel<false>, grid, tile_block, 0, st, fr, g, Lf, roots, off, sf, cap);
        }
    }
    return 0;
}

// =================================================================================================================
// rirb_label_movie: events, the connected components of the whole (t, y, x) volume
// =================================================================================================================
// 6-, 18- and 26-connectivity are 4-, 8- and 8-connectivity in the plane plus, to the neighbouring frame, the same
// pixel, the same pixel and its 4 edge neighbours, or the 3 x 3 block.  So the 2-D passes above label every frame at
// the in-plane connectivity (labels = 2-D labels 1..K_t, counts = K_t), and what is left is a union-find over the
// 2-D components:
//   ids:     base[t] = K_0 + .. + K_{t-1} (exclusive scan); component (t, l) has id g = base[t] + l - 1, C = sum K_t.
//   link:    for every foreground pixel of frame t >= 1 and every foreground stencil neighbour in frame t - 1, union
//            the two ids (union_g on a 64-bit parent array: the smaller root becomes the parent).  A lane skips a pair
//            that the lane before it (pixel x - 1 of the same row) or its own previous union already joined, and
//            union_g finds both roots before any atomic, so an all-foreground volume does one union per warp and tile.
//   roots:   each id is pointed at its root (path halving first, so a chain of unions through every frame is walked
//            once, not once per member); root flags.
//   scan:    inclusive scan of the flags: ids[r] = 1 + roots before r for a root r; ids[C] = K.  Then every non-root
//            takes its root's number (read-only finds; roots' entries are never written, so the pass does not race).
//   final:   labels[t][y][x] = ids[base[t] + l - 1] in place; with statistics, each CTA folds its tile per event in a
//            shared hash (warps pre-reduce equal-event runs of a row) before one set of global atomics per event and
//            tile.  A last kernel splits the packed (max value, argmax) column.
// Why this numbering is scipy.ndimage.label's on the volume: the order of g is (t, raster order of the component's
// first pixel).  Take an event E and its first voxel v in (t, y, x) raster order, in frame t0, the first frame E
// touches.  Every other 2-D component of E lies in a later frame, or in frame t0 with its first pixel after v, so the
// component holding v has the smallest g of E, and it is E's root.  Two events are then in the order of their roots'
// g, i.e. of (t0, raster position of v): the 3-D raster order of their first voxels.
// Traffic beyond the 2-D passes: link 4 B/px read (the previous frame's labels come from L2) plus 8 B per union,
// final 4 B/px read + 4 B/px written (+ 2 B/px read with statistics) plus 8 B per 2-D component.
constexpr int LM_COLS = 13;
constexpr unsigned long long LM_IDX_MASK = (1ull << 48) - 1;  // argmax indices; the entry refuses movies of >= 2^48 voxels

static size_t align256(size_t b) { return (b + 255) & ~(size_t)255; }

static unsigned flat_grid(long long n)
{
    const long long b = ceil_div(n, 256), cap = 8LL * sm_count();
    return (unsigned)(b < 1 ? 1 : b < cap ? b : cap);
}
static unsigned tile_grid(long long items)
{
    const long long cap = 32LL * sm_count();
    return (unsigned)(items < cap ? items : cap);
}

__global__ void __launch_bounds__(256) movie_init_kernel(long long* __restrict__ P, long long C)
{
    for (long long c = (long long)blockIdx.x * blockDim.x + threadIdx.x; c < C; c += (long long)gridDim.x * blockDim.x) P[c] = c;
}

// K_t (int, from launch_label) -> base[t] (int64, scanned in place), base[n] = 0
__global__ void __launch_bounds__(256) movie_widen_kernel(const int* __restrict__ kt, long long* __restrict__ base, long long n)
{
    for (long long t = (long long)blockIdx.x * blockDim.x + threadIdx.x; t <= n; t += (long long)gridDim.x * blockDim.x)
        base[t] = t < n ? kt[t] : 0;
}

// ---- 7. links between consecutive frames -----------------------------------------------------------------------
// Work item wi: tile (wi % tiles) of frame 1 + wi / tiles, joined to frame t - 1.
template <int CONN>
__global__ void __launch_bounds__(LB_TW* LB_BY, 4)  // without a floor on the CTAs per SM, ptxas caps it at 32 registers and spills
movie_link_kernel(LabelGeom g, const int* __restrict__ labels, const long long* __restrict__ base, long long* __restrict__ P,
                  long long items)
{
    const int lx = threadIdx.x;
    for (long long wi = blockIdx.x; wi < items; wi += gridDim.x) {
        const long long t = 1 + wi / g.tiles;
        const int tile = (int)(wi - (t - 1) * g.tiles);
        const int tx0 = (tile % g.tiles_x) * LB_TW, ty0 = (tile / g.tiles_x) * LB_TH;
        const int* Lc = labels + t * g.npx;
        const int* Lp = Lc - g.npx;
        const long long gc = base[t] - 1, gp = base[t - 1] - 1;
        const int x = tx0 + lx;
        int last_a = 0, last_b = 0;  // this thread's last union
        for (int ly = threadIdx.y; ly < LB_TH; ly += LB_BY) {
            const int y = ty0 + ly;
            const int a = (x < g.w && y < g.h) ? __ldg(Lc + (size_t)y * g.w + x) : 0;
            if (!__any_sync(0xFFFFFFFFu, a > 0)) continue;
#pragma unroll
            for (int dy = -1; dy <= 1; ++dy) {
#pragma unroll
                for (int dx = -1; dx <= 1; ++dx) {
                    if ((CONN == 6 && (dy || dx)) || (CONN == 18 && dy && dx)) continue;
                    const int ny = y + dy, nx = x + dx;
                    const int b = (a > 0 && ny >= 0 && ny < g.h && nx >= 0 && nx < g.w) ? __ldg(Lp + (size_t)ny * g.w + nx) : 0;
                    const int pa = __shfl_up_sync(0xFFFFFFFFu, a, 1), pb = __shfl_up_sync(0xFFFFFFFFu, b, 1);
                    if (b > 0 && !(lx > 0 && pa == a && pb == b) && !(a == last_a && b == last_b)) {
                        union_g(P, gc + a, gp + b);
                        last_a = a;
                        last_b = b;
                    }
                }
            }
        }
    }
}

// ---- 8. roots and their flags (ids[C] = 0, so that the inclusive scan leaves K there) ---------------------------
__global__ void __launch_bounds__(256) movie_roots_kernel(long long* __restrict__ P, long long* __restrict__ ids, long long C)
{
    for (long long c = (long long)blockIdx.x * blockDim.x + threadIdx.x; c <= C; c += (long long)gridDim.x * blockDim.x) {
        if (c == C) {
            ids[C] = 0;
            continue;
        }
        const long long r = find_g(P, c);
        if (r != c) __stcg(P + c, r);
        ids[c] = r == c;
    }
}

// ---- 9. event numbers of the non-roots, the count, the statistics rows reset -------------------------------------
__global__ void __launch_bounds__(256)
movie_number_kernel(const long long* __restrict__ P, long long* __restrict__ ids, long long C, int* __restrict__ count,
                    long long* __restrict__ stats, int cap)
{
    const long long K = ids[C];
    const long long rows = K < cap ? K : cap;
    const long long n = C > rows ? C : rows;
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x) {
        if (i == 0) *count = (int)K;  // the launcher has checked K <= INT_MAX
        if (i < C) {
            const long long r = root_of(P, i);
            if (r != i) ids[i] = ids[r];
        }
        if (stats && i < rows) {
            long long* row = stats + i * LM_COLS;
            row[0] = 0;
            row[1] = LLONG_MAX;  // t first
            row[2] = -1;         // t last
            row[3] = row[4] = LLONG_MAX;
            row[5] = row[6] = -1;
            row[7] = row[8] = row[9] = row[10] = row[11] = row[12] = 0;
        }
    }
}

// ---- 10. labels in place + statistics ----------------------------------------------------------------------------
// A 32 x 32 tile holds at most 512 2-D components, so a hash of LB_TPX event slots (linear probing) never fills.
__device__ __forceinline__ int movie_slot(int* keys, int e)
{
    int s = (int)(((unsigned)e * 2654435761u) >> 22);  // LB_TPX = 2^10 slots
    for (;;) {
        const int k = atomicCAS(keys + s, 0, e);
        if (k == 0 || k == e) return s;
        s = (s + 1) & (LB_TPX - 1);
    }
}
__device__ __forceinline__ void movie_slot_reset(int* keys, unsigned (*acc)[LB_TPX], int k)
{
    keys[k] = 0;
#pragma unroll
    for (int a = 0; a < A_COUNT; ++a) acc[a][k] = (a == A_XMIN || a == A_YMIN) ? 0xFFFFFFFFu : 0u;
}

template <bool STATS>
__global__ void __launch_bounds__(LB_TW* LB_BY)
movie_final_kernel(const u16* __restrict__ frames, LabelGeom g, int* __restrict__ labels, const long long* __restrict__ base,
                   const long long* __restrict__ ids, long long* __restrict__ stats, int cap, long long items)
{
    __shared__ int keys[STATS ? LB_TPX : 1];
    __shared__ unsigned acc[STATS ? A_COUNT : 1][STATS ? LB_TPX : 1];
    const int lx = threadIdx.x, tid = threadIdx.y * LB_TW + lx;
    if constexpr (STATS) {
        for (int k = tid; k < LB_TPX; k += LB_TW * LB_BY) movie_slot_reset(keys, acc, k);
        __syncthreads();
    }
    for (long long wi = blockIdx.x; wi < items; wi += gridDim.x) {
        const long long t = wi / g.tiles;
        const int tile = (int)(wi - t * g.tiles);
        const int tx0 = (tile % g.tiles_x) * LB_TW, ty0 = (tile / g.tiles_x) * LB_TH;
        int* L = labels + t * g.npx;
        const long long* id = ids + base[t] - 1;  // id[l]: the event of 2-D component l of frame t
        const int x = tx0 + lx;
        for (int ly = threadIdx.y; ly < LB_TH; ly += LB_BY) {
            const int y = ty0 + ly;
            const size_t p = (size_t)y * g.w + x;
            const int l = (x < g.w && y < g.h) ? L[p] : 0;
            const int e = l > 0 ? (int)id[l] : 0;
            if (l > 0) L[p] = e;
            if constexpr (STATS) {
                // the lanes of one event in this row: one leader folds them into the event's slot
                const unsigned grp = __match_any_sync(0xFFFFFFFFu, e);
                if (e > 0) {
                    const unsigned val = frames[t * g.npx + p];
                    const unsigned sx = __reduce_add_sync(grp, (unsigned)lx);
                    const unsigned sv = __reduce_add_sync(grp, val);
                    const unsigned key = __reduce_max_sync(grp, val << 10 | (unsigned)(LB_TPX - 1 - (ly * LB_TW + lx)));
                    if (lx == __ffs(grp) - 1) {
                        const int s = movie_slot(keys, e);
                        const unsigned vol = __popc(grp);
                        atomicAdd(&acc[A_AREA][s], vol);
                        atomicAdd(&acc[A_SX][s], sx);
                        atomicAdd(&acc[A_SY][s], vol * ly);
                        atomicAdd(&acc[A_SV][s], sv);
                        atomicMin(&acc[A_XMIN][s], (unsigned)lx);
                        atomicMin(&acc[A_YMIN][s], (unsigned)ly);
                        atomicMax(&acc[A_XMAX][s], (unsigned)(31 - __clz(grp)));
                        atomicMax(&acc[A_YMAX][s], (unsigned)ly);
                        atomicMax(&acc[A_KEY][s], key);
                    }
                }
            }
        }
        if constexpr (STATS) {
            __syncthreads();
            for (int k = tid; k < LB_TPX; k += LB_TW * LB_BY) {
                const int e = keys[k];
                if (!e) continue;
                if (e <= cap) {
                    long long* r = stats + (size_t)(e - 1) * LM_COLS;
                    const unsigned long long vol = acc[A_AREA][k];
                    atomicAdd((unsigned long long*)r + 0, vol);
                    atomicMin(r + 1, t);
                    atomicMax(r + 2, t);
                    atomicMin(r + 3, (long long)(tx0 + (int)acc[A_XMIN][k]));
                    atomicMin(r + 4, (long long)(ty0 + (int)acc[A_YMIN][k]));
                    atomicMax(r + 5, (long long)(tx0 + (int)acc[A_XMAX][k]));
                    atomicMax(r + 6, (long long)(ty0 + (int)acc[A_YMAX][k]));
                    atomicAdd((unsigned long long*)r + 7, vol * (unsigned long long)t);
                    atomicAdd((unsigned long long*)r + 8, (unsigned long long)acc[A_SX][k] + vol * tx0);
                    atomicAdd((unsigned long long*)r + 9, (unsigned long long)acc[A_SY][k] + vol * ty0);
                    atomicAdd((unsigned long long*)r + 10, (unsigned long long)acc[A_SV][k]);
                    const unsigned key = acc[A_KEY][k];
                    const int li = LB_TPX - 1 - (int)(key & (LB_TPX - 1));
                    const unsigned long long at = (unsigned long long)t * g.npx + (unsigned long long)(ty0 + li / LB_TW) * g.w + tx0 + li % LB_TW;
                    // column 11 holds (max value << 48 | 2^48 - 1 - argmax) until movie_stats_split_kernel
                    atomicMax((unsigned long long*)r + 11, (unsigned long long)(key >> 10) << 48 | (LM_IDX_MASK - at));
                }
                movie_slot_reset(keys, acc, k);
            }
            __syncthreads();
        }
    }
}

// ---- 11. the packed (max value, argmax) column -> columns 11 and 12 -----------------------------------------------
__global__ void __launch_bounds__(256) movie_stats_split_kernel(long long* __restrict__ stats, const long long* __restrict__ K, int cap)
{
    const long long rows = *K < cap ? *K : cap;
    for (long long r = (long long)blockIdx.x * blockDim.x + threadIdx.x; r < rows; r += (long long)gridDim.x * blockDim.x) {
        long long* row = stats + r * LM_COLS;
        const unsigned long long key = (unsigned long long)row[11];
        row[11] = (long long)(key >> 48);
        row[12] = (long long)(LM_IDX_MASK - (key & LM_IDX_MASK));
    }
}

int launch_label_movie(const u16* frames, int w, int h, long long nframes, const u16* thr, int per_frame_thr, int connectivity,
                       int* labels, int* count, long long* stats, int cap, cudaStream_t st)
{
    const LabelGeom g = label_geom(w, h);
    if (cap <= 0) stats = nullptr;
    // K_t [n] | base [n + 1] | the scan's work space
    const long long n1 = nframes + 1;
    size_t tmp1 = 0;
    RIRB_CUDA_OK(cub::DeviceScan::ExclusiveSum(nullptr, tmp1, (long long*)nullptr, n1, st));
    const size_t o_base = align256((size_t)nframes * sizeof(int)), o_tmp1 = o_base + align256((size_t)n1 * sizeof(long long));
    char* frame_ws = (char*)scratch_buffer(o_tmp1 + tmp1);
    if (!frame_ws) return -1;
    int* kt = (int*)frame_ws;
    long long* base = (long long*)(frame_ws + o_base);
    if (launch_label(frames, w, h, nframes, thr, per_frame_thr, connectivity == 6 ? 4 : 8, labels, kt, nullptr, 0, st) != 0)
        return -1;
    RIRB_LAUNCH(movie_widen_kernel, flat_grid(n1), 256, 0, st, kt, base, nframes);
    RIRB_CUDA_OK(cub::DeviceScan::ExclusiveSum(frame_ws + o_tmp1, tmp1, base, n1, st));
    long long C = 0;  // 2-D components of the whole movie: the one read-back every call waits for
    RIRB_CUDA_OK(cudaMemcpyAsync(&C, base + nframes, sizeof C, cudaMemcpyDeviceToHost, st));
    RIRB_CUDA_OK(cudaStreamSynchronize(st));
    if (C == 0) {  // nothing above the thresholds: every label is already 0
        RIRB_CUDA_OK(cudaMemsetAsync(count, 0, sizeof(int), st));
        return 0;
    }
    // parents [C]; root flags -> event ids [C + 1] | the scan's work space
    size_t tmp2 = 0;
    RIRB_CUDA_OK(cub::DeviceScan::InclusiveSum(nullptr, tmp2, (long long*)nullptr, C + 1, st));
    const size_t o_tmp2 = align256((size_t)(C + 1) * sizeof(long long));
    long long* P = (long long*)scratch_buffer((size_t)C * sizeof(long long));
    char* event_ws = (char*)scratch_buffer(o_tmp2 + tmp2);
    if (!P || !event_ws) return -1;
    long long* ids = (long long*)event_ws;
    const dim3 tile_block(LB_TW, LB_BY);
    RIRB_LAUNCH(movie_init_kernel, flat_grid(C), 256, 0, st, P, C);
    if (nframes > 1) {
        const long long items = (nframes - 1) * g.tiles;
        if (connectivity == 6)
            RIRB_LAUNCH(movie_link_kernel<6>, tile_grid(items), tile_block, 0, st, g, labels, base, P, items);
        else if (connectivity == 18)
            RIRB_LAUNCH(movie_link_kernel<18>, tile_grid(items), tile_block, 0, st, g, labels, base, P, items);
        else
            RIRB_LAUNCH(movie_link_kernel<26>, tile_grid(items), tile_block, 0, st, g, labels, base, P, items);
    }
    RIRB_LAUNCH(movie_roots_kernel, flat_grid(C + 1), 256, 0, st, P, ids, C);
    RIRB_CUDA_OK(cub::DeviceScan::InclusiveSum(event_ws + o_tmp2, tmp2, ids, C + 1, st));
    if (C > INT_MAX) {  // only then can the events outnumber a 32-bit label
        long long K = 0;
        RIRB_CUDA_OK(cudaMemcpyAsync(&K, ids + C, sizeof K, cudaMemcpyDeviceToHost, st));
        RIRB_CUDA_OK(cudaStreamSynchronize(st));
        if (K > INT_MAX) {
            set_error("label_movie: %lld events, more than an int32 label can number", K);
            return -1;
        }
    }
    RIRB_LAUNCH(movie_number_kernel, flat_grid(C > cap ? C : cap), 256, 0, st, P, ids, C, count, stats, cap);
    const long long items = nframes * g.tiles;
    if (stats) {
        RIRB_LAUNCH(movie_final_kernel<true>, tile_grid(items), tile_block, 0, st, frames, g, labels, base, ids, stats, cap, items);
        RIRB_LAUNCH(movie_stats_split_kernel, flat_grid(cap), 256, 0, st, stats, ids + C, cap);
    } else {
        RIRB_LAUNCH(movie_final_kernel<false>, tile_grid(items), tile_block, 0, st, frames, g, labels, base, ids, stats, cap, items);
    }
    return 0;
}

}  // namespace rirb
