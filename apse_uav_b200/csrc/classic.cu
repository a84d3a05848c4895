// classic.cu -- CLASSIC candidate stage of aruco.detectMarkers (aruco_detect.py:267 with cornerRefinementMethod
// NONE / SUBPIX; north_star stages (2)-(4), BASELINE.json config 5; SURVEY.md rows a6.C1-a6.C4), batched, sm_100a.
//
//   C1  k_adaptive_threshold   box-mean threshold (MEAN_C, BINARY_INV) of one window size: gray tile + halo staged in
//                              shared memory, row prefix sums by warp shuffles, sliding column sums
//   C2  k_ccl_* (detect_apriltag.cu, full-range mode)  foreground 8-connected / background 4-connected components,
//                              root = raster-first pixel;  k_mark_outside flags the background components that touch
//                              the image edge;  k_border_jobs lists one border per foreground component (outer) and
//                              per enclosed background component (hole) -- exactly the borders Suzuki-Abe border
//                              following finds, without its sequential raster scan (SURVEY.md Appendix A.5)
//       k_trace_borders        one thread per border: border following with the dependency's start / direction
//                              conventions; borders inside the perimeter limits are stored
//   C3  k_approx_quads         one warp per stored border: closed Douglas-Peucker (3 farthest-point rounds,
//                              explicit stack, point-to-segment distance, clean-up pass), convexity, corner
//                              distance, clockwise order -> candidate quad + ordering key
//       k_rank_quads           dependency candidate order: window ascending, then descending raster order of
//                              the border's trigger pixel
//   C4  k_corner_subpix        cornerSubPix on the accepted markers (thread per corner, FP64 normal equations)
//
// Integer / FP64 arithmetic follows the dependency's evaluation order (-fmad=false); parity: tests/test_gpu_classic.py.
#include "common.cuh"
#include <math.h>
#include <float.h>

// ---------------------------------------------------------------------------------------------------------
// C1: adaptive threshold, ALL windows of the sweep from one staged tile.  Tile 64 x 32 outputs, 256 threads; the gray tile
// with the halo of the LARGEST window is staged once (replicated border) as row prefix sums in dynamic shared memory (warp
// per row, shuffle scan); every window then takes its horizontal box sums as prefix differences and slides them down the
// columns.  Prefix sums are kept modulo 2^16: a difference is exact while win * 255 < 2^16, i.e. for every window up to 255.
#define AT_TW 64
#define AT_TH 32
#define AT_MAX_WINDOWS 16
#define AT_MAX_WIN 255
struct AtWindows { int n; int win[AT_MAX_WINDOWS]; };

static inline size_t at_smem_bytes(int rmax) { return (size_t)(AT_TH + 2 * rmax) * (size_t)(AT_TW + 2 * rmax + 2) * sizeof(uint16_t); }

__global__ void __launch_bounds__(256) k_adaptive_threshold(const uint8_t *__restrict__ gray, int w, int h, AtWindows W, int rmax, int idelta,
                                                            uint8_t *__restrict__ out, size_t window_stride)
{
    extern __shared__ uint16_t at_P[];   // [sh][pitch] inclusive row prefix sums (mod 2^16), column 0 = 0
    const int sw = AT_TW + 2 * rmax, sh = AT_TH + 2 * rmax, pitch = sw + 2;
    const int f = blockIdx.z, x0 = blockIdx.x * AT_TW, y0 = blockIdx.y * AT_TH;
    const uint8_t *g = gray + (size_t)f * w * h;
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    // stage rows and turn each into prefix sums: one warp per row, chunks of 128 columns (4 per lane) with a running carry
    for (int ry = warp; ry < sh; ry += 8) {
        const int gy = min(max(y0 - rmax + ry, 0), h - 1);
        const uint8_t *row = g + (size_t)gy * w;
        uint16_t *P = at_P + (size_t)ry * pitch;
        int carry = 0;
        for (int c0 = 0; c0 < sw; c0 += 128) {
            int v[4], s = 0;
#pragma unroll
            for (int k = 0; k < 4; k++) {
                const int cx = c0 + lane * 4 + k;
                const int gx = min(max(x0 - rmax + cx, 0), w - 1);
                v[k] = cx < sw ? (int)__ldg(row + gx) : 0;
                s += v[k];
            }
            int inc = s;
            for (int d = 1; d < 32; d <<= 1) { int t = __shfl_up_sync(0xffffffffu, inc, d); if (lane >= d) inc += t; }
            int run = carry + inc - s;
#pragma unroll
            for (int k = 0; k < 4; k++) { run += v[k]; const int cx = c0 + lane * 4 + k; if (cx < sw) P[cx + 1] = (uint16_t)run; }
            carry += __shfl_sync(0xffffffffu, inc, 31);
        }
        if (lane == 0) P[0] = 0;
    }
    __syncthreads();
    // per window: column sums of the horizontal box sums: thread = (column, group of 8 output rows), sliding along y
    const int cx = tid & 63, yg = tid >> 6;
    const int x = x0 + cx;
    for (int wi = 0; wi < W.n; wi++) {
        const int win = W.win[wi], r = win >> 1, off = rmax - r;   // this window's box starts `off` inside the staged halo
        const int area = win * win;
        const uint16_t *Q = at_P + (size_t)off * pitch + off + cx;  // row 0 / left edge of the box of output (cx, 0)
        auto hbox = [&](int row) { return (int)(uint16_t)(Q[(size_t)row * pitch + win] - Q[(size_t)row * pitch]); };
        int s = 0;
        for (int k = 0; k < win; k++) s += hbox(yg * 8 + k);
        uint8_t *o = out + (size_t)wi * window_stride + (size_t)f * w * h;
#pragma unroll 1
        for (int j = 0; j < 8; j++) {
            const int oy = yg * 8 + j, y = y0 + oy;
            if (j > 0) s += hbox(oy + win - 1) - hbox(oy - 1);
            if (x < w && y < h) {
                // mean = round-half-even(s / area); area is odd, so no ties exist and floor((2s + area) / (2 area)) is exact
                const int mean = (2 * s + area) / (2 * area);
                o[(size_t)y * w + x] = ((int)g[(size_t)y * w + x] - mean <= -idelta) ? 255 : 0;
            }
        }
    }
}

// all windows of a sweep (ascending, odd) for a batch: out[wi] = out + wi * window_stride
static int launch_adaptive(apse_ctx *ctx, const uint8_t *gray, int w, int h, int batch, const AtWindows &W, int idelta, uint8_t *out,
                           size_t window_stride, cudaStream_t st)
{
    int wmax = 0;
    for (int i = 0; i < W.n; i++) wmax = W.win[i] > wmax ? W.win[i] : wmax;
    if (wmax > AT_MAX_WIN) CTX_FAIL(ctx, APSE_ERR_UNSUPPORTED, "adaptiveThreshold: block size %d exceeds the supported %d", wmax, AT_MAX_WIN);
    const int rmax = wmax >> 1;
    const size_t smem = at_smem_bytes(rmax);
    static size_t attr_bytes[64] = {0};
    if (smem > 48 * 1024 && smem > attr_bytes[ctx->device & 63]) {
        CUDA_TRY(ctx, cudaFuncSetAttribute(k_adaptive_threshold, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        attr_bytes[ctx->device & 63] = smem;
    }
    dim3 grid(div_up(w, AT_TW), div_up(h, AT_TH), batch);
    KLAUNCH(ctx, KID_ADAPTIVE, st, k_adaptive_threshold<<<grid, 256, smem, st>>>(gray, w, h, W, rmax, idelta, out, window_stride));
    return APSE_OK;
}

// ---------------------------------------------------------------------------------------------------------
// C2: border jobs
#define LBL_OUTSIDE 0x80000000u

// background components that touch the image edge are connected to the (virtual) outside: flag their root
__global__ void k_mark_outside(const uint8_t *__restrict__ bin, int w, int h, uint32_t *__restrict__ labels, int batch)
{
    const int per = 2 * (w + h);
    for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < per * batch; i += gridDim.x * blockDim.x) {
        int f = i / per, k = i - f * per, x, y;
        if (k < w) { x = k; y = 0; }
        else if (k < 2 * w) { x = k - w; y = h - 1; }
        else if (k < 2 * w + h) { x = 0; y = k - 2 * w; }
        else { x = w - 1; y = k - 2 * w - h; }
        size_t o = (size_t)f * w * h + (size_t)y * w + x;
        if (bin[o] == 0) {
            uint32_t root = labels[o] & ~LBL_OUTSIDE;
            atomicOr(&labels[(size_t)f * w * h + root], LBL_OUTSIDE);
        }
    }
}

// one job per border: trigger pixel index | hole flag (bit 31)
// Also writes, for every foreground pixel, the 8-bit mask of its foreground neighbours (bit s = direction s), so that
// a border-following step is ONE dependent load instead of up to eight.
__global__ void __launch_bounds__(256) k_border_jobs(const uint8_t *__restrict__ bin, int w, int h, const uint32_t *__restrict__ labels,
                                                     uint32_t *__restrict__ jobs, int job_cap, int32_t *__restrict__ counters,
                                                     uint8_t *__restrict__ nbr_mask)
{
    const int f = blockIdx.y;
    const size_t npx = (size_t)w * h;
    const uint8_t *b = bin + f * npx;
    uint8_t *M = nbr_mask + f * npx;
    const uint32_t *L = labels + f * npx;
    uint32_t *J = jobs + (size_t)f * job_cap;
    int32_t *cnt = counters + f * APSE_COUNTERS;
    const int lane = threadIdx.x & 31;
    for (size_t p0 = (size_t)blockIdx.x * blockDim.x; p0 < npx; p0 += (size_t)gridDim.x * blockDim.x) {
        size_t p = p0 + threadIdx.x;
        bool job = false;
        uint32_t enc = 0;
        if (p < npx) {
            uint32_t l = L[p];
            const bool is_fg = b[p] != 0;
            if ((l & ~LBL_OUTSIDE) == (uint32_t)p) {
                if (is_fg) { job = true; enc = (uint32_t)p; }
                else if (!(l & LBL_OUTSIDE)) { job = true; enc = (uint32_t)p | 0x80000000u; }
            }
            unsigned m = 0;
            if (is_fg) {
                const int y = (int)(p / w), x = (int)(p - (size_t)y * w);
                const bool n_ = y > 0, s_ = y + 1 < h, w_ = x > 0, e_ = x + 1 < w;
                m = (e_ && b[p + 1] ? 1u : 0u) | (n_ && e_ && b[p - w + 1] ? 2u : 0u) | (n_ && b[p - w] ? 4u : 0u) |
                    (n_ && w_ && b[p - w - 1] ? 8u : 0u) | (w_ && b[p - 1] ? 16u : 0u) | (s_ && w_ && b[p + w - 1] ? 32u : 0u) |
                    (s_ && b[p + w] ? 64u : 0u) | (s_ && e_ && b[p + w + 1] ? 128u : 0u);
            }
            M[p] = (uint8_t)m;
        }
        unsigned m = __ballot_sync(0xffffffffu, job);
        if (m) {
            int leader = __ffs(m) - 1, base = 0;
            if (lane == leader) base = atomicAdd(&cnt[0], __popc(m));
            base = __shfl_sync(0xffffffffu, base, leader);
            if (job) {
                int idx = base + __popc(m & ((1u << lane) - 1));
                if (idx < job_cap) J[idx] = enc; else atomicExch(&cnt[3], APSE_ERR_CAPACITY);
            }
        }
    }
}

// Border following (Suzuki-Abe) on the neighbour masks; directions 0..7 = E, NE, N, NW, W, SW, S, SE (y downwards).
__device__ __constant__ int8_t c_dx[8] = {1, 1, 0, -1, -1, -1, 0, 1};
__device__ __constant__ int8_t c_dy[8] = {0, -1, -1, -1, 0, 1, 1, 1};
__device__ __forceinline__ unsigned rotr8(unsigned m, int r) { return ((m >> r) | (m << (8 - r))) & 0xffu; }
// c_dx / c_dy without the dependent constant-memory load: (d + 1) packed two bits per direction
__device__ __forceinline__ int dir_dx(int s) { return (int)((0x901Au >> (2 * s)) & 3u) - 1; }   // {1, 1, 0, -1, -1, -1, 0, 1} + 1 = {2, 2, 1, 0, 0, 0, 1, 2}
__device__ __forceinline__ int dir_dy(int s) { return (int)((0xA901u >> (2 * s)) & 3u) - 1; }   // {0, -1, -1, -1, 0, 1, 1, 1} + 1 = {1, 0, 0, 0, 1, 2, 2, 2}

template <bool STORE>
__device__ int trace_border(const uint8_t *__restrict__ M, int w, int x0, int y0, bool hole, int max_n, uint32_t *out)
{
    const int s0 = hole ? 0 : 4;
    unsigned m = M[(size_t)y0 * w + x0];
    if (m == 0) {   // isolated pixel
        if (STORE) out[0] = (uint32_t)x0 | ((uint32_t)y0 << 16);
        return 1;
    }
    // first neighbour clockwise from s0 - 1: candidate k <-> direction (s0 - 1 - k) & 7
    int s = (s0 - 1 - (__ffs(rotr8(__brev(m) >> 24, (8 - s0) & 7)) - 1)) & 7;
    const int x1 = x0 + dir_dx(s), y1 = y0 + dir_dy(s);
    int cx = x0, cy = y0, n = 0;
    for (;;) {
        // next neighbour counter-clockwise from s + 1: candidate k <-> direction (s + 1 + k) & 7
        const int base = (s + 1) & 7;
        s = (base + __ffs(rotr8(m, base)) - 1) & 7;
        const int nx = cx + dir_dx(s), ny = cy + dir_dy(s);
        if (STORE) out[n] = (uint32_t)cx | ((uint32_t)cy << 16);
        n++;
        if (nx == x0 && ny == y0 && cx == x1 && cy == y1) break;
        if (n > max_n) break;   // longer than the perimeter limit: the caller drops it
        cx = nx; cy = ny;
        m = M[(size_t)cy * w + cx];
        s = (s + 4) & 7;
    }
    return n;
}

struct ContourDesc { uint32_t offset, count, trigger, hole; };   // same footprint as ClusterDesc (scratch is shared)

// Borders are followed in two kernels.  k_trace_borders: one thread per border, for the ~10^5 short borders of a noisy frame; a
// border that is still open after TRACE_SHORT steps is handed to k_trace_long: one WARP per border, lane 0 follows it while all
// lanes keep the mask bytes around the current position in L1 (prefetch of the 32 rows x 2 lines around it every TRACE_PF
// steps).  A step is one dependent load; from L2 that is ~340 cycles, and the longest border of a frame (up to the perimeter
// limit, 15 360 steps at 4K) used to set the duration of the whole stage.
#define TRACE_SHORT 256
#define TRACE_PF 12
#define TRACE_LONG_CAP (1 << 16)
#define TW_W 64                       // shared-memory window of k_trace_long
#define TW_H 32

__device__ __forceinline__ void store_border(const uint8_t *I, int w, uint32_t e, int n, int32_t *cnt, uint32_t *P, int pts_cap, ContourDesc *D,
                                             int desc_cap, int max_px)
{
    const bool hole = (e >> 31) != 0;
    const uint32_t trig = e & 0x7fffffffu;
    const int ty = trig / w, tx = trig - ty * w;
    const int x0 = hole ? tx - 1 : tx, y0 = ty;
    const int di = atomicAdd(&cnt[1], 1);
    const int off = atomicAdd(&cnt[5], n);
    if (di >= desc_cap || off + n > pts_cap) { atomicExch(&cnt[3], APSE_ERR_CAPACITY); return; }
    trace_border<true>(I, w, x0, y0, hole, max_px, P + off);
    D[di] = ContourDesc{(uint32_t)off, (uint32_t)n, trig, hole ? 1u : 0u};
}

__global__ void __launch_bounds__(128) k_trace_borders(const uint8_t *__restrict__ bin, int w, int h, const uint32_t *__restrict__ jobs,
                                                       int job_cap, int32_t *__restrict__ counters, int min_px, int max_px,
                                                       uint32_t *__restrict__ pts, int pts_cap, ContourDesc *__restrict__ descs,
                                                       int desc_cap, int batch, uint32_t *__restrict__ long_jobs)
{
    const int f = blockIdx.y;
    int32_t *cnt = counters + f * APSE_COUNTERS;
    const int njobs = min(cnt[0], job_cap);
    const uint8_t *I = bin + (size_t)f * w * h;   // neighbour masks
    const uint32_t *J = jobs + (size_t)f * job_cap;
    uint32_t *P = pts + (size_t)f * pts_cap;
    ContourDesc *D = descs + (size_t)f * desc_cap;
    const int short_max = (w % 16 == 0 && w >= TW_W && h >= TW_H) ? min(max_px, TRACE_SHORT) : max_px;   // else: every border in this kernel
    for (int j = blockIdx.x * blockDim.x + threadIdx.x; j < njobs; j += gridDim.x * blockDim.x) {
        uint32_t e = J[j];
        bool hole = (e >> 31) != 0;
        uint32_t trig = e & 0x7fffffffu;
        int ty = trig / w, tx = trig - ty * w;
        int x0 = hole ? tx - 1 : tx, y0 = ty;
        int n = trace_border<false>(I, w, x0, y0, hole, short_max, nullptr);
        if (n > short_max) {
            if (short_max < max_px) {   // still open: a long border
                const int k = atomicAdd(&cnt[6], 1);
                if (k < TRACE_LONG_CAP) long_jobs[(size_t)f * TRACE_LONG_CAP + k] = e;
                else atomicExch(&cnt[3], APSE_ERR_CAPACITY);
            }
            continue;
        }
        if (n < min_px) continue;
        store_border(I, w, e, n, cnt, P, pts_cap, D, desc_cap, max_px);
    }
}

// lane 0 follows the border ONCE, writing the points to this warp's temporary strip.  The neighbour masks around the current
// position live in a per-warp shared-memory window (TW_W x TW_H bytes, loaded by the whole warp with 16-byte loads and re-centred
// whenever the walker leaves it), and the next direction comes from a 2 KB table indexed by (mask, incoming direction): a step is
// two shared-memory look-ups and a handful of integer instructions instead of a dependent global load.  Needs w % 16 == 0.
// Returns the length (> max_n: over the perimeter limit).
__device__ int trace_border_warp(const uint8_t *__restrict__ M, int w, int h, int x0, int y0, bool hole, int max_n, uint32_t *tmp,
                                 uint8_t *win /* [TW_H][TW_W] */, const uint8_t *next_dir /* [256][8] */)
{
    const int lane = threadIdx.x & 31;
    const int s0 = hole ? 0 : 4;
    unsigned m = M[(size_t)y0 * w + x0];
    int s = (s0 - 1 - (__ffs(rotr8(__brev(m) >> 24, (8 - s0) & 7)) - 1)) & 7;
    const int x1 = x0 + dir_dx(s), y1 = y0 + dir_dy(s);
    int cx = x0, cy = y0, n = 0;
    bool done = false;
    while (!done) {
        // re-centre the window on (cx, cy): lane = window row, four 16-byte loads per lane
        const int wx0 = min(max((cx - TW_W / 2) & ~15, 0), w - TW_W), wy0 = min(max(cy - TW_H / 2, 0), h - TW_H);
        {
            const uint4 *src = reinterpret_cast<const uint4 *>(M + (size_t)(wy0 + lane) * w + wx0);
            uint4 *dst = reinterpret_cast<uint4 *>(win + lane * TW_W);
#pragma unroll
            for (int k = 0; k < TW_W / 16; k++) dst[k] = __ldg(src + k);
        }
        __syncwarp();
        if (lane == 0) {
            int lx = cx - wx0, ly = cy - wy0;
            for (;;) {
                s = next_dir[m * 8 + s];                                   // next neighbour counter-clockwise from s + 1
                const int dx = dir_dx(s), dy = dir_dy(s);
                const int nx = cx + dx, ny = cy + dy;
                tmp[n] = (uint32_t)cx | ((uint32_t)cy << 16);
                n++;
                if (nx == x0 && ny == y0 && cx == x1 && cy == y1) { done = true; break; }
                if (n > max_n) { done = true; break; }
                cx = nx; cy = ny; lx += dx; ly += dy;
                s = (s + 4) & 7;
                if ((unsigned)lx >= (unsigned)TW_W || (unsigned)ly >= (unsigned)TW_H) { m = 0x100u; break; }   // left the window
                m = win[ly * TW_W + lx];
            }
        }
        done = __shfl_sync(0xffffffffu, done, 0);
        cx = __shfl_sync(0xffffffffu, cx, 0);
        cy = __shfl_sync(0xffffffffu, cy, 0);
        if (!done && lane == 0) m = M[(size_t)cy * w + cx];   // (the mask of the pixel the walker stands on, from the new window's centre)
        __syncwarp();
    }
    return __shfl_sync(0xffffffffu, n, 0);
}

__global__ void __launch_bounds__(128) k_trace_long(const uint8_t *__restrict__ bin, int w, int h, const uint32_t *__restrict__ long_jobs,
                                                    int32_t *__restrict__ counters, int min_px, int max_px, uint32_t *__restrict__ pts, int pts_cap,
                                                    ContourDesc *__restrict__ descs, int desc_cap, uint32_t *__restrict__ strips)
{
    __shared__ __align__(16) uint8_t s_win[4][TW_H * TW_W];
    __shared__ uint8_t s_next[256 * 8];
    // next direction for (neighbour mask m, incoming direction s): first neighbour counter-clockwise from s + 1
    for (int i = threadIdx.x; i < 256 * 8; i += blockDim.x) {
        const unsigned m = (unsigned)i >> 3;
        const int base = ((i & 7) + 1) & 7;
        s_next[i] = m ? (uint8_t)((base + __ffs(rotr8(m, base)) - 1) & 7) : 0;
    }
    __syncthreads();
    const int f = blockIdx.y, lane = threadIdx.x & 31;
    int32_t *cnt = counters + f * APSE_COUNTERS;
    const int njobs = min(cnt[6], TRACE_LONG_CAP);
    const uint8_t *I = bin + (size_t)f * w * h;
    uint32_t *P = pts + (size_t)f * pts_cap;
    ContourDesc *D = descs + (size_t)f * desc_cap;
    const int warps = blockDim.x >> 5;
    uint32_t *tmp = strips + ((size_t)(blockIdx.y * gridDim.x + blockIdx.x) * warps + (threadIdx.x >> 5)) * (size_t)(max_px + 2);
    for (int j = blockIdx.x * warps + (threadIdx.x >> 5); j < njobs; j += gridDim.x * warps) {
        const uint32_t e = long_jobs[(size_t)f * TRACE_LONG_CAP + j];
        const bool hole = (e >> 31) != 0;
        const uint32_t trig = e & 0x7fffffffu;
        const int ty = trig / w, tx = trig - ty * w;
        const int x0 = hole ? tx - 1 : tx, y0 = ty;
        const int n = trace_border_warp(I, w, h, x0, y0, hole, max_px, tmp, s_win[threadIdx.x >> 5], s_next);
#ifdef TRACE_DEBUG
        if (lane == 0 && (n > 3000)) printf("long border f=%d j=%d x0=%d y0=%d hole=%d n=%d njobs=%d\n", f, j, x0, y0, (int)hole, n, njobs);
#endif
        if (n < min_px || n > max_px) continue;
        int di = 0, off = 0;
        if (lane == 0) { di = atomicAdd(&cnt[1], 1); off = atomicAdd(&cnt[5], n); }
        di = __shfl_sync(0xffffffffu, di, 0); off = __shfl_sync(0xffffffffu, off, 0);
        if (di >= desc_cap || off + n > pts_cap) { if (lane == 0) atomicExch(&cnt[3], APSE_ERR_CAPACITY); continue; }
        __syncwarp();
        for (int i = lane; i < n; i += 32) P[off + i] = tmp[i];   // (lane 0's stores are visible to the warp after the barrier)
        if (lane == 0) D[di] = ContourDesc{(uint32_t)off, (uint32_t)n, trig, hole ? 1u : 0u};
        __syncwarp();
    }
}

// ---------------------------------------------------------------------------------------------------------
// C3: polygon approximation + quad filters, one warp per stored border
#define AQ_WARPS 8
#define AQ_STACK 96
#define AQ_MAXV 128

__device__ __forceinline__ int pt_x(uint32_t p) { return (int)(p & 0xffffu); }
__device__ __forceinline__ int pt_y(uint32_t p) { return (int)(p >> 16); }

// squared point-to-segment distance (FP64, the dependency's expression order)
__device__ __forceinline__ double seg_dist2(int ax, int ay, int bx, int by, int px_, int py_, double dx, double dy, double len2)
{
    double px = px_ - ax, py = py_ - ay;
    double proj = px * dx + py * dy;
    if (proj < 0) return px * px + py * py;
    if (proj > len2) { double qx = px_ - bx, qy = py_ - by; return qx * qx + qy * qy; }
    double cr = py * dx - px * dy;
    return cr * cr / len2;
}

struct ClassicArgs {
    const uint32_t *pts;
    int pts_cap;
    const ContourDesc *descs;
    int desc_cap;
    int32_t *counters;
    float *quads;
    float *refined;              // nullable: CORNER_REFINE_CONTOUR corners of every candidate, parallel to quads
    unsigned long long *quad_keys;
    int quad_cap;
    int w, h, window_index;
    double accuracy_rate, min_corner_rate;
};

// CORNER_REFINE_CONTOUR of one candidate (dependency: _refineCandidateLines, _interpolate2Dline, _getCrossPoint), one warp.
// The contour points are grouped by the corner they follow in contour order (points ahead of the first corner join the group
// that is open at the end), one least-squares line per group, refined corner = intersection of the two lines meeting at it.
// Arithmetic of cv2 4.13, bit for bit: exact sums (double), the 2 x 2 normal equations and their LU with partial pivoting in
// float32, Matx22f::solve's closed form in float32 (the CPU restatement of the same arithmetic is pinned to cv2 in tests/).  marks: >= 128 words of scratch.
#define RC_MAX_MARKS 60
__device__ void refine_candidate_lines(const uint32_t *__restrict__ src, int count, const float (&c)[8], float *__restrict__ out, uint32_t *marks)
{
    const int lane = threadIdx.x & 31;
    // positions where the contour passes through a corner, in contour order: (position << 2 | corner)
    int nm = 0;
    for (int base = 0; base < count; base += 32) {
        const int i = base + lane;
        int hit = -1;
        if (i < count) {
            const uint32_t p = src[i];
            const float x = (float)pt_x(p), y = (float)pt_y(p);
#pragma unroll
            for (int j = 0; j < 4; j++) if (c[2 * j] == x && c[2 * j + 1] == y) hit = j;
        }
        const unsigned m = __ballot_sync(0xffffffffu, hit >= 0);
        if (hit >= 0) {
            const int k = nm + __popc(m & ((1u << lane) - 1));
            if (k < RC_MAX_MARKS) marks[k] = ((uint32_t)i << 2) | (uint32_t)hit;
        }
        nm += __popc(m);
    }
    __syncwarp();
    int idx[4] = {-1, -1, -1, -1};
    const int nmk = min(nm, RC_MAX_MARKS);
    for (int k = 0; k < nmk; k++) idx[marks[k] & 3u] = (int)(marks[k] >> 2);   // last occurrence wins
    if (nm > RC_MAX_MARKS || idx[0] < 0 || idx[1] < 0 || idx[2] < 0 || idx[3] < 0) {   // (not seen on real contours) keep the corners
        if (lane < 8) out[lane] = c[lane];
        return;
    }
    const int last_group = (int)(marks[nmk - 1] & 3u);
    // per group: n, sum x, sum y, sum xx, sum yy, sum xy (exact in double), extents
    double S[4][6];
    int mn_x[4], mx_x[4], mn_y[4], mx_y[4];
#pragma unroll
    for (int g = 0; g < 4; g++) { for (int k = 0; k < 6; k++) S[g][k] = 0; mn_x[g] = mn_y[g] = INT32_MAX; mx_x[g] = mx_y[g] = INT32_MIN; }
    for (int i = lane; i < count; i += 32) {
        // group of point i: the corner of the last mark at or before i; ahead of the first mark: the group open at the end
        int g = last_group;
        for (int k = 0; k < nmk; k++) { if ((int)(marks[k] >> 2) <= i) g = (int)(marks[k] & 3u); else break; }
        const uint32_t p = src[i];
        const int xi = pt_x(p), yi = pt_y(p);
        const double x = xi, y = yi;
#pragma unroll
        for (int gg = 0; gg < 4; gg++)
            if (gg == g) {
                S[gg][0] += 1; S[gg][1] += x; S[gg][2] += y; S[gg][3] += x * x; S[gg][4] += y * y; S[gg][5] += x * y;
                mn_x[gg] = min(mn_x[gg], xi); mx_x[gg] = max(mx_x[gg], xi); mn_y[gg] = min(mn_y[gg], yi); mx_y[gg] = max(mx_y[gg], yi);
            }
    }
    float L[4][3];
#pragma unroll
    for (int g = 0; g < 4; g++) {
#pragma unroll
        for (int k = 0; k < 6; k++)
            for (int o = 16; o > 0; o >>= 1) S[g][k] += __shfl_xor_sync(0xffffffffu, S[g][k], o);
        mn_x[g] = __reduce_min_sync(0xffffffffu, mn_x[g]); mx_x[g] = __reduce_max_sync(0xffffffffu, mx_x[g]);
        mn_y[g] = __reduce_min_sync(0xffffffffu, mn_y[g]); mx_y[g] = __reduce_max_sync(0xffffffffu, mx_y[g]);
        const bool horiz = (float)mx_x[g] - (float)mn_x[g] > (float)mx_y[g] - (float)mn_y[g];
        float A00 = (float)(horiz ? S[g][3] : S[g][4]), A01 = (float)(horiz ? S[g][1] : S[g][2]), A10 = A01, A11 = (float)S[g][0];
        float B0 = (float)S[g][5], B1 = (float)(horiz ? S[g][2] : S[g][1]);
        if (fabsf(A10) > fabsf(A00)) { float t = A00; A00 = A10; A10 = t; t = A01; A01 = A11; A11 = t; t = B0; B0 = B1; B1 = t; }
        float x0 = 0.f, x1 = 0.f;
        if (!(fabsf(A00) < FLT_EPSILON)) {
            const float d = __fdiv_rn(-1.f, A00), alpha = __fmul_rn(A10, d);
            A11 = __fadd_rn(A11, __fmul_rn(alpha, A01));
            B1 = __fadd_rn(B1, __fmul_rn(alpha, B0));
            if (!(fabsf(A11) < FLT_EPSILON)) {
                x1 = __fdiv_rn(B1, A11);
                x0 = __fdiv_rn(__fsub_rn(B0, __fmul_rn(A01, x1)), A00);
            }
        }
        if (horiz) { L[g][0] = x0; L[g][1] = -1.f; L[g][2] = x1; }
        else { L[g][0] = -1.f; L[g][1] = x0; L[g][2] = x1; }
    }
    int inc = 1;
    if (idx[0] > idx[1] && idx[3] > idx[0]) inc = -1;
    if (idx[2] > idx[3] && idx[1] > idx[2]) inc = -1;
    if (lane < 4) {
        const int i = lane, j = inc < 0 ? (i + 1) & 3 : (i + 3) & 3;
        float a0, a1, a2, b0_, b1_, b2;
        // (register arrays indexed by a lane-dependent value: select explicitly)
        a0 = i == 0 ? L[0][0] : i == 1 ? L[1][0] : i == 2 ? L[2][0] : L[3][0];
        a1 = i == 0 ? L[0][1] : i == 1 ? L[1][1] : i == 2 ? L[2][1] : L[3][1];
        a2 = i == 0 ? L[0][2] : i == 1 ? L[1][2] : i == 2 ? L[2][2] : L[3][2];
        b0_ = j == 0 ? L[0][0] : j == 1 ? L[1][0] : j == 2 ? L[2][0] : L[3][0];
        b1_ = j == 0 ? L[0][1] : j == 1 ? L[1][1] : j == 2 ? L[2][1] : L[3][1];
        b2 = j == 0 ? L[0][2] : j == 1 ? L[1][2] : j == 2 ? L[2][2] : L[3][2];
        const float r0 = -a2, r1 = -b2;
        const float det = __fsub_rn(__fmul_rn(a0, b1_), __fmul_rn(a1, b0_));
        float ox = 0.f, oy = 0.f;   // Matx::solve fails on a singular system: the zero vector comes back
        if (det != 0.f) {
            const float dinv = __fdiv_rn(1.f, det);
            ox = __fmul_rn(__fsub_rn(__fmul_rn(r0, b1_), __fmul_rn(r1, a1)), dinv);
            oy = __fmul_rn(__fsub_rn(__fmul_rn(r1, a0), __fmul_rn(r0, b0_)), dinv);
        }
        out[2 * i] = ox; out[2 * i + 1] = oy;
    }
}

// after the decode stage: every accepted marker takes the refined corners of its candidate -- the first candidate in the
// dependency's order with the same corners up to the rotation the identification applied.  One CTA per frame.
__global__ void __launch_bounds__(256) k_contour_refine_out(const float *__restrict__ quads, const float *__restrict__ refined,
                                                            const uint32_t *__restrict__ quad_order, const int32_t *__restrict__ counters, int quad_cap,
                                                            apse_detections out)
{
    __shared__ unsigned s_best;
    const int f = blockIdx.x;
    const int nq = min(counters[f * APSE_COUNTERS + 2], quad_cap), nm = min(out.n_markers[f], out.max_markers);
    const float *Q = quads + (size_t)f * quad_cap * 8, *R = refined + (size_t)f * quad_cap * 8;
    const uint32_t *O = quad_order + (size_t)f * quad_cap;
    for (int m = 0; m < nm; m++) {
        float *oc = out.corners + ((size_t)f * out.max_markers + m) * 8;
        if (threadIdx.x == 0) s_best = 0xffffffffu;
        __syncthreads();
        float c[8];
        for (int k = 0; k < 8; k++) c[k] = oc[k];
        for (int qi = threadIdx.x; qi < nq; qi += blockDim.x) {
            const float *q = Q + 8 * qi;
            for (int sh = 0; sh < 4; sh++) {
                bool same = true;
                for (int k = 0; k < 4 && same; k++) { const int s2 = (k + sh) & 3; same = q[2 * s2] == c[2 * k] && q[2 * s2 + 1] == c[2 * k + 1]; }
                if (same) { atomicMin(&s_best, (O[qi] << 14) | ((unsigned)qi << 2) | (unsigned)sh); break; }
            }
        }
        __syncthreads();
        const unsigned best = s_best;
        __syncthreads();
        if (best != 0xffffffffu && threadIdx.x < 4) {
            const int qi = (int)((best >> 2) & 0xfffu), sh = (int)(best & 3u), k = threadIdx.x, s2 = (k + sh) & 3;
            oc[2 * k] = R[8 * qi + 2 * s2];
            oc[2 * k + 1] = R[8 * qi + 2 * s2 + 1];
        }
        __syncthreads();
    }
}

__global__ void __launch_bounds__(AQ_WARPS * 32) k_approx_quads(ClassicArgs A)
{
    __shared__ int2 s_stack[AQ_WARPS][AQ_STACK];
    __shared__ uint32_t s_out[AQ_WARPS][AQ_MAXV];
    const int f = blockIdx.y, lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
    int32_t *cnt = A.counters + f * APSE_COUNTERS;
    const int ndesc = min(cnt[1], A.desc_cap);
    const uint32_t *P = A.pts + (size_t)f * A.pts_cap;
    const ContourDesc *D = A.descs + (size_t)f * A.desc_cap;
    int2 *stack = s_stack[wid];
    uint32_t *outv = s_out[wid];
    for (int ci = blockIdx.x * AQ_WARPS + wid; ci < ndesc; ci += gridDim.x * AQ_WARPS) {
        const ContourDesc cd = D[ci];
        const uint32_t *src = P + cd.offset;
        const int count = (int)cd.count;
        const double eps = (double)count * A.accuracy_rate, eps2 = eps * eps;
        // ---- farthest point from the current start, three rounds (first maximum wins)
        int pos = 0, right_start = 0, start_idx = 0;
        bool le_eps = false;
        for (int it = 0; it < 3; it++) {
            pos = (pos + right_start) % count;
            start_idx = pos;
            const uint32_t sp = src[start_idx];
            const int sx = pt_x(sp), sy = pt_y(sp);
            int best = 0, best_j = 0;   // max_dist starts at 0: j is only taken on a strictly larger distance
            for (int j = 1 + lane; j < count; j += 32) {
                int q = start_idx + j;
                if (q >= count) q -= count;
                const uint32_t pp = src[q];
                const int dx = pt_x(pp) - sx, dy = pt_y(pp) - sy, d = dx * dx + dy * dy;
                if (d > best) { best = d; best_j = j; }
            }
            for (int o = 16; o > 0; o >>= 1) {
                int ob = __shfl_xor_sync(0xffffffffu, best, o), oj = __shfl_xor_sync(0xffffffffu, best_j, o);
                if (ob > best || (ob == best && ob > 0 && oj < best_j)) { best = ob; best_j = oj; }
            }
            if (best > 0) right_start = best_j;
            le_eps = (double)best <= eps2;
            pos = start_idx;   // the read position is back at the start point after a full round
        }
        int nout = 0, top = 0;
        bool overflow = false;
        if (!le_eps) {
            int slice_start = pos % count;
            int slice_end = (right_start + slice_start) % count;
            // right slice pushed first, left slice processed first
            if (lane == 0) { stack[0] = make_int2(slice_end, slice_start); stack[1] = make_int2(slice_start, slice_end); }
            top = 2;
        } else {
            if (lane == 0) outv[0] = src[start_idx];
            nout = 1;
        }
        __syncwarp();
        while (top > 0) {
            const int2 sl = stack[--top];
            __syncwarp();
            const uint32_t ep = src[sl.y], sp = src[sl.x];
            const int ex = pt_x(ep), ey = pt_y(ep), sx = pt_x(sp), sy = pt_y(sp);
            int first = sl.x + 1;
            if (first >= count) first = 0;
            bool ok;
            int split = 0;
            if (first != sl.y) {
                const double dx = ex - sx, dy = ey - sy, len2 = dx * dx + dy * dy;
                int m = sl.y - first;
                if (m < 0) m += count;            // interior points first .. end-1 (cyclic)
                double best = 0;
                int best_k = -1;
                for (int k = lane; k < m; k += 32) {
                    int q = first + k;
                    if (q >= count) q -= count;
                    const uint32_t pp = src[q];
                    double d = seg_dist2(sx, sy, ex, ey, pt_x(pp), pt_y(pp), dx, dy, len2);
                    if (d > best) { best = d; best_k = k; }
                }
                for (int o = 16; o > 0; o >>= 1) {
                    double ob = __shfl_xor_sync(0xffffffffu, best, o);
                    int ok_ = __shfl_xor_sync(0xffffffffu, best_k, o);
                    if (ob > best || (ob == best && ok_ >= 0 && (best_k < 0 || ok_ < best_k))) { best = ob; best_k = ok_; }
                }
                ok = best <= eps2;
                if (!ok) { split = first + best_k; if (split >= count) split -= count; }
            } else {
                ok = true;
            }
            if (ok) {
                if (nout < AQ_MAXV) { if (lane == 0) outv[nout] = sp; } else overflow = true;
                nout++;
            } else {
                if (top + 2 <= AQ_STACK) {
                    if (lane == 0) { stack[top] = make_int2(split, sl.y); stack[top + 1] = make_int2(sl.x, split); }
                    top += 2;
                } else { overflow = true; top = 0; }
            }
            __syncwarp();
        }
        if (overflow) { if (lane == 0) atomicExch(&cnt[3], APSE_ERR_CAPACITY); continue; }
        // ---- clean-up pass + filters: sequential, lane 0
        int emitted = -1;             // index of the quad this contour produced (lane 0)
        float ec[8] = {0, 0, 0, 0, 0, 0, 0, 0};
        if (lane == 0) {
            int cntv = nout, new_count = nout;
            if (cntv >= 3) {
                int rp = cntv - 1, wpos;
                auto rd = [&](int &x, int &y) { uint32_t v = outv[rp]; x = pt_x(v); y = pt_y(v); if (++rp >= cntv) rp = 0; };
                int sx, sy, px, py, ex, ey;
                rd(sx, sy);
                wpos = rp;
                rd(px, py);
                for (int i = 0; i < cntv && new_count > 2; i++) {
                    rd(ex, ey);
                    double dx = ex - sx, dy = ey - sy;
                    double dist = fabs((double)(px - sx) * dy - (double)(py - sy) * dx);
                    double sip = (double)(px - sx) * (ex - px) + (double)(py - sy) * (ey - py);
                    if (dist * dist <= 0.5 * eps2 * (dx * dx + dy * dy) && dx != 0 && dy != 0 && sip >= 0) {
                        new_count--;
                        outv[wpos] = (uint32_t)ex | ((uint32_t)ey << 16);
                        sx = ex; sy = ey;
                        if (++wpos >= cntv) wpos = 0;
                        rd(px, py);
                        i++;
                        continue;
                    }
                    outv[wpos] = (uint32_t)px | ((uint32_t)py << 16);
                    sx = px; sy = py;
                    if (++wpos >= cntv) wpos = 0;
                    px = ex; py = ey;
                }
            }
            if (new_count == 4) {
                int qx[4], qy[4];
                for (int k = 0; k < 4; k++) { qx[k] = pt_x(outv[k]); qy[k] = pt_y(outv[k]); }
                // convexity (collinear / repeated vertices reject)
                bool convex = true;
                {
                    int prx = qx[2], pry = qy[2], cux = qx[3], cuy = qy[3];
                    long long dx0 = cux - prx, dy0 = cuy - pry;
                    int orient = 0;
                    for (int i = 0; i < 4; i++) {
                        prx = cux; pry = cuy; cux = qx[i]; cuy = qy[i];
                        long long dx = cux - prx, dy = cuy - pry;
                        long long dxdy0 = dx * dy0, dydx0 = dy * dx0;
                        orient |= (dydx0 > dxdy0) ? 1 : ((dydx0 < dxdy0) ? 2 : 3);
                        if (orient == 3) { convex = false; break; }
                        dx0 = dx; dy0 = dy;
                    }
                }
                if (convex) {
                    const int mx = max(A.w, A.h);
                    double min_d2 = (double)mx * mx;
                    for (int j = 0; j < 4; j++) {
                        int k = (j + 1) & 3;
                        double d = (double)(qx[j] - qx[k]) * (qx[j] - qx[k]) + (double)(qy[j] - qy[k]) * (qy[j] - qy[k]);
                        min_d2 = fmin(min_d2, d);
                    }
                    double min_corner = (double)count * A.min_corner_rate;
                    if (!(min_d2 < min_corner * min_corner)) {
                        int qi = atomicAdd(&cnt[2], 1);
                        if (qi < A.quad_cap) {
                            float *q = A.quads + ((size_t)f * A.quad_cap + qi) * 8;
                            float c[8];
                            for (int k = 0; k < 4; k++) { c[2 * k] = (float)qx[k]; c[2 * k + 1] = (float)qy[k]; }
                            double dx1 = c[2] - c[0], dy1 = c[3] - c[1], dx2 = c[4] - c[0], dy2 = c[5] - c[1];
                            if (dx1 * dy2 - dy1 * dx2 < 0.0) { float tx = c[2], ty = c[3]; c[2] = c[6]; c[3] = c[7]; c[6] = tx; c[7] = ty; }
                            for (int k = 0; k < 8; k++) { q[k] = c[k]; ec[k] = c[k]; }
                            emitted = qi;
                            // candidate order of the dependency: window ascending, then descending trigger pixel
                            A.quad_keys[(size_t)f * A.quad_cap + qi] =
                                ((unsigned long long)A.window_index << 32) | (unsigned long long)(0xffffffffu - cd.trigger);
                        } else {
                            atomicExch(&cnt[3], APSE_ERR_CAPACITY);
                        }
                    }
                }
            }
        }
        __syncwarp();
        // ---- CORNER_REFINE_CONTOUR: refined corners of this candidate from its contour (whole warp)
        if (A.refined) {
            emitted = __shfl_sync(0xffffffffu, emitted, 0);
            if (emitted >= 0) {
#pragma unroll
                for (int k = 0; k < 8; k++) ec[k] = __shfl_sync(0xffffffffu, ec[k], 0);
                refine_candidate_lines(src, count, ec, A.refined + ((size_t)f * A.quad_cap + emitted) * 8, s_out[wid]);
            }
        }
        __syncwarp();
    }
}

// rank of every quad of a frame in key order -> quad_order (consumed by the decode stage).  Keys are unique within a frame
// (classic: window and trigger pixel; APRILTAG: the cluster's component pair), so the ranks are a permutation.
__global__ void k_rank_quads(const unsigned long long *__restrict__ keys, const int32_t *__restrict__ counters, int quad_cap,
                             uint32_t *__restrict__ quad_order)
{
    const int f = blockIdx.y;
    const int n = min(counters[f * APSE_COUNTERS + 2], quad_cap);
    const unsigned long long *K = keys + (size_t)f * quad_cap;
    for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) {
        unsigned long long k = K[i];
        int r = 0;
        for (int j = 0; j < n; j++) r += K[j] < k;
        quad_order[(size_t)f * quad_cap + i] = (uint32_t)r;
    }
}

// ---------------------------------------------------------------------------------------------------------
// C4: cornerSubPix on the accepted markers (thread per corner)
#define SP_MAXWIN 8
__device__ __forceinline__ float subpix_sample(const uint8_t *im, int w, int h, int x0, int y0, bool inside, float a11, float a12,
                                               float a21, float a22)
{
    int x1 = x0 + 1, y1 = y0 + 1;
    if (!inside) {
        x0 = min(max(x0, 0), w - 1); x1 = min(max(x1, 0), w - 1);
        y0 = min(max(y0, 0), h - 1); y1 = min(max(y1, 0), h - 1);
    }
    // ((p00 a11 + p01 a12) + p10 a21) + p11 a22, float32, no contraction
    float v = __fmul_rn((float)im[(size_t)y0 * w + x0], a11);
    v = __fadd_rn(v, __fmul_rn((float)im[(size_t)y0 * w + x1], a12));
    v = __fadd_rn(v, __fmul_rn((float)im[(size_t)y1 * w + x0], a21));
    v = __fadd_rn(v, __fmul_rn((float)im[(size_t)y1 * w + x1], a22));
    return v;
}

__global__ void __launch_bounds__(64) k_corner_subpix(const uint8_t *__restrict__ gray, int w, int h, float *__restrict__ corners,
                                                     const int32_t *__restrict__ n_markers, int batch, int max_markers, int marker_cells,
                                                     float rel_win, int max_win, int max_iter, double eps)
{
    const int t = blockIdx.x * blockDim.x + threadIdx.x;
    const bool in_range = t < batch * max_markers * 4;
    const int f = in_range ? t / (max_markers * 4) : 0, r = t - f * max_markers * 4, m = r >> 2, k = r & 3;
    const bool active = in_range && m < n_markers[f];
    const uint8_t *im = gray + (size_t)f * w * h;
    float *c = corners + ((size_t)f * max_markers + m) * 8;
    // the four corners of a marker are refined by four lanes of one warp: all of them read the unrefined corners
    // (window size) before any of them writes its result
    float c0[8];
    for (int i = 0; i < 8; i++) c0[i] = active ? c[i] : 0.f;
    __syncwarp();
    if (!active) return;
    // window from the marker's average module size (float32, the dependency's order)
    float side = 0.f;
    for (int i = 0; i < 4; i++) {
        int j = (i + 1) & 3;
        float dx = c0[2 * i] - c0[2 * j], dy = c0[2 * i + 1] - c0[2 * j + 1];
        side = __fadd_rn(side, sqrtf(__fadd_rn(__fmul_rn(dx, dx), __fmul_rn(dy, dy))));
    }
    float module = side / (4.f * (float)marker_cells);
    int win = max(1, __float2int_rn(__fmul_rn(rel_win, module)));
    win = min(min(win, max_win), SP_MAXWIN);
    const int ww = 2 * win + 1, pw = ww + 2;
    float mk[2 * SP_MAXWIN + 1];
    for (int i = 0; i < ww; i++) {
        float x = (float)(i - win) / (float)win;
        mk[i] = (float)exp((double)(-__fmul_rn(x, x)));
    }
    const float ctx = c0[2 * k], cty = c0[2 * k + 1];
    float cix = ctx, ciy = cty;
    const double eps2 = eps * eps;
    int iter = 0;
    double err = 0;
    do {
        float fx = cix - (float)(pw - 1) * 0.5f, fy = ciy - (float)(pw - 1) * 0.5f;
        int ipx = (int)floorf(fx), ipy = (int)floorf(fy);
        float a = fx - (float)ipx, b = fy - (float)ipy;
        float a11 = __fmul_rn(1.f - a, 1.f - b), a12 = __fmul_rn(a, 1.f - b), a21 = __fmul_rn(1.f - a, b), a22 = __fmul_rn(a, b);
        bool inside = ipx >= 0 && ipx + pw < w && ipy >= 0 && ipy + pw < h;
        double sa = 0, sb = 0, sc = 0, bb1 = 0, bb2 = 0;
        for (int i = 0; i < ww; i++) {
            double py = i - win;
            // gradient taps of patch row i+1: keep a sliding window of three patch rows' samples per column
            for (int j = 0; j < ww; j++) {
                float l = subpix_sample(im, w, h, ipx + j, ipy + i + 1, inside, a11, a12, a21, a22);
                float rr = subpix_sample(im, w, h, ipx + j + 2, ipy + i + 1, inside, a11, a12, a21, a22);
                float u = subpix_sample(im, w, h, ipx + j + 1, ipy + i, inside, a11, a12, a21, a22);
                float d = subpix_sample(im, w, h, ipx + j + 1, ipy + i + 2, inside, a11, a12, a21, a22);
                double mm = __fmul_rn(mk[j], mk[i]);
                double tgx = __fsub_rn(rr, l), tgy = __fsub_rn(d, u);
                double gxx = tgx * tgx * mm, gxy = tgx * tgy * mm, gyy = tgy * tgy * mm;
                double px = j - win;
                sa += gxx; sb += gxy; sc += gyy;
                bb1 += gxx * px + gxy * py;
                bb2 += gxy * px + gyy * py;
            }
        }
        double det = sa * sc - sb * sb;
        if (fabs(det) <= DBL_EPSILON * DBL_EPSILON) break;
        double scale = 1.0 / det;
        float nx = (float)(cix + sc * scale * bb1 - sb * scale * bb2);
        float ny = (float)(ciy - sb * scale * bb1 + sa * scale * bb2);
        err = (double)(nx - cix) * (nx - cix) + (double)(ny - ciy) * (ny - ciy);
        cix = nx; ciy = ny;
        if (cix < 0 || cix >= w || ciy < 0 || ciy >= h) break;
    } while (++iter < max_iter && err > eps2);
    if (fabsf(cix - ctx) > win || fabsf(ciy - cty) > win) { cix = ctx; ciy = cty; }
    c[2 * k] = cix;
    c[2 * k + 1] = ciy;
}

// ---------------------------------------------------------------------------------------------------------
// host side
int apse_ccl_binary(apse_ctx *ctx, const uint8_t *bin, int w, int h, int batch, cudaStream_t st);   // detect_apriltag.cu

int apse_adaptive_threshold_impl(apse_ctx *ctx, const uint8_t *gray, int w, int h, int batch, int win, double c, uint8_t *out, cudaStream_t st)
{
    if (win % 2 == 0) win++;
    AtWindows W;
    W.n = 1; W.win[0] = win;
    return launch_adaptive(ctx, gray, w, h, batch, W, (int)floor(c), out, 0, st);
}

int apse_classic_quads(apse_ctx *ctx, const uint8_t *gray, int w, int h, int batch, cudaStream_t st)
{
    const apse_params &p = ctx->params;
    if (w > ctx->max_w || h > ctx->max_h || batch > ctx->max_batch)
        CTX_FAIL(ctx, APSE_ERR_INVALID_ARG, "detect: frame %dx%d x%d exceeds the context capacity", w, h, batch);
    if (w < 8 || h < 8 || w > 32767 || h > 32767) CTX_FAIL(ctx, APSE_ERR_INVALID_ARG, "detect: unsupported image size");
    const int n_scales = (p.adaptiveThreshWinSizeMax - p.adaptiveThreshWinSizeMin) / p.adaptiveThreshWinSizeStep + 1;
    const int mx = w > h ? w : h;
    const int min_px = (int)(unsigned)(p.minMarkerPerimeterRate * mx);
    long long max_px_ll = (long long)(p.maxMarkerPerimeterRate * mx);
    const int max_px = (int)(max_px_ll > 0x3fffffff ? 0x3fffffff : max_px_ll);
    const int idelta = (int)floor(p.adaptiveThreshConstant);
    // scratch shared with the APRILTAG path: thresh = binary image, labels, points = border jobs, sorted_pts = border
    // points, clusters = border descriptors; counters: [0] jobs, [1] borders kept, [2] quads, [3] status, [5] points
    const int job_cap = APSE_MAX_POINTS * 4, pts_cap = APSE_MAX_POINTS * 2, desc_cap = APSE_MAX_CLUSTERS;
    CUDA_TRY(ctx, cudaMemsetAsync(ctx->counters, 0, (size_t)batch * APSE_COUNTERS * sizeof(int32_t), st));
    if (!ctx->nbr_mask) CUDA_TRY(ctx, cudaMalloc((void **)&ctx->nbr_mask, (size_t)ctx->max_batch * ctx->max_w * ctx->max_h));
    if (!ctx->long_jobs) CUDA_TRY(ctx, cudaMalloc((void **)&ctx->long_jobs, (size_t)ctx->max_batch * TRACE_LONG_CAP * sizeof(uint32_t)));
    if (max_px > (1 << 18)) CTX_FAIL(ctx, APSE_ERR_UNSUPPORTED, "detect: maxMarkerPerimeterRate allows borders of %d points, more than the supported %d", max_px, 1 << 18);
    {   // one temporary strip of max_px + 2 points per resident warp of k_trace_long
        const size_t want = (size_t)ctx->max_batch * ctx->sm_count * 4 * (size_t)(max_px + 2) * sizeof(uint32_t);
        if (ctx->trace_strips_bytes < want) {
            CUDA_TRY(ctx, cudaStreamSynchronize(st));
            cudaFree(ctx->trace_strips);
            ctx->trace_strips = nullptr; ctx->trace_strips_bytes = 0;
            CUDA_TRY(ctx, cudaMalloc((void **)&ctx->trace_strips, want));
            ctx->trace_strips_bytes = want;
        }
    }
    // all binaries of the sweep from one staged gray tile (north_star stage 2): bin_all[window][batch][h][w]
    if (n_scales > AT_MAX_WINDOWS) CTX_FAIL(ctx, APSE_ERR_UNSUPPORTED, "detect: %d threshold windows exceed the supported %d", n_scales, AT_MAX_WINDOWS);
    const size_t win_stride = (size_t)batch * w * h;
    if (ctx->bin_all_bytes < (size_t)n_scales * win_stride) {
        CUDA_TRY(ctx, cudaStreamSynchronize(st));
        cudaFree(ctx->bin_all);
        ctx->bin_all = nullptr; ctx->bin_all_bytes = 0;
        const size_t want = (size_t)n_scales * (size_t)ctx->max_batch * ctx->max_w * ctx->max_h;
        CUDA_TRY(ctx, cudaMalloc((void **)&ctx->bin_all, want));
        ctx->bin_all_bytes = want;
    }
    {
        AtWindows W;
        W.n = n_scales;
        for (int s = 0; s < n_scales; s++) { int win = p.adaptiveThreshWinSizeMin + s * p.adaptiveThreshWinSizeStep; W.win[s] = win % 2 == 0 ? win + 1 : win; }
        int rc = launch_adaptive(ctx, gray, w, h, batch, W, idelta, ctx->bin_all, win_stride, st);
        if (rc) return rc;
    }
    for (int s = 0; s < n_scales; s++) {
        const uint8_t *bin = ctx->bin_all + (size_t)s * win_stride;
        int rc = apse_ccl_binary(ctx, bin, w, h, batch, st);
        if (rc) return rc;
        KLAUNCH(ctx, KID_BORDER_JOBS, st, k_mark_outside<<<div_up(2 * (w + h) * batch, 256), 256, 0, st>>>(bin, w, h, ctx->labels, batch));
        // per window: reset the job / border / point counters, keep quads and status
        KLAUNCH(ctx, KID_BORDER_JOBS, st, k_border_jobs<<<dim3(ctx->sm_count * 2, batch), 256, 0, st>>>(bin, w, h, ctx->labels, reinterpret_cast<uint32_t *>(ctx->points), job_cap, ctx->counters, ctx->nbr_mask));
        KLAUNCH(ctx, KID_TRACE, st, k_trace_borders<<<dim3(ctx->sm_count, batch), 128, 0, st>>>(ctx->nbr_mask, w, h, reinterpret_cast<uint32_t *>(ctx->points), job_cap, ctx->counters, min_px,
                                                                                max_px, reinterpret_cast<uint32_t *>(ctx->sorted_pts), pts_cap,
                                                                                reinterpret_cast<ContourDesc *>(ctx->clusters), desc_cap, batch, ctx->long_jobs));
        KLAUNCH(ctx, KID_TRACE, st, k_trace_long<<<dim3(ctx->sm_count, batch), 128, 0, st>>>(ctx->nbr_mask, w, h, ctx->long_jobs, ctx->counters, min_px, max_px,
                                                                             reinterpret_cast<uint32_t *>(ctx->sorted_pts), pts_cap,
                                                                             reinterpret_cast<ContourDesc *>(ctx->clusters), desc_cap, ctx->trace_strips));
        ClassicArgs A;
        A.pts = reinterpret_cast<uint32_t *>(ctx->sorted_pts); A.pts_cap = pts_cap;
        A.descs = reinterpret_cast<ContourDesc *>(ctx->clusters); A.desc_cap = desc_cap;
        A.counters = ctx->counters; A.quads = ctx->quads; A.quad_keys = ctx->quad_keys; A.quad_cap = APSE_MAX_QUADS;
        A.refined = nullptr;
        if (p.cornerRefinementMethod == 2) {   // CORNER_REFINE_CONTOUR: the line fits need the contour, which only lives in this loop
            if (!ctx->quads_refined) CUDA_TRY(ctx, cudaMalloc((void **)&ctx->quads_refined, (size_t)ctx->max_batch * APSE_MAX_QUADS * 8 * sizeof(float)));
            A.refined = ctx->quads_refined;
        }
        A.w = w; A.h = h; A.window_index = s;
        A.accuracy_rate = p.polygonalApproxAccuracyRate; A.min_corner_rate = p.minCornerDistanceRate;
        KLAUNCH(ctx, KID_APPROX, st, k_approx_quads<<<dim3(ctx->sm_count, batch), AQ_WARPS * 32, 0, st>>>(A));
        // counters [0] (jobs), [1] (borders), [5] (points) restart for the next window
        CUDA_TRY(ctx, cudaMemset2DAsync(ctx->counters, APSE_COUNTERS * sizeof(int32_t), 0, 2 * sizeof(int32_t), batch, st));
        CUDA_TRY(ctx, cudaMemset2DAsync(ctx->counters + 5, APSE_COUNTERS * sizeof(int32_t), 0, 2 * sizeof(int32_t), batch, st));   // [5] points, [6] long borders
    }
    return apse_rank_quads(ctx, batch, st);
}

// both candidate paths: the decode stage breaks perimeter ties by this rank, so it has to be the dependency's candidate order
int apse_rank_quads(apse_ctx *ctx, int batch, cudaStream_t st)
{
    const int kid = ctx->params.cornerRefinementMethod == 3 ? KID_FIT_QUADS : KID_APPROX;   // timed with the stage that made the quads
    KLAUNCH(ctx, kid, st, k_rank_quads<<<dim3(8, batch), 256, 0, st>>>(ctx->quad_keys, ctx->counters, APSE_MAX_QUADS, ctx->quad_order));
    return APSE_OK;
}

int apse_contour_refine(apse_ctx *ctx, int batch, apse_detections *out, cudaStream_t st)
{
    if (!ctx->quads_refined) CTX_FAIL(ctx, APSE_ERR_NOT_CONFIGURED, "detect: no refined candidates (CORNER_REFINE_CONTOUR)");
    KLAUNCH(ctx, KID_SUBPIX, st, k_contour_refine_out<<<batch, 256, 0, st>>>(ctx->quads, ctx->quads_refined, ctx->quad_order, ctx->counters, APSE_MAX_QUADS, *out));
    return APSE_OK;
}

int apse_corner_subpix(apse_ctx *ctx, const uint8_t *gray, int w, int h, int batch, apse_detections *out, cudaStream_t st)
{
    const apse_params &p = ctx->params;
    if (p.cornerRefinementWinSize > SP_MAXWIN)
        CTX_FAIL(ctx, APSE_ERR_UNSUPPORTED, "detect: cornerRefinementWinSize %d exceeds the supported %d", p.cornerRefinementWinSize, SP_MAXWIN);
    if (p.cornerRefinementWinSize < 1 || p.cornerRefinementMaxIterations < 1 || p.cornerRefinementMinAccuracy <= 0)
        CTX_FAIL(ctx, APSE_ERR_INVALID_ARG, "detect: cornerRefinement{WinSize,MaxIterations,MinAccuracy} must be positive");
    const int total = batch * out->max_markers * 4;
    KLAUNCH(ctx, KID_SUBPIX, st, k_corner_subpix<<<div_up(total, 64), 64, 0, st>>>(gray, w, h, out->corners, out->n_markers, batch, out->max_markers,
                                                                        ctx->marker_size + 2 * p.markerBorderBits, p.relativeCornerRefinmentWinSize,
                                                                        p.cornerRefinementWinSize, p.cornerRefinementMaxIterations,
                                                                        p.cornerRefinementMinAccuracy));
    return APSE_OK;
}
