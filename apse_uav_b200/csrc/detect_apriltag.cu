// detect_apriltag.cu -- candidate stage of aruco.detectMarkers in CORNER_REFINE_APRILTAG mode
// (aruco_detect.py:266-267; SURVEY.md section 8 rows a6.A1-a6.A4), batched over frames, sm_100a.
//
//   K2  k_tile_minmax / k_threshold       4x4-tile min/max, 3x3 tile dilation, ternary {0,127,255} image
//   K3  k_ccl_local / merge / flatten     union-find components (white 8-conn, black 4-conn, 127 skipped);
//                                         block-local union-find in shared memory + boundary merge
//   K4  k_emit_points / k_cluster_scan / k_scatter_points
//                                         black/white boundary points grouped by component pair through a
//                                         per-frame hash table (counting sort by cluster, no global sort)
//   K5  k_fit_quads                       persistent kernel, one CTA per cluster: theta sort, dedup, FP64
//                                         prefix moments, error curve, maxima, 4-subset search, corners
//
// Parity notes: this file is compiled with -fmad=false.  All FP64/FP32 expressions are written in the
// evaluation order of the dependency (OpenCV's apriltag_quad_thresh) so that results are bit-identical:
// fastAtan2 polynomial, sequential (not tree) prefix sums of the moments, and cosf/sinf evaluated with the
// same double-precision polynomial the host libm uses.
#include "common.cuh"
#include <math.h>
#include <float.h>
#include <stdlib.h>

#define FQ_THREADS 128
#define MAXIMA_CAP 16  // aprilTagMaxNmaxima supported up to this value

// ---------------------------------------------------------------------------------------------------------
// K2: threshold
__global__ void k_tile_minmax(const uint8_t *__restrict__ gray, int w, int h, int tw, int th, uint16_t *__restrict__ tmm)
{
    int tx = blockIdx.x * blockDim.x + threadIdx.x, ty = blockIdx.y * blockDim.y + threadIdx.y, f = blockIdx.z;
    if (tx >= tw || ty >= th) return;
    const uint8_t *g = gray + (size_t)f * w * h;
    unsigned mn = 255, mx = 0;
    if ((w & 3) == 0 && (reinterpret_cast<uintptr_t>(gray) & 3) == 0) {   // 32-bit loads: every row 4-byte aligned
#pragma unroll
        for (int dy = 0; dy < 4; dy++) {
            uint32_t v = __ldg(reinterpret_cast<const uint32_t *>(g + (size_t)(ty * 4 + dy) * w + tx * 4));
            unsigned a = v & 255, b = (v >> 8) & 255, c = (v >> 16) & 255, d = v >> 24;
            mn = min(mn, min(min(a, b), min(c, d)));
            mx = max(mx, max(max(a, b), max(c, d)));
        }
    } else {
        for (int dy = 0; dy < 4; dy++)
            for (int dx = 0; dx < 4; dx++) {
                unsigned v = g[(size_t)(ty * 4 + dy) * w + tx * 4 + dx];
                mn = min(mn, v);
                mx = max(mx, v);
            }
    }
    tmm[(size_t)f * tw * th + (size_t)ty * tw + tx] = (uint16_t)(mn | (mx << 8));
}

__device__ __forceinline__ void dilated_minmax(const uint16_t *tmm, int tw, int th, int tx, int ty, int &mn, int &mx)
{
    mn = 255; mx = 0;
    for (int dy = -1; dy <= 1; dy++) {
        int yy = ty + dy;
        if (yy < 0 || yy >= th) continue;
        for (int dx = -1; dx <= 1; dx++) {
            int xx = tx + dx;
            if (xx < 0 || xx >= tw) continue;
            int v = __ldg(tmm + (size_t)yy * tw + xx);
            mn = min(mn, v & 255);
            mx = max(mx, v >> 8);
        }
    }
}

// CCL tiles (CCL_TW x CCL_TH px) that contain at least one non-127 pixel are flagged here and compacted into a work
// list, so that the component / boundary kernels only ever touch the ~1-20 % of the image that has contrast.
#define CCL_TW 32
#define CCL_TH 16
// ---- active-tile list ("A-list") -------------------------------------------------------------------------------
// Everything after the threshold decision works on the 4x4 tiles that are not low-contrast (1 % of a sparse frame,
// ~16 % of a dense one): k_threshold_scan appends them to a list, and the pixel work of the threshold itself, the reset
// of the ternary image before the next batch and the search for black/white crossings run over that list with full
// warps instead of over whole 32x16 CCL tiles in which four pixels out of five are background.
// Entry: tx | ty << 13 | frame << 26 (frames per launch <= 64, tile coordinates < 8192); alist_thr[i] = threshold.
// (ATILE / ATILE_TX / ATILE_TY / ATILE_F: common.cuh)

// One thread = 8 consecutive tiles of a tile row (one 128-bit load of the extrema per tile row when the row stride
// allows it) plus the two outer columns: 3x3 dilation of the tile extrema in registers; high-contrast tiles are
// appended to the A-list (one atomic per warp) and flag their CCL tile.  No pixel is touched here.
#define THR_TPT 8
__global__ void __launch_bounds__(128) k_threshold_scan(int w, int h, int tw, int th, const uint16_t *__restrict__ tmm, int min_wb_diff,
                                                        uint32_t *__restrict__ alist, uint8_t *__restrict__ alist_thr,
                                                        int *__restrict__ acount, int acap,
                                                        uint8_t *__restrict__ tile_active, int ctw, int cth)
{
    const int groups = (tw + THR_TPT - 1) / THR_TPT;
    const int gi = blockIdx.x * blockDim.x + threadIdx.x, ty = blockIdx.y, f = blockIdx.z, lane = threadIdx.x & 31;
    const int tx0 = gi * THR_TPT;
    const uint16_t *T = tmm + (size_t)f * tw * th;
    unsigned on = 0;       // bit c: tile tx0 + c is high-contrast
    uint32_t thr8[2] = {0, 0};
    if ((tw % THR_TPT) == 0) {
        // rows are 16-byte aligned and every group is complete: two tiles per register, 16-bit SIMD min / max
        // (VIMNMX3.U16x2).  hmn[j] / hmx[j] = dilated extrema of tiles tx0 + 2j (low half) and tx0 + 2j + 1 (high half).
        uint32_t hmn[4], hmx[4];
        if (gi < groups) {
            uint32_t mn[3][5], mx[3][5];   // [row][pair 0..3, 4 = {left column, right column}]
#pragma unroll
            for (int r = 0; r < 3; r++) {
                const int yy = ty + r - 1;
                uint32_t wv[5] = {0x00ff00ffu, 0x00ff00ffu, 0x00ff00ffu, 0x00ff00ffu, 0x00ff00ffu};   // (min 255, max 0)
                if (yy >= 0 && yy < th) {
                    const uint16_t *row = T + (size_t)yy * tw;
                    const uint4 q = __ldg(reinterpret_cast<const uint4 *>(row + tx0));
                    wv[0] = q.x; wv[1] = q.y; wv[2] = q.z; wv[3] = q.w;
                    const uint32_t l = tx0 > 0 ? __ldg(row + tx0 - 1) : 0x00ffu, rr = tx0 + THR_TPT < tw ? __ldg(row + tx0 + THR_TPT) : 0x00ffu;
                    wv[4] = l | (rr << 16);
                }
#pragma unroll
                for (int c = 0; c < 5; c++) { mn[r][c] = wv[c] & 0x00ff00ffu; mx[r][c] = __byte_perm(wv[c], 0u, 0x4341); }
            }
            uint32_t vmn[5], vmx[5];
#pragma unroll
            for (int c = 0; c < 5; c++) { vmn[c] = __vimin3_u16x2(mn[0][c], mn[1][c], mn[2][c]); vmx[c] = __vimax3_u16x2(mx[0][c], mx[1][c], mx[2][c]); }
#pragma unroll
            for (int c = 0; c < 4; c++) {
                const uint32_t ln = c == 0 ? __byte_perm(vmn[4], vmn[0], 0x5410) : __byte_perm(vmn[c - 1], vmn[c], 0x5432);
                const uint32_t rn = c == 3 ? __byte_perm(vmn[3], vmn[4], 0x7632) : __byte_perm(vmn[c], vmn[c + 1], 0x5432);
                const uint32_t lx_ = c == 0 ? __byte_perm(vmx[4], vmx[0], 0x5410) : __byte_perm(vmx[c - 1], vmx[c], 0x5432);
                const uint32_t rx = c == 3 ? __byte_perm(vmx[3], vmx[4], 0x7632) : __byte_perm(vmx[c], vmx[c + 1], 0x5432);
                hmn[c] = __vimin3_u16x2(ln, vmn[c], rn);
                hmx[c] = __vimax3_u16x2(lx_, vmx[c], rx);
            }
            // range >= diff  <=>  bit 15 of (0x8000 + range - diff) per 16-bit lane.  The range is in [-255, 255]: neighbourhoods
            // made of neutral tiles only (min 255, max 0 -- the sparse evaluation writes them for tiles that cannot be
            // high-contrast) have max < min, so bit 15 is set BEFORE the subtraction and no lane ever borrows from its neighbour
            const int d = min(max(min_wb_diff, 0), 256);
            const uint32_t kk = (uint32_t)d * 0x00010001u;
#pragma unroll
            for (int c = 0; c < 4; c++) {
                const uint32_t t = ((hmx[c] | 0x80008000u) - hmn[c]) - kk;
                on |= ((t >> 15) & 1u) << (2 * c) | (t >> 31) << (2 * c + 1);
            }
        }
        if (!__any_sync(0xffffffffu, on != 0)) return;
#pragma unroll
        for (int c = 0; c < THR_TPT; c++) {
            if (!((on >> c) & 1u)) continue;
            const uint32_t a = (hmn[c >> 1] >> ((c & 1) * 16)) & 0xffffu, b = (hmx[c >> 1] >> ((c & 1) * 16)) & 0xffffu;
            thr8[c >> 2] |= (a + (b - a) / 2) << ((c & 3) * 8);
        }
    } else {
        int cmn[THR_TPT + 2], cmx[THR_TPT + 2];   // vertical extrema of columns tx0 - 1 .. tx0 + 8
#pragma unroll
        for (int c = 0; c < THR_TPT + 2; c++) { cmn[c] = 255; cmx[c] = 0; }
        if (gi < groups) {
#pragma unroll
            for (int dy = -1; dy <= 1; dy++) {
                const int yy = ty + dy;
                if (yy < 0 || yy >= th) continue;
                const uint16_t *row = T + (size_t)yy * tw;
#pragma unroll
                for (int c = 0; c < THR_TPT + 2; c++) {
                    const int xx = tx0 + c - 1;
                    if (xx < 0 || xx >= tw) continue;
                    const int e = __ldg(row + xx);
                    cmn[c] = min(cmn[c], e & 255); cmx[c] = max(cmx[c], e >> 8);
                }
            }
        }
#pragma unroll
        for (int c = 0; c < THR_TPT; c++) {
            const int mn = min(cmn[c], min(cmn[c + 1], cmn[c + 2])), mx = max(cmx[c], max(cmx[c + 1], cmx[c + 2]));
            if (gi < groups && tx0 + c < tw && (mx - mn) >= min_wb_diff) {
                on |= 1u << c;
                thr8[c >> 2] |= (uint32_t)(mn + (mx - mn) / 2) << ((c & 3) * 8);
            }
        }
        if (!__any_sync(0xffffffffu, on != 0)) return;
    }
    const int cnt = __popc(on);
    int inc = cnt;
#pragma unroll
    for (int d = 1; d < 32; d <<= 1) { int t = __shfl_up_sync(0xffffffffu, inc, d); if (lane >= d) inc += t; }
    int base = 0;
    if (lane == 31) base = atomicAdd(acount, inc);
    base = __shfl_sync(0xffffffffu, base, 31) + inc - cnt;
#pragma unroll
    for (int c = 0; c < THR_TPT; c++) {
        if (!((on >> c) & 1u)) continue;
        const int tx = tx0 + c;
        if (base < acap) { alist[base] = ATILE(f, tx, ty); alist_thr[base] = (uint8_t)(thr8[c >> 2] >> ((c & 3) * 8)); }
        base++;
        tile_active[((size_t)f * cth + (ty * 4) / CCL_TH) * ctw + (tx * 4) / CCL_TW] = 1;
    }
}

// Sparse evaluation: only the tiles of the E-list carry real extrema (every other tile is neutral and cannot be high-contrast), so
// the threshold decision runs over that list (7 % of the tiles of a sparse frame) instead of over all tiles: one thread per
// listed tile, 3x3 dilation of the extrema, high-contrast tiles appended to the A-list (one atomic per warp).
__global__ void __launch_bounds__(256) k_threshold_scan_list(int tw, int th, const uint16_t *__restrict__ tmm, const uint32_t *__restrict__ elist,
                                                             const int *__restrict__ ecount, int min_wb_diff, uint32_t *__restrict__ alist,
                                                             uint8_t *__restrict__ alist_thr, int *__restrict__ acount, int acap,
                                                             uint8_t *__restrict__ tile_active, int ctw, int cth)
{
    const int n = *ecount, lane = threadIdx.x & 31;
    for (int base = blockIdx.x * blockDim.x; base < n; base += gridDim.x * blockDim.x) {   // whole warps stay in the loop together
        const int i = base + threadIdx.x;
        bool on = false;
        uint32_t e = 0;
        int thr = 0;
        if (i < n) {
            e = __ldg(elist + i);
            const int tx = ATILE_TX(e), ty = ATILE_TY(e), f = ATILE_F(e);
            int mn, mx;
            dilated_minmax(tmm + (size_t)f * tw * th, tw, th, tx, ty, mn, mx);
            on = mx - mn >= min_wb_diff;
            thr = mn + (mx - mn) / 2;
        }
        const unsigned m = __ballot_sync(0xffffffffu, on);
        if (m) {
            int b0 = 0;
            if (lane == 0) b0 = atomicAdd(acount, __popc(m));
            b0 = __shfl_sync(0xffffffffu, b0, 0);
            if (on) {
                const int k = b0 + __popc(m & ((1u << lane) - 1));
                if (k < acap) { alist[k] = e; alist_thr[k] = (uint8_t)thr; }
                tile_active[((size_t)ATILE_F(e) * cth + (ATILE_TY(e) * 4) / CCL_TH) * ctw + (ATILE_TX(e) * 4) / CCL_TW] = 1;
            }
        }
    }
}

// ternary pixels of the listed tiles: one thread per tile row (a 32-bit word of gray in, a word of {0, 255} out)
__global__ void __launch_bounds__(256) k_threshold_apply(const uint8_t *__restrict__ gray, int w, int h, int tw, int th,
                                                         const uint32_t *__restrict__ alist, const uint8_t *__restrict__ alist_thr,
                                                         const int *__restrict__ acount, int acap, uint8_t *__restrict__ out)
{
    const int n = min(*acount, acap);
    for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < 4 * n; i += gridDim.x * blockDim.x) {
        const uint32_t e = alist[i >> 2];
        const int tx = ATILE_TX(e), ty = ATILE_TY(e), f = ATILE_F(e), dy = i & 3;
        if (tx >= tw || ty >= th) continue;   // partial edge tiles are written by k_threshold_edges
        const unsigned thr = alist_thr[i >> 2];
        const size_t p = (size_t)f * w * h + (size_t)(ty * 4 + dy) * w + tx * 4;
        if ((w & 3) == 0 && (reinterpret_cast<uintptr_t>(gray) & 3) == 0) {   // out (thresh) is the context's own, aligned
            const uint32_t v = __ldg(reinterpret_cast<const uint32_t *>(gray + p));
            const uint32_t r = ((v & 255) > thr ? 0xffu : 0u) | (((v >> 8) & 255) > thr ? 0xff00u : 0u) |
                               (((v >> 16) & 255) > thr ? 0xff0000u : 0u) | ((v >> 24) > thr ? 0xff000000u : 0u);
            *reinterpret_cast<uint32_t *>(out + p) = r;
        } else {
            for (int dx = 0; dx < 4; dx++) out[p + dx] = gray[p + dx] > thr ? 255 : 0;
        }
    }
}

// back to 127 on every tile of the previous batch's A-list (runs at the start of the next batch)
__global__ void __launch_bounds__(256) k_reset_thresh(uint8_t *__restrict__ thresh, int w, int h, const uint32_t *__restrict__ alist,
                                                      const int *__restrict__ acount, int acap)
{
    const int n = min(*acount, acap);
    for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < 4 * n; i += gridDim.x * blockDim.x) {
        const uint32_t e = alist[i >> 2];
        const int x = ATILE_TX(e) * 4, y = ATILE_TY(e) * 4 + (i & 3), f = ATILE_F(e);
        if (y >= h) continue;
        uint8_t *p = thresh + (size_t)f * w * h + (size_t)y * w + x;
        if ((w & 3) == 0) *reinterpret_cast<uint32_t *>(p) = 0x7f7f7f7fu;
        else for (int dx = 0; dx < 4 && x + dx < w; dx++) p[dx] = 127;
    }
}

// The per-tile CCL kernels below run as 128-thread CTAs: lane = tile column, warp wy owns the tile rows wy, wy + 4, wy + 8,
// wy + 12, i.e. four pixels per thread whose global loads are independent and in flight together (these kernels are
// latency-bound: a tile is 512 B of ternary image and 2 KB of labels), 16 resident CTAs = 16 tiles in flight per SM.
#define CCL_THREADS 128
#define CCL_RPT (CCL_TH / (CCL_THREADS / 32))   // rows per thread = 4

// right / bottom partial tiles: nearest full tile's dilated threshold, never marked 127; every partial tile goes to
// the A-list (coordinates tx == tw or ty == th; the list consumers clip to the image)
__global__ void k_threshold_edges(const uint8_t *__restrict__ gray, int w, int h, int tw, int th,
                                  const uint16_t *__restrict__ tmm,
                                  uint8_t *__restrict__ out, uint8_t *__restrict__ tile_active, int ctw, int cth,
                                  uint32_t *__restrict__ alist, uint8_t *__restrict__ alist_thr, int *__restrict__ acount, int acap)
{
    int f = blockIdx.z;
    int nright = w - tw * 4, nbottom = h - th * 4;
    int total = nright * (th * 4) + nbottom * w;
    const uint8_t *g = gray + (size_t)f * w * h;
    uint8_t *o = out + (size_t)f * w * h;
    for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < total; i += gridDim.x * blockDim.x) {
        int x, y;
        if (i < nright * (th * 4)) { y = i / nright; x = tw * 4 + i % nright; }
        else { int j = i - nright * (th * 4); y = th * 4 + j / w; x = j % w; }
        int ty = min(y / 4, th - 1), tx = min(x / 4, tw - 1), mn, mx;
        dilated_minmax(tmm + (size_t)f * tw * th, tw, th, tx, ty, mn, mx);
        int thr = mn + (mx - mn) / 2;
        o[(size_t)y * w + x] = g[(size_t)y * w + x] > thr ? 255 : 0;
        tile_active[((size_t)f * cth + y / CCL_TH) * ctw + x / CCL_TW] = 1;
        if ((x & 3) == 0 && (y & 3) == 0) {   // first pixel of a partial tile
            int k = atomicAdd(acount, 1);
            if (k < acap) { alist[k] = ATILE(f, x / 4, y / 4); alist_thr[k] = (uint8_t)thr; }
        }
    }
}

// compaction of the flagged tiles of the whole batch into list[] = frame << 20 | tile index (warp-aggregated append)
__global__ void k_compact_tiles(const uint8_t *__restrict__ tile_active, int ntiles_total, int tiles_per_frame,
                                uint32_t *__restrict__ list, int *__restrict__ n_active)
{
    int i = blockIdx.x * blockDim.x + threadIdx.x;
    bool on = i < ntiles_total && tile_active[i];
    unsigned m = __ballot_sync(0xffffffffu, on);
    if (!m) return;
    int lane = threadIdx.x & 31, leader = __ffs(m) - 1, base = 0;
    if (lane == leader) base = atomicAdd(n_active, __popc(m));
    base = __shfl_sync(0xffffffffu, base, leader);
    if (on) list[base + __popc(m & ((1u << lane) - 1))] = ((uint32_t)(i / tiles_per_frame) << 20) | (uint32_t)(i % tiles_per_frame);
}

// ---------------------------------------------------------------------------------------------------------
// K3: connected components.  Union rule of the dependency: for x in [1,w-2], y in [0,h-2], v != 127:
// join (x+1,y), (x,y+1) when equal; for v == 255 also (x-1,y+1), (x+1,y+1).  Root = smallest pixel index.
template <typename T>
__device__ __forceinline__ T uf_find(const volatile T *L, T x)
{
    T p = L[x];
    while (p != x) { x = p; p = L[x]; }
    return x;
}

__device__ __forceinline__ void uf_union_smem(int *L, int a, int b)
{
    for (;;) {
        a = uf_find<int>(L, a);
        b = uf_find<int>(L, b);
        if (a == b) return;
        if (a > b) { int t = a; a = b; b = t; }
        int old = atomicMin(&L[b], a);
        if (old == b) return;
        b = old;
    }
}

// root walk with path halving: every visited node is re-pointed at its grandparent.  The plain stores race with the
// atomicMin of a concurrent union only on nodes that have a parent already; they always store an ancestor, and a union
// whose atomicMin loses a link follows up on the old parent, so the sets come out the same -- but the trees stay shallow
// (without it a component that spans hundreds of 4x4 tiles is a chain hundreds of links deep).
__device__ __forceinline__ uint32_t uf_find_halve(uint32_t *L, uint32_t x)
{
    volatile uint32_t *V = L;
    uint32_t p = V[x];
    while (p != x) {
        const uint32_t gp = V[p];
        if (gp != p) V[x] = gp;
        x = p;
        p = gp;
    }
    return x;
}

__device__ __forceinline__ void uf_union_gmem(uint32_t *L, uint32_t a, uint32_t b)
{
    for (;;) {
        a = uf_find_halve(L, a);
        b = uf_find_halve(L, b);
        if (a == b) return;
        if (a > b) { uint32_t t = a; a = b; b = t; }
        uint32_t old = atomicMin(&L[b], a);
        if (old == b) return;
        b = old;
    }
}

// One CTA = one 32x16 tile per iteration.  Horizontal runs are labelled with a warp ballot (no atomics); the
// vertical / diagonal joins are union-find merges of run roots, skipping the joins that a left neighbour of the
// same run already implies, so a solid tile costs ~16 atomics instead of ~1500.
__global__ void __launch_bounds__(CCL_THREADS) k_ccl_local(const uint8_t *__restrict__ thresh, int w, int h,
                                                           uint32_t *__restrict__ labels,
                                                           const uint32_t *__restrict__ list, const int *__restrict__ n_active,
                                                           int ctw, int full)
{
    __shared__ int L[CCL_TW * CCL_TH];
    __shared__ uint8_t V[CCL_TH][CCL_TW + 1];
    __shared__ uint32_t JR[CCL_TH];   // bit x of JR[y]: pixel (x,y) is joined with (x+1,y)
    const int lx = threadIdx.x & 31, wy = threadIdx.x >> 5;
    const int n = *n_active;
    for (int it = blockIdx.x; it < n; it += gridDim.x) {
        const uint32_t e = list[it];
        const int f = e >> 20, tile = e & 0xfffff, tyb = tile / ctw, txb = tile - tyb * ctw;
        const int x = txb * CCL_TW + lx;
        const uint8_t *t = thresh + (size_t)f * w * h;
        int v[CCL_RPT];
        uint32_t jr[CCL_RPT];
        bool src[CCL_RPT];
#pragma unroll
        for (int r = 0; r < CCL_RPT; r++) {
            const int y = tyb * CCL_TH + wy + 4 * r;
            v[r] = (x < w && y < h) ? t[(size_t)y * w + x] : 127;
        }
#pragma unroll
        for (int r = 0; r < CCL_RPT; r++) {
            const int ly = wy + 4 * r, y = tyb * CCL_TH + ly;
            if (!__any_sync(0xffffffffu, v[r] != 127)) {   // background row: only what the rows above / below read of it
                V[ly][lx] = 127;
                if (lx == 0) JR[ly] = 0;
                src[r] = false; jr[r] = 0;
                continue;
            }
            // pixel may initiate joins (full = classic path: every pixel; otherwise the dependency's AprilTag loop ranges)
            src[r] = v[r] != 127 && (full || (x >= 1 && x <= w - 2 && y <= h - 2));
            const int vr = __shfl_down_sync(0xffffffffu, v[r], 1);
            const bool join_r = src[r] && lx + 1 < CCL_TW && vr == v[r];
            jr[r] = __ballot_sync(0xffffffffu, join_r);
            const uint32_t starts = ~(jr[r] << 1);                                 // bit i: pixel i starts a run
            const int start = 31 - __clz(starts & (0xffffffffu >> (31 - lx)));
            V[ly][lx] = (uint8_t)v[r];
            L[ly * CCL_TW + lx] = ly * CCL_TW + start;
            if (lx == 0) JR[ly] = jr[r];
        }
        __syncthreads();
#pragma unroll
        for (int r = 0; r < CCL_RPT; r++) {
            const int ly = wy + 4 * r, li = ly * CCL_TW + lx;
            if (!__any_sync(0xffffffffu, src[r])) continue;   // rows without foreground cost nothing (warp-uniform)
            if (src[r] && ly + 1 < CCL_TH) {
                const uint32_t jr_b = JR[ly + 1];
                const bool s_same = V[ly + 1][lx] == v[r];
                const bool left_same_run = lx > 0 && ((jr[r] >> (lx - 1)) & 1u);
                if (s_same) {
                    const bool implied = left_same_run && V[ly + 1][lx - 1] == v[r] && ((jr_b >> (lx - 1)) & 1u);
                    if (!implied) uf_union_smem(L, li, li + CCL_TW);
                }
                if (v[r] == 255) {
                    if (lx > 0 && V[ly + 1][lx - 1] == v[r] && !(s_same && ((jr_b >> (lx - 1)) & 1u))) uf_union_smem(L, li, li + CCL_TW - 1);
                    if (lx + 1 < CCL_TW && V[ly + 1][lx + 1] == v[r] && !(s_same && ((jr_b >> lx) & 1u))) uf_union_smem(L, li, li + CCL_TW + 1);
                }
            }
        }
        __syncthreads();
#pragma unroll
        for (int r = 0; r < CCL_RPT; r++) {
            const int ly = wy + 4 * r, y = tyb * CCL_TH + ly;
            if (!__any_sync(0xffffffffu, v[r] != 127)) continue;
            if (x < w && y < h && v[r] != 127) {
                int rt = uf_find<int>(L, ly * CCL_TW + lx);
                int ry = tyb * CCL_TH + rt / CCL_TW, rx = txb * CCL_TW + rt % CCL_TW;
                labels[(size_t)f * w * h + (size_t)y * w + x] = (uint32_t)(ry * w + rx);
            }
        }
        __syncthreads();
    }
}

// unions across tile boundaries, per active tile: sources on its last row (S, SW, SE cross), on its last
// column (E, SE cross) and on its first column (SW crosses).  64 threads per tile.
__global__ void k_ccl_merge(const uint8_t *__restrict__ thresh, int w, int h, uint32_t *__restrict__ labels,
                            const uint32_t *__restrict__ list, const int *__restrict__ n_active, int ctw, int full)
{
    const int n = *n_active;
    const int per_block = blockDim.x / 64, sub = threadIdx.x / 64, k = threadIdx.x % 64;
    for (int it = blockIdx.x * per_block + sub; it < n; it += gridDim.x * per_block) {
        const uint32_t e = list[it];
        const int f = e >> 20, tile = e & 0xfffff, tyb = tile / ctw, txb = tile - tyb * ctw;
        const uint8_t *t = thresh + (size_t)f * w * h;
        uint32_t *L = labels + (size_t)f * w * h;
        int x, y, kind;
        if (k < 32) { kind = 0; x = txb * CCL_TW + k; y = tyb * CCL_TH + CCL_TH - 1; }
        else if (k < 48) { kind = 1; x = txb * CCL_TW + CCL_TW - 1; y = tyb * CCL_TH + (k - 32); }
        else { kind = 2; x = txb * CCL_TW; y = tyb * CCL_TH + (k - 48); }
        if (x >= w || y >= h) continue;
        if (!full && (x < 1 || x > w - 2 || y > h - 2)) continue;
        const int v = t[(size_t)y * w + x];
        if (v == 127) continue;
        const uint32_t o = (uint32_t)(y * w + x);
        const bool has_s = y + 1 < h, has_e = x + 1 < w, has_w = x >= 1;   // always true inside the AprilTag ranges
        // A union is skipped when other unions already join the same two components: pixels that are neighbours in a row (or a
        // column) of ONE tile with equal values were joined by k_ccl_local, so only the first pixel of a run that continues across
        // the boundary does the (global, latency-bound) union, and a diagonal crossing is only needed where the straight one is
        // not there.  The unions relied upon must lie inside the AprilTag ranges (initiators x in [1, w-2], y in [0, h-2]); next
        // to the image frame the plain rule stays.
        if (kind == 0) {
            const bool s_eq = has_s && t[o + w] == v;
            const bool dedupe = full || (x >= 2 && y + 1 <= h - 2);
            if (s_eq) {
                const bool left_pair = dedupe && k > 0 && has_w && t[o - 1] == v && t[o + w - 1] == v;
                if (!left_pair) uf_union_gmem(L, o, o + w);
            }
            if (v == 255 && has_s && !(s_eq && dedupe)) {
                if (has_w && t[o + w - 1] == v) uf_union_gmem(L, o, o + w - 1);
                if (has_e && t[o + w + 1] == v) uf_union_gmem(L, o, o + w + 1);
            }
        } else if (kind == 1) {
            const bool e_eq = has_e && t[o + 1] == v;
            const bool dedupe = full || x + 1 <= w - 2;
            if (e_eq) {
                const bool up_pair = dedupe && k > 32 && t[o - w] == v && t[o - w + 1] == v;
                if (!up_pair) uf_union_gmem(L, o, o + 1);
            }
            if (v == 255 && has_e && has_s && !(e_eq && dedupe) && t[o + w + 1] == v) uf_union_gmem(L, o, o + w + 1);
        } else {
            if (v == 255 && has_w && has_s && t[o + w - 1] == v) uf_union_gmem(L, o, o + w - 1);
        }
    }
}

__global__ void __launch_bounds__(CCL_THREADS) k_ccl_flatten(const uint8_t *__restrict__ thresh, int w, int h,
                                                             uint32_t *__restrict__ labels,
                                                             const uint32_t *__restrict__ list,
                                                             const int *__restrict__ n_active, int ctw)
{
    const int n = *n_active;
    const int lx = threadIdx.x & 31, wy = threadIdx.x >> 5;
    for (int it = blockIdx.x; it < n; it += gridDim.x) {
        const uint32_t e = list[it];
        const int f = e >> 20, tile = e & 0xfffff, tyb = tile / ctw, txb = tile - tyb * ctw;
        const int x = txb * CCL_TW + lx;
        const uint8_t *t = thresh + (size_t)f * w * h;
        uint32_t *L = labels + (size_t)f * w * h;
        uint32_t o[CCL_RPT], cur[CCL_RPT];
        bool act[CCL_RPT];
#pragma unroll
        for (int r = 0; r < CCL_RPT; r++) {
            const int y = tyb * CCL_TH + wy + 4 * r;
            o[r] = (uint32_t)(y * w + x);
            act[r] = x < w && y < h && t[o[r]] != 127;
        }
        if (!__any_sync(0xffffffffu, act[0] | act[1] | act[2] | act[3])) continue;
#pragma unroll
        for (int r = 0; r < CCL_RPT; r++) cur[r] = act[r] ? L[o[r]] : 0u;
        // the four root walks advance together: one independent load per pixel and round
        bool walk[CCL_RPT];
#pragma unroll
        for (int r = 0; r < CCL_RPT; r++) walk[r] = act[r];
        for (;;) {
            bool any = false;
            uint32_t par[CCL_RPT];
#pragma unroll
            for (int r = 0; r < CCL_RPT; r++) par[r] = walk[r] ? const_cast<const volatile uint32_t *>(L)[cur[r]] : cur[r];
#pragma unroll
            for (int r = 0; r < CCL_RPT; r++) {
                if (walk[r]) {
                    if (par[r] == cur[r]) walk[r] = false;
                    else { cur[r] = par[r]; any = true; }
                }
            }
            if (!any) break;
        }
#pragma unroll
        for (int r = 0; r < CCL_RPT; r++)
            if (act[r]) L[o[r]] = cur[r];  // racing writers store roots of the same tree; finds stay correct
    }
}

// ---------------------------------------------------------------------------------------------------------
// K4: boundary points -> clusters
__device__ __forceinline__ uint32_t hash64(unsigned long long k)
{
    k ^= k >> 33; k *= 0xff51afd7ed558ccdULL; k ^= k >> 33; k *= 0xc4ceb9fe1a85ec53ULL; k ^= k >> 33;
    return (uint32_t)k;
}
#define HASH_EMPTY 0xffffffffffffffffULL

// Phase 1: one thread per pixel of an A-list tile (16 lanes per tile) looks at the E, S, SW, SE neighbours (tiles that
// are not listed hold 127) and appends one record per black/white crossing to the frame's point array:
// {x | y << 16, k | (v0 == 255) << 8, -, -}.  One atomic per tile with crossings.
__global__ void __launch_bounds__(256) k_emit_scan(const uint8_t *__restrict__ thresh, int w, int h, const uint32_t *__restrict__ alist,
                                                   const int *__restrict__ acount, int acap, uint4 *__restrict__ points,
                                                   int32_t *__restrict__ counters)
{
    const int n = min(*acount, acap);
    const int lane = threadIdx.x & 31, sub = lane & 15;
    // uniform trip count per warp: both half-warps stay together for the shuffles
    for (int it = (blockIdx.x * blockDim.x + threadIdx.x) >> 4; it - (lane >> 4) < n; it += (gridDim.x * blockDim.x) >> 4) {
        const bool live = it < n;
        const uint32_t e = live ? alist[it] : 0u;
        const int f = ATILE_F(e), x = ATILE_TX(e) * 4 + (sub & 3), y = ATILE_TY(e) * 4 + (sub >> 2);
        const uint8_t *t = thresh + (size_t)f * w * h;
        const bool src = live && x >= 1 && x <= w - 2 && y >= 1 && y <= h - 2;
        const int v0 = src ? t[(size_t)y * w + x] : 127;
        unsigned mask = 0;
        if (src && v0 != 127) {
            const int want = 255 - v0;
            const uint8_t *r1 = t + (size_t)(y + 1) * w + x;
            mask = (t[(size_t)y * w + x + 1] == want ? 1u : 0u) | (r1[0] == want ? 2u : 0u) | (r1[-1] == want ? 4u : 0u) | (r1[1] == want ? 8u : 0u);
        }
        const int cnt = __popc(mask);
        int inc = cnt;
#pragma unroll
        for (int d = 1; d < 16; d <<= 1) { int tv = __shfl_up_sync(0xffffffffu, inc, d, 16); if (sub >= d) inc += tv; }
        const int total = __shfl_sync(0xffffffffu, inc, 15, 16);
        int pos = 0;
        if (sub == 15 && total) pos = atomicAdd(&counters[f * APSE_COUNTERS], total);
        pos = __shfl_sync(0xffffffffu, pos, 15, 16) + inc - cnt;
        uint4 *pts = points + (size_t)f * APSE_MAX_POINTS;
#pragma unroll
        for (int k = 0; k < 4; k++) {
            if (!((mask >> k) & 1u)) continue;
            if (pos < APSE_MAX_POINTS) pts[pos] = make_uint4((uint32_t)x | ((uint32_t)y << 16), (uint32_t)k | (v0 == 255 ? 256u : 0u), 0u, 0u);
            else atomicExch(&counters[f * APSE_COUNTERS + 3], APSE_ERR_CAPACITY);
            pos++;
        }
    }
}

// Phase 2: one thread per record: component pair -> cluster hash slot and rank, record rewritten in place as
// {slot, rank, 2x + dx | (2y + dy) << 16, gx | gy << 16}.  Every lane has a point.
__global__ void __launch_bounds__(256) k_emit_insert(int w, int h, uint32_t *__restrict__ labels,
                                                     unsigned long long *__restrict__ hash_keys, uint32_t *__restrict__ hash_count,
                                                     uint32_t *__restrict__ used_slots, uint4 *__restrict__ points,
                                                     int32_t *__restrict__ counters, int batch)
{
    const int DX[4] = {1, 0, -1, 1}, DY[4] = {0, 1, 1, 1};
    for (int f = blockIdx.y; f < batch; f += gridDim.y) {
        int32_t *cnt = counters + f * APSE_COUNTERS;
        const int n = min(cnt[0], APSE_MAX_POINTS);
        uint32_t *L = labels + (size_t)f * w * h;
        unsigned long long *hk = hash_keys + (size_t)f * APSE_HASH_SLOTS;
        uint32_t *hc = hash_count + (size_t)f * APSE_HASH_SLOTS;
        uint4 *pts = points + (size_t)f * APSE_MAX_POINTS;
        for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) {
            const uint4 rec = pts[i];
            const int x = rec.x & 0xffff, y = rec.x >> 16, k = rec.y & 3, v0 = (rec.y & 256u) ? 255 : 0, v1 = 255 - v0;
            const int dx = DX[k], dy = DY[k];
            // component ids: root walks from the two pixels (pixel -> tile-local root -> roots merged across tiles), with the
            // root written back to the pixel; only crossing pixels ever pay for this, there is no flatten pass over all pixels
            const uint32_t pa = (uint32_t)(y * w + x), pb = (uint32_t)((y + dy) * w + x + dx);
            const uint32_t ra = uf_find_halve(L, pa), rb = uf_find_halve(L, pb);
            if (L[pa] != ra) L[pa] = ra;
            if (L[pb] != rb) L[pb] = rb;
            const unsigned long long a = ra, b = rb;
            const unsigned long long key = a < b ? (b << 32) + a : (a << 32) + b;
            uint32_t slot = hash64(key) & (APSE_HASH_SLOTS - 1);
            bool ok = true;
            int probes = 0;
            for (;;) {
                unsigned long long prev = atomicCAS(&hk[slot], HASH_EMPTY, key);
                if (prev == HASH_EMPTY) {  // this thread created the cluster: list the slot for the scan kernel
                    used_slots[(size_t)f * APSE_HASH_SLOTS + atomicAdd(&cnt[6], 1)] = slot;
                    break;
                }
                if (prev == key) break;
                slot = (slot + 1) & (APSE_HASH_SLOTS - 1);
                if (++probes >= APSE_HASH_SLOTS) { atomicExch(&cnt[3], APSE_ERR_CAPACITY); ok = false; break; }
            }
            if (!ok) { pts[i] = make_uint4(0xffffffffu, 0u, 0u, 0u); continue; }
            const uint32_t rank = atomicAdd(&hc[slot], 1u);
            const int gx = dx * (v1 - v0), gy = dy * (v1 - v0);
            pts[i] = make_uint4(slot, rank, (uint32_t)(2 * x + dx) | ((uint32_t)(2 * y + dy) << 16), ((uint32_t)gx & 0xffffu) | ((uint32_t)gy << 16));
        }
    }
}

// one block per frame: size filter + exclusive scan of the kept clusters' counts over the list of used hash slots;
// the slots are reset here (their last reader), so the tables never need a memset between batches
__global__ void __launch_bounds__(1024) k_cluster_scan(unsigned long long *__restrict__ hash_keys, uint32_t *__restrict__ hash_count,
                                                       uint32_t *__restrict__ hash_offset, const uint32_t *__restrict__ used_slots,
                                                       ClusterDesc *__restrict__ clusters, int32_t *__restrict__ counters,
                                                       int min_px, int max_px)
{
    const int f = blockIdx.x, tid = threadIdx.x;
    unsigned long long *hk = hash_keys + (size_t)f * APSE_HASH_SLOTS;
    uint32_t *hc = hash_count + (size_t)f * APSE_HASH_SLOTS;
    uint32_t *ho = hash_offset + (size_t)f * APSE_HASH_SLOTS;
    const uint32_t *us = used_slots + (size_t)f * APSE_HASH_SLOTS;
    ClusterDesc *cl = clusters + (size_t)f * APSE_MAX_CLUSTERS;
    int32_t *cnt = counters + f * APSE_COUNTERS;
    const int n_used = cnt[6];
    __shared__ uint32_t s_pts[1024], s_cl[1024];
    uint32_t npts = 0, ncl = 0;
    for (int i = tid; i < n_used; i += 1024) {
        uint32_t c = hc[us[i]];
        if ((int)c >= min_px && (int)c <= max_px) { npts += c; ncl++; }
    }
    s_pts[tid] = npts; s_cl[tid] = ncl;
    __syncthreads();
    for (int d = 1; d < 1024; d <<= 1) {  // Hillis-Steele inclusive scan
        uint32_t a = 0, b = 0;
        if (tid >= d) { a = s_pts[tid - d]; b = s_cl[tid - d]; }
        __syncthreads();
        s_pts[tid] += a; s_cl[tid] += b;
        __syncthreads();
    }
    uint32_t off = s_pts[tid] - npts, ci = s_cl[tid] - ncl;
    for (int i = tid; i < n_used; i += 1024) {
        const uint32_t sl = us[i], c = hc[sl];
        if ((int)c >= min_px && (int)c <= max_px) {
            ho[sl] = off;
            if (ci < APSE_MAX_CLUSTERS) {
                unsigned long long k = hk[sl];
                cl[ci] = ClusterDesc{off, c, (uint32_t)k, (uint32_t)(k >> 32)};
            }
            off += c; ci++;
        } else {
            ho[sl] = 0xffffffffu;
        }
        hk[sl] = HASH_EMPTY;
        hc[sl] = 0;
    }
    if (tid == 1023) {
        if (s_cl[1023] > APSE_MAX_CLUSTERS) cnt[3] = APSE_ERR_CAPACITY;
        cnt[1] = (int32_t)min(s_cl[1023], (uint32_t)APSE_MAX_CLUSTERS);
        cnt[4] = n_used;
        cnt[5] = (int32_t)s_pts[1023];
    }
}

__global__ void k_scatter_points(const uint4 *__restrict__ points, const uint32_t *__restrict__ hash_offset,
                                 const int32_t *__restrict__ counters, uint2 *__restrict__ sorted_pts, int batch)
{
    for (int f = blockIdx.y; f < batch; f += gridDim.y) {
        int n = min(counters[f * APSE_COUNTERS], APSE_MAX_POINTS);
        const uint4 *pts = points + (size_t)f * APSE_MAX_POINTS;
        const uint32_t *ho = hash_offset + (size_t)f * APSE_HASH_SLOTS;
        uint2 *sp = sorted_pts + (size_t)f * APSE_MAX_POINTS;
        for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) {
            uint4 p = pts[i];
            if (p.x == 0xffffffffu) continue;   // hash table full (status already set)
            uint32_t off = ho[p.x];
            if (off != 0xffffffffu) sp[off + p.y] = make_uint2(p.z, p.w);
        }
    }
}

// ---------------------------------------------------------------------------------------------------------
// K5: quad fit
__device__ __forceinline__ float fast_atan2_deg(float y, float x)
{
    // OpenCV's fastAtan2 (scalar path), float32, no FMA
    const float k = (float)(180 / 3.14159265358979323846);
    const float p1 = 0.9997878412794807f * k, p3 = -0.3258083974640975f * k;
    const float p5 = 0.1555786518463281f * k, p7 = -0.04432655554792128f * k;
    float ax = fabsf(x), ay = fabsf(y), a, c, c2;
    if (ax >= ay) {
        c = ay / (ax + (float)DBL_EPSILON);
        c2 = c * c;
        a = (((p7 * c2 + p5) * c2 + p3) * c2 + p1) * c;
    } else {
        c = ax / (ay + (float)DBL_EPSILON);
        c2 = c * c;
        a = 90.f - (((p7 * c2 + p5) * c2 + p3) * c2 + p1) * c;
    }
    if (x < 0) a = 180.f - a;
    if (y < 0) a = 360.f - a;
    return a;
}

// cosf / sinf evaluated with the double-precision polynomials of the host libm (glibc >= 2.28 sincosf), so
// that the float results are bit-identical to the CPU reference.  Valid for |y| < 120 (here y in [0, pi]).
__device__ __forceinline__ float libm_poly(double x, double x2, bool flip, int n)
{
    const double C0 = 0x1p0, C1 = -0x1.ffffffd0c621cp-2, C2 = 0x1.55553e1068f19p-5, C3 = -0x1.6c087e89a359dp-10,
                 C4 = 0x1.99343027bf8c3p-16;
    const double S1 = -0x1.555545995a603p-3, S2 = 0x1.1107605230bc4p-7, S3 = -0x1.994eb3774cf24p-13;
    if ((n & 1) == 0) {
        double x3 = x * x2, s1 = S2 + x2 * S3, x7 = x3 * x2, s = x + x3 * S1;
        return (float)(s + x7 * s1);
    }
    const double f = flip ? -1.0 : 1.0;  // second table of the libm: cosine coefficients negated
    double x4 = x2 * x2, c2 = (f * C3) + x2 * (f * C4), c1 = (f * C0) + x2 * (f * C1), x6 = x4 * x2;
    double c = c1 + x4 * (f * C2);
    return (float)(c + x6 * c2);
}

__device__ __forceinline__ void libm_sincosf(float y, float *sp, float *cp)
{
    const double hpi_inv = 0x1.45F306DC9C883p+23, hpi = 0x1.921FB54442D18p0;
    double x = y;
    unsigned top = (__float_as_uint(y) >> 20) & 0x7ff;
    if (top < ((__float_as_uint(0x1.921FB6p-1f) >> 20) & 0x7ff)) {
        if (top < ((__float_as_uint(0x1p-12f) >> 20) & 0x7ff)) { *sp = y; *cp = 1.0f; return; }
        double x2 = x * x;
        *sp = libm_poly(x, x2, false, 0);
        *cp = libm_poly(x, x2, false, 1);
        return;
    }
    double r = x * hpi_inv;
    int n = ((int)r + 0x800000) >> 24;
    x = x - n * hpi;
    double s = ((n & 3) == 1 || (n & 3) == 2) ? -1.0 : 1.0;
    bool flip = (n & 2) != 0;
    double x2 = x * x;
    *sp = libm_poly(x * s, x2, flip, n);
    *cp = libm_poly(x * s, x2, flip, n ^ 1);
}

struct LineFit { double Ex, Ey, nx, ny, err, mse; };

// lfps: inclusive prefix sums [sz][6] = {Mx, My, Mxx, Mxy, Myy, W}
__device__ void fit_line(const double *__restrict__ l, int sz, int i0, int i1, LineFit &o)
{
    double Mx, My, Mxx, Mxy, Myy, W;
    int N;
    const double *a = l + (size_t)i1 * 6;
    if (i0 < i1) {
        N = i1 - i0 + 1;
        Mx = a[0]; My = a[1]; Mxx = a[2]; Mxy = a[3]; Myy = a[4]; W = a[5];
        if (i0 > 0) {
            const double *b = l + (size_t)(i0 - 1) * 6;
            Mx -= b[0]; My -= b[1]; Mxx -= b[2]; Mxy -= b[3]; Myy -= b[4]; W -= b[5];
        }
    } else {
        const double *e = l + (size_t)(sz - 1) * 6, *b = l + (size_t)(i0 - 1) * 6;
        Mx = e[0] - b[0]; My = e[1] - b[1]; Mxx = e[2] - b[2]; Mxy = e[3] - b[3]; Myy = e[4] - b[4]; W = e[5] - b[5];
        Mx += a[0]; My += a[1]; Mxx += a[2]; Mxy += a[3]; Myy += a[4]; W += a[5];
        N = sz - i0 + i1 + 1;
    }
    double Ex = Mx / W, Ey = My / W;
    double Cxx = Mxx / W - Ex * Ex, Cxy = Mxy / W - Ex * Ey, Cyy = Myy / W - Ey * Ey;
    float normal_theta = (float)(.5f * (3.14159265358979323846 / 180)) * fast_atan2_deg((float)(-2 * Cxy), (float)(Cyy - Cxx));
    float sn, cs;
    libm_sincosf(normal_theta, &sn, &cs);
    double nx = cs, ny = sn;
    o.Ex = Ex; o.Ey = Ey; o.nx = nx; o.ny = ny;
    o.err = nx * nx * N * Cxx + 2 * nx * ny * N * Cxy + ny * ny * N * Cyy;
    o.mse = nx * nx * Cxx + 2 * nx * ny * Cxy + ny * ny * Cyy;
}

__device__ __forceinline__ double sq(double v) { return v * v; }

// block-wide helpers (FQ_THREADS threads)
__device__ __forceinline__ int block_scan_excl(int v, int *s_warp, int &total)
{
    int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
    int inc = v;
    for (int d = 1; d < 32; d <<= 1) { int t = __shfl_up_sync(0xffffffffu, inc, d); if (lane >= d) inc += t; }
    if (lane == 31) s_warp[wid] = inc;
    __syncthreads();
    int base = 0, tot = 0;
    for (int i = 0; i < FQ_THREADS / 32; i++) { int t = s_warp[i]; if (i < wid) base += t; tot += t; }
    __syncthreads();
    total = tot;
    return base + inc - v;
}

struct FitArgs {
    const uint8_t *gray;
    int w, h, batch;
    const ClusterDesc *clusters;
    uint2 *sorted_pts;
    unsigned long long *sort_keys;
    double *lfps, *errs;
    int32_t *counters;
    float *quads;
    unsigned long long *quad_keys;
    int *work_counter;
    int max_nmaxima;
    float critical_rad, max_line_fit_mse;
    double max_dot;
};

__device__ void bitonic_sort_u64(unsigned long long *keys, int npow2)
{
    for (int k = 2; k <= npow2; k <<= 1)
        for (int j = k >> 1; j > 0; j >>= 1) {
            for (int i = threadIdx.x; i < npow2; i += FQ_THREADS) {
                int ixj = i ^ j;
                if (ixj > i) {
                    unsigned long long a = keys[i], b = keys[ixj];
                    bool up = (i & k) == 0;
                    if ((a > b) == up) { keys[i] = b; keys[ixj] = a; }
                }
            }
            __syncthreads();
        }
}

// 40 registers (a few hundred bytes of spills in this latency-bound kernel): a CTA then needs 5 K registers and fits beside the
// three resident preprocess CTAs of an SM instead of displacing one of them for the ~0.3 ms it lives
__global__ void __maxnreg__(40) k_fit_quads(FitArgs A)
{
    __shared__ unsigned long long s_keys[APSE_SORT_SMEM];
    __shared__ int s_prefix[65];       // cluster count prefix over frames (batch <= 64 per launch)
    __shared__ int s_item;
    __shared__ int s_warp[FQ_THREADS / 32];
    __shared__ int s_i4[8];
    __shared__ double s_d[FQ_THREADS / 32];
    __shared__ int s_max_idx[MAXIMA_CAP + 1];
    __shared__ double s_max_err[MAXIMA_CAP + 1];
    __shared__ LineFit s_pair[MAXIMA_CAP][MAXIMA_CAP];
    __shared__ double s_best_err[FQ_THREADS];
    __shared__ unsigned s_best_combo[FQ_THREADS];
    const int tid = threadIdx.x, lane = tid & 31, wid = tid >> 5;

    if (tid == 0) {
        int acc = 0;
        for (int f = 0; f < A.batch; f++) { s_prefix[f] = acc; acc += A.counters[f * APSE_COUNTERS + 1]; }
        s_prefix[A.batch] = acc;
    }
    __syncthreads();
    const int total_items = s_prefix[A.batch];

    for (;;) {
        __syncthreads();
        if (tid == 0) s_item = atomicAdd(A.work_counter, 1);
        __syncthreads();
        const int item = s_item;
        if (item >= total_items) break;
        int f = 0;
        while (s_prefix[f + 1] <= item) f++;
        const int ci = item - s_prefix[f];
        const ClusterDesc cd = A.clusters[(size_t)f * APSE_MAX_CLUSTERS + ci];
        const int n = (int)cd.count;
        uint2 *pts = A.sorted_pts + (size_t)f * APSE_MAX_POINTS + cd.offset;
        const uint8_t *im = A.gray + (size_t)f * A.w * A.h;
        double *lf = A.lfps + ((size_t)f * APSE_MAX_POINTS + cd.offset) * 6;
        double *e0 = A.errs + ((size_t)f * APSE_MAX_POINTS + cd.offset) * 2, *e1 = e0 + n;

        // ---- bounding box
        int xmin = INT32_MAX, xmax = 0, ymin = INT32_MAX, ymax = 0;
        for (int i = tid; i < n; i += FQ_THREADS) {
            uint32_t xy = pts[i].x;
            int x = xy & 0xffff, y = xy >> 16;
            xmin = min(xmin, x); xmax = max(xmax, x); ymin = min(ymin, y); ymax = max(ymax, y);
        }
        for (int d = 16; d > 0; d >>= 1) {
            xmin = min(xmin, __shfl_xor_sync(0xffffffffu, xmin, d)); xmax = max(xmax, __shfl_xor_sync(0xffffffffu, xmax, d));
            ymin = min(ymin, __shfl_xor_sync(0xffffffffu, ymin, d)); ymax = max(ymax, __shfl_xor_sync(0xffffffffu, ymax, d));
        }
        if (tid == 0) { s_i4[0] = INT32_MAX; s_i4[1] = 0; s_i4[2] = INT32_MAX; s_i4[3] = 0; }
        __syncthreads();
        if (lane == 0) { atomicMin(&s_i4[0], xmin); atomicMax(&s_i4[1], xmax); atomicMin(&s_i4[2], ymin); atomicMax(&s_i4[3], ymax); }
        __syncthreads();
        const double cx = (s_i4[0] + s_i4[1]) * 0.5 + 0.05118, cy = (s_i4[2] + s_i4[3]) * 0.5 + -0.028581;

        // ---- theta keys + orientation test (black inside white)
        int npow2 = 1;
        while (npow2 < n) npow2 <<= 1;
        unsigned long long *keys = npow2 <= APSE_SORT_SMEM ? s_keys : A.sort_keys + (size_t)f * APSE_MAX_POINTS * 2 + 2 * (size_t)cd.offset;
        double dot = 0;
        for (int i = tid; i < npow2; i += FQ_THREADS) {
            unsigned long long key = 0xffffffffffffffffULL;
            if (i < n) {
                uint2 p = pts[i];
                int x = p.x & 0xffff, y = p.x >> 16;
                int gx = (int)(short)(p.y & 0xffff), gy = (int)(short)(p.y >> 16);
                double dx = x - cx, dy = y - cy;
                float theta = fast_atan2_deg((float)dy, (float)dx) * (float)(3.14159265358979323846 / 180);
                dot += dx * gx + dy * gy;
                key = ((unsigned long long)__float_as_uint(theta) << 32) | p.x;
            }
            keys[i] = key;
        }
        for (int d = 16; d > 0; d >>= 1) dot += __shfl_xor_sync(0xffffffffu, dot, d);
        if (lane == 0) s_d[wid] = dot;
        __syncthreads();
        dot = 0;
        for (int i = 0; i < FQ_THREADS / 32; i++) dot += s_d[i];
        if (dot < 0) continue;

        // ---- sort by theta (ties: packed y,x), drop adjacent duplicates
        bitonic_sort_u64(keys, npow2);
        uint32_t *uniq = reinterpret_cast<uint32_t *>(pts);  // reuse the cluster's point segment (n uint2 = 2n u32)
        int sz = 0;
        for (int base = 0; base < n; base += FQ_THREADS) {
            int i = base + tid;
            uint32_t xy = 0;
            int flag = 0;
            if (i < n) {
                xy = (uint32_t)keys[i];
                flag = (i == 0) || ((uint32_t)keys[i - 1] != xy);
            }
            int tot;
            int pos = block_scan_excl(flag, s_warp, tot);
            if (flag) uniq[sz + pos] = xy;
            sz += tot;
        }
        __syncthreads();
        if (sz < 4) continue;
        const int ksz = min(20, sz / 12);
        if (ksz < 2) continue;

        // ---- weighted moments: terms in parallel, then exact sequential prefix sums (one thread per moment)
        for (int i = tid; i < sz; i += FQ_THREADS) {
            uint32_t xy = uniq[i];
            double x = (xy & 0xffff) * .5 + 0.5, y = (xy >> 16) * .5 + 0.5;
            int ix = (int)x, iy = (int)y;
            double W = 1;
            if (ix > 0 && ix + 1 < A.w && iy > 0 && iy + 1 < A.h) {
                int gx = (int)im[(size_t)iy * A.w + ix + 1] - (int)im[(size_t)iy * A.w + ix - 1];
                int gy = (int)im[(size_t)(iy + 1) * A.w + ix] - (int)im[(size_t)(iy - 1) * A.w + ix];
                W = sqrt((double)(gx * gx + gy * gy)) + 1;
            }
            double *t = lf + (size_t)i * 6;
            t[0] = W * x; t[1] = W * y; t[2] = W * x * x; t[3] = W * x * y; t[4] = W * y * y; t[5] = W;
        }
        __syncthreads();
        if (tid < 6) {
            // sequential on purpose (the dependency's summation order); 8 independent loads are in flight per step of
            // the dependent add chain
            double acc = 0;
            for (int base = 0; base < sz; base += 8) {
                double v[8];
#pragma unroll
                for (int k = 0; k < 8; k++) v[k] = base + k < sz ? lf[(size_t)(base + k) * 6 + tid] : 0.;
#pragma unroll
                for (int k = 0; k < 8; k++) { acc = acc + v[k]; v[k] = acc; }
#pragma unroll
                for (int k = 0; k < 8; k++)
                    if (base + k < sz) lf[(size_t)(base + k) * 6 + tid] = v[k];
            }
        }
        __syncthreads();

        // ---- line-fit error curve, 7-tap Gaussian (sigma 1) low-pass
        for (int i = tid; i < sz; i += FQ_THREADS) {
            LineFit lfit;
            fit_line(lf, sz, (i + sz - ksz) % sz, (i + ksz) % sz, lfit);
            e0[i] = lfit.err;
        }
        __syncthreads();
        {
            // f[j] = (float)exp(-j*j/2) for j = -3..3
            const float fw[7] = {0.011108996f, 0.13533528f, 0.60653067f, 1.0f, 0.60653067f, 0.13533528f, 0.011108996f};
            for (int i = tid; i < sz; i += FQ_THREADS) {
                double acc = 0;
#pragma unroll
                for (int t = 0; t < 7; t++) acc += e0[(i + t - 3 + sz) % sz] * fw[t];
                e1[i] = acc;
            }
        }
        __syncthreads();

        // ---- strict local maxima
        int nloc = 0;
        for (int i = tid; i < sz; i += FQ_THREADS) {
            double e = e1[i];
            nloc += (e > e1[(i + 1) % sz] && e > e1[(i + sz - 1) % sz]) ? 1 : 0;
        }
        int nmaxima;
        (void)block_scan_excl(nloc, s_warp, nmaxima);
        if (nmaxima < 4) continue;
        double thresh = -HUGE_VAL;  // keep maxima with err > thresh
        if (nmaxima > A.max_nmaxima) {
            // (max_nmaxima+1)-th largest maximum, duplicates counted: remove one instance per round
            for (int r = 0; r <= A.max_nmaxima; r++) {
                double best = -HUGE_VAL;
                int bi = -1;
                for (int i = tid; i < sz; i += FQ_THREADS) {
                    double e = e1[i];
                    if (!(e > e1[(i + 1) % sz] && e > e1[(i + sz - 1) % sz])) continue;
                    bool removed = false;
                    for (int q = 0; q < r; q++) removed |= (s_max_idx[q] == i);
                    if (removed) continue;
                    if (e > best || (e == best && i < bi)) { best = e; bi = i; }
                }
                for (int d = 16; d > 0; d >>= 1) {   // (largest error, smallest index) over the warp, then over the 4 warps
                    double ob = __shfl_xor_sync(0xffffffffu, best, d);
                    int oi = __shfl_xor_sync(0xffffffffu, bi, d);
                    if (oi >= 0 && (bi < 0 || ob > best || (ob == best && oi < bi))) { best = ob; bi = oi; }
                }
                if (lane == 0) { s_best_err[wid] = best; s_best_combo[wid] = (unsigned)bi; }
                __syncthreads();
                if (tid == 0) {
                    double b = -HUGE_VAL; int idx = -1;
                    for (int t = 0; t < FQ_THREADS / 32; t++) {
                        int ti = (int)s_best_combo[t];
                        if (ti < 0) continue;
                        if (idx < 0 || s_best_err[t] > b || (s_best_err[t] == b && ti < idx)) { b = s_best_err[t]; idx = ti; }
                    }
                    s_max_idx[r] = idx;
                    s_max_err[r] = b;
                }
                __syncthreads();
            }
            thresh = s_max_err[A.max_nmaxima];
            __syncthreads();
        }
        // gather kept maxima in index order (at most MAXIMA_CAP)
        if (tid == 0) s_i4[4] = 0;
        __syncthreads();
        for (int base = 0; base < sz; base += FQ_THREADS) {
            int i = base + tid;
            int flag = 0;
            if (i < sz) {
                double e = e1[i];
                flag = (e > e1[(i + 1) % sz] && e > e1[(i + sz - 1) % sz] && e > thresh) ? 1 : 0;
            }
            int tot;
            int pos = block_scan_excl(flag, s_warp, tot);
            int start = s_i4[4];
            if (flag && start + pos < MAXIMA_CAP) s_max_idx[start + pos] = i;
            __syncthreads();
            if (tid == 0) s_i4[4] = start + tot;
            __syncthreads();
        }
        const int m = min(s_i4[4], MAXIMA_CAP);
        if (m < 4) continue;

        // ---- line fits between all ordered pairs of maxima, then the 4-subset search
        for (int p = tid; p < m * m; p += FQ_THREADS) {
            int a = p / m, b = p % m;
            if (a != b) fit_line(lf, sz, s_max_idx[a], s_max_idx[b], s_pair[a][b]);
        }
        __syncthreads();
        double best_err = HUGE_VAL;
        unsigned best_combo = 0xffffffffu;
        const double mse_max = A.max_line_fit_mse;
        for (int p = tid; p < m * m; p += FQ_THREADS) {
            int m0 = p / m, m1 = p % m;
            if (m1 <= m0) continue;
            const LineFit &l01 = s_pair[m0][m1];
            if (l01.mse > mse_max) continue;
            for (int m2 = m1 + 1; m2 < m - 1; m2++) {
                const LineFit &l12 = s_pair[m1][m2];
                if (l12.mse > mse_max) continue;
                double dt = l01.nx * l12.nx + l01.ny * l12.ny;
                if (fabs(dt) > A.max_dot) continue;
                for (int m3 = m2 + 1; m3 < m; m3++) {
                    const LineFit &l23 = s_pair[m2][m3];
                    if (l23.mse > mse_max) continue;
                    const LineFit &l30 = s_pair[m3][m0];
                    if (l30.mse > mse_max) continue;
                    double err = l01.err + l12.err + l23.err + l30.err;
                    unsigned combo = ((unsigned)m0 << 24) | ((unsigned)m1 << 16) | ((unsigned)m2 << 8) | (unsigned)m3;
                    if (err < best_err || (err == best_err && combo < best_combo)) { best_err = err; best_combo = combo; }
                }
            }
        }
        for (int d = 16; d > 0; d >>= 1) {   // (smallest error, smallest combination) over the warp, then over the 4 warps
            double oe = __shfl_xor_sync(0xffffffffu, best_err, d);
            unsigned oc = __shfl_xor_sync(0xffffffffu, best_combo, d);
            if (oc != 0xffffffffu && (best_combo == 0xffffffffu || oe < best_err || (oe == best_err && oc < best_combo))) { best_err = oe; best_combo = oc; }
        }
        if (lane == 0) { s_best_err[wid] = best_err; s_best_combo[wid] = best_combo; }
        __syncthreads();
        if (tid == 0) {
            double be = HUGE_VAL;
            unsigned bc = 0xffffffffu;
            for (int t = 0; t < FQ_THREADS / 32; t++)
                if (s_best_combo[t] != 0xffffffffu && (bc == 0xffffffffu || s_best_err[t] < be || (s_best_err[t] == be && s_best_combo[t] < bc))) {
                    be = s_best_err[t]; bc = s_best_combo[t];
                }
            bool ok = bc != 0xffffffffu && (be / sz < (double)A.max_line_fit_mse);
            float quad[4][2];
            if (ok) {
                int idx[4] = {s_max_idx[bc >> 24], s_max_idx[(bc >> 16) & 255], s_max_idx[(bc >> 8) & 255], s_max_idx[bc & 255]};
                LineFit L[4];
                for (int i = 0; i < 4 && ok; i++) {
                    fit_line(lf, sz, idx[i], idx[(i + 1) & 3], L[i]);
                    if (L[i].mse > (double)A.max_line_fit_mse) ok = false;
                }
                for (int i = 0; i < 4 && ok; i++) {
                    int j = (i + 1) & 3;
                    double A00 = L[i].ny, A01 = -L[j].ny, A10 = -L[i].nx, A11 = L[j].nx;
                    double B0 = -L[i].Ex + L[j].Ex, B1 = -L[i].Ey + L[j].Ey;
                    double det = A00 * A11 - A10 * A01;
                    if (fabs(det) < 0.001) { ok = false; break; }
                    double det_inv = 1.0 / det;
                    double W00 = A11 * det_inv, W01 = -A01 * det_inv;
                    double L0 = W00 * B0 + W01 * B1;
                    quad[i][0] = (float)(L[i].Ex + L0 * A00);
                    quad[i][1] = (float)(L[i].Ey + L0 * A10);
                }
            }
            if (ok) {
                double area = 0, len[3], p;
                for (int i = 0; i < 3; i++) {
                    int a = i, b = (i + 1) % 3;
                    len[i] = sqrt(sq(quad[b][0] - quad[a][0]) + sq(quad[b][1] - quad[a][1]));
                }
                p = (len[0] + len[1] + len[2]) / 2;
                area += sqrt(p * (p - len[0]) * (p - len[1]) * (p - len[2]));
                const int idxs[4] = {2, 3, 0, 2};
                for (int i = 0; i < 3; i++) {
                    int a = idxs[i], b = idxs[i + 1];
                    len[i] = sqrt(sq(quad[b][0] - quad[a][0]) + sq(quad[b][1] - quad[a][1]));
                }
                p = (len[0] + len[1] + len[2]) / 2;
                area += sqrt(p * (p - len[0]) * (p - len[1]) * (p - len[2]));
                if (area < 64) ok = false;
            }
            if (ok) {
                double total = 0;
                bool res = true;
                for (int i = 0; i < 4; i++) {
                    int i0 = i, i1 = (i + 1) & 3, i2 = (i + 2) & 3;
                    double t0 = atan2f(quad[i0][1] - quad[i1][1], quad[i0][0] - quad[i1][0]);
                    double t1 = atan2f(quad[i2][1] - quad[i1][1], quad[i2][0] - quad[i1][0]);
                    double dth = t0 - t1;
                    if (dth < 0) dth += 2 * 3.14159265358979323846;
                    if (dth < A.critical_rad || dth > (3.14159265358979323846 - A.critical_rad)) res = false;
                    total += dth;
                }
                if (total < 6.2 || total > 6.4) res = false;
                ok = res;
            }
            if (ok) {
                int32_t *cnt = A.counters + f * APSE_COUNTERS;
                int qi = atomicAdd(&cnt[2], 1);
                if (qi < APSE_MAX_QUADS) {
                    float *q = A.quads + ((size_t)f * APSE_MAX_QUADS + qi) * 8;
                    const int order[4] = {3, 0, 1, 2};
                    for (int k = 0; k < 4; k++) { q[2 * k] = quad[order[k]][0]; q[2 * k + 1] = quad[order[k]][1]; }
                    // the dependency's candidate order is ascending cluster key (apse_rank_quads); qi follows thread scheduling
                    A.quad_keys[(size_t)f * APSE_MAX_QUADS + qi] = ((unsigned long long)cd.key_hi << 32) | cd.key_lo;
                } else {
                    atomicExch(&cnt[3], APSE_ERR_CAPACITY);
                }
            }
        }
    }
}

// ---------------------------------------------------------------------------------------------------------
// host side
struct DetectExtra {
    int prev_w = 0, prev_h = 0;      // geometry of the batch whose active tiles are still marked in thresh (0 = none)
    bool thresh_full = true;         // thresh holds arbitrary data everywhere (first use / after the classic path)
    uint8_t *tile_active;
    uint32_t *tile_list;
    uint32_t *used_slots;
    int *work_counter;   // [0] quad-fit work counter, [1] number of active CCL tiles, [2], [3] entries of the two A-lists
    // A-list of high-contrast 4x4 tiles, double-buffered: the list of batch k drives the reset at the start of batch k + 1
    uint32_t *alist[2] = {nullptr, nullptr};
    uint8_t *alist_thr[2] = {nullptr, nullptr};
    int acap = 0, acur = 0;
};

int apse_detect_alloc(apse_ctx *ctx)
{
    size_t B = ctx->max_batch, npx = (size_t)ctx->max_w * ctx->max_h;
    size_t ntiles = (size_t)div_up(ctx->max_w, 4) * div_up(ctx->max_h, 4);
    CUDA_TRY(ctx, cudaMalloc((void **)&ctx->thresh, B * npx));
    for (TileSlot &s : ctx->slot) CUDA_TRY(ctx, cudaMalloc((void **)&s.tmm, B * ntiles * sizeof(uint16_t)));
    CUDA_TRY(ctx, cudaMalloc((void **)&ctx->labels, B * npx * sizeof(uint32_t)));
    CUDA_TRY(ctx, cudaMalloc((void **)&ctx->points, B * APSE_MAX_POINTS * sizeof(uint4)));
    CUDA_TRY(ctx, cudaMalloc((void **)&ctx->hash_keys, B * APSE_HASH_SLOTS * sizeof(unsigned long long)));
    CUDA_TRY(ctx, cudaMalloc((void **)&ctx->hash_count, B * APSE_HASH_SLOTS * sizeof(uint32_t)));
    CUDA_TRY(ctx, cudaMalloc((void **)&ctx->hash_offset, B * APSE_HASH_SLOTS * sizeof(uint32_t)));
    CUDA_TRY(ctx, cudaMalloc((void **)&ctx->sorted_pts, B * APSE_MAX_POINTS * sizeof(uint2)));
    CUDA_TRY(ctx, cudaMalloc((void **)&ctx->sort_keys, B * APSE_MAX_POINTS * 2 * sizeof(unsigned long long)));
    CUDA_TRY(ctx, cudaMalloc((void **)&ctx->lfps, B * APSE_MAX_POINTS * 6 * sizeof(double)));
    CUDA_TRY(ctx, cudaMalloc((void **)&ctx->errs, B * APSE_MAX_POINTS * 2 * sizeof(double)));
    CUDA_TRY(ctx, cudaMalloc((void **)&ctx->clusters, B * APSE_MAX_CLUSTERS * sizeof(ClusterDesc)));
    CUDA_TRY(ctx, cudaMalloc((void **)&ctx->counters, B * APSE_COUNTERS * sizeof(int32_t)));
    CUDA_TRY(ctx, cudaMalloc((void **)&ctx->quads, B * APSE_MAX_QUADS * 8 * sizeof(float)));
    CUDA_TRY(ctx, cudaMalloc((void **)&ctx->quad_order, B * APSE_MAX_QUADS * sizeof(uint32_t)));
    CUDA_TRY(ctx, cudaMalloc((void **)&ctx->quad_keys, B * APSE_MAX_QUADS * sizeof(unsigned long long)));
    DetectExtra *ex = new DetectExtra();
    size_t nct = (size_t)div_up(ctx->max_w, CCL_TW) * div_up(ctx->max_h, CCL_TH);
    CUDA_TRY(ctx, cudaMalloc((void **)&ex->tile_active, B * nct));
    CUDA_TRY(ctx, cudaMalloc((void **)&ex->tile_list, B * nct * sizeof(uint32_t)));
    CUDA_TRY(ctx, cudaMalloc((void **)&ex->work_counter, 4 * sizeof(int)));
    CUDA_TRY(ctx, cudaMemset(ex->work_counter, 0, 4 * sizeof(int)));
    ex->acap = (int)(B * ntiles + B * (size_t)(div_up(ctx->max_w, 4) + div_up(ctx->max_h, 4) + 1));   // + partial edge tiles
    for (int k = 0; k < 2; k++) {
        CUDA_TRY(ctx, cudaMalloc((void **)&ex->alist[k], (size_t)ex->acap * sizeof(uint32_t)));
        CUDA_TRY(ctx, cudaMalloc((void **)&ex->alist_thr[k], (size_t)ex->acap));
    }
    CUDA_TRY(ctx, cudaMalloc((void **)&ex->used_slots, B * APSE_HASH_SLOTS * sizeof(uint32_t)));
    // the hash tables are cleared once; k_cluster_scan resets exactly the slots a batch used
    CUDA_TRY(ctx, cudaMemset(ctx->hash_keys, 0xff, B * APSE_HASH_SLOTS * sizeof(unsigned long long)));
    CUDA_TRY(ctx, cudaMemset(ctx->hash_count, 0, B * APSE_HASH_SLOTS * sizeof(uint32_t)));
    ctx->point_rank = reinterpret_cast<uint32_t *>(ex);  // opaque slot reused to carry the extra pointers
    return APSE_OK;
}

void apse_detect_free(apse_ctx *ctx)
{
    cudaFree(ctx->thresh); cudaFree(ctx->slot[0].tmm); cudaFree(ctx->slot[1].tmm); cudaFree(ctx->labels); cudaFree(ctx->points);
    cudaFree(ctx->hash_keys); cudaFree(ctx->hash_count); cudaFree(ctx->hash_offset); cudaFree(ctx->sorted_pts);
    cudaFree(ctx->sort_keys); cudaFree(ctx->lfps); cudaFree(ctx->errs); cudaFree(ctx->clusters); cudaFree(ctx->counters);
    cudaFree(ctx->quads); cudaFree(ctx->quad_order); cudaFree(ctx->quad_keys);
    DetectExtra *ex = reinterpret_cast<DetectExtra *>(ctx->point_rank);
    if (ex) {
        cudaFree(ex->tile_active); cudaFree(ex->tile_list); cudaFree(ex->used_slots); cudaFree(ex->work_counter);
        for (int k = 0; k < 2; k++) { cudaFree(ex->alist[k]); cudaFree(ex->alist_thr[k]); }
        delete ex;
    }
    ctx->point_rank = nullptr;
}

// persistent grid of the work-list kernels: 2 CTAs per SM
static int chain_grid(const apse_ctx *ctx)
{
    return ctx->sm_count * 2;
}

// runs K2..K5 for `batch` gray frames; leaves quads / counters in the context scratch
int apse_apriltag_quads(apse_ctx *ctx, const uint8_t *gray, int w, int h, int batch, const DeviceParams &dp, cudaStream_t st,
                        const TileSlot *tiles, uint16_t *tmm_scratch, bool flat_labels)
{
    if (w > ctx->max_w || h > ctx->max_h || batch > ctx->max_batch || batch > 64)
        CTX_FAIL(ctx, APSE_ERR_INVALID_ARG, "detect: frame %dx%d x%d exceeds the context capacity %dx%d x%d (64 max)", w, h,
                 batch, ctx->max_w, ctx->max_h, ctx->max_batch);
    if (w < 8 || h < 8 || w > 32767 || h > 32767 || (long long)div_up(w, CCL_TW) * div_up(h, CCL_TH) >= (1 << 20))
        CTX_FAIL(ctx, APSE_ERR_INVALID_ARG, "detect: unsupported image size");
    DetectExtra *ex = reinterpret_cast<DetectExtra *>(ctx->point_rank);
    int tw = w / 4, th = h / 4;
    // ternary image invariant: 127 everywhere except the tiles of the previous batch's A-list -> reset exactly those
    const int prev = ex->acur, cur = prev ^ 1;
    ex->acur = cur;
    if (ex->thresh_full || ex->prev_w != w || ex->prev_h != h) {
        if (ex->thresh_full || ex->prev_w != 0)
            CUDA_TRY(ctx, cudaMemsetAsync(ctx->thresh, 127, (size_t)ctx->max_batch * ctx->max_w * ctx->max_h, st));
        ex->thresh_full = false;
    } else {
        KLAUNCH(ctx, KID_THRESHOLD, st, k_reset_thresh<<<chain_grid(ctx), 256, 0, st>>>(ctx->thresh, w, h, ex->alist[prev], ex->work_counter + 2 + prev, ex->acap));
    }
    ex->prev_w = w; ex->prev_h = h;
    CUDA_TRY(ctx, cudaMemsetAsync(ctx->counters, 0, (size_t)batch * APSE_COUNTERS * sizeof(int32_t), st));
    CUDA_TRY(ctx, cudaMemsetAsync(ex->work_counter, 0, 2 * sizeof(int), st));
    CUDA_TRY(ctx, cudaMemsetAsync(ex->work_counter + 2 + cur, 0, sizeof(int), st));
    const int ctw = div_up(w, CCL_TW), cth = div_up(h, CCL_TH), nct = ctw * cth;
    CUDA_TRY(ctx, cudaMemsetAsync(ex->tile_active, 0, (size_t)batch * nct, st));
    int *acount = ex->work_counter + 2 + cur;
    {
        dim3 block(32, 8), grid(div_up(tw, 32), div_up(th, 8), batch);
        uint16_t *tmm = tiles ? tiles->tmm : tmm_scratch;
        if (!tiles)
            KLAUNCH(ctx, KID_TILE_MINMAX, st, k_tile_minmax<<<grid, block, 0, st>>>(gray, w, h, tw, th, tmm));
        if (tiles && tiles->bgr && tw * 4 == w && th * 4 == h) {   // sparse batch: scan only its exact tiles
            KLAUNCH(ctx, KID_THRESHOLD, st, k_threshold_scan_list<<<chain_grid(ctx), 256, 0, st>>>(tw, th, tmm, tiles->elist, tiles->ecount,
                                                                                             dp.min_white_black_diff, ex->alist[cur], ex->alist_thr[cur], acount,
                                                                                             ex->acap, ex->tile_active, ctw, cth));
        } else {
            dim3 tgrid(div_up(div_up(tw, THR_TPT), 128), th, batch);
            KLAUNCH(ctx, KID_THRESHOLD, st, k_threshold_scan<<<tgrid, 128, 0, st>>>(w, h, tw, th, tmm, dp.min_white_black_diff, ex->alist[cur],
                                                                                   ex->alist_thr[cur], acount, ex->acap, ex->tile_active, ctw, cth));
        }
        if (tw * 4 != w || th * 4 != h) {
            KLAUNCH(ctx, KID_THRESHOLD, st, k_threshold_edges<<<dim3(64, 1, batch), 256, 0, st>>>(gray, w, h, tw, th, tmm, ctx->thresh,
                                                                                     ex->tile_active, ctw, cth, ex->alist[cur], ex->alist_thr[cur],
                                                                                     acount, ex->acap));
        }
        KLAUNCH(ctx, KID_THRESHOLD, st, k_threshold_apply<<<chain_grid(ctx), 256, 0, st>>>(gray, w, h, tw, th, ex->alist[cur], ex->alist_thr[cur], acount,
                                                                                      ex->acap, ctx->thresh));
    }
    {
        // 32x16 CCL tiles (shared-memory union-find); flat_labels (debug entry point): every pixel labelled with its
        // component root.  Also the path of the classic detector (apse_ccl_binary).  Components over the 4x4 A-list tiles
        // (register flood + global border joins) gave the same results but ran 1 % slower on sparse and 10 % slower on
        // dense frames: the border joins of 4x4 tiles are four times as many global union-find operations.
        int *n_active = ex->work_counter + 1;
        KLAUNCH(ctx, KID_THRESHOLD, st, k_compact_tiles<<<div_up(batch * nct, 256), 256, 0, st>>>(ex->tile_active, batch * nct, nct, ex->tile_list, n_active));
        const int block = CCL_THREADS;
        const int grid = chain_grid(ctx) * 4;   // persistent: 16 CTAs of 128 threads per SM, tiles taken round-robin from the list
        KLAUNCH(ctx, KID_CCL_LOCAL, st, k_ccl_local<<<grid, block, 0, st>>>(ctx->thresh, w, h, ctx->labels, ex->tile_list, n_active, ctw, 0));
        KLAUNCH(ctx, KID_CCL_MERGE, st, k_ccl_merge<<<chain_grid(ctx) * 2, 256, 0, st>>>(ctx->thresh, w, h, ctx->labels, ex->tile_list, n_active, ctw, 0));
        if (flat_labels)
            KLAUNCH(ctx, KID_CCL_FLATTEN, st, k_ccl_flatten<<<grid, block, 0, st>>>(ctx->thresh, w, h, ctx->labels, ex->tile_list, n_active, ctw));
        KLAUNCH(ctx, KID_EMIT, st, k_emit_scan<<<chain_grid(ctx), 256, 0, st>>>(ctx->thresh, w, h, ex->alist[cur], acount, ex->acap, ctx->points, ctx->counters));
        KLAUNCH(ctx, KID_EMIT, st, k_emit_insert<<<dim3(ctx->sm_count, min(batch, 8)), 256, 0, st>>>(w, h, ctx->labels, ctx->hash_keys, ctx->hash_count, ex->used_slots,
                                                                                         ctx->points, ctx->counters, batch));
    }
    KLAUNCH(ctx, KID_CLUSTER_SCAN, st, k_cluster_scan<<<batch, 1024, 0, st>>>(ctx->hash_keys, ctx->hash_count, ctx->hash_offset, ex->used_slots, ctx->clusters, ctx->counters,
                                           dp.min_cluster_pixels, dp.max_cluster_points));
    KLAUNCH(ctx, KID_SCATTER, st, k_scatter_points<<<dim3(ctx->sm_count, min(batch, 8)), 256, 0, st>>>(ctx->points, ctx->hash_offset, ctx->counters, ctx->sorted_pts, batch));
    FitArgs A;
    A.gray = gray; A.w = w; A.h = h; A.batch = batch; A.clusters = ctx->clusters; A.sorted_pts = ctx->sorted_pts;
    A.sort_keys = ctx->sort_keys; A.lfps = ctx->lfps; A.errs = ctx->errs; A.counters = ctx->counters; A.quads = ctx->quads;
    A.quad_keys = ctx->quad_keys; A.work_counter = ex->work_counter; A.max_nmaxima = dp.max_nmaxima;
    A.critical_rad = dp.critical_rad; A.max_line_fit_mse = dp.max_line_fit_mse; A.max_dot = dp.max_dot;
    KLAUNCH(ctx, KID_FIT_QUADS, st, k_fit_quads<<<chain_grid(ctx) * 2, FQ_THREADS, 0, st>>>(A));   // one cluster per CTA at a time: dense frames have thousands
    return apse_rank_quads(ctx, batch, st);
}

// Components of a binary image for the classic path (classic.cu): foreground (255) 8-connected, background (0)
// 4-connected, every pixel in range, root = raster-first pixel of the component.  Labels go to ctx->labels.
int apse_ccl_binary(apse_ctx *ctx, const uint8_t *bin, int w, int h, int batch, cudaStream_t st)
{
    if ((long long)div_up(w, CCL_TW) * div_up(h, CCL_TH) >= (1 << 20)) CTX_FAIL(ctx, APSE_ERR_INVALID_ARG, "detect: unsupported image size");
    DetectExtra *ex = reinterpret_cast<DetectExtra *>(ctx->point_rank);
    ex->thresh_full = true;   // ctx->thresh is the binary image of this path: the APRILTAG invariant (127 background) is gone
    const int ctw = div_up(w, CCL_TW), cth = div_up(h, CCL_TH), nct = ctw * cth;
    int *n_active = ex->work_counter + 1;
    CUDA_TRY(ctx, cudaMemsetAsync(ex->work_counter, 0, 2 * sizeof(int), st));
    CUDA_TRY(ctx, cudaMemsetAsync(ex->tile_active, 1, (size_t)batch * nct, st));   // no low-contrast class: all tiles
    KLAUNCH(ctx, KID_THRESHOLD, st, k_compact_tiles<<<div_up(batch * nct, 256), 256, 0, st>>>(ex->tile_active, batch * nct, nct, ex->tile_list, n_active));
    const int block = CCL_THREADS;
    const int grid = chain_grid(ctx) * 4;
    KLAUNCH(ctx, KID_CCL_LOCAL, st, k_ccl_local<<<grid, block, 0, st>>>(bin, w, h, ctx->labels, ex->tile_list, n_active, ctw, 1));
    KLAUNCH(ctx, KID_CCL_MERGE, st, k_ccl_merge<<<chain_grid(ctx) * 2, 256, 0, st>>>(bin, w, h, ctx->labels, ex->tile_list, n_active, ctw, 1));
    KLAUNCH(ctx, KID_CCL_FLATTEN, st, k_ccl_flatten<<<grid, block, 0, st>>>(bin, w, h, ctx->labels, ex->tile_list, n_active, ctw));
    return APSE_OK;
}
