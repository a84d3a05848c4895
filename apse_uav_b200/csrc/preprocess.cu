// preprocess.cu -- stage 1 of the marker pipeline on B200 (sm_100a):
//   K0  build_undistort_map   aruco_detect.py:568  cv2.initUndistortRectifyMap
//   K1  preprocess_fused      aruco_detect.py:250-259 + :592  remap + RGB2LAB + LUT(L) + LAB2RGB + BGR2GRAY
//   stand-alone remap / cvtColor / LUT kernels for the drop-in cv2-shaped API
//   k_yuv420_to_bgr: a video decoder's YUV 4:2:0 frames (NV12 / NV21 / I420 / YV12) -> BGR, cv2.cvtColor-exact
// Integer pipeline, bit-exact with the dependency's 8-bit paths (SURVEY.md A.1, A.2).  HBM-bound by design:
// one pass over the BGR frame (24.9 MB read) producing gray (8.3 MB) and optionally the corrected BGR frame.
#include "common.cuh"
#include "chain.cuh"
#include <cuda.h>
#include <math.h>
#include <string.h>
#include <stdlib.h>

// ---------------------------------------------------------------------------------------------------------
// host: integer colour tables (values are what OpenCV's RGB2Lab_b / Lab2RGBinteger tables hold)
static void build_lab_tables_host(LabTables &T, const uint8_t *lut /* nullable = identity */)
{
    for (int i = 0; i < 256; i++) {
        float x = i * (1.f / 255.f);
        double g = x <= 0.04045f ? (double)(x * (1.f / 12.92f)) : (double)(float)pow((double)(x + 0.055) * (1. / 1.055), 2.4);
        T.gamma[i] = (uint16_t)lrint(2040.0 * g);
    }
    for (int i = 0; i < 3072; i++) {
        float x = i * (1.f / 2040.f);
        double c = x < 0.008856f ? (double)(x * 7.787f + 0.13793103448275862f) : cbrt((double)x);
        T.cbrt[i] = (uint16_t)lrint(32768.0 * c);
    }
    // float32 cube-root approximation of the dependency rounds these two entries the other way
    T.cbrt[49] = 9454;
    T.cbrt[628] = 22126;
    uint16_t ly[256], lf[256];
    const int BASE = 16384;
    for (int i = 0; i < 256; i++) {
        int y, f;
        if (i <= 20) {
            y = (int)lrintf((float)(i * BASE * 100) * 27.f / (float)(255 * 24389));
            f = (int)lrintf((float)BASE * (16.f / 116.f + (float)(i * 100 * 841) * 27.f / (float)(255 * 24389) / 108.f));
        } else {
            float fy = ((float)(i * 100) / 255.f + 16.f) / 116.f;
            f = (int)lrintf((float)BASE * fy);
            y = (int)lrintf((float)BASE * fy * fy * fy);
        }
        ly[i] = (uint16_t)y;
        lf[i] = (uint16_t)f;
    }
    for (int i = 0; i < 256; i++) {  // compose with the gamma LUT on L (aruco_detect.py:256)
        int j = lut ? lut[i] : i;
        T.ly[i] = ly[j];
        T.lf[i] = lf[j];
    }
    for (int i = 0; i < 4096; i++) {
        float x = i * (1.f / 4096.f);
        double v = x <= 0.0031308 ? x * 12.92 : 1.055 * pow((double)x, 1. / 2.4) - 0.055;
        long r = lrint(255.0 * v);
        T.invgamma[i] = (uint8_t)(r < 0 ? 0 : r > 255 ? 255 : r);
    }
}

int apse_upload_tables(apse_ctx *ctx, const uint8_t *lut, LabTables **dev, cudaStream_t st)
{
    LabTables T;
    build_lab_tables_host(T, lut);
    if (!*dev) CUDA_TRY(ctx, cudaMalloc((void **)dev, sizeof(LabTables)));
    CUDA_TRY(ctx, cudaMemcpyAsync(*dev, &T, sizeof(LabTables), cudaMemcpyHostToDevice, st));
    CUDA_TRY(ctx, cudaStreamSynchronize(st));  // T is a stack object
    return APSE_OK;
}

// ---------------------------------------------------------------------------------------------------------
// device: colour chain on one pixel (channel 0 is treated as "R" exactly as COLOR_RGB2LAB does on BGR data)
struct SmemTables {
    uint16_t gamma[256];
    uint16_t cbrt[3072];
    uint16_t ly[256];
    uint16_t lf[256];
    uint8_t invgamma[4096];
};

__device__ __forceinline__ void load_tables(SmemTables *s, const LabTables *g)
{
    const uint32_t *src = reinterpret_cast<const uint32_t *>(g);
    uint32_t *dst = reinterpret_cast<uint32_t *>(s);
    for (int i = threadIdx.x; i < (int)(sizeof(SmemTables) / 4); i += blockDim.x) dst[i] = src[i];
}

__device__ __forceinline__ int clip255(int v) { return min(max(v, 0), 255); }

__device__ __forceinline__ void rgb2lab_px(const SmemTables *T, int c0, int c1, int c2, int &L, int &a, int &b)
{
    int R = T->gamma[c0], G = T->gamma[c1], B = T->gamma[c2];
    int fX = T->cbrt[(R * 1777 + G * 1541 + B * 778 + 2048) >> 12];
    int fY = T->cbrt[(R * 871 + G * 2929 + B * 296 + 2048) >> 12];
    int fZ = T->cbrt[(R * 73 + G * 448 + B * 3575 + 2048) >> 12];
    L = clip255((296 * fY - 1336934 + 16384) >> 15);
    a = clip255((500 * (fX - fY) + 128 * 32768 + 16384) >> 15);
    b = clip255((200 * (fY - fZ) + 128 * 32768 + 16384) >> 15);
}

__device__ __forceinline__ int ab_to_xz(int v)
{
    // integer divisions truncate toward zero, as in the dependency's table construction
    return v <= 3390 ? v * 108 / 841 - 290 : v * v / 16384 * v / 16384;
}

__device__ __forceinline__ void lab2rgb_px(const SmemTables *T, int L, int a, int b, int &o0, int &o1, int &o2)
{
    int y = T->ly[L], f = T->lf[L];
    int adiv = ((5 * a * 53687 + 128) >> 13) - 4194;
    int bdiv = ((b * 41943 + 16) >> 9) - 10485 + 1;
    int X = ab_to_xz(f + adiv), Z = ab_to_xz(f - bdiv);
    int r0 = (12615 * X - 6296 * y - 2223 * Z + 8192) >> 14;
    int r1 = (-3773 * X + 7684 * y + 185 * Z + 8192) >> 14;
    int r2 = (217 * X - 836 * y + 4715 * Z + 8192) >> 14;
    o0 = T->invgamma[min(max(r0, 0), 4095)];
    o1 = T->invgamma[min(max(r1, 0), 4095)];
    o2 = T->invgamma[min(max(r2, 0), 4095)];
}

// ---------------------------------------------------------------------------------------------------------
// K0: undistort map (FP64 per pixel, init only)
__global__ void k_build_undistort_map(int w, int h, double fx, double fy, double u0, double v0, double k1, double k2,
                                      double p1, double p2, double k3, double k4, double k5, double k6, double s1,
                                      double s2, double s3, double s4, float *__restrict__ mapx,
                                      float *__restrict__ mapy)
{
    int j = blockIdx.x * blockDim.x + threadIdx.x, i = blockIdx.y;
    if (j >= w || i >= h) return;
    double ir0 = 1.0 / fx, ir2 = -u0 / fx, ir4 = 1.0 / fy, ir5 = -v0 / fy;
    double x = __dadd_rn(__dmul_rn(j, ir0), ir2), y = __dadd_rn(__dmul_rn(i, ir4), ir5);
    double x2 = __dmul_rn(x, x), y2 = __dmul_rn(y, y);
    double r2 = __dadd_rn(x2, y2), _2xy = __dmul_rn(__dmul_rn(2, x), y);
    double num = __dadd_rn(1, __dmul_rn(__dadd_rn(__dmul_rn(__dadd_rn(__dmul_rn(k3, r2), k2), r2), k1), r2));
    double den = __dadd_rn(1, __dmul_rn(__dadd_rn(__dmul_rn(__dadd_rn(__dmul_rn(k6, r2), k5), r2), k4), r2));
    double kr = __ddiv_rn(num, den);
    double xd = __dadd_rn(__dadd_rn(__dadd_rn(__dadd_rn(__dmul_rn(x, kr), __dmul_rn(p1, _2xy)),
                                              __dmul_rn(p2, __dadd_rn(r2, __dmul_rn(2, x2)))),
                                    __dmul_rn(s1, r2)),
                          __dmul_rn(__dmul_rn(s2, r2), r2));
    double yd = __dadd_rn(__dadd_rn(__dadd_rn(__dadd_rn(__dmul_rn(y, kr), __dmul_rn(p1, __dadd_rn(r2, __dmul_rn(2, y2)))),
                                              __dmul_rn(p2, _2xy)),
                                    __dmul_rn(s3, r2)),
                          __dmul_rn(__dmul_rn(s4, r2), r2));
    size_t o = (size_t)i * w + j;
    mapx[o] = (float)__dadd_rn(__dmul_rn(fx, xd), u0);
    mapy[o] = (float)__dadd_rn(__dmul_rn(fy, yd), v0);
}

int apse_init_undistort_map(apse_ctx *ctx, const double K[9], const double D[14], int w, int h, float *mapx,
                            float *mapy, void *stream)
{
    if (!ctx || !K || !D || !mapx || !mapy || w <= 0 || h <= 0) CTX_FAIL(ctx, APSE_ERR_INVALID_ARG, "init_undistort_map: bad argument");
    if (D[12] != 0 || D[13] != 0) CTX_FAIL(ctx, APSE_ERR_UNSUPPORTED, "tilted sensor model (tauX/tauY) is not supported");
    dim3 block(256), grid(div_up(w, 256), h);
    KLAUNCH(ctx, KID_BUILD_MAP, (cudaStream_t)stream, k_build_undistort_map<<<grid, block, 0, (cudaStream_t)stream>>>(w, h, K[0], K[4], K[2], K[5], D[0], D[1], D[2], D[3],
                                                                    D[4], D[5], D[6], D[7], D[8], D[9], D[10], D[11],
                                                                    mapx, mapy));
    return APSE_OK;
}

// K1: fused preprocess.  Block = 256 threads = 8 rows x 32 lanes, each lane 4 consecutive pixels (128 x 8 tile).
// The map of the tile is read once and kept in registers while the block walks `fpb` frames of the batch, so
// map traffic is amortised over the batch; gray is written as one 32-bit word per lane (128 B per warp).
#define K1_PX 4
__global__ void __launch_bounds__(256, 4) k_preprocess_fused(const uint8_t *__restrict__ bgr, uint8_t *__restrict__ bgr_out,
                                                          uint8_t *__restrict__ gray, const float *__restrict__ mapx,
                                                          const float *__restrict__ mapy, const LabTables *__restrict__ tables,
                                                          int w, int h, int batch, int fpb)
{
    __shared__ SmemTables T;
    load_tables(&T, tables);
    __syncthreads();
    int lane = threadIdx.x & 31, row = threadIdx.x >> 5;
    int x0 = (blockIdx.x * 32 + lane) * K1_PX, y = blockIdx.y * 8 + row;
    if (y >= h || x0 >= w) return;
    Taps taps[K1_PX];
    int npx = min(K1_PX, w - x0);
#pragma unroll
    for (int k = 0; k < K1_PX; k++) {
        int xx = min(x0 + k, w - 1);
        size_t o = (size_t)y * w + xx;
        taps[k] = make_taps(__ldg(mapx + o), __ldg(mapy + o), w, h, 3);
    }
    size_t frame_px = (size_t)w * h;
    int f0 = blockIdx.z * fpb, f1 = min(batch, f0 + fpb);
    for (int f = f0; f < f1; f++) {
        const uint8_t *src = bgr + (size_t)f * frame_px * 3;
        int g[K1_PX], o0[K1_PX], o1[K1_PX], o2[K1_PX];
#pragma unroll
        for (int k = 0; k < K1_PX; k++) {
            int c0 = sample(src, taps[k], w * 3, 3, 0);
            int c1 = sample(src, taps[k], w * 3, 3, 1);
            int c2 = sample(src, taps[k], w * 3, 3, 2);
            int L, a, b;
            rgb2lab_px(&T, c0, c1, c2, L, a, b);
            lab2rgb_px(&T, L, a, b, o0[k], o1[k], o2[k]);
            g[k] = gray_px(o0[k], o1[k], o2[k]);
        }
        size_t o = (size_t)f * frame_px + (size_t)y * w + x0;
        // 32-bit stores need 4-byte aligned rows: the caller's buffers may start anywhere
        if (npx == K1_PX && (w & 3) == 0 && (reinterpret_cast<uintptr_t>(gray) & 3) == 0 &&
            (reinterpret_cast<uintptr_t>(bgr_out) & 3) == 0) {
            *reinterpret_cast<uint32_t *>(gray + o) = (uint32_t)g[0] | ((uint32_t)g[1] << 8) | ((uint32_t)g[2] << 16) | ((uint32_t)g[3] << 24);
            if (bgr_out) {
                uint32_t *d = reinterpret_cast<uint32_t *>(bgr_out + o * 3);
                d[0] = (uint32_t)o0[0] | ((uint32_t)o1[0] << 8) | ((uint32_t)o2[0] << 16) | ((uint32_t)o0[1] << 24);
                d[1] = (uint32_t)o1[1] | ((uint32_t)o2[1] << 8) | ((uint32_t)o0[2] << 16) | ((uint32_t)o1[2] << 24);
                d[2] = (uint32_t)o2[2] | ((uint32_t)o0[3] << 8) | ((uint32_t)o1[3] << 16) | ((uint32_t)o2[3] << 24);
            }
        } else {
            for (int k = 0; k < npx; k++) {
                gray[o + k] = (uint8_t)g[k];
                if (bgr_out) {
                    bgr_out[(o + k) * 3] = (uint8_t)o0[k];
                    bgr_out[(o + k) * 3 + 1] = (uint8_t)o1[k];
                    bgr_out[(o + k) * 3 + 2] = (uint8_t)o2[k];
                }
            }
        }
    }
}

// ---------------------------------------------------------------------------------------------------------
// K1t: TMA-staged fused preprocess (the hot-path variant; k_preprocess_fused above stays as the generic path).
//
// One CTA (384 threads) owns a 64x24 output tile and walks `fpb` frames of the batch.  The bilinear taps of the
// tile (smem offset + two packed Q10 weight pairs per pixel) are computed once from the undistort map and stay in
// registers.  Per frame the bounding box of the tile's source pixels (<= 74 x 32 px for this camera; the map is
// smooth) is fetched by ONE bulk tensor copy (TMA, 3-D map over [batch][h][w*3/4] u32 words, out-of-image words
// zero-filled = BORDER_CONSTANT 0) into one of two staging buffers and sampled in place: three aligned 32-bit LDS per
// tap row, a funnel shift to the tap's byte offset, PRMT, and IDP.2A (16-bit weight x 8-bit pixel dot products).
// The next frame's box is in flight while the current one is being processed.  The colour chain uses tables composed on the host
// (P2Tables): idxY -> {cbrt, y, f}, (fX-fY) -> a-contribution, (fY-fZ) -> b-contribution, so the 8-bit Lab
// round trip costs 11 shared-memory look-ups per pixel and no clip / divide instructions.
// Tiles whose source box does not fit (folded corners of the rational model) take the direct-gather path.
// The kernel also emits the 4x4-tile min / max of gray that the APRILTAG threshold needs (a6.A1), so the
// candidate stage does not have to re-read gray for it.
#define P2_TW 64
#ifndef P2_TH
#define P2_TH 24                              // 2160 = 90 x 24: no partial block row at 4K
#define P2_THREADS 384                        // 12 warps; 3 CTAs per SM at 48 registers
#endif
#define P2_NPX 4
#define P2_BOX_WORDS 64                       // 256 B = 85 px + 1 B per box row
#ifndef P2_BOX_H
#define P2_BOX_H 32
#endif
#define P2_BOX_PX 85
#define P2_RAW_BYTES (P2_BOX_WORDS * 4 * P2_BOX_H)
#define P2_RAW_STRIDE (P2_RAW_BYTES + 128)    // staging buffers (a ring over frames), 128 B slack each
// ring depth: the full colour chain (MODE 0) spends ~2 us per frame and CTA, which covers the latency of one bulk copy; the
// bounds pass (MODE 1) is 3.4 x shorter per frame and needs more copies in flight
#define P2_STAGES(MODE) ((MODE) ? 4 : 2)
#define P2_OFF_TABLES_N(NS) ((NS) * P2_RAW_STRIDE)
// MODE 0: colour tables (P2Tables), gray + exact tile extrema out.  MODE 1 (sparse evaluation, see "sparse evaluation" below):
// the 16 KB gray-bound table, only per-tile BOUNDS of gray out.
#define SB_ENTRIES (16 * 32 * 32)             // cells of the bound table: (c0 >> 4, c1 >> 3, c2 >> 3), 32 KB
#define P2_TABLE_BYTES(MODE) ((MODE) ? SB_ENTRIES * 2 : (int)sizeof(P2Tables))
#define P2_OFF_MISC_N(MODE, NS) (P2_OFF_TABLES_N(NS) + P2_TABLE_BYTES(MODE))
#define P2_SMEM_BYTES_N(MODE, NS) (P2_OFF_MISC_N(MODE, NS) + 16 * (NS) + 16)   // full[NS], empty[NS] mbarriers, source box
#define P2_SMEM_BYTES_M(MODE) P2_SMEM_BYTES_N(MODE, P2_STAGES(MODE))
#define P2_SMEM_BYTES P2_SMEM_BYTES_M(0)
#define P2_CTA_THREADS (P2_THREADS + 32)       // 12 consumer warps + 1 TMA producer warp

static void build_p2_tables_host(P2Tables &P, const LabTables &T)
{
    memcpy(P.gamma, T.gamma, sizeof P.gamma);
    memcpy(P.invgamma, T.invgamma, sizeof P.invgamma);
    memset(P.cb, 0, sizeof P.cb);
    for (int i = 0; i <= 2040; i++) P.cb[i] = T.cbrt[i];
    for (int L = 0; L < 256; L++) P.yf[L] = (uint32_t)T.ly[L] | ((uint32_t)T.lf[L] << 16);   // ly / lf: gamma LUT on L composed in
}

int apse_upload_p2_tables(apse_ctx *ctx, const uint8_t *lut, P2Tables **dev, cudaStream_t st)
{
    LabTables T;
    build_lab_tables_host(T, lut);
    P2Tables *P = new P2Tables();
    build_p2_tables_host(*P, T);
    cudaError_t e = cudaSuccess;
    if (!*dev) e = cudaMalloc((void **)dev, sizeof(P2Tables));
    if (e == cudaSuccess) e = cudaMemcpyAsync(*dev, P, sizeof(P2Tables), cudaMemcpyHostToDevice, st);
    if (e == cudaSuccess) e = cudaStreamSynchronize(st);
    delete P;
    CUDA_TRY(ctx, e);
    return APSE_OK;
}

__device__ __forceinline__ uint32_t smem_u32(const void *p) { return (uint32_t)__cvta_generic_to_shared(p); }

__device__ __forceinline__ void mbar_wait(uint32_t mbar, uint32_t parity)
{
    asm volatile(
        "{\n"
        ".reg .pred p;\n"
        "W_%=:\n"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n"
        "@p bra D_%=;\n"
        "bra W_%=;\n"
        "D_%=:\n"
        "}\n" ::"r"(mbar), "r"(parity) : "memory");
}

__device__ __forceinline__ void tma_load_box(uint32_t dst, const CUtensorMap *tmap, int c0, int c1, int c2, uint32_t mbar)
{
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;\n" ::"r"(mbar), "r"((uint32_t)P2_RAW_BYTES) : "memory");
    asm volatile(
        "cp.async.bulk.tensor.3d.shared::cluster.global.tile.mbarrier::complete_tx::bytes [%0], [%1, {%2, %3, %4}], [%5];\n" ::"r"(dst),
        "l"(tmap), "r"(c0), "r"(c1), "r"(c2), "r"(mbar)
        : "memory");
}

// the packed tap pairs of ONE staged row at byte address a (the aligned word holding the first tap byte; shf brings that byte to
// bit 0): bytes b .. b+5 of the row are (c0 c1 c2 of tap ix, c0 c1 c2 of tap ix+1) -> T = (c0, c0', c1, c1'), U = (c2, c2', ..).
// A pixel's three channel sums (Q10) are IDP.2A of its two rows' pairs with the packed weights wA (top row) and wB (bottom row).
__device__ __forceinline__ void k1t_row(uint32_t a, uint32_t shf, uint32_t &T, uint32_t &U)
{
    uint32_t r0, r1, r2;
    asm volatile("ld.shared.u32 %0, [%1];" : "=r"(r0) : "r"(a));
    asm volatile("ld.shared.u32 %0, [%1+4];" : "=r"(r1) : "r"(a));
    asm volatile("ld.shared.u32 %0, [%1+8];" : "=r"(r2) : "r"(a));
    const uint32_t X0 = __funnelshift_r(r0, r1, shf), X1 = __funnelshift_r(r1, r2, shf);
    T = __byte_perm(X0, X1, 0x4130);
    U = __byte_perm(X0, X1, 0x5252);
}

// one thread, one frame: the four pixels of the thread's column sampled from staging buffer `boff` and pushed through the
// colour chain
template <bool WANT_BGR>
__device__ __forceinline__ void k1t_pixels(const P2Tables *T, const uint32_t (&addr)[P2_NPX], const uint32_t (&shf)[P2_NPX],
                                           const uint32_t (&wA)[P2_NPX], const uint32_t (&wB)[P2_NPX], uint32_t boff, unsigned brk,
                                           int (&g)[P2_NPX], int (&o0)[P2_NPX], int (&o1)[P2_NPX], int (&o2)[P2_NPX])
{
    uint32_t Tp = 0, Up = 0;
#pragma unroll
    for (int k = 0; k < P2_NPX; k++) {
        if (k == 0 || ((brk >> (k - 1)) & 1u)) k1t_row(addr[k] + boff, shf[k], Tp, Up);   // warp-uniform (see brk)
        uint32_t Tn, Un;
        k1t_row(addr[k] + boff + (uint32_t)(P2_BOX_WORDS * 4), shf[k], Tn, Un);
        const uint32_t d0 = __dp2a_lo(wA[k], Tp, __dp2a_lo(wB[k], Tn, 512u));
        const uint32_t d1 = __dp2a_hi(wA[k], Tp, __dp2a_hi(wB[k], Tn, 512u));
        const uint32_t d2 = __dp2a_lo(wA[k], Up, __dp2a_lo(wB[k], Un, 512u));
        g[k] = chain_px(T, (int)(d0 >> 10), (int)(d1 >> 10), (int)(d2 >> 10), o0[k], o1[k], o2[k]);
        Tp = Tn; Up = Un;
    }
}

// ---- sparse evaluation ------------------------------------------------------------------------------------------
// The detector reads gray only (a) as 4x4-tile extrema for the threshold decision (a6.A1: a tile whose 3x3-dilated range is
// below aprilTagMinWhiteBlackDiff becomes 127 and is never looked at again: 99 % of a sparse frame), (b) at the pixels of the
// remaining tiles and their 1-pixel surroundings (threshold, gradient weights of fit_quad), (c) at the 48x48 samples of every
// candidate quad.  So the colour chain (90 of K1t's 119 instructions per pixel) is needed on a few percent of the frame.
// Which few percent is decided RIGOROUSLY: BoundTable[c0 >> 4][c1 >> 3][c2 >> 3] = (min, max) of the chain's gray over all
// colours of the cell, computed by brute force over all 2^24 colours from the chain itself when the LUT is set.  K1t in MODE 1
// samples every pixel (the remap is unchanged) and reduces the cell bounds to per-tile bounds; k_sparse_flags marks the tiles
// whose dilated BOUND range reaches the threshold (P, a superset of the truly high-contrast tiles) plus a one-tile ring (E);
// k_sparse_exact runs the exact chain on E (gray + exact extrema); all other tiles get the neutral extrema (255, 0), which
// leaves every dilated range that matters untouched (every neighbour of a P tile is in E).  Results are bit-identical to the
// dense path by construction; tests/test_gpu_sparse.py checks the table against a brute-force CPU evaluation of all 2^24 colours
// and the detections against MODE 0.
// packed (lo | (255 - hi) << 16) of the cell of one pixel (d = Q10 channel sums)
__device__ __forceinline__ uint32_t bound_px(uint32_t tbl, uint32_t d0, uint32_t d1, uint32_t d2)
{
    // 2 * (c0>>4 << 10 | c1>>3 << 5 | c2>>3) + tbl; the sums are below 2^18, so the shifts leave clean fields, and the fields are
    // merged by two multiply-adds on the FMA pipe (the kernel is bound by the ALU pipe: shifts, PRMT, LOP3, VIMNMX)
    uint32_t a;
    asm("mad.lo.u32 %0, %1, 64, %2;" : "=r"(a) : "r"(d1 >> 13), "r"((d2 >> 13) << 1));
    asm("mad.lo.u32 %0, %1, 2048, %2;" : "=r"(a) : "r"(d0 >> 14), "r"(a + tbl));
    uint32_t e;
    asm volatile("ld.shared.u16 %0, [%1];" : "=r"(e) : "r"(a));
    return __byte_perm(e, 0u, 0x4140);
}

// WC: compile-time frame width (0 = run-time): row offsets of the stores become immediates for the 3840-px footage
// MODE 1: `tables` is the bound table, `tmm` receives per-tile BOUNDS (lo | hi << 8), gray / bgr_out are not touched
template <bool WANT_BGR, int NREG, int WC, bool FULL = false, int MODE = 0, int NSTAGES = 0>   // FULL: every thread of every CTA has pixels (w % 64 == 0, h % 24 == 0)
__global__ void __maxnreg__(NREG)
k_preprocess_tma(const __grid_constant__ CUtensorMap tmap, const uint8_t *__restrict__ bgr, uint8_t *__restrict__ bgr_out,
                 uint8_t *__restrict__ gray, uint16_t *__restrict__ tmm,
                 const float *__restrict__ mapx, const float *__restrict__ mapy, const void *__restrict__ tables, int w_rt, int h,
                 int batch, int fpb)
{
    extern __shared__ __align__(128) uint8_t smem[];
    constexpr int NS = NSTAGES ? NSTAGES : P2_STAGES(MODE);
    P2Tables *T = reinterpret_cast<P2Tables *>(smem + P2_OFF_TABLES_N(NS));
    unsigned long long *mbar_p = reinterpret_cast<unsigned long long *>(smem + P2_OFF_MISC_N(MODE, NS));   // full[NS], empty[NS]
    int *box = reinterpret_cast<int *>(smem + P2_OFF_MISC_N(MODE, NS) + 16 * NS);   // xmin, xmax, ymin, ymax
    const int w = WC ? WC : w_rt;
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const uint32_t mbar0 = smem_u32(mbar_p), raw0 = smem_u32(smem);
    const uint32_t tbl0 = smem_u32(smem + P2_OFF_TABLES_N(NS));

    {   // tables -> shared memory
        const uint4 *src = reinterpret_cast<const uint4 *>(tables);
        uint4 *dst = reinterpret_cast<uint4 *>(T);
        for (int i = tid; i < P2_TABLE_BYTES(MODE) / 16; i += P2_CTA_THREADS) dst[i] = __ldg(src + i);
    }
    if (tid == 0) {
        for (int b = 0; b < NS; b++) {
            asm volatile("mbarrier.init.shared::cta.b64 [%0], 1;\n" ::"r"(mbar0 + 8 * b));          // full[b]: the producer's expect_tx arrival
            asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;\n" ::"r"(mbar0 + 8 * (NS + b)), "r"(P2_THREADS / 32));   // empty[b]: one arrival per consumer warp
        }
        asm volatile("fence.mbarrier_init.release.cluster;\n" ::: "memory");
        box[0] = INT32_MAX; box[1] = INT32_MIN; box[2] = INT32_MAX; box[3] = INT32_MIN;
    }
    __syncthreads();

    // ---- taps of this thread's 4 pixels: column x, rows y0..y0+3
    const int x = blockIdx.x * P2_TW + (warp & 1) * 32 + lane;
    const int y0 = blockIdx.y * P2_TH + (warp >> 1) * 4;
    const bool producer = warp == P2_THREADS / 32;   // 13th warp: issues the bulk tensor copies, owns no pixels
    const bool valid = !producer && (FULL || (x < w && y0 < h));   // h % 4 == 0: a 4-row group is inside or outside as a whole
    int ixs[P2_NPX], iys[P2_NPX];
    uint32_t wA[P2_NPX], wB[P2_NPX];
    int xmin = INT32_MAX, xmax = INT32_MIN, ymin = INT32_MAX, ymax = INT32_MIN;
#pragma unroll
    for (int k = 0; k < P2_NPX; k++) {
        ixs[k] = iys[k] = 0; wA[k] = wB[k] = 0;
        if (valid) {
            size_t o = (size_t)(y0 + k) * w + x;
            int sx = q5(__ldg(mapx + o)), sy = q5(__ldg(mapy + o));
            int ix = sx >> 5, iy = sy >> 5, fx = sx & 31, fy = sy & 31;
            // taps completely outside the image contribute 0: clamp them next to the image so that the box stays small
            ix = min(max(ix, -2), w + 1); iy = min(max(iy, -2), h + 1);
            ixs[k] = ix; iys[k] = iy;
            wA[k] = (uint32_t)((32 - fy) * (32 - fx)) | ((uint32_t)((32 - fy) * fx) << 16);
            wB[k] = (uint32_t)(fy * (32 - fx)) | ((uint32_t)(fy * fx) << 16);
            xmin = min(xmin, ix); xmax = max(xmax, ix + 1); ymin = min(ymin, iy); ymax = max(ymax, iy + 1);
        }
    }
    xmin = __reduce_min_sync(0xffffffffu, xmin); xmax = __reduce_max_sync(0xffffffffu, xmax);
    ymin = __reduce_min_sync(0xffffffffu, ymin); ymax = __reduce_max_sync(0xffffffffu, ymax);
    if (lane == 0 && xmin != INT32_MAX) { atomicMin(&box[0], xmin); atomicMax(&box[1], xmax); atomicMin(&box[2], ymin); atomicMax(&box[3], ymax); }
    __syncthreads();
    const int bx0 = box[0] & ~15, by0 = box[2];   // TMA: the innermost start coordinate must be 16-byte aligned (16 px = 48 B)
    const int bw = box[1] - bx0 + 1, bh = box[3] - by0 + 1;
    const bool fast = bw <= P2_BOX_PX && bh <= P2_BOX_H;   // CTA-uniform
    // per pixel: shared-memory byte address (buffer 0) of the aligned word holding the first tap byte, and the funnel
    // shift (0 / 8 / 16 / 24) that brings that byte to bit 0
    uint32_t addr[P2_NPX], shf[P2_NPX];
#pragma unroll
    for (int k = 0; k < P2_NPX; k++) {
        int b = valid ? (ixs[k] - bx0) * 3 : 0, r = valid ? iys[k] - by0 : 0;
        addr[k] = raw0 + (uint32_t)(r * (P2_BOX_WORDS * 4) + (b & ~3));
        shf[k] = (uint32_t)(b & 3) * 8;
    }
    // Where pixel k + 1 of every thread of the warp sits in the source column of pixel k, one row further down (most of an
    // undistortion map), the bottom tap row of pixel k is the top tap row of pixel k + 1 and is staged once.  brk: bit k set =
    // somewhere in the warp that does not hold between pixels k and k + 1 (warp-uniform, so the branches below do not diverge)
    // MODE 0 stages all eight rows (measured: sharing does not pay there -- the dense kernel runs out of shared-memory
    // wavefronts in the colour chain, config 1 went from 26.6 k to 26.2 k frames/s)
    unsigned brk = MODE ? 0u : 7u;
    if (MODE) {
#pragma unroll
        for (int k = 0; k + 1 < P2_NPX; k++) {
            const bool same = addr[k + 1] == addr[k] + P2_BOX_WORDS * 4 && shf[k + 1] == shf[k];
            if (__any_sync(0xffffffffu, valid && !same)) brk |= 1u << k;
        }
    }

    const size_t frame_px = (size_t)w * h;
    const int f0 = blockIdx.z * fpb, f1 = min(batch, f0 + fpb);
    const int tw4 = w >> 2;
    const int c0x = (bx0 * 3) >> 2;
    // output cursors of this thread, advanced by one frame per iteration
    uint8_t *gp = MODE ? nullptr : gray + (size_t)f0 * frame_px + (size_t)(valid ? y0 : 0) * w + (valid ? x : 0);
    uint8_t *cp = WANT_BGR ? bgr_out + ((size_t)f0 * frame_px + (size_t)(valid ? y0 : 0) * w + (valid ? x : 0)) * 3 : nullptr;
    const size_t tile_stride = (size_t)(h >> 2) * tw4;
    uint16_t *tp = tmm ? tmm + (size_t)f0 * tile_stride + (size_t)((valid ? y0 : 0) >> 2) * tw4 + ((valid ? x : 0) >> 2) : nullptr;
    const bool tile_writer = valid && (lane & 3) == 0;

    // 4x4-tile reduction of the packed (min | (255 - max) << 16) of this thread's column over the 4 lanes of the tile
    auto tile_out = [&](uint32_t pk) {
        pk = __vminu2(pk, __shfl_xor_sync(0xffffffffu, pk, 1));
        pk = __vminu2(pk, __shfl_xor_sync(0xffffffffu, pk, 2));
        if (tile_writer) *tp = (uint16_t)((pk & 0xffu) | ((255u - (pk >> 16)) << 8));
        tp += tile_stride;
    };
    // stores of one frame + the 4x4-tile extrema (this thread holds one column of a tile, 4 lanes hold its columns),
    // then advance the cursors
    auto finish = [&](const int (&g)[P2_NPX], const int (&o0)[P2_NPX], const int (&o1)[P2_NPX], const int (&o2)[P2_NPX]) {
        if (valid) {
#pragma unroll
            for (int k = 0; k < P2_NPX; k++) {
                gp[(size_t)k * w] = (uint8_t)g[k];
                if (WANT_BGR) {
                    uint8_t *d = cp + (size_t)k * w * 3;
                    d[0] = (uint8_t)o0[k]; d[1] = (uint8_t)o1[k]; d[2] = (uint8_t)o2[k];
                }
            }
        }
        if (tmm) {
            int mn = 255, mx = 0;
            if (valid) {
                mn = min(min(g[0], g[1]), min(g[2], g[3]));
                mx = max(max(g[0], g[1]), max(g[2], g[3]));
            }
            // min and (255 - max) side by side in one register: one shuffle + one VIMNMX.U16x2 per butterfly step
            tile_out((uint32_t)mn | ((uint32_t)(255 - mx) << 16));
        }
        gp += frame_px;
        if (WANT_BGR) cp += frame_px * 3;
    };
    // MODE 1: cell bounds of the four pixels sampled from staging buffer `boff`, reduced to the tile
    auto bounds_frame = [&](uint32_t boff) {
        uint32_t pk = 0x00ff00ffu;   // (min 255, max 0)
        if (valid) {
            uint32_t Tp = 0, Up = 0;
#pragma unroll
            for (int k = 0; k < P2_NPX; k++) {
                if (k == 0 || ((brk >> (k - 1)) & 1u)) k1t_row(addr[k] + boff, shf[k], Tp, Up);   // warp-uniform
                uint32_t Tn, Un;
                k1t_row(addr[k] + boff + (uint32_t)(P2_BOX_WORDS * 4), shf[k], Tn, Un);
                const uint32_t d0 = __dp2a_lo(wA[k], Tp, __dp2a_lo(wB[k], Tn, 512u));
                const uint32_t d1 = __dp2a_hi(wA[k], Tp, __dp2a_hi(wB[k], Tn, 512u));
                const uint32_t d2 = __dp2a_lo(wA[k], Up, __dp2a_lo(wB[k], Un, 512u));
                pk = __vminu2(pk, bound_px(tbl0, d0, d1, d2));
                Tp = Tn; Up = Un;
            }
        }
        return pk;
    };
    if (fast) {
        // Producer / consumer over two staging buffers with full / empty mbarriers; no CTA-wide barrier in the frame loop, so
        // the consumer warps drift apart and hide each other's shared-memory latency.
        //   producer (one lane): wait until the 12 consumer warps have released buffer b, arm full[b], issue the copy of frame i
        //   consumer warp:       wait full[b], sample + colour chain + stores, release buffer b (one arrival per warp)
        const int nf = f1 - f0;
        if (producer) {
            if (lane == 0) {
                for (int i = 0; i < nf; i++) {
                    const int b = i % NS;
                    if (i >= NS) mbar_wait(mbar0 + 8 * (NS + b), (uint32_t)(i / NS - 1) & 1u);
                    tma_load_box(raw0 + b * P2_RAW_STRIDE, &tmap, c0x, by0, f0 + i, mbar0 + 8 * b);
                }
            }
            return;
        }
        // NS frames per trip: staging buffer and barriers of a frame are compile-time constants
        for (int i = 0; i < nf; i += NS) {
            const uint32_t ph = (uint32_t)(i / NS) & 1u;
#pragma unroll
            for (int b = 0; b < NS; b++) {
                if (i + b >= nf) break;
                mbar_wait(mbar0 + 8 * b, ph);
                if (MODE) {
                    const uint32_t pk = bounds_frame((uint32_t)(b * P2_RAW_STRIDE));
                    __syncwarp();
                    if (lane == 0) asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];\n" ::"r"(mbar0 + 8 * (NS + b)) : "memory");
                    tile_out(pk);
                } else {
                    int g[P2_NPX], o0[P2_NPX], o1[P2_NPX], o2[P2_NPX];
                    if (valid) k1t_pixels<WANT_BGR>(T, addr, shf, wA, wB, (uint32_t)(b * P2_RAW_STRIDE), brk, g, o0, o1, o2);
                    __syncwarp();
                    if (lane == 0) asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];\n" ::"r"(mbar0 + 8 * (NS + b)) : "memory");
                    finish(g, o0, o1, o2);
                }
            }
        }
    } else if (!producer) {
        // direct-gather path (source box larger than the staging buffer: folded corners of the rational model)
        for (int f = f0; f < f1; f++) {
            int g[P2_NPX], o0[P2_NPX], o1[P2_NPX], o2[P2_NPX];
            uint32_t pk = 0x00ff00ffu;
            if (valid) {
                const uint8_t *src = bgr + (size_t)f * frame_px * 3;
#pragma unroll
                for (int k = 0; k < P2_NPX; k++) {
                    size_t o = (size_t)(y0 + k) * w + x;
                    Taps t = make_taps(__ldg(mapx + o), __ldg(mapy + o), w, h, 3);
                    int c0 = sample(src, t, w * 3, 3, 0), c1 = sample(src, t, w * 3, 3, 1), c2 = sample(src, t, w * 3, 3, 2);
                    if (MODE) pk = __vminu2(pk, bound_px(tbl0, (uint32_t)c0 << 10, (uint32_t)c1 << 10, (uint32_t)c2 << 10));
                    else g[k] = chain_px(T, c0, c1, c2, o0[k], o1[k], o2[k]);
                }
            }
            if (MODE) tile_out(pk);
            else finish(g, o0, o1, o2);
        }
    }
}

typedef CUresult (*PFN_tmapEncodeTiled)(CUtensorMap *, CUtensorMapDataType, cuuint32_t, void *, const cuuint64_t *, const cuuint64_t *,
                                        const cuuint32_t *, const cuuint32_t *, CUtensorMapInterleave, CUtensorMapSwizzle,
                                        CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

static PFN_tmapEncodeTiled get_tmap_encoder()
{
    static PFN_tmapEncodeTiled fn = nullptr;
    static bool tried = false;
    if (!tried) {
        tried = true;
        void *p = nullptr;
        cudaDriverEntryPointQueryResult q;
        if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &q) == cudaSuccess && q == cudaDriverEntryPointSuccess)
            fn = (PFN_tmapEncodeTiled)p;
    }
    return fn;
}

// fused preprocess of a batch; tmm (nullable) receives the 4x4-tile extrema of gray (min | max << 8): [batch][h/4][w/4]
int apse_preprocess_ex(apse_ctx *ctx, const uint8_t *bgr, uint8_t *bgr_out, uint8_t *gray, uint16_t *tmm, int batch,
                       cudaStream_t st)
{
    int w = ctx->w, h = ctx->h;
    PFN_tmapEncodeTiled enc = get_tmap_encoder();
    bool tma_ok = enc && (w % 4) == 0 && (h % 4) == 0 && ((w * 3) % 16) == 0 && w >= P2_TW && h >= P2_TH && ((uintptr_t)bgr % 16) == 0 && ctx->tables2;
    CUtensorMap tmap;
    if (tma_ok) {
        // every global stride must be a multiple of 16 bytes (checked above); an encoder that still refuses the frame geometry
        // sends the batch to the generic kernel instead of failing the call
        cuuint64_t dims[3] = {(cuuint64_t)(w * 3 / 4), (cuuint64_t)h, (cuuint64_t)batch};
        cuuint64_t strides[2] = {(cuuint64_t)w * 3, (cuuint64_t)w * 3 * h};
        cuuint32_t boxd[3] = {P2_BOX_WORDS, P2_BOX_H, 1}, estr[3] = {1, 1, 1};
        CUresult r = enc(&tmap, CU_TENSOR_MAP_DATA_TYPE_UINT32, 3, (void *)bgr, dims, strides, boxd, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
                         CU_TENSOR_MAP_SWIZZLE_NONE, CU_TENSOR_MAP_L2_PROMOTION_L2_128B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
        if (r != CUDA_SUCCESS) tma_ok = false;
    }
    if (!tma_ok) {
        int fpb = batch >= 8 ? 8 : batch;
        dim3 grid(div_up(w, 32 * K1_PX), div_up(h, 8), div_up(batch, fpb));
        KLAUNCH(ctx, KID_PREPROCESS, st, k_preprocess_fused<<<grid, 256, 0, st>>>(bgr, bgr_out, gray, ctx->mapx, ctx->mapy, ctx->tables, w, h, batch, fpb));
        return 1;   // tile extrema not produced
    }
    // registers per thread at 4K: at 64 the resident preprocess CTAs fill the register file and every CTA of the
    // candidate / decode / pose chain on the other streams displaces one of them; 48 (no spills, 9 % fewer instructions than
    // the 40-register build) = three 384-thread CTAs per SM with 10 K registers left for chain CTAs
    if (!ctx->k1_attr_set) {
        CUDA_TRY(ctx, cudaFuncSetAttribute(k_preprocess_tma<false, 64, 0>, cudaFuncAttributeMaxDynamicSharedMemorySize, P2_SMEM_BYTES));
        CUDA_TRY(ctx, cudaFuncSetAttribute(k_preprocess_tma<true, 64, 0>, cudaFuncAttributeMaxDynamicSharedMemorySize, P2_SMEM_BYTES));
        CUDA_TRY(ctx, cudaFuncSetAttribute(k_preprocess_tma<false, 48, 3840>, cudaFuncAttributeMaxDynamicSharedMemorySize, P2_SMEM_BYTES));
        CUDA_TRY(ctx, cudaFuncSetAttribute(k_preprocess_tma<false, 48, 3840, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, P2_SMEM_BYTES));
        ctx->k1_attr_set = true;
    }
    // frames per CTA: the tap set-up (map reads, box reduction, table load) is amortised over up to 20 frames
    const int nz = div_up(batch, 20), fpb = div_up(batch, nz);
    dim3 grid(div_up(w, P2_TW), div_up(h, P2_TH), nz);
#define K1T_ARGS tmap, bgr, bgr_out, gray, tmm, ctx->mapx, ctx->mapy, ctx->tables2, w, h, batch, fpb
    if (bgr_out)
        KLAUNCH(ctx, KID_PREPROCESS, st, k_preprocess_tma<true, 64, 0><<<grid, P2_CTA_THREADS, P2_SMEM_BYTES, st>>>(K1T_ARGS));
    else if (w == 3840 && h % P2_TH == 0)
        KLAUNCH(ctx, KID_PREPROCESS, st, k_preprocess_tma<false, 48, 3840, true><<<grid, P2_CTA_THREADS, P2_SMEM_BYTES, st>>>(K1T_ARGS));
    else if (w == 3840)
        KLAUNCH(ctx, KID_PREPROCESS, st, k_preprocess_tma<false, 48, 3840><<<grid, P2_CTA_THREADS, P2_SMEM_BYTES, st>>>(K1T_ARGS));
    else
        KLAUNCH(ctx, KID_PREPROCESS, st, k_preprocess_tma<false, 64, 0><<<grid, P2_CTA_THREADS, P2_SMEM_BYTES, st>>>(K1T_ARGS));
#undef K1T_ARGS
    return APSE_OK;
}

// ---------------------------------------------------------------------------------------------------------
// sparse evaluation: bound table, tile flags, exact chain on the flagged tiles (see the comment above bound_px)

// one CTA per cell of the bound table: the exact chain on the cell's 16 x 8 x 8 colours, min / max of gray
__global__ void __launch_bounds__(256) k_build_bounds(const P2Tables *__restrict__ tables, uint16_t *__restrict__ out)
{
    __shared__ P2Tables T;
    __shared__ int s_mn[8], s_mx[8];
    {
        const uint4 *src = reinterpret_cast<const uint4 *>(tables);
        uint4 *dst = reinterpret_cast<uint4 *>(&T);
        for (int i = threadIdx.x; i < (int)(sizeof(P2Tables) / 16); i += blockDim.x) dst[i] = __ldg(src + i);
    }
    __syncthreads();
    const int cell = blockIdx.x, i0 = cell >> 10, i1 = (cell >> 5) & 31, i2 = cell & 31;
    int mn = 255, mx = 0;
    for (int j = threadIdx.x; j < 16 * 8 * 8; j += blockDim.x) {
        int o0, o1, o2;
        const int g = chain_px(&T, i0 * 16 + (j >> 6), i1 * 8 + ((j >> 3) & 7), i2 * 8 + (j & 7), o0, o1, o2);
        mn = min(mn, g); mx = max(mx, g);
    }
    mn = __reduce_min_sync(0xffffffffu, mn); mx = __reduce_max_sync(0xffffffffu, mx);
    if ((threadIdx.x & 31) == 0) { s_mn[threadIdx.x >> 5] = mn; s_mx[threadIdx.x >> 5] = mx; }
    __syncthreads();
    if (threadIdx.x == 0) {
        for (int i = 1; i < 8; i++) { mn = min(mn, s_mn[i]); mx = max(mx, s_mx[i]); }
        out[cell] = (uint16_t)(mn | ((255 - mx) << 8));
    }
}

int apse_build_bound_table(apse_ctx *ctx, cudaStream_t st)
{
    if (!ctx->btable) CUDA_TRY(ctx, cudaMalloc((void **)&ctx->btable, SB_ENTRIES * sizeof(uint16_t)));
    KLAUNCH(ctx, KID_SPARSE_FLAGS, st, k_build_bounds<<<SB_ENTRIES, 256, 0, st>>>(ctx->tables2, ctx->btable));
    return APSE_OK;
}

// P = tiles whose 3x3-dilated BOUND range reaches the threshold; E = P dilated by one tile.  E tiles go to the list of the
// exact pass; every tile of the frame first gets the neutral extrema (min 255, max 0), the exact pass overwrites those of E.
// One thread = 8 consecutive tiles of a tile row, walking down SFL_ROWS rows: the horizontally dilated bounds of the five rows
// around the current one slide through registers (one new row per step), two tiles per register, 16-bit SIMD min / max
// (VIMNMX3.U16x2), no shared memory.  Requires tw % 8 == 0.
#define SFL_ROWS 6
struct FlagRow { uint32_t mn[6], mx[6]; };   // horizontally dilated bounds, column pair j = (tx0 - 2 + 2j, tx0 - 1 + 2j)

__device__ __forceinline__ void flag_row_load(const uint16_t *__restrict__ T, int tw, int th, int tx0, int yy, FlagRow &R)
{
    uint32_t wv[6] = {0x00ff00ffu, 0x00ff00ffu, 0x00ff00ffu, 0x00ff00ffu, 0x00ff00ffu, 0x00ff00ffu};   // (min 255, max 0) pairs
    if (yy >= 0 && yy < th) {
        const uint16_t *row = T + (size_t)yy * tw;
        const uint4 q = __ldg(reinterpret_cast<const uint4 *>(row + tx0));
        wv[1] = q.x; wv[2] = q.y; wv[3] = q.z; wv[4] = q.w;
        if (tx0 > 0) wv[0] = __ldg(reinterpret_cast<const uint32_t *>(row + tx0 - 2));
        if (tx0 + 8 < tw) wv[5] = __ldg(reinterpret_cast<const uint32_t *>(row + tx0 + 8));
    }
    uint32_t mn[6], mx[6];
#pragma unroll
    for (int j = 0; j < 6; j++) { mn[j] = wv[j] & 0x00ff00ffu; mx[j] = __byte_perm(wv[j], 0u, 0x4341); }
#pragma unroll
    for (int j = 0; j < 6; j++) {
        // neighbours of pair j: (col 2j-1, col 2j) and (col 2j+1, col 2j+2); outside the 12 columns: neutral
        const uint32_t ln = j == 0 ? __byte_perm(0x00ffu, mn[0], 0x5410) : __byte_perm(mn[j - 1], mn[j], 0x5432);
        const uint32_t rn = j == 5 ? __byte_perm(mn[5], 0x00ffu, 0x5432) : __byte_perm(mn[j], mn[j + 1], 0x5432);
        const uint32_t lx = j == 0 ? __byte_perm(0u, mx[0], 0x5410) : __byte_perm(mx[j - 1], mx[j], 0x5432);
        const uint32_t rx = j == 5 ? __byte_perm(mx[5], 0u, 0x5432) : __byte_perm(mx[j], mx[j + 1], 0x5432);
        R.mn[j] = __vimin3_u16x2(ln, mn[j], rn);
        R.mx[j] = __vimax3_u16x2(lx, mx[j], rx);
    }
}

// P of one tile row for the 12 columns (bit c: column tx0 - 2 + c; the outer two are incomplete and masked by the caller)
__device__ __forceinline__ unsigned flag_row_p(const FlagRow &A, const FlagRow &B, const FlagRow &C, uint32_t kk)
{
    unsigned p = 0;
#pragma unroll
    for (int j = 0; j < 6; j++) {
        const uint32_t vmn = __vimin3_u16x2(A.mn[j], B.mn[j], C.mn[j]), vmx = __vimax3_u16x2(A.mx[j], B.mx[j], C.mx[j]);
        const uint32_t t = ((vmx | 0x80008000u) - vmn) - kk;   // bit 15 / 31: range >= diff (k_threshold_scan)
        p |= ((t >> 15) & 1u) << (2 * j) | (t >> 31) << (2 * j + 1);
    }
    return p;
}

__global__ void __launch_bounds__(128) k_sparse_flags(const uint16_t *__restrict__ tb, int tw, int th, int min_wb_diff,
                                                      uint16_t *__restrict__ tmm, uint8_t *__restrict__ eflag,
                                                      uint32_t *__restrict__ elist, int *__restrict__ ecount)
{
    const int groups = tw >> 3;
    const int gi = blockIdx.x * blockDim.x + threadIdx.x, f = blockIdx.z, lane = threadIdx.x & 31;
    const int tx0 = gi * 8, ty0 = blockIdx.y * SFL_ROWS, ty1 = min(th, ty0 + SFL_ROWS);
    const uint16_t *T = tb + (size_t)f * tw * th;
    const bool live = gi < groups;
    const uint32_t kk = (uint32_t)min(max(min_wb_diff, 0), 256) * 0x00010001u;
    unsigned colmask = 0x7feu;   // P is complete for columns tx0 - 1 .. tx0 + 8 = bits 1 .. 10; columns outside the image never count
    if (tx0 == 0) colmask &= ~2u;
    if (tx0 + 8 >= tw) colmask &= ~(1u << 10);
    // rows ty - 2 .. ty + 1 of the first tile row; P of rows ty - 1 and ty
    FlagRow r0, r1, r2, r3;
    unsigned p_prev = 0, p_cur = 0;
    if (live) {
        flag_row_load(T, tw, th, tx0, ty0 - 2, r0);
        flag_row_load(T, tw, th, tx0, ty0 - 1, r1);
        flag_row_load(T, tw, th, tx0, ty0, r2);
        flag_row_load(T, tw, th, tx0, ty0 + 1, r3);
        if (ty0 - 1 >= 0) p_prev = flag_row_p(r0, r1, r2, kk) & colmask;
        p_cur = flag_row_p(r1, r2, r3, kk) & colmask;
    }
    for (int ty = ty0; ty < ty1; ty++) {
        unsigned e8 = 0;
        if (live) {
            r1 = r2; r2 = r3;                                   // r1 = row ty, r2 = row ty + 1
            flag_row_load(T, tw, th, tx0, ty + 2, r3);
            const unsigned p_next = ty + 1 < th ? flag_row_p(r1, r2, r3, kk) & colmask : 0u;
            const unsigned prow = p_prev | p_cur | p_next;
            p_prev = p_cur; p_cur = p_next;
            e8 = ((prow >> 1) | (prow >> 2) | (prow >> 3)) & 0xffu;   // bit c: tile tx0 + c is within one tile of a P tile
            const size_t o = (size_t)f * tw * th + (size_t)ty * tw + tx0;
            uint2 fl;
            fl.x = ((e8 & 1u) ? 1u : 0u) | ((e8 & 2u) ? 0x100u : 0u) | ((e8 & 4u) ? 0x10000u : 0u) | ((e8 & 8u) ? 0x1000000u : 0u);
            fl.y = ((e8 & 16u) ? 1u : 0u) | ((e8 & 32u) ? 0x100u : 0u) | ((e8 & 64u) ? 0x10000u : 0u) | ((e8 & 128u) ? 0x1000000u : 0u);
            *reinterpret_cast<uint2 *>(eflag + o) = fl;
            *reinterpret_cast<uint4 *>(tmm + o) = make_uint4(0x00ff00ffu, 0x00ff00ffu, 0x00ff00ffu, 0x00ff00ffu);
        }
        if (!__any_sync(0xffffffffu, e8 != 0)) continue;
        const int cnt = __popc(e8);
        int inc = cnt;
#pragma unroll
        for (int d = 1; d < 32; d <<= 1) { int t = __shfl_up_sync(0xffffffffu, inc, d); if (lane >= d) inc += t; }
        int base = 0;
        if (lane == 31) base = atomicAdd(ecount, inc);
        base = __shfl_sync(0xffffffffu, base, 31) + inc - cnt;
#pragma unroll
        for (int c = 0; c < 8; c++)
            if ((e8 >> c) & 1u) elist[base++] = ATILE(f, tx0 + c, ty);
    }
}

// exact chain on the listed tiles: 4 lanes per tile, a lane = one column of the tile (4 pixels), so that the list entry, the
// frame base and the tile reduction are paid once per 4 pixels and the tap rows of vertically adjacent pixels are shared where
// the map allows (as in K1t): 5 gathered rows instead of 8.  Interior taps through aligned 32-bit loads + funnel shift + PRMT +
// IDP.2A with Q10 weights (rows of the frame are 4-byte aligned: w % 4 == 0); a column with a tap on or beyond the frame border
// takes the general sampler.  The gray bytes of a tile are transposed over its 4 lanes (2 shuffles) and leave as one 32-bit
// store per row.  Each 256-thread CTA loads the 9.7 KB of colour tables into shared memory once.
__device__ __forceinline__ void gather_row(const uint8_t *__restrict__ p, uint32_t shf, uint32_t &T, uint32_t &U)
{
    const uint32_t *r = reinterpret_cast<const uint32_t *>(p);
    const uint32_t r0 = __ldg(r), r1 = __ldg(r + 1), r2 = __ldg(r + 2);
    const uint32_t X0 = __funnelshift_r(r0, r1, shf), X1 = __funnelshift_r(r1, r2, shf);
    T = __byte_perm(X0, X1, 0x4130);
    U = __byte_perm(X0, X1, 0x5252);
}

__global__ void __launch_bounds__(256) k_sparse_exact(const uint8_t *__restrict__ bgr, const float *__restrict__ mapx, const float *__restrict__ mapy,
                                                      const P2Tables *tables, int w, int h, const uint32_t *__restrict__ elist,
                                                      const int *__restrict__ ecount, uint8_t *__restrict__ gray, uint16_t *__restrict__ tmm)
{
    __shared__ P2Tables Ts;
    {
        const uint4 *src = reinterpret_cast<const uint4 *>(tables);
        uint4 *dst = reinterpret_cast<uint4 *>(&Ts);
        for (int i = threadIdx.x; i < (int)(sizeof(P2Tables) / 16); i += blockDim.x) dst[i] = __ldg(src + i);
    }
    __syncthreads();
    tables = &Ts;
    const int n = *ecount, tw = w >> 2, th = h >> 2, col = threadIdx.x & 3;
    const size_t frame_px = (size_t)w * h;
    const uint32_t rowb = (uint32_t)w * 3u;
    for (int base = blockIdx.x * 64; base < n; base += gridDim.x * 64) {   // whole warps iterate together (shuffles below)
        const int it = base + (threadIdx.x >> 2);
        const bool live = it < n;
        const uint32_t e = live ? __ldg(elist + it) : 0u;
        const int tx = ATILE_TX(e), ty = ATILE_TY(e), f = ATILE_F(e);
        const int x = tx * 4 + col, y0 = ty * 4;
        const uint8_t *src = bgr + (size_t)f * frame_px * 3;
        int g[4] = {0, 0, 0, 0};
        if (live) {
            int sx[4], sy[4];
            bool interior = true;
#pragma unroll
            for (int k = 0; k < 4; k++) {
                const uint32_t o = (uint32_t)(y0 + k) * (uint32_t)w + (uint32_t)x;
                sx[k] = q5(__ldg(mapx + o)); sy[k] = q5(__ldg(mapy + o));
                const int ix = sx[k] >> 5, iy = sy[k] >> 5;
                interior = interior && ix >= 0 && ix + 4 < w && iy >= 0 && iy + 1 < h;
            }
            if (interior) {
                uint32_t Tp = 0, Up = 0;
                int pix = 0, piy = 0;
#pragma unroll
                for (int k = 0; k < 4; k++) {
                    const int ix = sx[k] >> 5, iy = sy[k] >> 5, fx = sx[k] & 31, fy = sy[k] & 31;
                    const uint32_t wA = (uint32_t)((32 - fy) * (32 - fx)) | ((uint32_t)((32 - fy) * fx) << 16);
                    const uint32_t wB = (uint32_t)(fy * (32 - fx)) | ((uint32_t)(fy * fx) << 16);
                    const uint32_t b = (uint32_t)ix * 3u, shf = (b & 3u) * 8u;
                    const uint8_t *r0 = src + (size_t)((uint32_t)iy * rowb + (b & ~3u));
                    if (k == 0 || ix != pix || iy != piy + 1) gather_row(r0, shf, Tp, Up);   // else: the previous pixel's bottom row
                    uint32_t Tn, Un;
                    gather_row(r0 + rowb, shf, Tn, Un);
                    const int c0 = (int)(__dp2a_lo(wA, Tp, __dp2a_lo(wB, Tn, 512u)) >> 10);
                    const int c1 = (int)(__dp2a_hi(wA, Tp, __dp2a_hi(wB, Tn, 512u)) >> 10);
                    const int c2 = (int)(__dp2a_lo(wA, Up, __dp2a_lo(wB, Un, 512u)) >> 10);
                    int o0, o1, o2;
                    g[k] = chain_px(tables, c0, c1, c2, o0, o1, o2);
                    Tp = Tn; Up = Un; pix = ix; piy = iy;
                }
            } else {
#pragma unroll
                for (int k = 0; k < 4; k++) g[k] = exact_gray_px(src, mapx, mapy, tables, w, h, x, y0 + k);
            }
        }
        // tile extrema over the 4 lanes, min and (255 - max) side by side
        const int mn = min(min(g[0], g[1]), min(g[2], g[3])), mx = max(max(g[0], g[1]), max(g[2], g[3]));
        uint32_t pk = (uint32_t)mn | ((uint32_t)(255 - mx) << 16);
        pk = __vminu2(pk, __shfl_xor_sync(0xffffffffu, pk, 1));
        pk = __vminu2(pk, __shfl_xor_sync(0xffffffffu, pk, 2));
        // 4 x 4 byte transpose over the 4 lanes: this lane's column (bytes = rows) -> row `col` of the tile (bytes = columns)
        uint32_t G = (uint32_t)g[0] | ((uint32_t)g[1] << 8) | ((uint32_t)g[2] << 16) | ((uint32_t)g[3] << 24);
        uint32_t P = __shfl_xor_sync(0xffffffffu, G, 1);
        G = __byte_perm(G, P, (col & 1) ? 0x3715 : 0x6240);
        P = __shfl_xor_sync(0xffffffffu, G, 2);
        G = __byte_perm(G, P, (col & 2) ? 0x3276 : 0x5410);
        if (live) {
            *reinterpret_cast<uint32_t *>(gray + (size_t)f * frame_px + (size_t)(y0 + col) * w + (size_t)tx * 4) = G;
            if (col == 0) tmm[(size_t)f * tw * th + (size_t)ty * tw + tx] = (uint16_t)((pk & 0xffu) | ((255u - (pk >> 16)) << 8));
        }
    }
}

void apse_sparse_free(apse_ctx *ctx)
{
    cudaFree(ctx->btable);
    if (ctx->aux_stream) { cudaStreamDestroy(ctx->aux_stream); cudaEventDestroy(ctx->aux_ev[0]); cudaEventDestroy(ctx->aux_ev[1]); }
    for (TileSlot &s : ctx->slot) { cudaFree(s.tbounds); cudaFree(s.eflag); cudaFree(s.elist); cudaFree(s.ecount); }
}

int apse_preprocess_sparse(apse_ctx *ctx, TileSlot &slot, const uint8_t *bgr, uint8_t *gray, int batch, int min_wb_diff, cudaStream_t st)
{
    const int w = ctx->w, h = ctx->h;
    PFN_tmapEncodeTiled enc = get_tmap_encoder();
    const bool tma_ok = enc && (w % 4) == 0 && (h % 4) == 0 && ((w * 3) % 16) == 0 && w >= P2_TW && h >= P2_TH &&
                        ((uintptr_t)bgr % 16) == 0 && ctx->tables2 && ctx->btable && batch <= 64 && (w % 32) == 0 &&   // k_sparse_flags: 8 tiles per thread
                        ((uintptr_t)gray % 4) == 0;                                                                  // k_sparse_exact: 32-bit stores
    if (!tma_ok) return 1;
    CUtensorMap tmap;
    {
        cuuint64_t dims[3] = {(cuuint64_t)(w * 3 / 4), (cuuint64_t)h, (cuuint64_t)batch};
        cuuint64_t strides[2] = {(cuuint64_t)w * 3, (cuuint64_t)w * 3 * h};
        cuuint32_t boxd[3] = {P2_BOX_WORDS, P2_BOX_H, 1}, estr[3] = {1, 1, 1};
        CUresult r = enc(&tmap, CU_TENSOR_MAP_DATA_TYPE_UINT32, 3, (void *)bgr, dims, strides, boxd, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
                         CU_TENSOR_MAP_SWIZZLE_NONE, CU_TENSOR_MAP_L2_PROMOTION_L2_128B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
        if (r != CUDA_SUCCESS) return 1;
    }
    const int tw = w / 4, th = h / 4;
    const size_t ntiles = (size_t)ctx->max_batch * (ctx->max_w / 4) * (ctx->max_h / 4);
    if (!slot.tbounds) {
        CUDA_TRY(ctx, cudaMalloc((void **)&slot.tbounds, ntiles * sizeof(uint16_t)));
        CUDA_TRY(ctx, cudaMalloc((void **)&slot.eflag, ntiles));
        CUDA_TRY(ctx, cudaMalloc((void **)&slot.elist, ntiles * sizeof(uint32_t)));
        CUDA_TRY(ctx, cudaMalloc((void **)&slot.ecount, sizeof(int)));
    }
    // 4K bounds pass: 40 registers per thread (leaves 15 K registers per SM to co-resident chain CTAs; 48 has no spill) and a
    // staging ring of 3
    static bool attr_set[64] = {false};
    if (!attr_set[ctx->device & 63]) {
        CUDA_TRY(ctx, cudaFuncSetAttribute(k_preprocess_tma<false, 40, 3840, true, 1, 3>, cudaFuncAttributeMaxDynamicSharedMemorySize, P2_SMEM_BYTES_N(1, 3)));
        CUDA_TRY(ctx, cudaFuncSetAttribute(k_preprocess_tma<false, 48, 0, false, 1>, cudaFuncAttributeMaxDynamicSharedMemorySize, P2_SMEM_BYTES_M(1)));
        attr_set[ctx->device & 63] = true;
    }
    const int nz = div_up(batch, 20), fpb = div_up(batch, nz);
    dim3 grid(div_up(w, P2_TW), div_up(h, P2_TH), nz);
    CUDA_TRY(ctx, cudaMemsetAsync(slot.ecount, 0, sizeof(int), st));
#define K1B_ARGS tmap, bgr, nullptr, nullptr, slot.tbounds, ctx->mapx, ctx->mapy, ctx->btable, w, h, batch, fpb
    if (w == 3840 && h % P2_TH == 0)
        KLAUNCH(ctx, KID_PREPROCESS, st, k_preprocess_tma<false, 40, 3840, true, 1, 3><<<grid, P2_CTA_THREADS, P2_SMEM_BYTES_N(1, 3), st>>>(K1B_ARGS));
    else
        KLAUNCH(ctx, KID_PREPROCESS, st, k_preprocess_tma<false, 48, 0, false, 1><<<grid, P2_CTA_THREADS, P2_SMEM_BYTES_M(1), st>>>(K1B_ARGS));
#undef K1B_ARGS
    // The two short kernels that follow gate the detector chain of this batch.  In a multi-stream pipeline they would share the
    // GPU with the bounds pass of the NEXT batch at its priority (0.2 - 0.6 ms instead of 0.04 + 0.10 ms, profiles/r02d_timeline.txt),
    // so they go to a high-priority stream of the context, fenced by two events: `st` sees them as if they had run on it.
    if (!ctx->aux_stream) {
        int lo_prio = 0, hi_prio = 0;
        CUDA_TRY(ctx, cudaDeviceGetStreamPriorityRange(&lo_prio, &hi_prio));
        CUDA_TRY(ctx, cudaStreamCreateWithPriority(&ctx->aux_stream, cudaStreamNonBlocking, hi_prio));
        CUDA_TRY(ctx, cudaEventCreateWithFlags(&ctx->aux_ev[0], cudaEventDisableTiming));
        CUDA_TRY(ctx, cudaEventCreateWithFlags(&ctx->aux_ev[1], cudaEventDisableTiming));
    }
    cudaStream_t sx = ctx->aux_stream;
    CUDA_TRY(ctx, cudaEventRecord(ctx->aux_ev[0], st));
    CUDA_TRY(ctx, cudaStreamWaitEvent(sx, ctx->aux_ev[0], 0));
    KLAUNCH(ctx, KID_SPARSE_FLAGS, sx, k_sparse_flags<<<dim3(div_up(tw / 8, 128), div_up(th, SFL_ROWS), batch), 128, 0, sx>>>(
                slot.tbounds, tw, th, min_wb_diff, slot.tmm, slot.eflag, slot.elist, slot.ecount));
    KLAUNCH(ctx, KID_SPARSE_EXACT, sx, k_sparse_exact<<<ctx->sm_count * 6, 256, 0, sx>>>(bgr, ctx->mapx, ctx->mapy, ctx->tables2, w, h, slot.elist,
                                                                                      slot.ecount, gray, slot.tmm));
    CUDA_TRY(ctx, cudaEventRecord(ctx->aux_ev[1], sx));
    CUDA_TRY(ctx, cudaStreamWaitEvent(st, ctx->aux_ev[1], 0));
    return APSE_OK;
}

int apse_preprocess(apse_ctx *ctx, const uint8_t *bgr, uint8_t *bgr_out, uint8_t *gray, int batch, void *stream)
{
    if (!ctx || !bgr || !gray || batch <= 0) CTX_FAIL(ctx, APSE_ERR_INVALID_ARG, "preprocess: bad argument");
    if (!ctx->has_camera || !ctx->has_lut) CTX_FAIL(ctx, APSE_ERR_NOT_CONFIGURED, "preprocess: set_camera and set_lut first");
    int rc = apse_preprocess_ex(ctx, bgr, bgr_out, gray, nullptr, batch, (cudaStream_t)stream);
    return rc < 0 ? rc : APSE_OK;
}

// ---------------------------------------------------------------------------------------------------------
// stand-alone kernels for the cv2-shaped drop-in calls
__global__ void k_remap(const uint8_t *__restrict__ src, int sw, int sh, int cn, const float *__restrict__ mapx,
                        const float *__restrict__ mapy, int dw, int dh, uint8_t *__restrict__ dst)
{
    int x = blockIdx.x * blockDim.x + threadIdx.x, y = blockIdx.y;
    if (x >= dw || y >= dh) return;
    size_t o = (size_t)y * dw + x;
    Taps t = make_taps(__ldg(mapx + o), __ldg(mapy + o), sw, sh, cn);
    for (int c = 0; c < cn; c++) dst[o * cn + c] = (uint8_t)sample(src, t, sw * cn, cn, c);
}

int apse_remap(apse_ctx *ctx, const uint8_t *src, int sw, int sh, int cn, const float *mapx, const float *mapy, int dw,
               int dh, uint8_t *dst, void *stream)
{
    if (!ctx || !src || !mapx || !mapy || !dst || sw <= 0 || sh <= 0 || dw <= 0 || dh <= 0)
        CTX_FAIL(ctx, APSE_ERR_INVALID_ARG, "remap: bad argument");
    if (cn != 1 && cn != 3) CTX_FAIL(ctx, APSE_ERR_UNSUPPORTED, "remap: only 1- or 3-channel 8-bit images");
    if ((int64_t)sw * sh * cn >= (1ll << 31)) CTX_FAIL(ctx, APSE_ERR_UNSUPPORTED, "remap: source image too large");
    dim3 grid(div_up(dw, 256), dh);
    KLAUNCH(ctx, KID_REMAP, (cudaStream_t)stream, k_remap<<<grid, 256, 0, (cudaStream_t)stream>>>(src, sw, sh, cn, mapx, mapy, dw, dh, dst));
    return APSE_OK;
}

// cv2.undistort (SURVEY.md row a2 note, dcnn/scripts/tests/visualize_uav.py:62): the dependency builds CV_16SC2 maps, i.e. the
// FP64 source coordinate is scaled by 32 and rounded to the Q5 grid directly (no float32 map in between), then the same
// Q15 bilinear remap with BORDER_CONSTANT 0.  Map and sample in one pass; A = new camera matrix (fx', fy', cx', cy').
__global__ void k_undistort(const uint8_t *__restrict__ src, int w, int h, int cn, double fx, double fy, double u0, double v0,
                            double afx, double afy, double au0, double av0, double k1, double k2, double p1, double p2, double k3,
                            double k4, double k5, double k6, double s1, double s2, double s3, double s4, uint8_t *__restrict__ dst)
{
    int j = blockIdx.x * blockDim.x + threadIdx.x, i = blockIdx.y;
    if (j >= w || i >= h) return;
    double ir0 = 1.0 / afx, ir2 = -au0 / afx, ir4 = 1.0 / afy, ir5 = -av0 / afy;
    double x = __dadd_rn(__dmul_rn(j, ir0), ir2), y = __dadd_rn(__dmul_rn(i, ir4), ir5);
    double x2 = __dmul_rn(x, x), y2 = __dmul_rn(y, y);
    double r2 = __dadd_rn(x2, y2), _2xy = __dmul_rn(__dmul_rn(2, x), y);
    double num = __dadd_rn(1, __dmul_rn(__dadd_rn(__dmul_rn(__dadd_rn(__dmul_rn(k3, r2), k2), r2), k1), r2));
    double den = __dadd_rn(1, __dmul_rn(__dadd_rn(__dmul_rn(__dadd_rn(__dmul_rn(k6, r2), k5), r2), k4), r2));
    double kr = __ddiv_rn(num, den);
    double xd = __dadd_rn(__dadd_rn(__dadd_rn(__dadd_rn(__dmul_rn(x, kr), __dmul_rn(p1, _2xy)),
                                              __dmul_rn(p2, __dadd_rn(r2, __dmul_rn(2, x2)))),
                                    __dmul_rn(s1, r2)),
                          __dmul_rn(__dmul_rn(s2, r2), r2));
    double yd = __dadd_rn(__dadd_rn(__dadd_rn(__dadd_rn(__dmul_rn(y, kr), __dmul_rn(p1, __dadd_rn(r2, __dmul_rn(2, y2)))),
                                              __dmul_rn(p2, _2xy)),
                                    __dmul_rn(s3, r2)),
                          __dmul_rn(__dmul_rn(s4, r2), r2));
    double u = __dadd_rn(__dmul_rn(fx, xd), u0), v = __dadd_rn(__dmul_rn(fy, yd), v0);
    int sx = __double2int_rn(__dmul_rn(u, 32.0)), sy = __double2int_rn(__dmul_rn(v, 32.0));   // saturating, round-half-even
    int ix = sx >> 5, iy = sy >> 5, fxq = sx & 31, fyq = sy & 31;
    Taps t;
    t.w00 = min(32767, (32 - fyq) * (32 - fxq) * 32);
    t.w01 = (32 - fyq) * fxq * 32;
    t.w10 = fyq * (32 - fxq) * 32;
    t.w11 = fyq * fxq * 32;
    // far-away coordinates (saturated) have no tap inside; the 64-bit offset below is never dereferenced then
    bool x0 = ix >= 0 && ix < w, x1 = ix + 1 >= 0 && ix + 1 < w && ix < w;
    bool y0 = iy >= 0 && iy < h, y1 = iy + 1 >= 0 && iy + 1 < h && iy < h;
    t.mask = (x0 && y0 ? 1u : 0u) | (x1 && y0 ? 2u : 0u) | (x0 && y1 ? 4u : 0u) | (x1 && y1 ? 8u : 0u);
    if (t.mask == 0) {
        for (int c = 0; c < cn; c++) dst[((size_t)i * w + j) * cn + c] = 0;
        return;
    }
    t.off00 = (iy * w + ix) * cn;
    for (int c = 0; c < cn; c++) dst[((size_t)i * w + j) * cn + c] = (uint8_t)sample(src, t, w * cn, cn, c);
}

int apse_undistort(apse_ctx *ctx, const uint8_t *src, int w, int h, int cn, const double K[9], const double D[14], const double newK[9],
                   uint8_t *dst, void *stream)
{
    if (!ctx || !src || !dst || !K || !D || w <= 0 || h <= 0) CTX_FAIL(ctx, APSE_ERR_INVALID_ARG, "undistort: bad argument");
    if (cn != 1 && cn != 3) CTX_FAIL(ctx, APSE_ERR_UNSUPPORTED, "undistort: only 1- or 3-channel 8-bit images");
    if ((int64_t)w * h * cn >= (1ll << 31)) CTX_FAIL(ctx, APSE_ERR_UNSUPPORTED, "undistort: image too large");
    if (D[12] != 0 || D[13] != 0) CTX_FAIL(ctx, APSE_ERR_UNSUPPORTED, "tilted sensor model (tauX/tauY) is not supported");
    const double *A = newK ? newK : K;
    dim3 grid(div_up(w, 256), h);
    KLAUNCH(ctx, KID_REMAP, (cudaStream_t)stream, k_undistort<<<grid, 256, 0, (cudaStream_t)stream>>>(src, w, h, cn, K[0], K[4], K[2], K[5], A[0], A[4], A[2], A[5],
                                                                                            D[0], D[1], D[2], D[3], D[4], D[5], D[6], D[7], D[8], D[9],
                                                                                            D[10], D[11], dst));
    return APSE_OK;
}

__global__ void __launch_bounds__(256) k_rgb2lab(const uint8_t *__restrict__ src, int64_t npx, uint8_t *__restrict__ dst,
                                                 const LabTables *__restrict__ tables)
{
    __shared__ SmemTables T;
    load_tables(&T, tables);
    __syncthreads();
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < npx; i += (int64_t)gridDim.x * blockDim.x) {
        int L, a, b;
        rgb2lab_px(&T, src[3 * i], src[3 * i + 1], src[3 * i + 2], L, a, b);
        dst[3 * i] = (uint8_t)L;
        dst[3 * i + 1] = (uint8_t)a;
        dst[3 * i + 2] = (uint8_t)b;
    }
}

__global__ void __launch_bounds__(256) k_lab2rgb(const uint8_t *__restrict__ src, int64_t npx, uint8_t *__restrict__ dst,
                                                 const LabTables *__restrict__ tables)
{
    __shared__ SmemTables T;
    load_tables(&T, tables);
    __syncthreads();
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < npx; i += (int64_t)gridDim.x * blockDim.x) {
        int o0, o1, o2;
        lab2rgb_px(&T, src[3 * i], src[3 * i + 1], src[3 * i + 2], o0, o1, o2);
        dst[3 * i] = (uint8_t)o0;
        dst[3 * i + 1] = (uint8_t)o1;
        dst[3 * i + 2] = (uint8_t)o2;
    }
}

__global__ void k_bgr2gray(const uint8_t *__restrict__ src, int64_t npx, uint8_t *__restrict__ dst)
{
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < npx; i += (int64_t)gridDim.x * blockDim.x)
        dst[i] = (uint8_t)gray_px(src[3 * i], src[3 * i + 1], src[3 * i + 2]);
}

__global__ void k_lut(const uint8_t *__restrict__ src, int64_t n, int sstride, const uint8_t *__restrict__ lut,
                      uint8_t *__restrict__ dst, int dstride)
{
    __shared__ uint8_t L[256];
    if (threadIdx.x < 256) L[threadIdx.x] = lut[threadIdx.x];
    __syncthreads();
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x)
        dst[i * dstride] = L[src[i * sstride]];
}

// ---------------------------------------------------------------------------------------------------------
// cv2.cvtColor(src, COLOR_YUV2BGR_{NV12,NV21,I420,YV12}): BT.601 limited range in 20-bit fixed point, no chroma
// interpolation (the four pixels of a 2x2 block share one (U, V) pair).  Integer only, so bit-exact by construction.
// One kernel for the four layouts: u / v point at the first chroma sample of frame 0, cstep is the element step of a chroma
// row (2: interleaved, 1: planar), cstride its row stride; frames are fsz = w * h * 3 / 2 bytes apart.
struct YuvTerms { int r, g, b; };

__device__ __forceinline__ YuvTerms yuv_chroma(int U, int V)
{
    const int uu = U - 128, vv = V - 128, half = 1 << 19;
    return {half + 1673527 * vv, half - 852492 * vv - 409993 * uu, half + 2116026 * uu};
}

__device__ __forceinline__ uint32_t yuv_px(int Y, const YuvTerms &c, int which)   // which: 0 B, 1 G, 2 R
{
    const int y = max(Y - 16, 0) * 1220542;
    return (uint32_t)clip255((y + (which == 0 ? c.b : which == 1 ? c.g : c.r)) >> 20);
}

// scalar path: one thread per 2x2 block
__global__ void __launch_bounds__(256) k_yuv420_to_bgr(const uint8_t *__restrict__ yp, const uint8_t *__restrict__ up,
                                                       const uint8_t *__restrict__ vp, int cstep, int cstride, int w, int h,
                                                       int batch, int64_t fsz, uint8_t *__restrict__ bgr)
{
    const int bw = w >> 1, nblk = bw * (h >> 1);
    for (int f = blockIdx.y; f < batch; f += gridDim.y) {
        for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < nblk; i += gridDim.x * blockDim.x) {
            const int cy = i / bw, cx = i - cy * bw;
            const int64_t co = f * fsz + (int64_t)cy * cstride + (int64_t)cx * cstep;
            const YuvTerms c = yuv_chroma(up[co], vp[co]);
#pragma unroll
            for (int r = 0; r < 2; r++) {
                const int64_t yo = (int64_t)f * fsz + (int64_t)(2 * cy + r) * w + 2 * cx;
                uint8_t *d = bgr + ((int64_t)f * h * w + (int64_t)(2 * cy + r) * w + 2 * cx) * 3;
#pragma unroll
                for (int k = 0; k < 2; k++) {
                    const int Y = yp[yo + k];
                    d[3 * k] = (uint8_t)yuv_px(Y, c, 0);
                    d[3 * k + 1] = (uint8_t)yuv_px(Y, c, 1);
                    d[3 * k + 2] = (uint8_t)yuv_px(Y, c, 2);
                }
            }
        }
    }
}

// vector path (w % 16 == 0, 16-byte aligned source and destination): one thread = 2 rows x 16 columns.  Two 16-byte Y loads,
// 16 bytes of interleaved chroma or 8 + 8 bytes from the two planes, 8 chroma triples, six 16-byte stores.
template <int CSTEP>
__global__ void __launch_bounds__(256) k_yuv420_to_bgr_v16(const uint8_t *__restrict__ yp, const uint8_t *__restrict__ up,
                                                           const uint8_t *__restrict__ vp, int cstride, int w, int h, int batch,
                                                           int64_t fsz, uint8_t *__restrict__ bgr)
{
    const int gw = w >> 4, ngrp = gw * (h >> 1);
    for (int f = blockIdx.y; f < batch; f += gridDim.y) {
        for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < ngrp; i += gridDim.x * blockDim.x) {
            const int cy = i / gw, gx = i - cy * gw;
            const int64_t co = f * fsz + (int64_t)cy * cstride + (int64_t)gx * 8 * CSTEP;
            uint8_t U[8], V[8];
            if (CSTEP == 2) {   // interleaved: up and vp are one byte apart, the lower of the two is 16-byte aligned
                const uint4 q = __ldg(reinterpret_cast<const uint4 *>((up < vp ? up : vp) + co));
                const uint32_t wd[4] = {q.x, q.y, q.z, q.w};
                const int su = up < vp ? 0 : 8, sv = 8 - su;
#pragma unroll
                for (int k = 0; k < 8; k++) {
                    U[k] = (uint8_t)(wd[k >> 1] >> ((k & 1) * 16 + su));
                    V[k] = (uint8_t)(wd[k >> 1] >> ((k & 1) * 16 + sv));
                }
            } else {
                const uint2 qu = __ldg(reinterpret_cast<const uint2 *>(up + co));
                const uint2 qv = __ldg(reinterpret_cast<const uint2 *>(vp + co));
#pragma unroll
                for (int k = 0; k < 8; k++) {
                    U[k] = (uint8_t)((k < 4 ? qu.x : qu.y) >> ((k & 3) * 8));
                    V[k] = (uint8_t)((k < 4 ? qv.x : qv.y) >> ((k & 3) * 8));
                }
            }
            YuvTerms c[8];
#pragma unroll
            for (int k = 0; k < 8; k++) c[k] = yuv_chroma(U[k], V[k]);
#pragma unroll
            for (int r = 0; r < 2; r++) {
                const int row = 2 * cy + r;
                const uint4 qy = __ldg(reinterpret_cast<const uint4 *>(yp + f * fsz + (int64_t)row * w + gx * 16));
                const uint32_t yw[4] = {qy.x, qy.y, qy.z, qy.w};
                uint32_t o[12];
#pragma unroll
                for (int j = 0; j < 12; j++) o[j] = 0;
#pragma unroll
                for (int p = 0; p < 16; p++) {
                    const int Y = (int)((yw[p >> 2] >> ((p & 3) * 8)) & 0xffu);
#pragma unroll
                    for (int ch = 0; ch < 3; ch++) {
                        const int byte = 3 * p + ch;
                        o[byte >> 2] |= yuv_px(Y, c[p >> 1], ch) << ((byte & 3) * 8);
                    }
                }
                uint4 *d = reinterpret_cast<uint4 *>(bgr + ((int64_t)f * h * w + (int64_t)row * w + gx * 16) * 3);
                d[0] = make_uint4(o[0], o[1], o[2], o[3]);
                d[1] = make_uint4(o[4], o[5], o[6], o[7]);
                d[2] = make_uint4(o[8], o[9], o[10], o[11]);
            }
        }
    }
}

int apse_cvt_yuv420_bgr(apse_ctx *ctx, const uint8_t *yuv, int w, int h, int batch, int layout, uint8_t *bgr, void *stream)
{
    if (!ctx || !yuv || !bgr || w <= 0 || h <= 0 || (w & 1) || (h & 1) || batch < 1 || layout < APSE_YUV_NV12 || layout > APSE_YUV_YV12)
        CTX_FAIL(ctx, APSE_ERR_INVALID_ARG, "cvt_yuv420_bgr: bad argument (w %d, h %d, batch %d, layout %d)", w, h, batch, layout);
    const int64_t ysz = (int64_t)w * h, fsz = ysz * 3 / 2;
    const uint8_t *up, *vp;
    int cstep, cstride;
    if (layout == APSE_YUV_NV12 || layout == APSE_YUV_NV21) {
        up = yuv + ysz + (layout == APSE_YUV_NV21);
        vp = yuv + ysz + (layout == APSE_YUV_NV12);
        cstep = 2; cstride = w;
    } else {   // planar: each chroma plane is (h/2) * (w/2) contiguous bytes (a byte offset: it may start mid-row of a w-wide view)
        const int64_t csz = ysz / 4;
        up = yuv + ysz + (layout == APSE_YUV_YV12 ? csz : 0);
        vp = yuv + ysz + (layout == APSE_YUV_I420 ? csz : 0);
        cstep = 1; cstride = w / 2;
    }
    cudaStream_t st = (cudaStream_t)stream;
    const int gy = batch < 65535 ? batch : 65535;
    // 16-byte accesses need the caller's buffers 16-byte aligned and rows of whole 16-pixel groups; then every row, chroma row
    // and frame of the batch starts aligned as well
    if ((w & 15) == 0 && ((uintptr_t)yuv & 15) == 0 && ((uintptr_t)bgr & 15) == 0) {
        const int n = (w >> 4) * (h >> 1), gx = div_up(n, 256);
        if (cstep == 2)
            KLAUNCH(ctx, KID_YUV2BGR, st, k_yuv420_to_bgr_v16<2><<<dim3(gx, gy), 256, 0, st>>>(yuv, up, vp, cstride, w, h, batch, fsz, bgr));
        else
            KLAUNCH(ctx, KID_YUV2BGR, st, k_yuv420_to_bgr_v16<1><<<dim3(gx, gy), 256, 0, st>>>(yuv, up, vp, cstride, w, h, batch, fsz, bgr));
    } else {
        const int n = (w >> 1) * (h >> 1), gx = div_up(n, 256);
        KLAUNCH(ctx, KID_YUV2BGR, st, k_yuv420_to_bgr<<<dim3(gx, gy), 256, 0, st>>>(yuv, up, vp, cstep, cstride, w, h, batch, fsz, bgr));
    }
    return APSE_OK;
}

static int grid_for(const apse_ctx *ctx, int64_t n) { const int64_t cap = (int64_t)ctx->sm_count * 16; return (int)((n + 255) / 256 < cap ? (n + 255) / 256 : cap); }

int apse_cvt_rgb2lab(apse_ctx *ctx, const uint8_t *src, int64_t npx, uint8_t *dst, void *stream)
{
    if (!ctx || !src || !dst || npx <= 0) CTX_FAIL(ctx, APSE_ERR_INVALID_ARG, "cvt_rgb2lab: bad argument");
    KLAUNCH(ctx, KID_CVT, (cudaStream_t)stream, k_rgb2lab<<<grid_for(ctx, npx), 256, 0, (cudaStream_t)stream>>>(src, npx, dst, ctx->tables_id));
    return APSE_OK;
}
int apse_cvt_lab2rgb(apse_ctx *ctx, const uint8_t *src, int64_t npx, uint8_t *dst, void *stream)
{
    if (!ctx || !src || !dst || npx <= 0) CTX_FAIL(ctx, APSE_ERR_INVALID_ARG, "cvt_lab2rgb: bad argument");
    KLAUNCH(ctx, KID_CVT, (cudaStream_t)stream, k_lab2rgb<<<grid_for(ctx, npx), 256, 0, (cudaStream_t)stream>>>(src, npx, dst, ctx->tables_id));
    return APSE_OK;
}
int apse_cvt_bgr2gray(apse_ctx *ctx, const uint8_t *src, int64_t npx, uint8_t *dst, void *stream)
{
    if (!ctx || !src || !dst || npx <= 0) CTX_FAIL(ctx, APSE_ERR_INVALID_ARG, "cvt_bgr2gray: bad argument");
    KLAUNCH(ctx, KID_CVT, (cudaStream_t)stream, k_bgr2gray<<<grid_for(ctx, npx), 256, 0, (cudaStream_t)stream>>>(src, npx, dst));
    return APSE_OK;
}
int apse_lut(apse_ctx *ctx, const uint8_t *src, int64_t n, int src_stride, const uint8_t *lut_dev, uint8_t *dst,
             int dst_stride, void *stream)
{
    if (!ctx || !src || !dst || !lut_dev || n <= 0 || src_stride <= 0 || dst_stride <= 0)
        CTX_FAIL(ctx, APSE_ERR_INVALID_ARG, "lut: bad argument");
    KLAUNCH(ctx, KID_LUT, (cudaStream_t)stream, k_lut<<<grid_for(ctx, n), 256, 0, (cudaStream_t)stream>>>(src, n, src_stride, lut_dev, dst, dst_stride));
    return APSE_OK;
}
