// common.cuh -- context, error plumbing and launch helpers shared by the libapse_b200 translation units.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>
#include <string>
#include "../../include/apse_b200.h"

// ---------------------------------------------------------------------------------------------------------
// capacities of the per-frame work buffers of the APRILTAG candidate path (overflow => APSE_ERR_CAPACITY)
#define APSE_MAX_POINTS (1 << 20)       // boundary points per frame
#define APSE_HASH_SLOTS (1 << 17)       // cluster hash slots per frame (power of two)
#define APSE_MAX_CLUSTERS (1 << 14)     // clusters passing the size filter per frame
#define APSE_MAX_QUADS 4096             // candidate quads per frame (classic path, dense frames: ~1000)
#define APSE_MAX_MAXIMA 512             // local maxima of the line-fit error curve kept per cluster
#define APSE_SORT_SMEM 4096             // points sorted in shared memory; larger clusters sort in global

struct LabTables {  // integer sRGB<->Lab tables (SURVEY.md A.2); ly/lf already composed with the gamma LUT
    uint16_t gamma[256];
    uint16_t cbrt[3072];
    uint16_t ly[256];
    uint16_t lf[256];
    uint8_t invgamma[4096];
};

struct P2Tables {   // tables of the TMA-staged preprocess kernel (preprocess.cu, K1t), 8.8 KB of shared memory
    uint16_t gamma[256];     // 8-bit sRGB -> linear * 2040
    uint16_t cb[2048];       // cube-root table on the 0..2040 index range
    uint32_t yf[256];        // L -> y | f << 16: the gamma LUT on L and LabToYF composed
    uint8_t invgamma[4096];
};

// tile list entry: tx | ty << 13 | frame << 26 (frames per launch <= 64, tile coordinates < 8192)
#define ATILE(f, tx, ty) ((uint32_t)(tx) | ((uint32_t)(ty) << 13) | ((uint32_t)(f) << 26))
#define ATILE_TX(e) ((int)((e) & 0x1fffu))
#define ATILE_TY(e) ((int)(((e) >> 13) & 0x1fffu))
#define ATILE_F(e) ((int)((e) >> 26))

struct SparseSrc {   // sparse evaluation (preprocess.cu): what a consumer needs to compute the gray of a pixel on demand
    const uint8_t *bgr;       // [batch][h][w][3] source frames of the batch
    const float *mapx, *mapy;
    const P2Tables *tables;   // device (global memory) copy of the colour tables
    const uint8_t *eflag;     // [batch][h/4][w/4]: non-zero = the gray buffer holds the exact values of this tile
    int tw, th;
};

struct ClusterDesc {
    uint32_t offset;  // into the frame's sorted point array
    uint32_t count;
    uint32_t key_lo, key_hi;
};

struct DeviceParams {  // what the detection kernels need of apse_params (+ derived values computed on host)
    int min_cluster_pixels, max_nmaxima, min_white_black_diff;
    float critical_rad, max_line_fit_mse;
    double max_dot;  // cos(critical_rad), evaluated on the host in double like the dependency does
    int max_cluster_points;
    // decode
    int marker_size, border_bits, cell_size, cell_margin_px, max_border_errors, max_correction;
    double min_otsu_stddev;
    int min_distance_to_border;
    float min_marker_distance_rate, min_group_distance;
    int n_markers, nbytes;
    int detect_inverted;   // detectInvertedMarker
};

enum KernelId {
    KID_BUILD_MAP = 0, KID_PREPROCESS, KID_REMAP, KID_CVT, KID_LUT, KID_TILE_MINMAX, KID_THRESHOLD, KID_CCL_LOCAL,
    KID_CCL_MERGE, KID_CCL_FLATTEN, KID_EMIT, KID_CLUSTER_SCAN, KID_SCATTER, KID_FIT_QUADS, KID_DECODE, KID_POSE,
    KID_PROJECT, KID_CLASSIC, KID_ADAPTIVE, KID_BORDER_JOBS, KID_TRACE, KID_APPROX, KID_SUBPIX, KID_DECODE_BITS, KID_SEQ_JOBS,
    KID_SPARSE_FLAGS, KID_SPARSE_EXACT, KID_DRAW, KID_COUNT
};
#define APSE_EVENT_POOL 2048

struct apse_ctx {
    int device = 0, max_w = 0, max_h = 0, max_batch = 0;
    int sm_count = 148;               // queried at apse_create; persistent grids are sized in multiples of it
    std::string err;
    int64_t launches = 0;
    // optional per-kernel CUDA-event timing (bench.py roofline): event pairs recorded around each launch
    bool timing = false;
    cudaEvent_t ev_start[APSE_EVENT_POOL], ev_stop[APSE_EVENT_POOL];
    int ev_kid[APSE_EVENT_POOL];
    int ev_used = 0, ev_created = 0;
    double kernel_ms[KID_COUNT] = {0};
    int64_t kernel_launches[KID_COUNT] = {0};
    double *trace = nullptr;          // optional launch trace rows {kid, start ms, end ms} (apse_timing_trace)
    int trace_cap = 0, trace_used = 0;
    // camera
    bool has_camera = false;
    int w = 0, h = 0;
    double K[9], D[14];
    float *mapx = nullptr, *mapy = nullptr;
    // colour tables
    bool has_lut = false;
    uint8_t lut[256];
    LabTables *tables = nullptr;      // device, composed with lut (fused preprocess)
    LabTables *tables_id = nullptr;   // device, identity lut (stand-alone cvtColor)
    P2Tables *tables2 = nullptr;      // device, composed tables of the TMA-staged fused kernel
    // dictionary
    bool has_dict = false;
    uint8_t *dict = nullptr;          // device [n_markers][4][nbytes]
    int n_markers = 0, marker_size = 0, max_corr_bits = 0, nbytes = 0;
    // parameters
    bool has_params = false;
    apse_params params;
    // APRILTAG scratch (sized for max_batch frames of max_w x max_h)
    uint8_t *thresh = nullptr;
    uint16_t *tmm = nullptr;          // 4x4-tile extrema of gray, min | max << 8, [batch][h/4][w/4] (= one of tmm_buf)
    uint16_t *tmm_buf[2] = {nullptr, nullptr};   // apse_preprocess_tiles alternates between them
    uint32_t *labels = nullptr;
    uint4 *points = nullptr;          // {key_lo, key_hi, xy, slot|g}
    uint32_t *point_rank = nullptr;
    unsigned long long *hash_keys = nullptr;
    uint32_t *hash_count = nullptr, *hash_offset = nullptr;
    uint2 *sorted_pts = nullptr;      // {x | y<<16, gx | gy<<16} per kept point, grouped by cluster
    unsigned long long *sort_keys = nullptr;
    double *lfps = nullptr;           // [P][6]
    double *errs = nullptr;           // [P][2]
    ClusterDesc *clusters = nullptr;
    int32_t *counters = nullptr;      // per frame: {n_points, n_clusters_kept, n_quads, status, n_clusters_total, n_kept_points}
    float *quads = nullptr;           // [batch][APSE_MAX_QUADS][8]
    unsigned long long *quad_keys = nullptr;   // [batch][APSE_MAX_QUADS] candidate-order key of each quad (both candidate paths)
    uint32_t *quad_order = nullptr;   // rank of each quad in the dependency's candidate order (apse_rank_quads)
    // decode scratch
    void *decode_scratch = nullptr;
    const uint8_t *tiles_gray[2] = {nullptr, nullptr};   // gray batch whose tile extrema are in tmm_buf[i] (apse_preprocess_tiles -> apse_detect_pose_frames)
    int tiles_batch[2] = {0, 0}, tiles_slot = 0;
    uint8_t *nbr_mask = nullptr;      // [max_batch][h][w] 8-neighbour foreground masks of the classic path (first use)
    uint8_t *gray_scratch = nullptr;  // [max_batch][h][w], allocated on first use by apse_process_frames(gray = NULL)
    void *seq_jobs = nullptr, *seq_results = nullptr;   // device staging of apse_sequence_jobs (grown on demand)
    int seq_cap = 0;
    // sparse evaluation (apse_preprocess_tiles_sparse / apse_process_frames without a gray output), one set per tiles slot
    uint16_t *btable = nullptr;       // [SB_ENTRIES] bound table: min | (255 - max) << 8 of gray over the colours of a cell
    cudaStream_t aux_stream = nullptr;   // high-priority stream of the flag / exact kernels of a sparse batch (first use)
    cudaEvent_t aux_ev[2] = {nullptr, nullptr};
    uint16_t *tbounds[2] = {nullptr, nullptr};   // [max_batch][h/4][w/4] per-tile bounds of gray (lo | hi << 8)
    uint8_t *eflag[2] = {nullptr, nullptr};      // [max_batch][h/4][w/4] 1 = tile evaluated exactly
    uint32_t *elist[2] = {nullptr, nullptr};     // tiles to evaluate exactly (ATILE entries), capacity = every tile of the batch
    int *ecount[2] = {nullptr, nullptr};
    const uint8_t *tiles_bgr[2] = {nullptr, nullptr};   // source frames of the batch in slot i (sparse batches only)
    bool tiles_sparse[2] = {false, false};
    const uint8_t *sparse_gray[2] = {nullptr, nullptr};   // gray buffer a sparse batch was written into (partial: only valid with its slot)
    bool sparse_active = false;       // the detect call in flight reads gray through sparse_src
    SparseSrc sparse_src;
    const uint32_t *sparse_elist = nullptr;   // tiles of that batch that carry exact extrema (k_threshold_scan_list)
    const int *sparse_ecount = nullptr;
    // image of the quad detector when aprilTagQuadDecimate / aprilTagQuadSigma are set (quadim.cu), allocated on first use
    uint32_t *trace_strips = nullptr; // classic path: per-warp temporary point strips of k_trace_long
    size_t trace_strips_bytes = 0;
    uint32_t *long_jobs = nullptr;    // classic path: borders handed to the warp-per-border kernel [max_batch][2^16]
    uint8_t *bin_all = nullptr;       // classic path: the binaries of all threshold windows [window][batch][h][w] (first use)
    size_t bin_all_bytes = 0;
    float *quads_refined = nullptr;   // [max_batch][APSE_MAX_QUADS][8] CORNER_REFINE_CONTOUR corners of the candidates (first use)
    uint8_t *quad_im = nullptr, *quad_im2 = nullptr;
    uint16_t *quad_tmp = nullptr;
    void *area_tab = nullptr;         // tap tables of the non-integer INTER_AREA filter for (area_w, area_h, area_dec)
    size_t area_ofs[4] = {0, 0, 0, 0};
    int area_w = 0, area_h = 0;
    float area_dec = 0;
    bool k1_attr_set = false;         // dynamic shared-memory attribute of the K1t instantiations set on this context's device
};

#define APSE_COUNTERS 8

#define CTX_FAIL(ctx, code, ...)                                   \
    do {                                                           \
        char _b[512];                                              \
        snprintf(_b, sizeof _b, __VA_ARGS__);                      \
        if (ctx) (ctx)->err = _b;                                  \
        return (code);                                             \
    } while (0)

#define CUDA_TRY(ctx, expr)                                                                         \
    do {                                                                                            \
        cudaError_t _e = (expr);                                                                    \
        if (_e != cudaSuccess)                                                                      \
            CTX_FAIL(ctx, APSE_ERR_CUDA, "%s failed: %s (%s:%d)", #expr, cudaGetErrorString(_e), __FILE__, __LINE__); \
    } while (0)

int apse_timing_flush(apse_ctx *ctx);

// KLAUNCH(ctx, kernel id, stream, kernel<<<...>>>(...)): counts the launch, checks it, and -- when timing is
// enabled -- brackets it with CUDA events on the launching stream.
#define KLAUNCH(ctx, kid, st, ...)                                                          \
    do {                                                                                    \
        int _slot = -1, _dev = -1;                                                          \
        if (cudaGetDevice(&_dev) == cudaSuccess && _dev != (ctx)->device)                   \
            CTX_FAIL(ctx, APSE_ERR_INVALID_ARG, "the calling thread's current CUDA device is %d but this context lives on device %d", _dev, (ctx)->device); \
        if ((ctx)->timing) {                                                                \
            if ((ctx)->ev_used == APSE_EVENT_POOL) { int _r = apse_timing_flush(ctx); if (_r) return _r; } \
            _slot = (ctx)->ev_used++;                                                       \
            if (_slot >= (ctx)->ev_created) {                                               \
                CUDA_TRY(ctx, cudaEventCreate(&(ctx)->ev_start[_slot]));                    \
                CUDA_TRY(ctx, cudaEventCreate(&(ctx)->ev_stop[_slot]));                     \
                (ctx)->ev_created = _slot + 1;                                              \
            }                                                                               \
            (ctx)->ev_kid[_slot] = (kid);                                                   \
            CUDA_TRY(ctx, cudaEventRecord((ctx)->ev_start[_slot], (st)));                   \
        }                                                                                   \
        __VA_ARGS__;                                                                        \
        if (_slot >= 0) CUDA_TRY(ctx, cudaEventRecord((ctx)->ev_stop[_slot], (st)));        \
        (ctx)->launches++;                                                                  \
        CUDA_TRY(ctx, cudaGetLastError());                                                  \
    } while (0)

static __host__ __device__ inline int div_up(int a, int b) { return (a + b - 1) / b; }

// internal entry points implemented per translation unit
int apse_preprocess_ex(apse_ctx *ctx, const uint8_t *bgr, uint8_t *bgr_out, uint8_t *gray, uint16_t *tmm, int batch,
                       cudaStream_t st);   // returns 1 when the tile extrema were not produced (generic path)
// sparse evaluation: bounds pass + flags + exact chain on the flagged tiles; fills tmm and ctx->eflag[slot].  Returns 1 when the
// frame geometry has no TMA path (the caller falls back to the dense kernel)
int apse_preprocess_sparse(apse_ctx *ctx, const uint8_t *bgr, uint8_t *gray, uint16_t *tmm, int slot, int batch, int min_wb_diff,
                           cudaStream_t st);
int apse_build_bound_table(apse_ctx *ctx, cudaStream_t st);
bool apse_quad_image_needed(const apse_params &p);
int apse_quad_image(apse_ctx *ctx, const uint8_t *gray, int w, int h, int batch, const uint8_t **out, int *qw, int *qh, float *scale, cudaStream_t st);
int apse_scale_quads(apse_ctx *ctx, int batch, float f, cudaStream_t st);
void apse_sparse_free(apse_ctx *ctx);
int apse_detect_alloc(apse_ctx *ctx);
void apse_detect_free(apse_ctx *ctx);
int apse_decode_alloc(apse_ctx *ctx);
void apse_decode_free(apse_ctx *ctx);
int apse_fill_device_params(apse_ctx *ctx, DeviceParams *dp, int w, int h);
int apse_apriltag_quads(apse_ctx *ctx, const uint8_t *gray, int w, int h, int batch, const DeviceParams &dp,
                        cudaStream_t st, bool have_tile_minmax = false,    // true: ctx->tmm already holds this batch's tile extrema
                        bool flat_labels = false);                         // true: ctx->labels fully flattened (debug entry point)
int apse_decode_big_scratch(apse_ctx *ctx);
int apse_adaptive_threshold_impl(apse_ctx *ctx, const uint8_t *gray, int w, int h, int batch, int win, double c, uint8_t *out, cudaStream_t st);
int apse_classic_quads(apse_ctx *ctx, const uint8_t *gray, int w, int h, int batch, cudaStream_t st);
int apse_rank_quads(apse_ctx *ctx, int batch, cudaStream_t st);   // ctx->quad_keys -> ctx->quad_order (keys unique per frame)
int apse_contour_refine(apse_ctx *ctx, int batch, apse_detections *out, cudaStream_t st);
int apse_corner_subpix(apse_ctx *ctx, const uint8_t *gray, int w, int h, int batch, apse_detections *out, cudaStream_t st);
int apse_decode_tap(apse_ctx *ctx, const uint8_t *gray, int w, int h, const float *corners, int n, const DeviceParams &dp, uint8_t *img_out,
                    uint8_t *bits_out, int32_t *res_out, cudaStream_t st);
int apse_decode_candidates(apse_ctx *ctx, const uint8_t *gray, int w, int h, int batch, const DeviceParams &dp,
                           apse_detections *out, cudaStream_t st);
