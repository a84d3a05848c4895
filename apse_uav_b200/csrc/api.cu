// api.cu -- C ABI of libapse_b200.so (include/apse_b200.h): context life cycle, configuration, and the
// batched detectMarkers entry point that chains the candidate (detect_apriltag.cu) and decode (decode.cu) stages.
#include "common.cuh"
#include <math.h>
#include <string.h>
#include <new>

int apse_upload_tables(apse_ctx *ctx, const uint8_t *lut, LabTables **dev, cudaStream_t st);  // preprocess.cu
int apse_upload_p2_tables(apse_ctx *ctx, const uint8_t *lut, P2Tables **dev, cudaStream_t st);

// cached tile extrema (apse_preprocess_tiles) never survive another entry point
static void drop_handoffs(apse_ctx *ctx) { for (TileSlot &s : ctx->slot) s.gray = nullptr; }

// the slot the last apse_preprocess_tiles[_sparse] call filled
static TileSlot &last_slot(apse_ctx *ctx) { return ctx->slot[ctx->next_slot ^ 1]; }

extern "C" {

int apse_abi_version(void) { return APSE_ABI_VERSION; }

void apse_params_default(apse_params *p)
{
    if (!p) return;
    memset(p, 0, sizeof *p);
    p->adaptiveThreshWinSizeMin = 3; p->adaptiveThreshWinSizeMax = 23; p->adaptiveThreshWinSizeStep = 10;
    p->adaptiveThreshConstant = 7;
    p->minMarkerPerimeterRate = 0.03; p->maxMarkerPerimeterRate = 4.;
    p->polygonalApproxAccuracyRate = 0.03; p->minCornerDistanceRate = 0.05;
    p->minDistanceToBorder = 3;
    p->minMarkerDistanceRate = 0.125;
    p->minGroupDistance = 0.21f;
    p->cornerRefinementMethod = 0;
    p->cornerRefinementWinSize = 5;
    p->relativeCornerRefinmentWinSize = 0.3f;
    p->cornerRefinementMaxIterations = 30;
    p->cornerRefinementMinAccuracy = 0.1;
    p->markerBorderBits = 1;
    p->perspectiveRemovePixelPerCell = 4;
    p->perspectiveRemoveIgnoredMarginPerCell = 0.13;
    p->maxErroneousBitsInBorderRate = 0.35;
    p->minOtsuStdDev = 5.0;
    p->errorCorrectionRate = 0.6;
    p->aprilTagQuadDecimate = 0.f; p->aprilTagQuadSigma = 0.f;
    p->aprilTagMinClusterPixels = 5; p->aprilTagMaxNmaxima = 10;
    p->aprilTagCriticalRad = (float)(10 * M_PI / 180);
    p->aprilTagMaxLineFitMse = 10.f;
    p->aprilTagMinWhiteBlackDiff = 5; p->aprilTagDeglitch = 0;
    p->detectInvertedMarker = 0; p->useAruco3Detection = 0;
    p->minSideLengthCanonicalImg = 32;
    p->minMarkerLengthRatioOriginalImg = 0.f;
}

int apse_create(apse_ctx **out, int device, int max_w, int max_h, int max_batch)
{
    if (!out || max_w < 8 || max_h < 8 || max_batch < 1 || max_batch > 64) return APSE_ERR_INVALID_ARG;
    *out = nullptr;
    int ndev = 0;
    if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0 || device < 0 || device >= ndev) return APSE_ERR_CUDA;
    int caller_dev = -1;
    cudaGetDevice(&caller_dev);
    if (cudaSetDevice(device) != cudaSuccess) return APSE_ERR_CUDA;
    // the caller's current device is restored on every exit path: a context never changes the thread's device for good,
    // and every launch checks that the thread is on the context's device (KLAUNCH)
    struct Restore { int d; ~Restore() { if (d >= 0) cudaSetDevice(d); } } restore{caller_dev};
    apse_ctx *ctx = new (std::nothrow) apse_ctx();
    if (!ctx) return APSE_ERR_CUDA;
    ctx->device = device; ctx->max_w = max_w; ctx->max_h = max_h; ctx->max_batch = max_batch;
    if (cudaDeviceGetAttribute(&ctx->sm_count, cudaDevAttrMultiProcessorCount, device) != cudaSuccess || ctx->sm_count <= 0) ctx->sm_count = 148;
    apse_params_default(&ctx->params);
    int rc = apse_detect_alloc(ctx);
    if (rc == APSE_OK) rc = apse_decode_alloc(ctx);
    if (rc == APSE_OK) rc = apse_upload_tables(ctx, nullptr, &ctx->tables_id, 0);
    if (rc != APSE_OK) {
        fprintf(stderr, "apse_create: %s\n", ctx->err.c_str());
        apse_destroy(ctx);
        return rc;
    }
    *out = ctx;
    return APSE_OK;
}

void apse_destroy(apse_ctx *ctx)
{
    if (!ctx) return;
    int caller_dev = -1;
    cudaGetDevice(&caller_dev);
    cudaSetDevice(ctx->device);
    struct Restore { int d; ~Restore() { if (d >= 0) cudaSetDevice(d); } } restore{caller_dev};
    apse_detect_free(ctx);
    apse_decode_free(ctx);
    apse_sparse_free(ctx);
    for (int i = 0; i < ctx->ev_created; i++) { cudaEventDestroy(ctx->ev_start[i]); cudaEventDestroy(ctx->ev_stop[i]); }
    delete[] ctx->trace;
    cudaFree(ctx->mapx); cudaFree(ctx->mapy); cudaFree(ctx->tables); cudaFree(ctx->tables_id); cudaFree(ctx->tables2); cudaFree(ctx->dict); cudaFree(ctx->gray_scratch); cudaFree(ctx->nbr_mask); cudaFree(ctx->seq_jobs); cudaFree(ctx->seq_results);
    cudaFree(ctx->quad_im); cudaFree(ctx->quad_im2); cudaFree(ctx->quad_tmp); cudaFree(ctx->quads_refined); cudaFree(ctx->area_tab); cudaFree(ctx->bin_all); cudaFree(ctx->long_jobs); cudaFree(ctx->trace_strips);
    delete ctx;
}

const char *apse_last_error(apse_ctx *ctx) { return ctx ? ctx->err.c_str() : "null context"; }

int64_t apse_launch_count(apse_ctx *ctx) { return ctx ? ctx->launches : 0; }

static const char *KERNEL_NAMES[KID_COUNT] = {
    "k_build_undistort_map", "k_preprocess_fused", "k_remap", "k_cvt", "k_lut", "k_tile_minmax", "k_threshold",
    "k_ccl_local", "k_ccl_merge", "k_ccl_flatten", "k_emit_points", "k_cluster_scan", "k_scatter_points", "k_fit_quads",
    "k_decode", "k_pose", "k_project_points", "k_classic", "k_adaptive_threshold", "k_border_jobs", "k_trace_borders",
    "k_approx_quads", "k_corner_subpix", "k_decode_bits", "k_sequence_jobs", "k_sparse_flags", "k_sparse_exact", "k_draw_overlay",
    "k_yuv420_to_bgr"};

int apse_kernel_count(void) { return KID_COUNT; }
const char *apse_kernel_name(int kid) { return kid >= 0 && kid < KID_COUNT ? KERNEL_NAMES[kid] : ""; }

int apse_timing_enable(apse_ctx *ctx, int on)
{
    if (!ctx) return APSE_ERR_INVALID_ARG;
    if (!on && ctx->timing) { int rc = apse_timing_flush(ctx); if (rc) return rc; }
    ctx->timing = on != 0;
    return APSE_OK;
}

int apse_timing_collect(apse_ctx *ctx, double *ms, int64_t *launches, int reset)
{
    if (!ctx || !ms || !launches) CTX_FAIL(ctx, APSE_ERR_INVALID_ARG, "timing_collect: bad argument");
    int rc = apse_timing_flush(ctx);
    if (rc) return rc;
    for (int i = 0; i < KID_COUNT; i++) { ms[i] = ctx->kernel_ms[i]; launches[i] = ctx->kernel_launches[i]; }
    if (reset) for (int i = 0; i < KID_COUNT; i++) { ctx->kernel_ms[i] = 0; ctx->kernel_launches[i] = 0; }
    return APSE_OK;
}

int apse_set_camera(apse_ctx *ctx, const double K[9], const double D[14], int w, int h, void *stream)
{
    if (!ctx || !K || !D) CTX_FAIL(ctx, APSE_ERR_INVALID_ARG, "set_camera: bad argument");
    if (w > ctx->max_w || h > ctx->max_h || w < 8 || h < 8)
        CTX_FAIL(ctx, APSE_ERR_INVALID_ARG, "set_camera: %dx%d outside the context capacity %dx%d", w, h, ctx->max_w, ctx->max_h);
    if (!ctx->mapx) {
        CUDA_TRY(ctx, cudaMalloc((void **)&ctx->mapx, (size_t)ctx->max_w * ctx->max_h * sizeof(float)));
        CUDA_TRY(ctx, cudaMalloc((void **)&ctx->mapy, (size_t)ctx->max_w * ctx->max_h * sizeof(float)));
    }
    int rc = apse_init_undistort_map(ctx, K, D, w, h, ctx->mapx, ctx->mapy, stream);
    if (rc) return rc;
    drop_handoffs(ctx);
    memcpy(ctx->K, K, sizeof ctx->K);
    memcpy(ctx->D, D, sizeof ctx->D);
    ctx->w = w; ctx->h = h;
    ctx->has_camera = true;
    return APSE_OK;
}

int apse_set_lut(apse_ctx *ctx, const uint8_t lut[256], void *stream)
{
    if (!ctx || !lut) CTX_FAIL(ctx, APSE_ERR_INVALID_ARG, "set_lut: bad argument");
    memcpy(ctx->lut, lut, 256);
    drop_handoffs(ctx);
    int rc = apse_upload_tables(ctx, lut, &ctx->tables, (cudaStream_t)stream);
    if (rc) return rc;
    rc = apse_upload_p2_tables(ctx, lut, &ctx->tables2, (cudaStream_t)stream);
    if (!rc) rc = apse_build_bound_table(ctx, (cudaStream_t)stream);   // sparse evaluation: gray bounds per colour cell, from the chain itself
    if (rc) return rc;
    ctx->has_lut = true;
    return APSE_OK;
}

int apse_set_dictionary(apse_ctx *ctx, const uint8_t *bytes, int n_markers, int marker_size, int max_corr_bits, void *stream)
{
    if (!ctx || !bytes || n_markers <= 0 || marker_size < 3 || marker_size > 7 || max_corr_bits < 0)
        CTX_FAIL(ctx, APSE_ERR_INVALID_ARG, "set_dictionary: bad argument");
    int nbytes = (marker_size * marker_size + 7) / 8;
    size_t sz = (size_t)n_markers * 4 * nbytes;
    cudaFree(ctx->dict);
    ctx->dict = nullptr;
    CUDA_TRY(ctx, cudaMalloc((void **)&ctx->dict, sz));
    CUDA_TRY(ctx, cudaMemcpyAsync(ctx->dict, bytes, sz, cudaMemcpyHostToDevice, (cudaStream_t)stream));
    CUDA_TRY(ctx, cudaStreamSynchronize((cudaStream_t)stream));
    ctx->n_markers = n_markers; ctx->marker_size = marker_size; ctx->max_corr_bits = max_corr_bits; ctx->nbytes = nbytes;
    ctx->has_dict = true;
    return APSE_OK;
}

int apse_set_params(apse_ctx *ctx, const apse_params *p)
{
    if (!ctx || !p) CTX_FAIL(ctx, APSE_ERR_INVALID_ARG, "set_params: bad argument");
    // asserts the dependency enforces on DetectorParameters
    if (p->adaptiveThreshWinSizeMin < 3 || p->adaptiveThreshWinSizeMax < 3 ||
        p->adaptiveThreshWinSizeMax < p->adaptiveThreshWinSizeMin || p->adaptiveThreshWinSizeStep <= 0)
        CTX_FAIL(ctx, APSE_ERR_INVALID_ARG, "set_params: adaptiveThreshWinSize{Min,Max,Step} invalid");
    if (p->markerBorderBits <= 0) CTX_FAIL(ctx, APSE_ERR_INVALID_ARG, "set_params: markerBorderBits must be > 0");
    if (p->minMarkerDistanceRate < 0 || p->minDistanceToBorder < 0)
        CTX_FAIL(ctx, APSE_ERR_INVALID_ARG, "set_params: minMarkerDistanceRate / minDistanceToBorder must be >= 0");
    if (p->perspectiveRemovePixelPerCell <= 0 || p->perspectiveRemoveIgnoredMarginPerCell < 0 ||
        p->perspectiveRemoveIgnoredMarginPerCell > 0.5)
        CTX_FAIL(ctx, APSE_ERR_INVALID_ARG, "set_params: perspectiveRemove* invalid");
    if (p->aprilTagDeglitch != 0) CTX_FAIL(ctx, APSE_ERR_UNSUPPORTED, "set_params: aprilTagDeglitch is not supported");
    if (p->aprilTagQuadDecimate > 64) CTX_FAIL(ctx, APSE_ERR_UNSUPPORTED, "set_params: aprilTagQuadDecimate above 64 is not supported");
    if (fabsf(p->aprilTagQuadSigma) >= 8.25f) CTX_FAIL(ctx, APSE_ERR_UNSUPPORTED, "set_params: |aprilTagQuadSigma| must be below 8.25 (33 taps)");
    if (p->useAruco3Detection)
        CTX_FAIL(ctx, APSE_ERR_UNSUPPORTED, "set_params: useAruco3Detection is not supported");
    if (p->cornerRefinementMethod < 0 || p->cornerRefinementMethod > 3) CTX_FAIL(ctx, APSE_ERR_INVALID_ARG, "set_params: cornerRefinementMethod must be 0 .. 3");
    if (p->aprilTagMaxNmaxima < 4 || p->aprilTagMaxNmaxima > 16)
        CTX_FAIL(ctx, APSE_ERR_UNSUPPORTED, "set_params: aprilTagMaxNmaxima must be in [4,16]");
    drop_handoffs(ctx);
    ctx->params = *p;
    ctx->has_params = true;
    return APSE_OK;
}

}  // extern "C"

// waits for the recorded events and accumulates their durations per kernel id
// process-wide time origin of the launch trace (recorded once on the legacy stream)
static cudaEvent_t g_trace_base = nullptr;

int apse_timing_flush(apse_ctx *ctx)
{
    for (int i = 0; i < ctx->ev_used; i++) {
        CUDA_TRY(ctx, cudaEventSynchronize(ctx->ev_stop[i]));
        float ms = 0;
        CUDA_TRY(ctx, cudaEventElapsedTime(&ms, ctx->ev_start[i], ctx->ev_stop[i]));
        ctx->kernel_ms[ctx->ev_kid[i]] += ms;
        ctx->kernel_launches[ctx->ev_kid[i]]++;
        if (ctx->trace && ctx->trace_used < ctx->trace_cap && g_trace_base) {
            float t0 = 0;
            CUDA_TRY(ctx, cudaEventElapsedTime(&t0, g_trace_base, ctx->ev_start[i]));
            double *r = ctx->trace + 3 * (size_t)ctx->trace_used++;
            r[0] = ctx->ev_kid[i]; r[1] = t0; r[2] = t0 + ms;
        }
    }
    ctx->ev_used = 0;
    return APSE_OK;
}

// development aid: keep (kernel id, start ms, end ms) of every timed launch, relative to a process-wide origin, so that
// the overlap of the streams of several contexts can be drawn as one timeline (tools/timeline.py)
int apse_timing_trace(apse_ctx *ctx, double *out, int cap_rows)
{
    if (!ctx) return APSE_ERR_INVALID_ARG;
    if (!out) {   // (re)arm with a capacity of cap_rows launches
        delete[] ctx->trace;
        ctx->trace = cap_rows > 0 ? new double[3 * (size_t)cap_rows] : nullptr;
        ctx->trace_cap = cap_rows > 0 ? cap_rows : 0;
        ctx->trace_used = 0;
        if (!g_trace_base) {
            CUDA_TRY(ctx, cudaEventCreate(&g_trace_base));
            CUDA_TRY(ctx, cudaEventRecord(g_trace_base, 0));
            CUDA_TRY(ctx, cudaEventSynchronize(g_trace_base));
        }
        return APSE_OK;
    }
    int rc = apse_timing_flush(ctx);
    if (rc) return rc;
    int n = ctx->trace_used < cap_rows ? ctx->trace_used : cap_rows;
    memcpy(out, ctx->trace, sizeof(double) * 3 * (size_t)n);
    ctx->trace_used = 0;
    return n;
}

int apse_fill_device_params(apse_ctx *ctx, DeviceParams *dp, int w, int h)
{
    const apse_params &p = ctx->params;
    dp->min_cluster_pixels = p.aprilTagMinClusterPixels;
    dp->max_nmaxima = p.aprilTagMaxNmaxima;
    dp->min_white_black_diff = p.aprilTagMinWhiteBlackDiff;
    dp->critical_rad = p.aprilTagCriticalRad;
    dp->max_line_fit_mse = p.aprilTagMaxLineFitMse;
    dp->max_dot = cos((double)p.aprilTagCriticalRad);
    dp->max_cluster_points = 3 * (2 * w + 2 * h);
    dp->marker_size = ctx->marker_size;
    dp->border_bits = p.markerBorderBits;
    dp->cell_size = p.perspectiveRemovePixelPerCell;
    dp->cell_margin_px = (int)(p.perspectiveRemoveIgnoredMarginPerCell * p.perspectiveRemovePixelPerCell);
    dp->max_border_errors = (int)(ctx->marker_size * ctx->marker_size * p.maxErroneousBitsInBorderRate);
    dp->detect_inverted = p.detectInvertedMarker ? 1 : 0;
    dp->max_correction = (int)((double)ctx->max_corr_bits * p.errorCorrectionRate);
    dp->min_otsu_stddev = p.minOtsuStdDev;
    dp->min_distance_to_border = p.minDistanceToBorder;
    dp->min_marker_distance_rate = (float)p.minMarkerDistanceRate;
    dp->min_group_distance = p.minGroupDistance;
    dp->n_markers = ctx->n_markers;
    dp->nbytes = ctx->nbytes;
    return APSE_OK;
}

// candidates (APRILTAG quad detector or the classic threshold / contour path) -> grouping + decoding -> SUBPIX.  tiles: the slot
// holding this batch's tile extrema (and, for a sparse batch, its flags), or null.  Extrema the chain computes itself go to the
// handed slot (the only one it writes: Pipeline), else to slot 0 (the caller orders the call against pending work on the context).
static int apse_detect_impl(apse_ctx *ctx, const uint8_t *gray, int w, int h, int batch, apse_detections *out, cudaStream_t st,
                            const TileSlot *tiles)
{
    DeviceParams dp;
    apse_fill_device_params(ctx, &dp, w, h);
    const int mode = ctx->params.cornerRefinementMethod;
    uint16_t *tmm_scratch = (tiles ? tiles : &ctx->slot[0])->tmm;
    // both candidate paths can produce more than DEC_SMEMC candidates per frame (a 4K frame with a few hundred small markers
    // does on the APRILTAG path): the decode stage then needs its global candidate arrays, whatever ran on the context before
    int rc = apse_decode_big_scratch(ctx);
    if (rc) return rc;
    if (mode == 3 && apse_quad_image_needed(ctx->params)) {
        // aprilTagQuadDecimate / aprilTagQuadSigma: quads are found on the shrunk / blurred image and scaled back; the tile
        // extrema of the full-size gray (if any) do not apply
        const uint8_t *qim; int qw, qh; float qscale;
        rc = apse_quad_image(ctx, gray, w, h, batch, &qim, &qw, &qh, &qscale, st);
        if (rc) return rc;
        DeviceParams dq;
        apse_fill_device_params(ctx, &dq, qw, qh);
        rc = apse_apriltag_quads(ctx, qim, qw, qh, batch, dq, st, nullptr, tmm_scratch);
        if (!rc && qscale != 1.f) rc = apse_scale_quads(ctx, batch, qscale, st);
    } else if (mode == 3) {
        rc = apse_apriltag_quads(ctx, gray, w, h, batch, dp, st, tiles, tmm_scratch);
    } else {
        rc = apse_classic_quads(ctx, gray, w, h, batch, st);
    }
    if (rc) return rc;
    SparseSrc sparse;
    if (tiles && tiles->bgr) sparse = SparseSrc{tiles->bgr, ctx->mapx, ctx->mapy, ctx->tables2, tiles->eflag, w / 4, h / 4};
    rc = apse_decode_candidates(ctx, gray, w, h, batch, dp, tiles && tiles->bgr ? &sparse : nullptr, out, st);
    if (rc) return rc;
    if (mode == 1) rc = apse_corner_subpix(ctx, gray, w, h, batch, out, st);
    if (mode == 2) rc = apse_contour_refine(ctx, batch, out, st);
    return rc;
}

static int detect_pose(apse_ctx *ctx, const uint8_t *gray, int batch, const TileSlot *tiles, apse_detections *out, const float *marker_len,
                       float marker_len_all, double *rvec, double *tvec, void *stream)
{
    int rc = apse_detect_impl(ctx, gray, ctx->w, ctx->h, batch, out, (cudaStream_t)stream, tiles);
    if (rc) return rc;
    if (rvec && tvec)
        rc = apse_pose_frames(ctx, out->corners, out->n_markers, batch, out->max_markers, marker_len, marker_len_all, ctx->K, ctx->D, rvec, tvec, stream);
    return rc;
}

// K1 writes the 4x4-tile extrema of gray straight into the slot, for the candidate stage.  want_sparse: the caller does not need
// the gray frames, so they may come from the sparse evaluation (identical detections; gray is computed only where the detector
// reads it).  On return slot.gray says whether extrema were produced.
static int preprocess_into(apse_ctx *ctx, TileSlot &slot, const uint8_t *bgr, uint8_t *gray, int batch, cudaStream_t st, bool want_sparse)
{
    int rc = 1;
    slot.bgr = nullptr;
    if (want_sparse && ctx->params.cornerRefinementMethod == 3 && !apse_quad_image_needed(ctx->params)) {
        rc = apse_preprocess_sparse(ctx, slot, bgr, gray, batch, ctx->params.aprilTagMinWhiteBlackDiff, st);
        if (rc < 0) return rc;
        if (rc == APSE_OK) slot.bgr = bgr;
    }
    if (rc == 1) rc = apse_preprocess_ex(ctx, bgr, nullptr, gray, slot.tmm, batch, st);
    if (rc < 0) return rc;
    slot.gray = rc == APSE_OK ? gray : nullptr;
    slot.batch = batch;
    return APSE_OK;
}

extern "C" {

int apse_detect(apse_ctx *ctx, const uint8_t *gray, int w, int h, int batch, apse_detections *out, void *stream)
{
    if (!ctx || !gray || !out || batch <= 0) CTX_FAIL(ctx, APSE_ERR_INVALID_ARG, "detect: bad argument");
    if (!ctx->has_dict) CTX_FAIL(ctx, APSE_ERR_NOT_CONFIGURED, "detect: set_dictionary first");
    drop_handoffs(ctx);
    return apse_detect_impl(ctx, gray, w, h, batch, out, (cudaStream_t)stream, nullptr);
}

int apse_process_frames(apse_ctx *ctx, const uint8_t *bgr, uint8_t *gray, int batch, apse_detections *out, const float *marker_len,
                        float marker_len_all, double *rvec, double *tvec, void *stream)
{
    if (!ctx || !bgr || !out || batch <= 0) CTX_FAIL(ctx, APSE_ERR_INVALID_ARG, "process_frames: bad argument");
    if (!ctx->has_camera || !ctx->has_lut || !ctx->has_dict)
        CTX_FAIL(ctx, APSE_ERR_NOT_CONFIGURED, "process_frames: set_camera, set_lut and set_dictionary first");
    if (batch > ctx->max_batch) CTX_FAIL(ctx, APSE_ERR_INVALID_ARG, "process_frames: batch %d exceeds the context capacity %d", batch, ctx->max_batch);
    drop_handoffs(ctx);
    const bool want_sparse = gray == nullptr;
    if (!gray) {
        if (!ctx->gray_scratch) CUDA_TRY(ctx, cudaMalloc((void **)&ctx->gray_scratch, (size_t)ctx->max_batch * ctx->max_w * ctx->max_h));
        gray = ctx->gray_scratch;
    }
    // slot 0 on the caller's stream, handed straight to the detector; the refusal records (partial_gray) are left as they are
    TileSlot &slot = ctx->slot[0];
    int rc = preprocess_into(ctx, slot, bgr, gray, batch, (cudaStream_t)stream, want_sparse);
    if (rc) return rc;
    const bool have_extrema = slot.gray != nullptr;
    slot.gray = nullptr;
    return detect_pose(ctx, gray, batch, have_extrema ? &slot : nullptr, out, marker_len, marker_len_all, rvec, tvec, stream);
}

static int preprocess_tiles_impl(apse_ctx *ctx, const uint8_t *bgr, uint8_t *gray, int batch, void *stream, bool want_sparse)
{
    if (!ctx || !bgr || !gray || batch <= 0) CTX_FAIL(ctx, APSE_ERR_INVALID_ARG, "preprocess_tiles: bad argument");
    if (!ctx->has_camera || !ctx->has_lut) CTX_FAIL(ctx, APSE_ERR_NOT_CONFIGURED, "preprocess_tiles: set_camera and set_lut first");
    if (batch > ctx->max_batch) CTX_FAIL(ctx, APSE_ERR_INVALID_ARG, "preprocess_tiles: batch %d exceeds the context capacity %d", batch, ctx->max_batch);
    TileSlot &slot = ctx->slot[ctx->next_slot];
    ctx->next_slot ^= 1;
    for (TileSlot &s : ctx->slot) if (s.partial_gray == gray) s.partial_gray = nullptr;   // the buffer is rewritten now
    int rc = preprocess_into(ctx, slot, bgr, gray, batch, (cudaStream_t)stream, want_sparse);
    if (!rc && slot.bgr) slot.partial_gray = gray;
    return rc;
}

int apse_preprocess_tiles(apse_ctx *ctx, const uint8_t *bgr, uint8_t *gray, int batch, void *stream)
{
    return preprocess_tiles_impl(ctx, bgr, gray, batch, stream, false);
}

int apse_preprocess_tiles_sparse(apse_ctx *ctx, const uint8_t *bgr, uint8_t *gray, int batch, void *stream)
{
    return preprocess_tiles_impl(ctx, bgr, gray, batch, stream, true);
}

int apse_detect_pose_frames(apse_ctx *ctx, const uint8_t *gray, int batch, apse_detections *out, const float *marker_len,
                            float marker_len_all, double *rvec, double *tvec, void *stream)
{
    if (!ctx || !gray || !out || batch <= 0) CTX_FAIL(ctx, APSE_ERR_INVALID_ARG, "detect_pose_frames: bad argument");
    if (!ctx->has_camera || !ctx->has_dict) CTX_FAIL(ctx, APSE_ERR_NOT_CONFIGURED, "detect_pose_frames: set_camera and set_dictionary first");
    TileSlot *tiles = nullptr;
    for (TileSlot &s : ctx->slot)
        if (!tiles && s.gray == gray && s.batch == batch) tiles = &s;
    if (tiles) {
        tiles->gray = nullptr;                         // consumed: a later call on other data recomputes the extrema
        if (tiles->bgr) tiles->partial_gray = nullptr;
    } else if (ctx->slot[0].partial_gray == gray || ctx->slot[1].partial_gray == gray) {
        // a gray batch of the sparse evaluation is only complete together with its tile flags: without them (another entry
        // point came in between) the detector would read pixels that were never computed
        CTX_FAIL(ctx, APSE_ERR_INVALID_ARG, "detect_pose_frames: this gray batch comes from apse_preprocess_tiles_sparse and its tile flags are gone "
                                            "(another call on the context came in between); preprocess it again");
    }
    return detect_pose(ctx, gray, batch, tiles, out, marker_len, marker_len_all, rvec, tvec, stream);
}

int apse_adaptive_threshold(apse_ctx *ctx, const uint8_t *gray, int w, int h, int batch, int win, double c, uint8_t *out, void *stream)
{
    if (!ctx || !gray || !out || batch <= 0 || w <= 0 || h <= 0 || win < 3) CTX_FAIL(ctx, APSE_ERR_INVALID_ARG, "adaptive_threshold: bad argument");
    return apse_adaptive_threshold_impl(ctx, gray, w, h, batch, win, c, out, (cudaStream_t)stream);
}

int apse_debug_classic(apse_ctx *ctx, const uint8_t *gray, int w, int h, float *quads, uint32_t *order, int max_quads,
                       int64_t *stats_host, void *stream)
{
    if (!ctx || !gray) CTX_FAIL(ctx, APSE_ERR_INVALID_ARG, "debug_classic: bad argument");
    cudaStream_t st = (cudaStream_t)stream;
    int rc = apse_classic_quads(ctx, gray, w, h, 1, st);
    if (rc) return rc;
    int32_t cnt[APSE_COUNTERS];
    CUDA_TRY(ctx, cudaMemcpyAsync(cnt, ctx->counters, sizeof cnt, cudaMemcpyDeviceToHost, st));
    CUDA_TRY(ctx, cudaStreamSynchronize(st));
    if (cnt[3] != 0) CTX_FAIL(ctx, cnt[3], "debug_classic: work buffer capacity exceeded (quads %d)", cnt[2]);
    int nq = cnt[2] < max_quads ? cnt[2] : max_quads;
    if (quads && order && nq > 0) {
        CUDA_TRY(ctx, cudaMemcpyAsync(quads, ctx->quads, (size_t)nq * 8 * sizeof(float), cudaMemcpyDeviceToDevice, st));
        CUDA_TRY(ctx, cudaMemcpyAsync(order, ctx->quad_order, (size_t)nq * sizeof(uint32_t), cudaMemcpyDeviceToDevice, st));
        CUDA_TRY(ctx, cudaStreamSynchronize(st));
    }
    if (stats_host) { stats_host[0] = cnt[2]; stats_host[1] = 0; stats_host[2] = 0; stats_host[3] = 0; }
    return APSE_OK;
}

int apse_debug_decode(apse_ctx *ctx, const uint8_t *gray, int w, int h, const float *corners, int n, uint8_t *img, uint8_t *bits, int32_t *result, void *stream)
{
    if (!ctx || !gray || !corners || !img || !bits || !result || n <= 0) CTX_FAIL(ctx, APSE_ERR_INVALID_ARG, "debug_decode: bad argument");
    if (!ctx->has_dict) CTX_FAIL(ctx, APSE_ERR_NOT_CONFIGURED, "debug_decode: set_dictionary first");
    DeviceParams dp;
    apse_fill_device_params(ctx, &dp, w, h);
    return apse_decode_tap(ctx, gray, w, h, corners, n, dp, img, bits, result, (cudaStream_t)stream);
}

int apse_debug_sparse(apse_ctx *ctx, uint16_t *bound_table_host, uint8_t *eflag_dev, int batch, int *n_exact_host, void *stream)
{
    if (!ctx) return APSE_ERR_INVALID_ARG;
    cudaStream_t st = (cudaStream_t)stream;
    if (bound_table_host) {
        if (!ctx->btable) CTX_FAIL(ctx, APSE_ERR_NOT_CONFIGURED, "debug_sparse: set_lut first");
        CUDA_TRY(ctx, cudaMemcpyAsync(bound_table_host, ctx->btable, 16 * 32 * 32 * sizeof(uint16_t), cudaMemcpyDeviceToHost, st));
        CUDA_TRY(ctx, cudaStreamSynchronize(st));
    }
    const TileSlot &slot = last_slot(ctx);
    if (eflag_dev || n_exact_host) {
        if (!slot.eflag) CTX_FAIL(ctx, APSE_ERR_NOT_CONFIGURED, "debug_sparse: no sparse batch was preprocessed on this context");
        if (eflag_dev) CUDA_TRY(ctx, cudaMemcpyAsync(eflag_dev, slot.eflag, (size_t)batch * (ctx->w / 4) * (ctx->h / 4), cudaMemcpyDeviceToDevice, st));
        if (n_exact_host) CUDA_TRY(ctx, cudaMemcpyAsync(n_exact_host, slot.ecount, sizeof(int), cudaMemcpyDeviceToHost, st));
        CUDA_TRY(ctx, cudaStreamSynchronize(st));
    }
    return APSE_OK;
}

int apse_debug_tile_bounds(apse_ctx *ctx, uint16_t *bounds_dev, int batch, void *stream)
{
    if (!ctx || !bounds_dev || batch <= 0 || batch > ctx->max_batch) CTX_FAIL(ctx, APSE_ERR_INVALID_ARG, "debug_tile_bounds: bad argument");
    const TileSlot &slot = last_slot(ctx);
    if (!slot.tbounds) CTX_FAIL(ctx, APSE_ERR_NOT_CONFIGURED, "debug_tile_bounds: no sparse batch was preprocessed on this context");
    CUDA_TRY(ctx, cudaMemcpyAsync(bounds_dev, slot.tbounds, (size_t)batch * (ctx->w / 4) * (ctx->h / 4) * sizeof(uint16_t),
                                  cudaMemcpyDeviceToDevice, (cudaStream_t)stream));
    return APSE_OK;
}

int apse_debug_tile_extrema(apse_ctx *ctx, uint16_t *dst_dev, int batch, void *stream)
{
    if (!ctx || !dst_dev || batch <= 0 || batch > ctx->max_batch) CTX_FAIL(ctx, APSE_ERR_INVALID_ARG, "debug_tile_extrema: bad argument");
    const TileSlot &slot = last_slot(ctx);
    if (!slot.gray) CTX_FAIL(ctx, APSE_ERR_NOT_CONFIGURED, "debug_tile_extrema: the last preprocess_tiles batch left no tile extrema");
    if (batch > slot.batch) CTX_FAIL(ctx, APSE_ERR_INVALID_ARG, "debug_tile_extrema: batch %d exceeds the preprocessed batch %d", batch, slot.batch);
    CUDA_TRY(ctx, cudaMemcpyAsync(dst_dev, slot.tmm, (size_t)batch * (ctx->w / 4) * (ctx->h / 4) * sizeof(uint16_t),
                                  cudaMemcpyDeviceToDevice, (cudaStream_t)stream));
    return APSE_OK;
}

int apse_debug_apriltag(apse_ctx *ctx, const uint8_t *gray, int w, int h, uint8_t *thresh, uint32_t *labels, float *quads,
                        int max_quads, int64_t *stats_host, void *stream)
{
    if (!ctx || !gray) CTX_FAIL(ctx, APSE_ERR_INVALID_ARG, "debug_apriltag: bad argument");
    cudaStream_t st = (cudaStream_t)stream;
    DeviceParams dp;
    apse_fill_device_params(ctx, &dp, w, h);
    int rc = apse_apriltag_quads(ctx, gray, w, h, 1, dp, st, nullptr, ctx->slot[0].tmm, true);
    if (rc) return rc;
    size_t npx = (size_t)w * h;
    if (thresh) CUDA_TRY(ctx, cudaMemcpyAsync(thresh, ctx->thresh, npx, cudaMemcpyDeviceToDevice, st));
    if (labels) CUDA_TRY(ctx, cudaMemcpyAsync(labels, ctx->labels, npx * sizeof(uint32_t), cudaMemcpyDeviceToDevice, st));
    int32_t cnt[APSE_COUNTERS];
    CUDA_TRY(ctx, cudaMemcpyAsync(cnt, ctx->counters, sizeof cnt, cudaMemcpyDeviceToHost, st));
    CUDA_TRY(ctx, cudaStreamSynchronize(st));
    if (cnt[3] != 0) CTX_FAIL(ctx, cnt[3], "debug_apriltag: work buffer capacity exceeded (points %d, clusters %d, quads %d)", cnt[0], cnt[4], cnt[2]);
    int nq = cnt[2] < max_quads ? cnt[2] : max_quads;
    if (quads && nq > 0) {
        CUDA_TRY(ctx, cudaMemcpyAsync(quads, ctx->quads, (size_t)nq * 8 * sizeof(float), cudaMemcpyDeviceToDevice, st));
        CUDA_TRY(ctx, cudaStreamSynchronize(st));
    }
    if (stats_host) { stats_host[0] = cnt[0]; stats_host[1] = cnt[4]; stats_host[2] = cnt[1]; stats_host[3] = cnt[2]; }
    return APSE_OK;
}

}  // extern "C"
