/* apse_b200.h -- C ABI of libapse_b200.so: B200 (sm_100a) CUDA implementation of the per-frame ArUco marker
 * pipeline of vision-agh/apse_uav's aruco_detect.py.
 *
 * The reference has no FFI of its own: its only language boundary is Python -> OpenCV C++ at each cv2.*
 * call (SURVEY.md section 3.2).  Every entry point below replaces one of those calls; the citation gives the
 * aruco_detect.py line of the call it stands in for.  All image / result pointers are DEVICE pointers unless
 * the parameter name ends in _host; all work is enqueued on the caller's stream (cudaStream_t passed as
 * void*, NULL = legacy default stream) and is asynchronous until the caller synchronises.
 *
 * Every function returns 0 on success or a negative apse_status; apse_last_error() returns the message.
 * Plain C types only (no torch / C++ types) so it can be bound from ctypes, cgo, JNI, ...
 */
#ifndef APSE_B200_H
#define APSE_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define APSE_ABI_VERSION 2

typedef enum {
    APSE_OK = 0,
    APSE_ERR_INVALID_ARG = -1,   /* NULL pointer, bad size, unsupported parameter value        */
    APSE_ERR_CUDA = -2,          /* a CUDA runtime call failed (message has the CUDA error)     */
    APSE_ERR_NOT_CONFIGURED = -3,/* camera / lut / dictionary / params not set before use       */
    APSE_ERR_CAPACITY = -4,      /* a fixed-capacity work buffer overflowed (never truncates silently) */
    APSE_ERR_UNSUPPORTED = -5    /* parameter combination outside the implemented hot path      */
} apse_status;

typedef struct apse_ctx apse_ctx;

/* POD mirror of cv2.aruco.DetectorParameters (aruco_detect.py:190-236; field names follow OpenCV).
 * apse_params_default() fills the cv2 4.13 defaults (SURVEY.md Appendix D). */
typedef struct apse_params {
    int adaptiveThreshWinSizeMin, adaptiveThreshWinSizeMax, adaptiveThreshWinSizeStep;
    double adaptiveThreshConstant;
    double minMarkerPerimeterRate, maxMarkerPerimeterRate;
    double polygonalApproxAccuracyRate, minCornerDistanceRate;
    int minDistanceToBorder;
    double minMarkerDistanceRate;
    float minGroupDistance;
    int cornerRefinementMethod;       /* 0 NONE, 1 SUBPIX, 2 CONTOUR, 3 APRILTAG */
    int cornerRefinementWinSize;
    float relativeCornerRefinmentWinSize;
    int cornerRefinementMaxIterations;
    double cornerRefinementMinAccuracy;
    int markerBorderBits;
    int perspectiveRemovePixelPerCell;
    double perspectiveRemoveIgnoredMarginPerCell;
    double maxErroneousBitsInBorderRate;
    double minOtsuStdDev;
    double errorCorrectionRate;
    float aprilTagQuadDecimate, aprilTagQuadSigma;   /* decimate: 0 / 1 (off) or any factor > 1 (the reference's example: 1.5); sigma: |sigma| < 8.25 */
    int aprilTagMinClusterPixels, aprilTagMaxNmaxima;
    float aprilTagCriticalRad, aprilTagMaxLineFitMse;
    int aprilTagMinWhiteBlackDiff, aprilTagDeglitch; /* deglitch must be 0 */
    int detectInvertedMarker;                        /* white markers: inverted bits tried when the border fits better; smallest candidate of a group is its main */
    int useAruco3Detection;                          /* must be 0 */
    int minSideLengthCanonicalImg;
    float minMarkerLengthRatioOriginalImg;
} apse_params;

/* Per-batch detection output (caller-owned DEVICE arrays, capacity max_markers per frame).
 * corners/rejected: [batch][max_markers][4][2] float32; ids: [batch][max_markers] int32;
 * n_markers / n_rejected / status: [batch] int32 (status != 0 -> capacity overflow code for that frame). */
typedef struct apse_detections {
    int max_markers;
    float *corners;
    int32_t *ids;
    int32_t *n_markers;
    float *rejected;      /* nullable */
    int32_t *n_rejected;  /* nullable iff rejected is NULL */
    int32_t *status;
} apse_detections;

int apse_abi_version(void);
void apse_params_default(apse_params *p);

/* Context: owns all scratch (labels, point lists, tables) sized here; no allocation on the hot path. */
int apse_create(apse_ctx **out, int device, int max_w, int max_h, int max_batch);
void apse_destroy(apse_ctx *ctx);
const char *apse_last_error(apse_ctx *ctx);

/* aruco_detect.py:92-103,568 -- camera model; builds the undistort maps on the device (initUndistortRectifyMap) */
int apse_set_camera(apse_ctx *ctx, const double K_host[9], const double D_host[14], int w, int h, void *stream);
/* aruco_detect.py:537-540 -- gamma look-up table applied to the Lab L channel */
int apse_set_lut(apse_ctx *ctx, const uint8_t lut_host[256], void *stream);
/* aruco_detect.py:263 -- dictionary bytesList [n_markers][4 rotations][nbytes] */
int apse_set_dictionary(apse_ctx *ctx, const uint8_t *bytes_host, int n_markers, int marker_size, int max_corr_bits,
                        void *stream);
/* aruco_detect.py:190-236,266 */
int apse_set_params(apse_ctx *ctx, const apse_params *p);

/* ---- stage entry points (device pointers) --------------------------------------------------------------- */
/* aruco_detect.py:568  cv2.initUndistortRectifyMap(K, D, None, K, (w,h), CV_32FC1) */
int apse_init_undistort_map(apse_ctx *ctx, const double K_host[9], const double D_host[14], int w, int h,
                            float *mapx, float *mapy, void *stream);
/* aruco_detect.py:252  cv2.remap(src, mapx, mapy, INTER_LINEAR), BORDER_CONSTANT 0; cn = 1 or 3 */
int apse_remap(apse_ctx *ctx, const uint8_t *src, int sw, int sh, int cn, const float *mapx, const float *mapy,
               int dw, int dh, uint8_t *dst, void *stream);

/* cv2.undistort(src, K, D, None, newK) (dcnn/scripts/tests/visualize_uav.py:62): FP64 source coordinate rounded to the Q5
 * grid directly (the dependency's CV_16SC2 maps) + the bilinear remap of apse_remap; newK == NULL means K.  Differs from
 * initUndistortRectifyMap(CV_32FC1) + remap (aruco_detect.py:568,252) in ~0.1 % of the pixels, exactly as in the dependency. */
int apse_undistort(apse_ctx *ctx, const uint8_t *src, int w, int h, int channels, const double K[9], const double D[14],
                   const double newK[9], uint8_t *dst, void *stream);
/* aruco_detect.py:255  cv2.cvtColor(.., COLOR_RGB2LAB) on 8-bit 3-channel pixels */
int apse_cvt_rgb2lab(apse_ctx *ctx, const uint8_t *src, int64_t npx, uint8_t *dst, void *stream);
/* aruco_detect.py:257  cv2.cvtColor(.., COLOR_LAB2RGB) */
int apse_cvt_lab2rgb(apse_ctx *ctx, const uint8_t *src, int64_t npx, uint8_t *dst, void *stream);
/* aruco_detect.py:592  cv2.cvtColor(.., COLOR_BGR2GRAY) */
int apse_cvt_bgr2gray(apse_ctx *ctx, const uint8_t *src, int64_t npx, uint8_t *dst, void *stream);
/* aruco_detect.py:256  cv2.LUT(src, lut) on a channel of an interleaved image: src/dst element stride in bytes */
int apse_lut(apse_ctx *ctx, const uint8_t *src, int64_t n, int src_stride, const uint8_t *lut_dev, uint8_t *dst,
             int dst_stride, void *stream);

/* YUV 4:2:0 layouts of cv2's single-array form [h*3/2][w] (what H.264 / HEVC decoders produce): Y plane, then
 * NV12: interleaved U V; NV21: interleaved V U; I420 (IYUV): U plane, V plane; YV12: V plane, U plane
 * (each chroma plane (h/2)*(w/2) contiguous bytes) */
typedef enum { APSE_YUV_NV12 = 0, APSE_YUV_NV21 = 1, APSE_YUV_I420 = 2, APSE_YUV_YV12 = 3 } apse_yuv_layout;
/* cv2.cvtColor(src, COLOR_YUV2BGR_{NV12,NV21,I420,YV12}) for a batch: yuv [batch][h*3/2][w], bgr [batch][h][w][3] (device).
 * w and h even.  Uses no context scratch: the frame size is not bounded by apse_create's max_w / max_h. */
int apse_cvt_yuv420_bgr(apse_ctx *ctx, const uint8_t *yuv, int w, int h, int batch, int layout, uint8_t *bgr, void *stream);

/* aruco_detect.py:250-259 + :592 fused: remap + Lab gamma + gray for a batch of frames
 * bgr: [batch][h][w][3]; bgr_out (nullable): same shape; gray: [batch][h][w] */
int apse_preprocess(apse_ctx *ctx, const uint8_t *bgr, uint8_t *bgr_out, uint8_t *gray, int batch, void *stream);

/* aruco_detect.py:267  aruco.detectMarkers(gray, dict, parameters=...) for a batch of gray frames [batch][h][w] */
int apse_detect(apse_ctx *ctx, const uint8_t *gray, int w, int h, int batch, apse_detections *out, void *stream);

/* aruco_detect.py:601  aruco.estimatePoseSingleMarkers(corners, markerLength, K, D)
 * corners: [n][4][2] float32 (device); marker_len: [n] float32 (device) or NULL to use marker_len_all;
 * rvec/tvec: [n][3] float64 (device) */
int apse_pose(apse_ctx *ctx, const float *corners, int n, const float *marker_len, float marker_len_all,
              const double K_host[9], const double D_host[14], double *rvec, double *tvec, void *stream);

/* Batched form of apse_pose over the output of apse_detect: corners [batch][max_markers][4][2], n_markers [batch];
 * marker_len: [batch] float32 (device, one length per frame -- aruco_detect.py:601 uses the global markerLength of
 * that frame) or NULL for marker_len_all; rvec/tvec: [batch][max_markers][3] float64; slots >= n_markers untouched */
int apse_pose_frames(apse_ctx *ctx, const float *corners, const int32_t *n_markers, int batch, int max_markers,
                     const float *marker_len, float marker_len_all, const double K_host[9], const double D_host[14],
                     double *rvec, double *tvec, void *stream);

/* aruco_detect.py:589-601 in one call for a batch of raw frames: preprocessFrame + BGR2GRAY + detectMarkers +
 * estimatePoseSingleMarkers (camera of apse_set_camera).  Same results as apse_preprocess -> apse_detect ->
 * apse_pose_frames; the fused kernel hands the 4x4-tile extrema of gray to the candidate stage directly.
 * bgr: [batch][h][w][3]; gray: [batch][h][w] or NULL (context scratch; the library then evaluates gray sparsely, see
 * apse_preprocess_tiles_sparse); rvec/tvec nullable (no pose) */
int apse_process_frames(apse_ctx *ctx, const uint8_t *bgr, uint8_t *gray, int batch, apse_detections *out,
                        const float *marker_len, float marker_len_all, double *rvec, double *tvec, void *stream);

/* The two halves of apse_process_frames as separate calls, so that a caller can put them on different streams
 * (bandwidth / issue-bound preprocess of batch k+1 on a low-priority stream under the latency-bound candidate /
 * decode / pose chain of batch k): apse_preprocess_tiles = aruco_detect.py:250-259,592 (+ tile extrema kept in the
 * context); apse_detect_pose_frames = :267 + :601 on that gray batch (the caller orders the two with an event). */
int apse_preprocess_tiles(apse_ctx *ctx, const uint8_t *bgr, uint8_t *gray, int batch, void *stream);
/* Sparse evaluation of the same half (CORNER_REFINE_APRILTAG only): identical detections, but the colour chain of
 * aruco_detect.py:255-257,592 runs only where the detector can read its result.  Every pixel is still remapped (:252) and
 * bounded through a table of (min, max) gray per colour cell that the library computes from the exact chain over all 2^24
 * colours when the LUT is set; tiles whose 3x3-dilated BOUND range cannot reach aprilTagMinWhiteBlackDiff (:200) are certain
 * to become 127 in the detector's threshold image and are skipped; the others (+ a one-tile ring) and the samples of
 * candidate quads get the exact chain.  `gray` is a work buffer afterwards: complete only on the evaluated tiles and only
 * meaningful to the apse_detect_pose_frames call that follows on this context.  apse_process_frames(gray = NULL) takes this
 * path as well.  Falls back to apse_preprocess_tiles for frame geometries without a TMA path. */
int apse_preprocess_tiles_sparse(apse_ctx *ctx, const uint8_t *bgr, uint8_t *gray, int batch, void *stream);
int apse_detect_pose_frames(apse_ctx *ctx, const uint8_t *gray, int batch, apse_detections *out, const float *marker_len,
                            float marker_len_all, double *rvec, double *tvec, void *stream);

/* aruco_detect.py:344,377,424,468  cv2.projectPoints(obj, rvec, tvec, K, D)
 * obj: [n][3] float64, rvec/tvec: [3] float64, img: [n][2] float64 -- all device pointers */
int apse_project_points(apse_ctx *ctx, const double *obj, int n, const double *rvec, const double *tvec,
                        const double K_host[9], const double D_host[14], double *img, void *stream);

/* Many projectPoints calls in one launch: point i uses pose pose_idx[i] of rvecs/tvecs [m][3] (all device) */
int apse_project_points_multi(apse_ctx *ctx, const double *obj, int n, const int32_t *pose_idx, const double *rvecs,
                              const double *tvecs, const double K_host[9], const double D_host[14], double *img,
                              void *stream);

/* Debug / parity taps of the APRILTAG candidate path for ONE frame (device pointers, nullable):
 * thresh [h][w] u8 ternary image, labels [h][w] u32 component representative (valid where thresh != 127),
 * quads [max_quads][8] float32 raw quads (cluster-key order), stats[4] int64 {points, clusters, fitted, quads} */
int apse_debug_apriltag(apse_ctx *ctx, const uint8_t *gray, int w, int h, uint8_t *thresh, uint32_t *labels,
                        float *quads, int max_quads, int64_t *stats_host, void *stream);

/* aruco_detect.py:352-358 (detectAndDrawLEDs): sums of the (2 half + 1)^2 gray neighbourhoods gray[y-half:y+half+1,
 * x-half:x+half+1] (numpy slicing rules at the image edges) of n points; pts: [n][3] int32 (frame, x, y), sums: [n]
 * int64 -- device pointers; gray: [frames][h][w] */
int apse_patch_sums(apse_ctx *ctx, const uint8_t *gray, int w, int h, const int32_t *pts, int n, int half, int64_t *sums,
                    void *stream);

/* cv2.adaptiveThreshold(gray, 255, ADAPTIVE_THRESH_MEAN_C, THRESH_BINARY_INV, win, c) for a batch [batch][h][w]: the
 * threshold step of the classic candidate path inside aruco.detectMarkers (aruco_detect.py:267 with
 * cornerRefinementMethod NONE / SUBPIX; north_star stage 2).  Even win is bumped to win + 1 as aruco does. */
int apse_adaptive_threshold(apse_ctx *ctx, const uint8_t *gray, int w, int h, int batch, int win, double c, uint8_t *out,
                            void *stream);

/* Debug / parity tap of the classic candidate path for ONE frame: quads [max_quads][8] float32 (unordered) and
 * order [max_quads] = rank of each quad in the dependency's candidate order; stats[0] = number of quads */
int apse_debug_classic(apse_ctx *ctx, const uint8_t *gray, int w, int h, float *quads, uint32_t *order, int max_quads,
                       int64_t *stats_host, void *stream);

/* ---- sequence post-pass (aruco_detect.py:598-782, CSV row :146-185) --------------------------------------------
 * The marker logic of the reference's frame loop over the per-frame results of apse_process_frames, for a whole
 * sequence at once.  Only the O(markers) state machine is sequential (apse_sequence_scan, host); every
 * cv2.projectPoints call of the loop (:344 LED strip, :468 vehicle outline) feeds outputs only and is deferred as a
 * job, evaluated for all frames in one launch (apse_sequence_jobs, device).  All arrays of the three host functions
 * are HOST pointers. */
typedef struct apse_seq_config {
    int start_frame, step_frame;                   /* aruco_detect.py:13,18; DIFF_MAX = 2/3 * step_frame * 2 (:524) */
    double marker_length_org, marker_div, div;     /* :520-523 */
    int width, height;                             /* :519 (field-of-view columns of the CSV) */
    int leds_threshold;                            /* LEDs_threshold (:36); < 0 = the default rule max(190 + int(tvec_z / marker_div), 240) */
    int leds;                                      /* 1 = emit LED read-out jobs (needs the corrected gray frames on the device) */
} apse_seq_config;

typedef struct apse_seq_job {                      /* one deferred projection job */
    int32_t frame;                                 /* index of the frame in the sequence */
    int32_t kind;                                  /* 0 = LED strip of the host vehicle (:338-373); 1..3 = distance host -> vehicle `kind` (:729-780) */
    double rvec[3], tvec[3];                       /* pose of the marker, tvec already divided by size_corr */
    double dim[4];                                 /* kind >= 1: scaled vehicle outline back, front, left, right (:406-420) */
    float src[2], tgt[2];                          /* kind >= 1: host-marker centre, vehicle-marker centre (:271-274) */
    double scale;                                  /* kind >= 1: markerLength / ((msp4 + msp_v) / 2)  (:489-490) */
    int32_t led_threshold, pad_;
} apse_seq_job;

typedef struct apse_seq_job_result {
    double dist_aruco, dist_bbox;                  /* kind >= 1, metres, unrounded */
    int32_t leds;                                  /* kind 0: the 8-bit LED code */
    int32_t valid;                                 /* 1 once a device has filled this result */
    int32_t nearest_px[2];                         /* kind >= 1: the outline point closest to the host marker (:466-481), for the renderer */
    int32_t outline_px[4][2];                      /* kind >= 1: projected outline corners in drawContours order (:421-425) */
} apse_seq_job_result;

typedef struct apse_seq_row {                      /* one CSV row (:146-185); float fields carry Python's round() */
    int32_t frame_id;
    int32_t detected[4];                           /* detected_ID[0..3] = vehicles 1, 2, 3, host */
    int32_t host_fields;                           /* 1: markerLength .. fov_height are written as floats, 0: the reference writes integer zeros */
    int32_t leds;
    int32_t job_led, job_dist[3];                  /* jobs whose results this frame takes (-1: value stays stale) */
    int32_t accepted_mask;                         /* bits 0-7: marker slot i of this frame passed the track gate (:613) -- what drawMarkers draws */
    double marker_length, altitude, fov_width, fov_height;
    double dist_aruco[3], dist_bbox[3];
} apse_seq_row;

void apse_seq_config_default(apse_seq_config *c);
/* Python's round(x, ndigits) on a float, as the CSV columns of :146-185 need it (exact half-to-even on the binary value) */
double apse_py_round(double x, int ndigits);
/* Sequential scan over n_frames frames: n_markers [F], ids [F][M] int32, corners [F][M][4][2] float32, rvec / tvec [F][M][3]
 * float64 (the layout apse_process_frames writes).  lengths (nullable) [F] receives the marker length the pose of each frame
 * must be computed with (:601 uses the global markerLength left by the previous frames).  rescale_tvec = 1: the poses were
 * computed with marker_length_org and tvec is scaled by markerLength / marker_length_org on the fly (first pass, only
 * `lengths` is meaningful).  rows / jobs / n_jobs nullable together (first pass).  Returns APSE_ERR_CAPACITY if job_cap is
 * too small (4 jobs per frame always suffice when marker ids are unique). */
int apse_sequence_scan(const apse_seq_config *cfg, int n_frames, int max_markers, const int32_t *n_markers, const int32_t *ids,
                       const float *corners, const double *rvec, const double *tvec, int rescale_tvec, double *lengths,
                       apse_seq_row *rows, apse_seq_job *jobs, int job_cap, int *n_jobs);
/* The same scan for a sequence that arrives in chunks (frames frame0 .. frame0 + n_frames - 1 of the sequence, chunks in order):
 * `state` carries the reference's module globals (:519-524, :782) from chunk to chunk; zero it before the first chunk.  Use one
 * state per pass (rescale_tvec = 1 / = 0).  Job and row indices are local to the chunk. */
typedef struct apse_seq_state { unsigned char opaque[512]; } apse_seq_state;
int apse_sequence_scan_chunk(const apse_seq_config *cfg, apse_seq_state *state, int frame0, int n_frames, int max_markers,
                             const int32_t *n_markers, const int32_t *ids, const float *corners, const double *rvec, const double *tvec,
                             int rescale_tvec, double *lengths, apse_seq_row *rows, apse_seq_job *jobs, int job_cap, int *n_jobs);
/* apse_sequence_finish for one chunk; the stale values (:729-780 leave the last distance / LED code in place) travel in the
 * state of the SECOND pass (the one apse_sequence_scan_chunk produced these rows with) */
int apse_sequence_finish_chunk(apse_seq_state *state, int n_frames, apse_seq_row *rows, const apse_seq_job_result *results, int n_jobs);
/* Evaluates the jobs on the device (one warp per job) and copies the results back; synchronous on `stream`.
 * gray (DEVICE, nullable): corrected gray frames [n_gray_frames][h][w] of the sequence frames frame0 .. frame0 + n_gray_frames - 1;
 * LED jobs of other frames are left with valid = 0 (frame-sharded runs: every rank fills the LED jobs of its own frames). */
int apse_sequence_jobs(apse_ctx *ctx, const apse_seq_job *jobs_host, int n_jobs, const uint8_t *gray, int frame0, int n_gray_frames,
                       int w, int h, const double K_host[9], const double D_host[14], apse_seq_job_result *results_host, void *stream);
/* Job results -> rows: values the reference leaves stale between frames stay stale; rounding of :146-185 */
int apse_sequence_finish(int n_frames, apse_seq_row *rows, const apse_seq_job_result *results, int n_jobs);
/* The CSV text of :131-139,146-185 (Python's str() of ints and floats); returns the number of bytes written or a negative status */
int64_t apse_sequence_csv(const apse_seq_row *rows, int n_frames, int with_header, char *buf, int64_t cap);

/* ---- annotated frames (aruco_detect.py:494-500,614-616,421-425: marker quads, vehicle outlines, distance lines, points) ---------
 * Overlay primitives drawn straight into device-resident BGR frames: a thick segment with round caps (what cv2.line /
 * cv2.drawContours produce up to their anti-aliasing-free edge rule) or a filled disc (cv2.circle, thickness -1).  Primitives of
 * one frame are drawn in list order (later ones on top); the list must be sorted by frame.  prims: DEVICE pointer. */
typedef struct apse_overlay_prim {
    int32_t frame;
    int32_t kind;                                  /* 0 = segment, 1 = disc */
    int32_t x0, y0, x1, y1;                        /* segment end points; disc: centre = (x0, y0) */
    int32_t thickness;                             /* segment: cv2 thickness; disc: radius */
    uint8_t bgr[4];
} apse_overlay_prim;
int apse_draw_overlay(apse_ctx *ctx, uint8_t *bgr, int w, int h, int batch, const apse_overlay_prim *prims, int n_prims, void *stream);

/* test tap of the identification stage in isolation (_extractBits + Dictionary::identify of ONE gray frame): for each of the n
 * candidate quads (corners [n][4][2] float32) the canonical image (img [n][64*64], the first S*S bytes, S = (markerSize + 2
 * border) * perspectiveRemovePixelPerCell), the cell bits (bits [n][256], first (markerSize + 2 border)^2) and result [n][4] =
 * {valid, id, rotation, Otsu threshold (-1: flat candidate, decided by its mean)}.  All pointers DEVICE. */
int apse_debug_decode(apse_ctx *ctx, const uint8_t *gray, int w, int h, const float *corners, int n, uint8_t *img, uint8_t *bits,
                      int32_t *result, void *stream);

/* test tap of the sparse evaluation: the bound table (HOST, 16*32*32 entries min | (255 - max) << 8, cell = (c0 >> 4, c1 >> 3,
 * c2 >> 3)), the tile flags of the last apse_preprocess_tiles_sparse batch (DEVICE, [batch][h/4][w/4], 1 = evaluated exactly)
 * and their count; every pointer nullable */
int apse_debug_sparse(apse_ctx *ctx, uint16_t *bound_table_host, uint8_t *eflag_dev, int batch, int *n_exact_host, void *stream);

/* test tap of the bounds pass of the last apse_preprocess_tiles_sparse batch: per-tile bounds of gray (DEVICE,
 * [batch][h/4][w/4], lo | hi << 8; every gray value the preprocess of aruco_detect.py:250-259,592 can produce inside the
 * tile lies in [lo, hi]) */
int apse_debug_tile_bounds(apse_ctx *ctx, uint16_t *bounds_dev, int batch, void *stream);

/* test tap of the 4x4-tile extrema of gray that the last apse_preprocess_tiles[_sparse] call left for the detector (DEVICE,
 * [batch][h/4][w/4], min | max << 8; after the sparse evaluation a tile that was not evaluated exactly holds (255, 0)).
 * APSE_ERR_NOT_CONFIGURED when that call produced no extrema (the frame geometry took the generic kernel) or when another call
 * on the context has dropped them since. */
int apse_debug_tile_extrema(apse_ctx *ctx, uint16_t *dst_dev, int batch, void *stream);

/* number of kernel launches issued through this context since creation (bench.py's gpu_launches) */
int64_t apse_launch_count(apse_ctx *ctx);

/* Optional per-kernel device timing: while enabled every launch is bracketed by CUDA events on the launching
 * stream; collect() synchronises and returns accumulated milliseconds / launch counts per kernel id. */
int apse_kernel_count(void);
const char *apse_kernel_name(int kid);
int apse_timing_enable(apse_ctx *ctx, int on);
int apse_timing_collect(apse_ctx *ctx, double *ms_host, int64_t *launches_host, int reset);
/* Development aid.  out == NULL: arm a trace of up to cap_rows launches.  Otherwise copy the rows {kernel id, start ms,
 * end ms} (relative to a process-wide origin) of the launches timed since, return their number and clear the trace. */
int apse_timing_trace(apse_ctx *ctx, double *out, int cap_rows);

#ifdef __cplusplus
}
#endif
#endif /* APSE_B200_H */
