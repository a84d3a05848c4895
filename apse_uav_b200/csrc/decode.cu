// decode.cu -- candidate post-filter, perspective bit sampling and dictionary matching of
// aruco.detectMarkers (aruco_detect.py:267, dictionary aruco_detect.py:263); SURVEY.md rows a6.A5-a6.A7,
// cv2 4.13 semantics.  One CTA per frame:
//   * quads ordered deterministically, border filter, stable sort by perimeter (descending)
//   * "too close" predicate for all pairs in parallel (centroid pre-test -> pair list -> exact test); the dependency's
//     order-dependent grouping walk restated as "first partner per candidate" (atomicMin) + chains to a mutual first pair
//   * every candidate decoded by one warp: FP64 homography, 48x48 nearest-neighbour gather, Otsu on a
//     shared-memory histogram, per-cell majority, border check, Hamming match against the dictionary
//   * nesting hierarchy + depth-ordered acceptance, corner rotation, output
// Compiled with -fmad=false (homography / Otsu arithmetic follows the dependency's evaluation order).
#include "common.cuh"
#include "chain.cuh"
#include <math.h>
#include <float.h>

#define DEC_THREADS 1024
#define DEC_WARPS (DEC_THREADS / 32)
#define DEC_MAX_S 64                      // canonical image side limit ((markerSize + 2*border) * cellSize)
#define DEC_SMEMC 512                     // candidates per frame handled entirely in shared memory
#define DEC_MIDC 1920                     // ... with everything but the too-close bit matrix in shared memory (classic path)
#define DEC_MAXC APSE_MAX_QUADS           // candidates per frame (beyond DEC_SMEMC the arrays live in global scratch)

// per-frame candidate arrays, carved out of shared memory (n <= DEC_SMEMC) or of a global scratch block
struct DecodeArrays {
    float (*c)[8];                        // candidate corners, sorted by perimeter (descending, stable)
    float *perim;
    uint32_t *key;                        // ordering key (rank in the dependency's candidate order) / scratch
    uint32_t *close_bits;                 // [cap][cap / 32] words of scratch (centroid-test operands, bounding boxes; once a bit matrix)
    uint32_t *pairs;                      // [cap * 8] pairs (i << 16 | j) that pass the centroid pre-test, unordered
    float *cxy;                           // [cap][2] scratch: perimeters before the sort, group member lists, nesting heights
    short *group_id, *next_in_group, *close_next, *parent, *depth, *sel, *sel_of, *dec_id, *use_c, *group_head, *group_tail;
    uint8_t *dec_valid, *dec_rot, *selected, *was, *valid;
    int cap;
};

__host__ __device__ inline size_t decode_arrays_bytes(int cap)
{
    return (size_t)cap * (8 * 4 + 4 + 4 + (cap / 32) * 4 + 8 * 4 + 2 * 4 + 11 * 2 + 5) + 64;
}

// bytes of everything but the too-close bit matrix (the middle tier keeps that matrix in global memory)
__host__ __device__ inline size_t decode_arrays_small_bytes(int cap)
{
    return (size_t)cap * (8 * 4 + 4 + 4 + 8 * 4 + 2 * 4 + 11 * 2 + 5) + 64;
}

// close_bits_ext != nullptr: the bit matrix lives there instead of behind `key`
__device__ inline void decode_arrays_carve(DecodeArrays &A, unsigned char *base, int cap, uint32_t *close_bits_ext = nullptr)
{
    A.cap = cap;
    unsigned char *p = base;
    A.c = reinterpret_cast<float(*)[8]>(p); p += (size_t)cap * 32;
    A.perim = reinterpret_cast<float *>(p); p += (size_t)cap * 4;
    A.key = reinterpret_cast<uint32_t *>(p); p += (size_t)cap * 4;
    if (close_bits_ext) A.close_bits = close_bits_ext;
    else { A.close_bits = reinterpret_cast<uint32_t *>(p); p += (size_t)cap * (cap / 32) * 4; }
    A.pairs = reinterpret_cast<uint32_t *>(p); p += (size_t)cap * 32;
    A.cxy = reinterpret_cast<float *>(p); p += (size_t)cap * 8;
    short **sp[11] = {&A.group_id, &A.next_in_group, &A.close_next, &A.parent, &A.depth, &A.sel, &A.sel_of, &A.dec_id, &A.use_c,
                      &A.group_head, &A.group_tail};
    for (int i = 0; i < 11; i++) { *sp[i] = reinterpret_cast<short *>(p); p += (size_t)cap * 2; }
    uint8_t **bp[5] = {&A.dec_valid, &A.dec_rot, &A.selected, &A.was, &A.valid};
    for (int i = 0; i < 5; i++) { *bp[i] = p; p += cap; }
}

// Top tier (up to DEC_MAXC candidates): the three big arrays -- corners, pair list, bit matrix -- in global scratch, every array the
// single-thread walks and the O(n^2) loops index per element (perimeters, centroids, group / nesting bookkeeping) in shared memory
__host__ __device__ inline size_t decode_arrays_top_bytes(int cap) { return (size_t)cap * (4 + 4 + 2 * 4 + 11 * 2 + 5) + 64; }
__device__ inline void decode_arrays_carve_top(DecodeArrays &A, unsigned char *smem, unsigned char *global, int cap)
{
    A.cap = cap;
    unsigned char *g = global, *p = smem;
    A.c = reinterpret_cast<float(*)[8]>(g); g += (size_t)cap * 32;
    A.close_bits = reinterpret_cast<uint32_t *>(g); g += (size_t)cap * (cap / 32) * 4;
    A.pairs = reinterpret_cast<uint32_t *>(g);
    A.perim = reinterpret_cast<float *>(p); p += (size_t)cap * 4;
    A.key = reinterpret_cast<uint32_t *>(p); p += (size_t)cap * 4;
    A.cxy = reinterpret_cast<float *>(p); p += (size_t)cap * 8;
    short **sp[11] = {&A.group_id, &A.next_in_group, &A.close_next, &A.parent, &A.depth, &A.sel, &A.sel_of, &A.dec_id, &A.use_c,
                      &A.group_head, &A.group_tail};
    for (int i = 0; i < 11; i++) { *sp[i] = reinterpret_cast<short *>(p); p += (size_t)cap * 2; }
    uint8_t **bp[5] = {&A.dec_valid, &A.dec_rot, &A.selected, &A.was, &A.valid};
    for (int i = 0; i < 5; i++) { *bp[i] = p; p += cap; }
}

// development aid (-DAPSE_DEC_PROFILE): cycles between the phases of k_decode, printed by frame 0
#ifdef APSE_DEC_PROFILE
#define DEC_T(i) do { __syncthreads(); if (threadIdx.x == 0 && blockIdx.x == 0) dbg_t[i] = clock64(); } while (0)
#else
#define DEC_T(i) do { } while (0)
#endif

struct DecodeSmem {
    int n, ns, ngroups;
    int pad;
    // followed by decode_arrays_bytes(DEC_SMEMC) bytes
};

__device__ __forceinline__ float sqf(float v) { return v * v; }

__device__ float perimeter_of(const float *c)
{
    float p = 0.f;
    for (int i = 0; i < 4; i++) {
        int j = (i + 1) % 4;
        p += sqrtf(sqf(c[2 * i] - c[2 * j]) + sqf(c[2 * i + 1] - c[2 * j + 1]));
    }
    return p;
}

__device__ float average_distance(const float *m1, const float *m2)
{
    float best = FLT_MAX;
    for (int fc = 0; fc < 4; fc++) {
        float d = 0;
        for (int c = 0; c < 4; c++) {
            int mc = (c + fc) % 4;
            float dx = m1[2 * mc] - m2[2 * c], dy = m1[2 * mc + 1] - m2[2 * c + 1];
            d += dx * dx + dy * dy;
        }
        d /= 4.f;
        best = fminf(best, d);
    }
    return sqrtf(best);
}

__device__ float average_module_size(const float *c, int ms, int bb)
{
    float a = 0.f;
    for (int i = 0; i < 4; i++) {
        int j = (i + 1) % 4;
        float dx = c[2 * i] - c[2 * j], dy = c[2 * i + 1] - c[2 * j + 1];
        a += sqrtf(dx * dx + dy * dy);
    }
    return a / (4.f * (ms + bb * 2));
}

// pointPolygonTest(poly, pt, false) > 0 for a 4-gon of float points
__device__ bool strictly_inside(const float *poly, float px, float py)
{
    int counter = 0;
    float vx = poly[6], vy = poly[7];
    for (int i = 0; i < 4; i++) {
        float v0x = vx, v0y = vy;
        vx = poly[2 * i]; vy = poly[2 * i + 1];
        if ((v0y <= py && vy <= py) || (v0y > py && vy > py) || (v0x < px && vx < px)) {
            if (py == vy && (px == vx || (py == v0y && ((v0x <= px && px <= vx) || (vx <= px && px <= v0x))))) return false;
            continue;
        }
        double dist = (double)(py - v0y) * (vx - v0x) - (double)(px - v0x) * (vy - v0y);
        if (dist == 0) return false;
        if (vy < v0y) dist = -dist;
        counter += dist > 0;
    }
    return (counter % 2) != 0;
}

// getPerspectiveTransform(corners -> canonical square) followed by the 3x3 inverse used by warpPerspective
__device__ void inverse_homography(const float *src, int S, double *Mi)
{
    double a[64], b[8];
    const float dstc[8] = {0.f, 0.f, (float)S - 1, 0.f, (float)S - 1, (float)S - 1, 0.f, (float)S - 1};
    for (int i = 0; i < 64; i++) a[i] = 0;
    for (int i = 0; i < 4; i++) {
        float sx = src[2 * i], sy = src[2 * i + 1], dx = dstc[2 * i], dy = dstc[2 * i + 1];
        a[i * 8 + 0] = a[(i + 4) * 8 + 3] = sx;
        a[i * 8 + 1] = a[(i + 4) * 8 + 4] = sy;
        a[i * 8 + 2] = a[(i + 4) * 8 + 5] = 1;
        // the dependency forms these products on float32 point members before widening to double
        a[i * 8 + 6] = __fmul_rn(-sx, dx);
        a[i * 8 + 7] = __fmul_rn(-sy, dx);
        a[(i + 4) * 8 + 6] = __fmul_rn(-sx, dy);
        a[(i + 4) * 8 + 7] = __fmul_rn(-sy, dy);
        b[i] = dx;
        b[i + 4] = dy;
    }
    bool ok = true;
    for (int i = 0; i < 8 && ok; i++) {  // LU, partial pivoting
        int k = i;
        for (int j = i + 1; j < 8; j++)
            if (fabs(a[j * 8 + i]) > fabs(a[k * 8 + i])) k = j;
        if (fabs(a[k * 8 + i]) < DBL_EPSILON) { ok = false; break; }
        if (k != i) {
            for (int j = i; j < 8; j++) { double t = a[i * 8 + j]; a[i * 8 + j] = a[k * 8 + j]; a[k * 8 + j] = t; }
            double t = b[i]; b[i] = b[k]; b[k] = t;
        }
        double d = -1 / a[i * 8 + i];
        for (int j = i + 1; j < 8; j++) {
            double alpha = a[j * 8 + i] * d;
            for (k = i + 1; k < 8; k++) a[j * 8 + k] += alpha * a[i * 8 + k];
            b[j] += alpha * b[i];
        }
    }
    if (ok)
        for (int i = 7; i >= 0; i--) {
            double s = b[i];
            for (int k = i + 1; k < 8; k++) s -= a[i * 8 + k] * b[k];
            b[i] = s / a[i * 8 + i];
        }
    else
        for (int i = 0; i < 8; i++) b[i] = 0;
    double m[9] = {b[0], b[1], b[2], b[3], b[4], b[5], b[6], b[7], 1.};
    double d = m[0] * (m[4] * m[8] - m[5] * m[7]) - m[1] * (m[3] * m[8] - m[5] * m[6]) + m[2] * (m[3] * m[7] - m[4] * m[6]);
    if (d == 0) { for (int i = 0; i < 9; i++) Mi[i] = 0; return; }
    d = 1. / d;
    Mi[0] = (m[4] * m[8] - m[5] * m[7]) * d; Mi[1] = (m[2] * m[7] - m[1] * m[8]) * d; Mi[2] = (m[1] * m[5] - m[2] * m[4]) * d;
    Mi[3] = (m[5] * m[6] - m[3] * m[8]) * d; Mi[4] = (m[0] * m[8] - m[2] * m[6]) * d; Mi[5] = (m[2] * m[3] - m[0] * m[5]) * d;
    Mi[6] = (m[3] * m[7] - m[4] * m[6]) * d; Mi[7] = (m[1] * m[6] - m[0] * m[7]) * d; Mi[8] = (m[0] * m[4] - m[1] * m[3]) * d;
}

// _identifyOneCandidate, two phases.
// (1) decode_sample: ALL threads of the CTA.  Nearest-neighbour warp (rint of the FP64 source coordinate, border 0) into img,
//     histogram, inner-region moments.  This is the latency of the candidate (2304 dependent gathers for a 48 x 48 canonical
//     image), so it is spread over the whole CTA.
// SPARSE: the gray buffer holds exact values only on the tiles flagged in S.eflag; every other sample is computed on demand
// from the source frame (same remap + colour chain as the preprocess kernels, bit-identical by construction)
template <bool SPARSE>
__device__ __forceinline__ void decode_sample(const uint8_t *__restrict__ im, int w, int h, const double *Mi, const DeviceParams &P,
                                              const SparseSrc &SS, int frame, uint8_t *img, int *hist, long long &s1, long long &s2)
{
    const int nb = P.marker_size + 2 * P.border_bits, cs = P.cell_size, S = nb * cs;
    const int c0 = cs / 2, c1 = S - cs / 2;
    s1 = 0; s2 = 0;
    for (int p = threadIdx.x; p < S * S; p += blockDim.x) {
        int y = p / S, x = p - y * S;
        double X0 = Mi[1] * y + Mi[2], Y0 = Mi[4] * y + Mi[5], W0 = Mi[7] * y + Mi[8];
        double W = W0 + Mi[6] * x;
        W = W ? 1. / W : 0;
        double fX = (X0 + Mi[0] * x) * W, fY = (Y0 + Mi[3] * x) * W;
        fX = fmin(fmax(fX, (double)INT32_MIN), (double)INT32_MAX);
        fY = fmin(fmax(fY, (double)INT32_MIN), (double)INT32_MAX);
        long long X = __double2ll_rn(fX), Y = __double2ll_rn(fY);
        int v = 0;
        if (X >= 0 && X < w && Y >= 0 && Y < h) {
            if (!SPARSE || SS.eflag[((size_t)frame * SS.th + ((int)Y >> 2)) * SS.tw + ((int)X >> 2)])
                v = im[(size_t)Y * w + X];
            else
                v = exact_gray_px(SS.bgr + (size_t)frame * w * h * 3, SS.mapx, SS.mapy, SS.tables, w, h, (int)X, (int)Y);
        }
        img[p] = (uint8_t)v;
        atomicAdd(&hist[v], 1);
        if (x >= c0 && x < c1 && y >= c0 && y < c1) { s1 += v; s2 += v * v; }
    }
}

// (2) decode_finish: ONE warp.  Otsu (sequential over the 256 bins in the dependency's order), cell majority, border check,
//     Hamming match against the dictionary.  Returns (valid, id, rot) on every lane.
__device__ void decode_finish(const DeviceParams &P, long long s1, long long s2, const uint8_t *__restrict__ dict, const uint8_t *img,
                              const int *hist, uint8_t *bits, bool &valid, int &id, int &rot, int *thr_out = nullptr)
{
    const int lane = threadIdx.x & 31;
    const int nb = P.marker_size + 2 * P.border_bits, cs = P.cell_size, S = nb * cs;
    const int c0 = cs / 2, c1 = S - cs / 2;
    const int cnt = (c1 - c0) * (c1 - c0);
    double mean = (double)s1 / cnt, var = (double)s2 / cnt - mean * mean;
    double sd = sqrt(var > 0 ? var : 0);
    if (sd < P.min_otsu_stddev) {
        for (int i = lane; i < nb * nb; i += 32) bits[i] = mean > 127 ? 1 : 0;
        if (thr_out && lane == 0) *thr_out = -1;   // flat candidate: no Otsu threshold
    } else {
        int thr = 0;
        if (lane == 0) {  // Otsu, sequential over the 256 bins in the dependency's order
            double mu = 0, scale = 1. / (S * S);
            for (int i = 0; i < 256; i++) mu += i * (double)hist[i];
            mu *= scale;
            double mu1 = 0, q1 = 0, max_sigma = 0;
            for (int i = 0; i < 256; i++) {
                double p_i = hist[i] * scale, q2, mu2, sigma;
                mu1 *= q1;
                q1 += p_i;
                q2 = 1. - q1;
                if (fmin(q1, q2) < FLT_EPSILON || fmax(q1, q2) > 1. - FLT_EPSILON) continue;
                mu1 = (mu1 + i * p_i) / q1;
                mu2 = (mu - q1 * mu1) / q2;
                sigma = q1 * q2 * (mu1 - mu2) * (mu1 - mu2);
                if (sigma > max_sigma) { max_sigma = sigma; thr = i; }
            }
        }
        thr = __shfl_sync(0xffffffffu, thr, 0);
        if (thr_out && lane == 0) *thr_out = thr;
        const int margin = P.cell_margin_px, inner = cs - 2 * margin;
        for (int cell = lane; cell < nb * nb; cell += 32) {
            int cy = cell / nb, cx = cell - cy * nb, nz = 0;
            for (int yy = 0; yy < inner; yy++)
                for (int xx = 0; xx < inner; xx++) nz += img[(cy * cs + margin + yy) * S + cx * cs + margin + xx] > thr;
            bits[cell] = nz > (inner * inner) / 2;
        }
    }
    __syncwarp();
    // border errors
    int e = 0;
    for (int cell = lane; cell < nb * nb; cell += 32) {
        int cy = cell / nb, cx = cell - cy * nb;
        bool border = cy < P.border_bits || cy >= nb - P.border_bits || cx < P.border_bits || cx >= nb - P.border_bits;
        e += (border && bits[cell]) ? 1 : 0;
    }
    for (int d = 16; d > 0; d >>= 1) e += __shfl_xor_sync(0xffffffffu, e, d);
    valid = false; id = -1; rot = 0;
    if (P.detect_inverted) {
        // detectInvertedMarker: a white marker is read through the inverted bits when its border fits better that way
        const int n_border = nb * nb - P.marker_size * P.marker_size;
        if (n_border - e < e) {
            for (int cell = lane; cell < nb * nb; cell += 32) bits[cell] = !bits[cell];
            e = n_border - e;
            __syncwarp();
        }
    }
    if (e > P.max_border_errors) return;
    // candidate bytes (MSB first, rows of inner bits)
    const int ms = P.marker_size, nbits = ms * ms, nbytes = P.nbytes;
    uint8_t cand[8];
    for (int b = 0; b < nbytes; b++) cand[b] = 0;
    {
        int cur_bit = 0, cur_byte = 0;
        for (int i = 0; i < nbits; i++) {
            int y = i / ms, x = i - y * ms;
            cand[cur_byte] = (uint8_t)(cand[cur_byte] << 1);
            if (bits[(y + P.border_bits) * nb + x + P.border_bits]) cand[cur_byte]++;
            if (++cur_bit == 8) { cur_bit = 0; cur_byte++; }
        }
    }
    // first marker (lowest index) whose best rotation is within the correction budget
    int best_m = 0x7fffffff, best_r = 0;
    for (int m = lane; m < P.n_markers; m += 32) {
        int bd = nbits + 1, br = -1;
        for (int r = 0; r < 4; r++) {
            int hd = 0;
            for (int b = 0; b < nbytes; b++) hd += __popc((unsigned)(dict[(m * 4 + r) * nbytes + b] ^ cand[b]));
            if (hd < bd) { bd = hd; br = r; }
        }
        if (bd <= P.max_correction && m < best_m) { best_m = m; best_r = br; }
    }
    int packed = best_m == 0x7fffffff ? 0x7fffffff : (best_m << 2) | best_r;
    for (int d = 16; d > 0; d >>= 1) packed = min(packed, __shfl_xor_sync(0xffffffffu, packed, d));
    if (packed != 0x7fffffff) { valid = true; id = packed >> 2; rot = packed & 3; }
}

// _identifyOneCandidate for every raw quad of the batch: one CTA per candidate at a time, grid = (candidate slots, frames).
// Results (valid | rot << 1 | id << 8) are indexed like the raw quads; k_decode picks them up after its sort.
#define DECB_THREADS 128
template <bool SPARSE>
__global__ void __launch_bounds__(DECB_THREADS) k_decode_bits(const uint8_t *__restrict__ gray, int w, int h, const float *__restrict__ quads,
                                                              const int32_t *__restrict__ counters, DeviceParams P,
                                                              const uint8_t *__restrict__ dict, int32_t *__restrict__ dec_raw, SparseSrc S)
{
    __shared__ uint8_t s_img[DEC_MAX_S * DEC_MAX_S];
    __shared__ int s_hist[256];
    __shared__ uint8_t s_bits[16 * 16];
    __shared__ double s_Mi[9];
    __shared__ long long s_sum[2][DECB_THREADS / 32];
    const int f = blockIdx.y, lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
    const int nq = min(counters[f * APSE_COUNTERS + 2], DEC_MAXC);
    const uint8_t *im = gray + (size_t)f * w * h;
    const int nbc = P.marker_size + 2 * P.border_bits;
    for (int i = blockIdx.x; i < nq; i += gridDim.x) {
        if (threadIdx.x == 0) {
            double Mi[9];
            inverse_homography(quads + ((size_t)f * APSE_MAX_QUADS + i) * 8, nbc * P.cell_size, Mi);
            for (int k = 0; k < 9; k++) s_Mi[k] = Mi[k];
        }
        for (int k = threadIdx.x; k < 256; k += DECB_THREADS) s_hist[k] = 0;
        __syncthreads();
        double Mi[9];
        for (int k = 0; k < 9; k++) Mi[k] = s_Mi[k];
        long long s1, s2;
        decode_sample<SPARSE>(im, w, h, Mi, P, S, f, s_img, s_hist, s1, s2);
        for (int d = 16; d > 0; d >>= 1) { s1 += __shfl_xor_sync(0xffffffffu, s1, d); s2 += __shfl_xor_sync(0xffffffffu, s2, d); }
        if (lane == 0) { s_sum[0][wid] = s1; s_sum[1][wid] = s2; }
        __syncthreads();
        if (wid == 0) {
            s1 = 0; s2 = 0;
            for (int k = 0; k < DECB_THREADS / 32; k++) { s1 += s_sum[0][k]; s2 += s_sum[1][k]; }
            bool v; int id, rot;
            decode_finish(P, s1, s2, dict, s_img, s_hist, s_bits, v, id, rot);
            if (lane == 0) dec_raw[(size_t)f * APSE_MAX_QUADS + i] = (v ? 1 : 0) | (rot << 1) | (id << 8);
        }
        __syncthreads();
    }
}

// test tap (a6.A6 / a6.A7 in isolation): one candidate -> canonical image, Otsu threshold, cell bits, identification
__global__ void __launch_bounds__(DECB_THREADS) k_decode_tap(const uint8_t *__restrict__ gray, int w, int h, const float *__restrict__ corners, int n,
                                                             DeviceParams P, const uint8_t *__restrict__ dict, uint8_t *__restrict__ img_out,
                                                             uint8_t *__restrict__ bits_out, int32_t *__restrict__ res_out)
{
    __shared__ uint8_t s_img[DEC_MAX_S * DEC_MAX_S];
    __shared__ int s_hist[256];
    __shared__ uint8_t s_bits[16 * 16];
    __shared__ double s_Mi[9];
    __shared__ long long s_sum[2][DECB_THREADS / 32];
    __shared__ int s_thr;
    const int i = blockIdx.x, lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
    if (i >= n) return;
    const int nbc = P.marker_size + 2 * P.border_bits, S = nbc * P.cell_size;
    if (threadIdx.x == 0) {
        double Mi[9];
        inverse_homography(corners + 8 * i, S, Mi);
        for (int k = 0; k < 9; k++) s_Mi[k] = Mi[k];
        s_thr = -2;
    }
    for (int k = threadIdx.x; k < 256; k += DECB_THREADS) s_hist[k] = 0;
    __syncthreads();
    double Mi[9];
    for (int k = 0; k < 9; k++) Mi[k] = s_Mi[k];
    long long s1, s2;
    decode_sample<false>(gray, w, h, Mi, P, SparseSrc{}, 0, s_img, s_hist, s1, s2);
    for (int d = 16; d > 0; d >>= 1) { s1 += __shfl_xor_sync(0xffffffffu, s1, d); s2 += __shfl_xor_sync(0xffffffffu, s2, d); }
    if (lane == 0) { s_sum[0][wid] = s1; s_sum[1][wid] = s2; }
    __syncthreads();
    if (wid == 0) {
        s1 = 0; s2 = 0;
        for (int k = 0; k < DECB_THREADS / 32; k++) { s1 += s_sum[0][k]; s2 += s_sum[1][k]; }
        bool v; int id, rot;
        decode_finish(P, s1, s2, dict, s_img, s_hist, s_bits, v, id, rot, &s_thr);
        __syncwarp();
        if (lane == 0) { res_out[4 * i] = v ? 1 : 0; res_out[4 * i + 1] = id; res_out[4 * i + 2] = rot; res_out[4 * i + 3] = s_thr; }
    }
    __syncthreads();
    for (int k = threadIdx.x; k < S * S; k += DECB_THREADS) img_out[(size_t)i * DEC_MAX_S * DEC_MAX_S + k] = s_img[k];
    for (int k = threadIdx.x; k < nbc * nbc; k += DECB_THREADS) bits_out[(size_t)i * 256 + k] = s_bits[k];
}

int apse_decode_tap(apse_ctx *ctx, const uint8_t *gray, int w, int h, const float *corners, int n, const DeviceParams &dp, uint8_t *img_out,
                    uint8_t *bits_out, int32_t *res_out, cudaStream_t st)
{
    int nb = dp.marker_size + 2 * dp.border_bits;
    if (nb * dp.cell_size > DEC_MAX_S || nb > 16 || dp.nbytes > 8) CTX_FAIL(ctx, APSE_ERR_UNSUPPORTED, "decode tap: canonical marker image too large");
    KLAUNCH(ctx, KID_DECODE_BITS, st, k_decode_tap<<<n, DECB_THREADS, 0, st>>>(gray, w, h, corners, n, dp, ctx->dict, img_out, bits_out, res_out));
    return APSE_OK;
}

// exclusive prefix sum of one int per thread over the CTA; s_scan[DEC_WARPS] = total.  s_scan is reusable after the call's barriers.
__device__ __forceinline__ int block_exclusive_scan(int v, int *s_scan)
{
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    int inc = v;
#pragma unroll
    for (int d = 1; d < 32; d <<= 1) { int t = __shfl_up_sync(0xffffffffu, inc, d); if (lane >= d) inc += t; }
    __syncthreads();   // previous readers of s_scan are done
    if (lane == 31) s_scan[warp] = inc;
    __syncthreads();
    if (warp == 0) {
        int w = lane < DEC_WARPS ? s_scan[lane] : 0, winc = w;
#pragma unroll
        for (int d = 1; d < 32; d <<= 1) { int t = __shfl_up_sync(0xffffffffu, winc, d); if (lane >= d) winc += t; }
        if (lane < DEC_WARPS) s_scan[lane] = winc - w;
        if (lane == 31) s_scan[DEC_WARPS] = winc;
    }
    __syncthreads();
    return s_scan[warp] + inc - v;
}

__global__ void __launch_bounds__(DEC_THREADS) k_decode(const uint8_t *__restrict__ gray, int w, int h, const float *__restrict__ quads,
                                                        const uint32_t *__restrict__ quad_order, int32_t *__restrict__ counters,
                                                        DeviceParams P, const int32_t *__restrict__ dec_raw,
                                                        unsigned char *__restrict__ big_scratch, size_t big_stride, int mid_tier, apse_detections out)
{
    extern __shared__ __align__(16) unsigned char smem_raw[];
    DecodeSmem &S = *reinterpret_cast<DecodeSmem *>(smem_raw);
    __shared__ DecodeArrays A;
#ifdef APSE_DEC_PROFILE
    __shared__ long long dbg_t[24];
    DEC_T(0);
#endif
    const int f = blockIdx.x, tid = threadIdx.x;
    int32_t *cnt = counters + f * APSE_COUNTERS;
    const int nq = min(cnt[2], DEC_MAXC);
    const float *q = quads + (size_t)f * APSE_MAX_QUADS * 8;
    const uint32_t *qo = quad_order + (size_t)f * APSE_MAX_QUADS;
    if (nq > DEC_SMEMC && !big_scratch) {   // apse_detect_impl always passes the scratch; without it such a frame is reported, not cut
        if (tid == 0) { out.n_markers[f] = 0; if (out.n_rejected) out.n_rejected[f] = 0; out.status[f] = APSE_ERR_CAPACITY; }
        return;
    }
    if (tid == 0) {
        // three tiers: everything in shared memory; the sequentially walked arrays in shared memory and the O(n^2) bit matrix in
        // global memory (the classic path's ~10^3 candidates per frame: its single-thread grouping walk is a chain of dependent
        // loads); everything in global memory
        if (nq <= DEC_SMEMC) decode_arrays_carve(A, smem_raw + sizeof(DecodeSmem), DEC_SMEMC);
        else if (nq <= DEC_MIDC && mid_tier) decode_arrays_carve(A, smem_raw + sizeof(DecodeSmem), DEC_MIDC, reinterpret_cast<uint32_t *>(big_scratch + (size_t)f * big_stride));
        else if (mid_tier) decode_arrays_carve_top(A, smem_raw + sizeof(DecodeSmem), big_scratch + (size_t)f * big_stride, DEC_MAXC);
        else decode_arrays_carve(A, big_scratch + (size_t)f * big_stride, DEC_MAXC);
    }
    __syncthreads();
    DEC_T(1);

    // ---- candidates sorted by perimeter (descending), ties in the deterministic candidate order (key).  n = nq: the
    // border-distance test comes AFTER the grouping (4.13: a border-touching quad still groups and, as a group main, takes its
    // group with it).  One rank pass over (perimeter, key), then one scatter straight from the quad list.
    const int n = nq;
    const int32_t *dr = dec_raw + (size_t)f * APSE_MAX_QUADS;
    float *perim0 = A.cxy;   // perimeters in quad-list order (the centroids are computed after the scatter)
    for (int i = tid; i < n; i += DEC_THREADS) { A.key[i] = qo[i]; perim0[i] = perimeter_of(q + 8 * i); }
    __syncthreads();
    DEC_T(2);
    for (int i = tid; i < n; i += DEC_THREADS) {
        const float p = perim0[i];
        const uint32_t k = A.key[i];
        int r = 0, j = 0;
        for (; j + 4 <= n; j += 4) {
            const float4 pj = *reinterpret_cast<const float4 *>(perim0 + j);
            const uint4 kj = *reinterpret_cast<const uint4 *>(A.key + j);
            r += (pj.x > p) || (pj.x == p && kj.x < k);
            r += (pj.y > p) || (pj.y == p && kj.y < k);
            r += (pj.z > p) || (pj.z == p && kj.z < k);
            r += (pj.w > p) || (pj.w == p && kj.w < k);
        }
        for (; j < n; j++) r += (perim0[j] > p) || (perim0[j] == p && A.key[j] < k);
        A.sel_of[i] = (short)r;
    }
    __syncthreads();
    DEC_T(3);
    for (int i = tid; i < n; i += DEC_THREADS) {
        const int r = A.sel_of[i];
        for (int k = 0; k < 8; k++) A.c[r][k] = q[8 * i + k];
        A.perim[r] = perim0[i];
        const int flags = dr[i] & 0xff;   // result of k_decode_bits for this quad
        A.dec_valid[r] = (uint8_t)(flags & 1); A.dec_rot[r] = (uint8_t)((flags >> 1) & 3); A.dec_id[r] = (short)(dr[i] >> 8);
    }
    __syncthreads();
    DEC_T(4);

    // ---- too-close predicate, avgDist(i,j) < perimeter[j] * rate for i < j, and the grouping it drives.
    // The dependency walks the close pairs in row-major order: both ungrouped -> new group; one grouped -> the other joins; both
    // grouped -> nothing.  A candidate is therefore assigned at the FIRST pair (in that order) it takes part in -- it is still
    // ungrouped there, and either its partner already has a group (it joins) or the partner is ungrouped too, which makes this the
    // partner's first pair as well (a new group).  The first pair of v is (i_min, v) with the smallest close i < v if there is one
    // (rows before row v), else (v, j_min).  So: first partner per candidate by atomicMin while the predicate is evaluated (no bit
    // matrix, no pair list, no sequential walk); groups = chains of first partners, ending in a mutual pair whose smaller index --
    // the smallest index of the whole group, the group's head -- labels the group.
    // avgDist^2 is a mean of squared corner distances, so it is never below the squared centroid distance (Jensen):
    // pairs whose centroids are clearly farther apart than the threshold are skipped without the 4-shift evaluation.
    const int lane = tid & 31, warp = tid >> 5;
    // centroid test operands, one array each (unit-stride reads), padded so that a row's last 128 columns need no bounds test
    const int sstride = A.cap + 128;
    float *thr2 = reinterpret_cast<float *>(A.close_bits), *cxs = thr2 + sstride, *cys = cxs + sstride;
    int *list_head = reinterpret_cast<int *>(A.cxy);   // per group (indexed by its head): unordered member list
    for (int i = tid; i < n + 128; i += DEC_THREADS) {
        if (i < n) {
            const float *c = A.c[i];
            cxs[i] = 0.25f * (c[0] + c[2] + c[4] + c[6]);
            cys[i] = 0.25f * (c[1] + c[3] + c[5] + c[7]);
            const float thr = A.perim[i] * P.min_marker_distance_rate;
            thr2[i] = thr * thr * 1.02f + 4.f;   // conservative: float rounding of the centroids
            A.key[i] = 0xffffffffu;   // first partner: u < v as u, u > v as 0x10000 + u (any smaller index wins over any larger one)
            list_head[i] = -1;
        } else { cxs[i] = 0.f; cys[i] = 0.f; thr2[i] = -1.f; }
    }
    if (tid == 0) S.n = 0;
    __syncthreads();
    DEC_T(5);
    // pass 1, warp per row i, lane = column: the pairs the centroid test cannot exclude go to a list (a few per candidate)
    const int pair_cap = A.cap * 8;
    for (int i = warp; i < n; i += DEC_WARPS) {
        const float cxi = cxs[i], cyi = cys[i];
        for (int jb = i & ~31; jb < n; jb += 128) {
            uint32_t m[4];
            bool cand[4];
#pragma unroll
            for (int u = 0; u < 4; u++) {
                const int j = jb + 32 * u + lane;
                const float dx = cxs[j] - cxi, dy = cys[j] - cyi;
                cand[u] = j > i && !(dx * dx + dy * dy > thr2[j]);
            }
#pragma unroll
            for (int u = 0; u < 4; u++) m[u] = __ballot_sync(0xffffffffu, cand[u]);
            if (m[0] | m[1] | m[2] | m[3]) {
                const int total = __popc(m[0]) + __popc(m[1]) + __popc(m[2]) + __popc(m[3]);
                int base = 0;
                if (lane == 0) base = atomicAdd(&S.n, total);
                base = __shfl_sync(0xffffffffu, base, 0);
#pragma unroll
                for (int u = 0; u < 4; u++) {
                    const int o = base + __popc(m[u] & ((1u << lane) - 1));
                    if (cand[u] && o < pair_cap) A.pairs[o] = ((uint32_t)i << 16) | (uint32_t)(jb + 32 * u + lane);
                    base += __popc(m[u]);
                }
            }
        }
    }
    __syncthreads();
    DEC_T(6);
    // pass 2, thread per listed pair: the exact predicate
    {
        const int np = S.n;
        if (np > pair_cap && tid == 0) cnt[3] = APSE_ERR_CAPACITY;   // reported through status; never truncated silently
        for (int k = tid; k < min(np, pair_cap); k += DEC_THREADS) {
            const uint32_t pr = A.pairs[k];
            const int i = pr >> 16, j = pr & 0xffff;
            if (average_distance(A.c[i], A.c[j]) < A.perim[j] * P.min_marker_distance_rate) {
                atomicMin(&A.key[j], (uint32_t)i);
                atomicMin(&A.key[i], 0x10000u + (uint32_t)j);
            }
        }
    }
    __syncthreads();
    DEC_T(7);
    for (int v = tid; v < n; v += DEC_THREADS) {
        const uint32_t k = A.key[v];
        int label = -1;
        if (k != 0xffffffffu) {
            int r = v, q1 = (int)(k & 0xffffu);
            for (int it = 0; it < n; it++) {   // the first-pair order strictly decreases along the chain
                const int q2 = (int)(A.key[q1] & 0xffffu);
                if (q2 == r) { label = min(r, q1); break; }
                r = q1; q1 = q2;
            }
        }
        A.group_id[v] = (short)label; A.selected[v] = label < 0;   // (a group's main is selected by its head thread below)
        A.close_next[v] = -1; A.parent[v] = -1; A.valid[v] = 0; A.use_c[v] = (short)v;
        A.next_in_group[v] = label >= 0 && label != v ? (short)atomicExch(&list_head[label], v) : (short)-1;
    }
    __syncthreads();
    DEC_T(8);
    // thread per group (its label = smallest index): the members in ascending index order (= largest perimeter first; with
    // detectInvertedMarker descending: the dependency then makes the SMALLEST candidate the group's main), the next one picked from
    // the unordered list each time -- groups are a handful of candidates; kept: the chain of members far enough from the previous one
    const bool desc = P.detect_inverted != 0;
    for (int g = tid; g < n; g += DEC_THREADS) {
        if (A.group_id[g] != g) continue;
        int head = g;
        if (desc) for (int m = list_head[g]; m >= 0; m = A.next_in_group[m]) head = max(head, m);
        A.selected[head] = 1;
        int cur = head, tail_close = -1, last = head;
        for (;;) {
            int id = desc ? -1 : 0x7fffffff;
            for (int m = list_head[g]; m >= 0; m = A.next_in_group[m]) if (desc ? (m < last && m > id) : (m > last && m < id)) id = m;
            if (desc && id < 0 && g < last) id = g;   // the label itself is the group's smallest index: last in descending order
            if (id < 0 || id == 0x7fffffff) break;
            last = id;
            float dist = average_distance(A.c[id], A.c[cur]);
            float msz = average_module_size(A.c[id], P.marker_size, P.border_bits);
            if (dist > P.min_group_distance * msz) {
                cur = id;
                if (tail_close < 0) A.close_next[head] = (short)id; else A.close_next[tail_close] = (short)id;
                tail_close = id;
            }
        }
    }
    __syncthreads();   // selected[] of the group mains
    DEC_T(9);
    // NB close_next chains start at the group's head; members never head a chain themselves.
    // Border-distance test on the selected (main) candidates only: a main too near the edge is dropped with its group.
    __shared__ int s_scan[DEC_WARPS + 1];
    const int chunk = (n + DEC_THREADS - 1) / DEC_THREADS, r0 = min(n, tid * chunk), r1 = min(n, r0 + chunk);
    {
        const float d = (float)P.min_distance_to_border;
        uint32_t keep = 0;
        for (int i = r0; i < r1; i++) {
            if (!A.selected[i]) continue;
            const float *c = A.c[i];
            bool near = false;
            for (int j = 0; j < 4; j++) near |= c[2 * j] < d || c[2 * j + 1] < d || c[2 * j] > w - 1 - d || c[2 * j + 1] > h - 1 - d;
            if (!near) keep |= 1u << (i - r0);
        }
        int off = block_exclusive_scan(__popc(keep), s_scan);
        for (int i = r0; i < r1; i++)
            if (keep >> (i - r0) & 1) { A.sel[off] = (short)i; A.sel_of[i] = (short)off; off++; }
        if (tid == 0) S.ns = s_scan[DEC_WARPS];
    }
    __syncthreads();
    DEC_T(10);
    const int ns = S.ns;

    // ---- nesting hierarchy among the selected candidates: parent = nearest smaller index that contains all 4 corners
    // (a point strictly inside a quad lies inside the quad's bounding box: the box test rejects almost every pair before the four
    // exact point-in-polygon tests; with ~10^3 candidates per frame on the classic path the plain O(n^2) loop was 0.8 ms per frame)
    float4 *box = reinterpret_cast<float4 *>(A.close_bits);   // bounding boxes (x0, x1, y0, y1) of the selected candidates
    for (int v = tid; v < ns; v += DEC_THREADS) {
        const float *a = A.c[A.sel[v]];
        box[v] = make_float4(fminf(fminf(a[0], a[2]), fminf(a[4], a[6])), fmaxf(fmaxf(a[0], a[2]), fmaxf(a[4], a[6])),
                             fminf(fminf(a[1], a[3]), fminf(a[5], a[7])), fmaxf(fmaxf(a[1], a[3]), fmaxf(a[5], a[7])));
    }
    __syncthreads();
    for (int v = tid; v < ns; v += DEC_THREADS) {
        const float *a = A.c[A.sel[v]];
        const float4 ba = box[v];
        int par = -1;
        for (int j = v - 1; j >= 0; j--) {
            const float4 bb = box[j];
            if (ba.x < bb.x || ba.y > bb.y || ba.z < bb.z || ba.w > bb.w) continue;
            const float *b = A.c[A.sel[j]];
            if (strictly_inside(b, a[0], a[1]) && strictly_inside(b, a[2], a[3]) && strictly_inside(b, a[4], a[5]) &&
                strictly_inside(b, a[6], a[7])) { par = j; break; }
        }
        A.parent[v] = (short)par;
    }
    // height of every node of the nesting forest (the dependency's "depth": longest chain of nested candidates below it) and the
    // "seen" marks of the acceptance loop, in the centroid scratch (no longer needed)
    DEC_T(11);
    int *hgt = reinterpret_cast<int *>(A.cxy);   // [2 v] height, [2 v + 1] seen
    __shared__ int s_lvl[2];                      // [0] number of candidates accounted for, [1] largest height
    for (int v = tid; v < ns; v += DEC_THREADS) { hgt[2 * v] = 0; hgt[2 * v + 1] = 0; }
    if (tid == 0) { s_lvl[0] = 0; s_lvl[1] = 0; }
    __syncthreads();
    for (int v = tid; v < ns; v += DEC_THREADS) {
        // a node that finds an ancestor already as high as it would make it stops: whoever raised that ancestor carries on upwards
        // (a frame-sized outer candidate is an ancestor of everything: without the test every thread would hit its counter)
        int k = 0;
        for (int p = A.parent[v]; p >= 0; p = A.parent[p]) {
            ++k;
            if (*reinterpret_cast<volatile int *>(&hgt[2 * p]) >= k) break;
            atomicMax(&hgt[2 * p], k);
            if (*reinterpret_cast<volatile int *>(&s_lvl[1]) < k) atomicMax(&s_lvl[1], k);
        }
    }
    __syncthreads();
    DEC_T(12);
    // Acceptance, level by level from the innermost candidates outwards, as the dependency does it: a level's candidates are tried
    // (the group's main first, then its far-enough members); every accepted one marks its not yet seen ancestors, and each mark
    // counts as a processed candidate -- as does, again, the ancestor itself when its own level comes.  The loop ends when the count
    // reaches the number of candidates, so outer candidates of a frame with nested markers may never be tried (and end up rejected).
    // Ancestors are strictly higher than their descendants, so the candidates of one level are independent of each other.
    const int max_depth = s_lvl[1];
    for (int dep = 0; dep <= max_depth; dep++) {
        if (s_lvl[0] >= ns) break;
        __syncthreads();
        int mine = 0;
        for (int v = tid; v < ns; v += DEC_THREADS) {
            if (hgt[2 * v] != dep) continue;
            mine++;
            const int head = A.sel[v];
            int use = -1;
            if (A.dec_valid[head]) use = head;
            else
                for (int c = A.close_next[head]; c >= 0; c = A.close_next[c])
                    if (A.dec_valid[c]) { use = c; break; }
            if (use < 0) continue;
            A.valid[v] = 1; A.use_c[v] = (short)use;
            for (int p = A.parent[v]; p >= 0; p = A.parent[p])
                if (atomicExch(&hgt[2 * p + 1], 1) == 0) mine++;
        }
        if (mine) atomicAdd(&s_lvl[0], mine);
        __syncthreads();
    }
    __syncthreads();
    DEC_T(13);

    // ---- output: accepted markers (corners rotated to the dictionary's orientation) and rejected candidates, in candidate order
    {
        const int cap = out.max_markers;
        float *oc = out.corners + (size_t)f * cap * 8;
        int32_t *oi = out.ids + (size_t)f * cap;
        float *orj = out.rejected ? out.rejected + (size_t)f * cap * 8 : nullptr;
        const int ochunk = (ns + DEC_THREADS - 1) / DEC_THREADS, v0 = min(ns, tid * ochunk), v1 = min(ns, v0 + ochunk);
        int nv = 0;
        for (int v = v0; v < v1; v++) nv += A.valid[v];
        int na = block_exclusive_scan(nv, s_scan);
        const int na_total = s_scan[DEC_WARPS];
        int nr = v0 - na;
        for (int v = v0; v < v1; v++) {
            if (A.valid[v]) {
                const int u = A.use_c[v];
                const float *c = A.c[u];
                if (na < cap) {
                    const int r = A.dec_rot[u];
                    for (int k = 0; k < 4; k++) {
                        const int s = (k + 4 - r) % 4;
                        oc[8 * na + 2 * k] = c[2 * s];
                        oc[8 * na + 2 * k + 1] = c[2 * s + 1];
                    }
                    oi[na] = A.dec_id[u];
                }
                na++;
            } else {
                const float *c = A.c[A.sel[v]];
                if (orj && nr < cap) for (int k = 0; k < 8; k++) orj[8 * nr + k] = c[k];
                nr++;
            }
        }
        if (tid == 0) {
            const int nr_total = ns - na_total;
            int status = cnt[3];
            if (na_total > cap || (orj && nr_total > cap)) status = APSE_ERR_CAPACITY;
            out.n_markers[f] = min(na_total, cap);
            if (out.n_rejected) out.n_rejected[f] = min(nr_total, cap);
            out.status[f] = status;
#ifdef APSE_DEC_PROFILE
            if (blockIdx.x == 0) {
                const long long t_end = clock64();
                const char *names[14] = {"carve", "perimeters", "rank", "scatter", "centroids", "pairs: centroid test", "pairs: exact", "labels", "groups", "border + scan", "nesting", "heights", "levels", "output"};
                for (int i = 1; i <= 13; i++) printf("%-22s %8lld cycles\n", names[i - 1], dbg_t[i] - dbg_t[i - 1]);
                printf("%-22s %8lld cycles; nq %d ns %d listed pairs %d\n", names[13], t_end - dbg_t[13], nq, ns, S.n);
            }
#endif
        }
    }
}

int apse_decode_alloc(apse_ctx *ctx)
{
    CUDA_TRY(ctx, cudaFuncSetAttribute(k_decode, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                       (int)(sizeof(DecodeSmem) + decode_arrays_small_bytes(DEC_MIDC))));
    return APSE_OK;
}
void apse_decode_free(apse_ctx *ctx) { cudaFree(ctx->decode_scratch); ctx->decode_scratch = nullptr; }

// global candidate arrays for frames with more than DEC_SMEMC quads (either candidate path); allocated on first use
int apse_decode_big_scratch(apse_ctx *ctx)
{
    if (!ctx->decode_scratch) CUDA_TRY(ctx, cudaMalloc(&ctx->decode_scratch, decode_arrays_bytes(DEC_MAXC) * ctx->max_batch));
    return APSE_OK;
}

int apse_decode_candidates(apse_ctx *ctx, const uint8_t *gray, int w, int h, int batch, const DeviceParams &dp,
                           apse_detections *out, cudaStream_t st)
{
    if (!out || !out->corners || !out->ids || !out->n_markers || !out->status || out->max_markers <= 0)
        CTX_FAIL(ctx, APSE_ERR_INVALID_ARG, "detect: incomplete apse_detections");
    if (out->rejected && !out->n_rejected) CTX_FAIL(ctx, APSE_ERR_INVALID_ARG, "detect: rejected without n_rejected");
    int nb = dp.marker_size + 2 * dp.border_bits;
    if (nb * dp.cell_size > DEC_MAX_S || nb > 16 || dp.nbytes > 8)
        CTX_FAIL(ctx, APSE_ERR_UNSUPPORTED, "detect: canonical marker image %d px exceeds the %d px limit", nb * dp.cell_size, DEC_MAX_S);
    // a quad that encloses an already decoded marker IS identified (cv2 4.13 on nested-marker frames, tests/test_gpu_detect.py)
    // hierarchy scratch of the quad fit is free at this point: [batch][APSE_MAX_QUADS] decode results
    int32_t *dec_raw = reinterpret_cast<int32_t *>(ctx->errs);
    const int cand_blocks = ctx->params.cornerRefinementMethod == 3 ? 64 : 512;   // CTAs per frame; a CTA without a candidate exits at once
    if (ctx->sparse_active)
        KLAUNCH(ctx, KID_DECODE_BITS, st, k_decode_bits<true><<<dim3(cand_blocks, batch), DECB_THREADS, 0, st>>>(gray, w, h, ctx->quads, ctx->counters, dp, ctx->dict, dec_raw, ctx->sparse_src));
    else
        KLAUNCH(ctx, KID_DECODE_BITS, st, k_decode_bits<false><<<dim3(cand_blocks, batch), DECB_THREADS, 0, st>>>(gray, w, h, ctx->quads, ctx->counters, dp, ctx->dict, dec_raw, SparseSrc{}));
    // the classic path (hundreds of candidates per frame) launches with the shared memory of the middle tier; the APRILTAG path keeps
    // the small footprint (its decode CTAs share SMs with the preprocess kernels of the next sub-batch)
    const int mid_tier = ctx->params.cornerRefinementMethod != 3 && ctx->decode_scratch ? 1 : 0;
    const size_t dec_smem = sizeof(DecodeSmem) + (mid_tier ? decode_arrays_small_bytes(DEC_MIDC) : decode_arrays_bytes(DEC_SMEMC));
    KLAUNCH(ctx, KID_DECODE, st, k_decode<<<batch, DEC_THREADS, dec_smem, st>>>(
                gray, w, h, ctx->quads, ctx->quad_order, ctx->counters, dp, dec_raw,
                (unsigned char *)ctx->decode_scratch, decode_arrays_bytes(DEC_MAXC), mid_tier, *out));
    return APSE_OK;
}
