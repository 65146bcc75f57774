// ORB front-end on the GPU: cv2.ORB_create().detectAndCompute with the reference's (default) parameters
// (feature_extractors/ORB.py:8 `orb = cv2.ORB_create()`, :10-21 extract_features_and_desc) — 500 features, scale
// 1.2f, 8 levels, edge 31, patch 31, FAST threshold 20, Harris score.  SURVEY 8(f) rank 1.
//
// STATUS: bit-identical to the CPU restatement pinned against OpenCV — on the host emulation of tests/cuda_emu.h
// (tests/test_orb_emulation.py) and on a B200 (tests/test_gpu_orb_frontend.py, tools/orb_bisect.py stage by stage).  Default
// extractor of feature_extractors/ORB.py and of DeviceLoop.push_image for byte-descriptor loops.
//
// Data layout: one unbordered 8-bit image per pyramid level, back to back in one buffer (keypoints stay >= 31 pixels
// from the border, so orientation / Harris / rBRIEF never leave a level; the Gaussian reflects indices).  Per level:
// a FAST score map (u8), a candidate list (FAST + 3x3 strict maximum + border filter), the survivors of
// retainBest(2 n) on the integer score (256-bin histogram), their Harris responses, the survivors of retainBest(n) on
// the response (4-pass radix select on the ordered float bits; ties kept, as OpenCV does), ranked by (y, x) so that the
// output order is deterministic: level-major, then row-major (OpenCV's own order depends on std::nth_element).
// Everything is HBM-bound integer / byte work: ~1.1 M pixels per 1241 x 376 frame over the 8 levels; the per-pixel
// kernels cover all levels in one launch each (17 launches per BGR frame, 7 of them the resize cascade).
//
// Batch (vo_orb_extract_batch): every kernel also runs over S images, the image index being the last grid dimension, so
// a call is 17 launches (BGR) whatever S is; vo_orb_extract is the S = 1 call.  Per-pixel buffers are level-major with
// the S images of a level back to back (image s of level l at img_ofs + s * w * h): level 0 of the batch is then one
// contiguous block and a gray batch arrives with one copy.  Keypoint lists, kept lists, angles and the 32-entry count
// block are image-major.  Image s's output rows are a prefix (level-major, then row-major) of what it alone would give.
//
// The rBRIEF point pairs below are OpenCV's learned pattern (modules/features2d/src/orb.cpp, bit_pattern_31_,
// Apache-2.0): data of the third-party library whose arithmetic the reference's plug-in runs.
#include "common.cuh"
#include "orb_math.cuh"
#include <math.h>
#include <vector>

namespace vo {
namespace {

__device__ const int8_t ORB_PATTERN[1024] = {
    8, -3, 9, 5, 4, 2, 7, -12, -11, 9, -8, 2, 7, -12, 12, -13, 2, -13, 2, 12, 1, -7, 1, 6, -2, -10, -2, -4, -13, -13, -11, -8,
    -13, -3, -12, -9, 10, 4, 11, 9, -13, -8, -8, -9, -11, 7, -9, 12, 7, 7, 12, 6, -4, -5, -3, 0, -13, 2, -12, -3, -9, 0, -7, 5,
    12, -6, 12, -1, -3, 6, -2, 12, -6, -13, -4, -8, 11, -13, 12, -8, 4, 7, 5, 1, 5, -3, 10, -3, 3, -7, 6, 12, -8, -7, -6, -2,
    -2, 11, -1, -10, -13, 12, -8, 10, -7, 3, -5, -3, -4, 2, -3, 7, -10, -12, -6, 11, 5, -12, 6, -7, 5, -6, 7, -1, 1, 0, 4, -5,
    9, 11, 11, -13, 4, 7, 4, 12, 2, -1, 4, 4, -4, -12, -2, 7, -8, -5, -7, -10, 4, 11, 9, 12, 0, -8, 1, -13, -13, -2, -8, 2,
    -3, -2, -2, 3, -6, 9, -4, -9, 8, 12, 10, 7, 0, 9, 1, 3, 7, -5, 11, -10, -13, -6, -11, 0, 10, 7, 12, 1, -6, -3, -6, 12,
    10, -9, 12, -4, -13, 8, -8, -12, -13, 0, -8, -4, 3, 3, 7, 8, 5, 7, 10, -7, -1, 7, 1, -12, 3, -10, 5, 6, 2, -4, 3, -10,
    -13, 0, -13, 5, -13, -7, -12, 12, -13, 3, -11, 8, -7, 12, -4, 7, 6, -10, 12, 8, -9, -1, -7, -6, -2, -5, 0, 12, -12, 5, -7, 5,
    3, -10, 8, -13, -7, -7, -4, 5, -3, -2, -1, -7, 2, 9, 5, -11, -11, -13, -5, -13, -1, 6, 0, -1, 5, -3, 5, 2, -4, -13, -4, 12,
    -9, -6, -9, 6, -12, -10, -8, -4, 10, 2, 12, -3, 7, 12, 12, 12, -7, -13, -6, 5, -4, 9, -3, 4, 7, -1, 12, 2, -7, 6, -5, 1,
    -13, 11, -12, 5, -3, 7, -2, -6, 7, -8, 12, -7, -13, -7, -11, -12, 1, -3, 12, 12, 2, -6, 3, 0, -4, 3, -2, -13, -1, -13, 1, 9,
    7, 1, 8, -6, 1, -1, 3, 12, 9, 1, 12, 6, -1, -9, -1, 3, -13, -13, -10, 5, 7, 7, 10, 12, 12, -5, 12, 9, 6, 3, 7, 11,
    5, -13, 6, 10, 2, -12, 2, 3, 3, 8, 4, -6, 2, 6, 12, -13, 9, -12, 10, 3, -8, 4, -7, 9, -11, 12, -4, -6, 1, 12, 2, -8,
    6, -9, 7, -4, 2, 3, 3, -2, 6, 3, 11, 0, 3, -3, 8, -8, 7, 8, 9, 3, -11, -5, -6, -4, -10, 11, -5, 10, -5, -8, -3, 12,
    -10, 5, -9, 0, 8, -1, 12, -6, 4, -6, 6, -11, -10, 12, -8, 7, 4, -2, 6, 7, -2, 0, -2, 12, -5, -8, -5, 2, 7, -6, 10, 12,
    -9, -13, -8, -8, -5, -13, -5, -2, 8, -8, 9, -13, -9, -11, -9, 0, 1, -8, 1, -2, 7, -4, 9, 1, -2, 1, -1, -4, 11, -6, 12, -11,
    -12, -9, -6, 4, 3, 7, 7, 12, 5, 5, 10, 8, 0, -4, 2, 8, -9, 12, -5, -13, 0, 7, 2, 12, -1, 2, 1, 7, 5, 11, 7, -9,
    3, 5, 6, -8, -13, -4, -8, 9, -5, 9, -3, -3, -4, -7, -3, -12, 6, 5, 8, 0, -7, 6, -6, 12, -13, 6, -5, -2, 1, -10, 3, 10,
    4, 1, 8, -4, -2, -2, 2, -13, 2, -12, 12, 12, -2, -13, 0, -6, 4, 1, 9, 3, -6, -10, -3, -5, -3, -13, -1, 1, 7, 5, 12, -11,
    4, -2, 5, -7, -13, 9, -9, -5, 7, 1, 8, 6, 7, -8, 7, 6, -7, -4, -7, 1, -8, 11, -7, -8, -13, 6, -12, -8, 2, 4, 3, 9,
    10, -5, 12, 3, -6, -5, -6, 7, 8, -3, 9, -8, 2, -12, 2, 8, -11, -2, -10, 3, -12, -13, -7, -9, -11, 0, -10, -5, 5, -3, 11, 8,
    -2, -13, -1, 12, -1, -8, 0, 9, -13, -11, -12, -5, -10, -2, -10, 11, -3, 9, -2, -13, 2, -3, 3, 2, -9, -13, -4, 0, -4, 6, -3, -10,
    -4, 12, -2, -7, -6, -11, -4, 9, 6, -3, 6, 11, -13, 11, -5, 5, 11, 11, 12, 6, 7, -5, 12, -2, -1, 12, 0, 7, -4, -8, -3, -2,
    -7, 1, -6, 7, -13, -12, -8, -13, -7, -2, -6, -8, -8, 5, -6, -9, -5, -1, -4, 5, -13, 7, -8, 10, 1, 5, 5, -13, 1, 0, 10, -13,
    9, 12, 10, -1, 5, -8, 10, -9, -1, 11, 1, -13, -9, -3, -6, 2, -1, -10, 1, 12, -13, 1, -8, -10, 8, -11, 10, -6, 2, -13, 3, -6,
    7, -13, 12, -9, -10, -10, -5, -7, -10, -8, -8, -13, 4, -6, 8, 5, 3, 12, 8, -13, -4, 2, -3, -3, 5, -13, 10, -12, 4, -13, 5, -1,
    -9, 9, -4, 3, 0, 3, 3, -9, -12, 1, -6, 1, 3, 2, 4, -8, -10, -10, -10, 9, 8, -13, 12, 12, -8, -12, -6, -5, 2, 2, 3, 7,
    10, 6, 11, -8, 6, 8, 8, -12, -7, 10, -6, 5, -3, -9, -3, 9, -1, -13, -1, 5, -3, -7, -3, 4, -8, -2, -8, 3, 4, 2, 12, 12,
    2, -5, 3, 11, 6, -9, 11, -13, 3, -1, 7, 12, 11, -1, 12, 4, -3, 0, -3, 6, 4, -11, 4, 12, 2, -4, 2, 1, -10, -6, -8, 1,
    -13, 7, -11, 1, -13, 12, -11, -13, 6, 0, 11, -13, 0, -1, 1, 4, -13, 3, -9, -2, -9, 8, -6, -3, -13, -6, -8, -2, 5, -9, 8, 10,
    2, 7, 3, -9, -1, -6, -1, -1, 9, 5, 11, -2, 11, -3, 12, -8, 3, 0, 3, 5, -1, 4, 0, 10, 3, -6, 4, 5, -13, 0, -10, 5,
    5, 8, 12, 11, 8, 9, 9, -6, 7, -4, 8, -12, -10, 4, -10, 9, 7, 3, 12, 4, 9, -7, 10, -2, 7, 0, 12, -2, -1, -6, 0, -11,
};

constexpr int ORB_MAX_LEVELS = 8;
constexpr int ORB_EDGE = 31;
constexpr int ORB_FINAL_CAP = 4096;   // keypoints kept per level (n_l + ties); more -> overflow flag

struct OrbLevel {
    int w, h;
    int n_feat;          // retainBest target of this level
    int cand_cap;        // w * h / 4 + 1: a strict 3x3 maximum cannot be denser
    float scale;
    size_t img_ofs;      // bytes into the pyramid / blurred / score buffers of image 0 (image s: + s * w * h)
    size_t cand_ofs;     // entries into the candidate / survivor lists of one image
};
struct OrbLevels {
    OrbLevel l[ORB_MAX_LEVELS];
    int n;
    int total_rows;      // sum of the level heights: per-pixel kernels run over all levels in one launch
    size_t cand_img;     // candidate / survivor entries of one image (image s starts at s * cand_img)
};

__device__ __forceinline__ size_t orb_img(const OrbLevel &lv, int s) { return lv.img_ofs + (size_t)s * lv.w * lv.h; }

// blockIdx.y of an all-level launch -> (level, row inside it).  The grid is as wide as level 0.
__device__ __forceinline__ bool orb_locate_row(const OrbLevels &L, int gy, int &lev, int &y) {
    for (lev = 0; lev < L.n; ++lev) {
        if (gy < L.l[lev].h) { y = gy; return true; }
        gy -= L.l[lev].h;
    }
    return false;
}

// blockIdx.y: image (level 0 of the batch is contiguous, n_px bytes per image)
__global__ void orb_gray_kernel(const uint8_t *__restrict__ bgr, uint8_t *__restrict__ gray, int n_px) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    const size_t o = (size_t)blockIdx.y * n_px + i;
    if (i < n_px) gray[o] = orb::bgr_to_gray(bgr[3 * o], bgr[3 * o + 1], bgr[3 * o + 2]);
}

// blockIdx.z: image; src / dst point at image 0's level, the next source image starts W * H bytes on, the next
// destination image dw * dh bytes on
__global__ void orb_resize_kernel(const uint8_t *__restrict__ src, int W, int H, uint8_t *__restrict__ dst, int dw, int dh) {
    const int x = blockIdx.x * blockDim.x + threadIdx.x, y = blockIdx.y;
    if (x >= dw) return;
    src += (size_t)blockIdx.z * W * H;
    dst += (size_t)blockIdx.z * dw * dh;
    int ox, cx, oy, cy;
    bool inx, iny;
    orb::linear_exact_coeff(x, dw, W, ox, cx, inx);
    orb::linear_exact_coeff(y, dh, H, oy, cy, iny);
    const int ox1 = min(ox + 1, W - 1), oy1 = min(oy + 1, H - 1);
    dst[(size_t)y * dw + x] = orb::linear_exact_pixel(src[(size_t)oy * W + ox], src[(size_t)oy * W + ox1],
                                                      src[(size_t)oy1 * W + ox], src[(size_t)oy1 * W + ox1], cx, inx, cy, iny);
}

// FAST-9/16 corner score of every pixel of every level (0 in the 3-pixel frame and for non-corners).  blockIdx.z: image
// (also in every kernel below).
__global__ void orb_fast_kernel(OrbLevels L, const uint8_t *__restrict__ pyr, int thr, uint8_t *__restrict__ score_all) {
    int lev, y;
    if (!orb_locate_row(L, blockIdx.y, lev, y)) return;
    const int w = L.l[lev].w, h = L.l[lev].h;
    const int x = blockIdx.x * blockDim.x + threadIdx.x;
    if (x >= w) return;
    const uint8_t *img = pyr + orb_img(L.l[lev], blockIdx.z);
    int s = 0;
    if (x >= 3 && x < w - 3 && y >= 3 && y < h - 3) {
        const uint8_t *p = img + (size_t)y * w + x;
        const int v = p[0];
        // opposite-pair quick reject (fast.cpp): a 9-arc contains one pixel of every opposite pair
        const int a = p[3 * w], b = p[-3 * w], c = p[3], d = p[-3];
        const bool dark = (a < v - thr || b < v - thr) && (c < v - thr || d < v - thr);
        const bool bright = (a > v + thr || b > v + thr) && (c > v + thr || d > v + thr);
        if (dark || bright) {
            uint8_t ring[16];
            const int dx[16] = {0, 1, 2, 3, 3, 3, 2, 1, 0, -1, -2, -3, -3, -3, -2, -1};
            const int dy[16] = {3, 3, 2, 1, 0, -1, -2, -3, -3, -3, -2, -1, 0, 1, 2, 3};
#pragma unroll
            for (int k = 0; k < 16; ++k) ring[k] = p[dy[k] * w + dx[k]];
            s = orb::fast_corner_score(v, ring, thr);
        }
    }
    score_all[orb_img(L.l[lev], blockIdx.z) + (size_t)y * w + x] = (uint8_t)s;
}

// Corners that are strict maxima of the score in their 3x3 neighbourhood and lie >= 31 pixels inside their level.
__global__ void orb_nms_kernel(OrbLevels L, const uint8_t *__restrict__ score_all, uint32_t *__restrict__ cand_xy,
                               uint8_t *__restrict__ cand_s, int32_t *__restrict__ cand_count) {
    int lev, y;
    if (!orb_locate_row(L, blockIdx.y, lev, y)) return;
    const OrbLevel lv = L.l[lev];
    const int w = lv.w, h = lv.h;
    const int x = blockIdx.x * blockDim.x + threadIdx.x;
    if (x < ORB_EDGE || x >= w - ORB_EDGE || y < ORB_EDGE || y >= h - ORB_EDGE) return;
    const uint8_t *p = score_all + orb_img(lv, blockIdx.z) + (size_t)y * w + x;
    const int s = p[0];
    if (s == 0) return;
    if (s > p[-1] && s > p[1] && s > p[-w - 1] && s > p[-w] && s > p[-w + 1] && s > p[w - 1] && s > p[w] && s > p[w + 1]) {
        const int i = atomicAdd(cand_count + 32 * blockIdx.z + lev, 1);
        const size_t c = blockIdx.z * L.cand_img + lv.cand_ofs + i;
        if (i < lv.cand_cap) { cand_xy[c] = (uint32_t)x | ((uint32_t)y << 16); cand_s[c] = (uint8_t)s; }
    }
}

// KeyPointsFilter::retainBest(2 n) on the FAST score: the 2 n best plus every tie with the 2 n-th.  One CTA per level
// (blockIdx.x) and image (blockIdx.y).
__global__ void __launch_bounds__(1024)
orb_select_fast_kernel(OrbLevels L, const uint32_t *__restrict__ cand_xy, const uint8_t *__restrict__ cand_s,
                       const int32_t *__restrict__ cand_count, uint32_t *__restrict__ surv_xy, int32_t *__restrict__ surv_count) {
    __shared__ int hist[256];
    __shared__ int thr_s, out_s;
    const OrbLevel lv = L.l[blockIdx.x];
    const size_t c0 = blockIdx.y * L.cand_img + lv.cand_ofs;
    const int m = min(cand_count[32 * blockIdx.y + blockIdx.x], lv.cand_cap), keep = 2 * lv.n_feat;
    const uint32_t *xy = cand_xy + c0;
    const uint8_t *sc = cand_s + c0;
    for (int i = threadIdx.x; i < 256; i += blockDim.x) hist[i] = 0;
    if (threadIdx.x == 0) { thr_s = 0; out_s = 0; }
    __syncthreads();
    if (m > keep && keep > 0) {
        for (int i = threadIdx.x; i < m; i += blockDim.x) atomicAdd(&hist[sc[i]], 1);
        __syncthreads();
        if (threadIdx.x == 0) {
            int acc = 0, t = 255;
            for (; t > 0; --t) { acc += hist[t]; if (acc >= keep) break; }
            thr_s = t;
        }
        __syncthreads();
    }
    const int thr = (keep > 0) ? thr_s : 256;   // keep == 0: retainBest clears the list
    for (int i = threadIdx.x; i < m; i += blockDim.x)
        if ((int)sc[i] >= thr) surv_xy[c0 + atomicAdd(&out_s, 1)] = xy[i];
    __syncthreads();
    if (threadIdx.x == 0) surv_count[32 * blockIdx.y + blockIdx.x] = out_s;
}

// Harris response of every survivor (orb.cpp HarrisResponses, 7x7 block).
__global__ void orb_harris_kernel(OrbLevels L, const uint8_t *__restrict__ pyr, const uint32_t *__restrict__ surv_xy,
                                  const int32_t *__restrict__ surv_count, float *__restrict__ resp) {
    const OrbLevel lv = L.l[blockIdx.y];
    const int m = surv_count[32 * blockIdx.z + blockIdx.y], w = lv.w;
    const uint8_t *img = pyr + orb_img(lv, blockIdx.z);
    const size_t c0 = blockIdx.z * L.cand_img + lv.cand_ofs;
    for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < m; i += gridDim.x * blockDim.x) {
    const uint32_t xy = surv_xy[c0 + i];
    const int x = xy & 0xffff, y = xy >> 16;
    int a = 0, b = 0, c = 0;
    for (int dy = -3; dy <= 3; ++dy)
        for (int dx = -3; dx <= 3; ++dx) {
            const uint8_t *p = img + (size_t)(y + dy) * w + (x + dx);
            const int ix = ((int)p[1] - (int)p[-1]) * 2 + ((int)p[-w + 1] - (int)p[-w - 1]) + ((int)p[w + 1] - (int)p[w - 1]);
            const int iy = ((int)p[w] - (int)p[-w]) * 2 + ((int)p[w - 1] - (int)p[-w - 1]) + ((int)p[w + 1] - (int)p[-w + 1]);
            a += ix * ix; b += iy * iy; c += ix * iy;
        }
    resp[c0 + i] = orb::harris_response(a, b, c);
    }
}

// retainBest(n) on the Harris response: exact n-th largest by a 4-pass radix select over the ordered float bits, every
// tie with it kept; the kept keypoints are then ranked by (y, x) and written in that order.  One CTA per level
// (blockIdx.x) and image (blockIdx.y); counts[24] of the image's block is its overflow flag.
__global__ void __launch_bounds__(1024)
orb_select_harris_kernel(OrbLevels L, const uint32_t *__restrict__ surv_xy, const float *__restrict__ resp,
                         const int32_t *__restrict__ surv_count, uint32_t *__restrict__ fin_xy, float *__restrict__ fin_resp,
                         int32_t *__restrict__ fin_count, int32_t *__restrict__ overflow) {
    __shared__ int hist[256];
    __shared__ uint32_t prefix_s;
    __shared__ int want_s, out_s;
    __shared__ uint32_t kxy[ORB_FINAL_CAP];
    __shared__ float kresp[ORB_FINAL_CAP];
    const int lev = blockIdx.x, img = blockIdx.y;
    const OrbLevel lv = L.l[lev];
    const int m = surv_count[32 * img + lev], keep = lv.n_feat;
    const size_t c0 = img * L.cand_img + lv.cand_ofs, f0 = ((size_t)img * L.n + lev) * ORB_FINAL_CAP;
    const uint32_t *xy = surv_xy + c0;
    const float *r = resp + c0;
    uint32_t thr_key = 0;   // keep everything
    if (m > keep && keep > 0) {
        if (threadIdx.x == 0) { prefix_s = 0; want_s = keep; }
        __syncthreads();
        for (int pass = 0; pass < 4; ++pass) {
            const int shift = 24 - 8 * pass;
            const uint32_t mask = pass == 0 ? 0u : (0xffffffffu << (shift + 8));
            for (int i = threadIdx.x; i < 256; i += blockDim.x) hist[i] = 0;
            __syncthreads();
            const uint32_t prefix = prefix_s;
            for (int i = threadIdx.x; i < m; i += blockDim.x) {
                const uint32_t k = float_to_ordered(r[i]);
                if ((k & mask) == prefix) atomicAdd(&hist[(k >> shift) & 255u], 1);
            }
            __syncthreads();
            if (threadIdx.x == 0) {
                int acc = 0, t = 255, want = want_s;
                for (; t > 0; --t) { if (acc + hist[t] >= want) break; acc += hist[t]; }
                want_s = want - acc;                       // rank of the threshold inside bin t
                prefix_s = prefix | ((uint32_t)t << shift);
            }
            __syncthreads();
        }
        thr_key = prefix_s;
    }
    if (threadIdx.x == 0) out_s = 0;
    __syncthreads();
    const bool none = keep <= 0;
    for (int i = threadIdx.x; i < m; i += blockDim.x) {
        if (!none && float_to_ordered(r[i]) >= thr_key) {
            const int o = atomicAdd(&out_s, 1);
            if (o < ORB_FINAL_CAP) { kxy[o] = xy[i]; kresp[o] = r[i]; }
        }
    }
    __syncthreads();
    const int n_out = min(out_s, ORB_FINAL_CAP);
    if (threadIdx.x == 0) {
        fin_count[32 * img + lev] = n_out;
        if (out_s > ORB_FINAL_CAP) atomicExch(overflow + 32 * img, 1);
    }
    // rank by (y << 16 | x): keys are distinct, so rank = number of smaller keys
    for (int i = threadIdx.x; i < n_out; i += blockDim.x) {
        const uint32_t k = kxy[i];
        int rank = 0;
        for (int j = 0; j < n_out; ++j) rank += kxy[j] < k;
        fin_xy[f0 + rank] = k;
        fin_resp[f0 + rank] = kresp[i];
    }
}

// Orientation (intensity centroid, fastAtan2) and the keypoint record.  One thread per kept keypoint; rows at or past
// out_rows are dropped.  count_out[img] = (rows written, flags: 1 = a level overflowed, 2 = rows were dropped).
__global__ void orb_finish_kernel(OrbLevels L, const uint8_t *__restrict__ pyr, const uint32_t *__restrict__ fin_xy,
                                  const float *__restrict__ fin_resp, const int32_t *__restrict__ fin_count,
                                  const int32_t *__restrict__ overflow, int out_rows, float *__restrict__ kp,
                                  float *__restrict__ aux, float *__restrict__ angle_out, int32_t *__restrict__ count_out) {
    const int lev = blockIdx.y, img = blockIdx.z;
    const OrbLevel lv = L.l[lev];
    fin_count += 32 * img;
    int base = 0, total = 0;
    for (int j = 0; j < L.n; ++j) { if (j < lev) base += fin_count[j]; total += fin_count[j]; }
    if (lev == 0 && blockIdx.x == 0 && threadIdx.x == 0) {
        count_out[2 * img] = min(total, out_rows);
        count_out[2 * img + 1] = overflow[32 * img] | (total > out_rows ? 2 : 0);
    }
    const int n_lev = min(fin_count[lev], out_rows - base), w = lv.w;
    const size_t f0 = ((size_t)img * L.n + lev) * ORB_FINAL_CAP, o0 = (size_t)img * out_rows;
    for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < n_lev; i += gridDim.x * blockDim.x) {
    const uint32_t xy = fin_xy[f0 + i];
    const int x = xy & 0xffff, y = xy >> 16;
    const uint8_t *c = pyr + orb_img(lv, img) + (size_t)y * w + x;
    int m01 = 0, m10 = 0;
    for (int u = -orb::HALF_PATCH; u <= orb::HALF_PATCH; ++u) m10 += u * (int)c[u];
    for (int v = 1; v <= orb::HALF_PATCH; ++v) {
        const int d = orb::umax(v);
        int vsum = 0;
        for (int u = -d; u <= d; ++u) {
            const int vp = c[u + v * w], vm = c[u - v * w];
            vsum += vp - vm;
            m10 += u * (vp + vm);
        }
        m01 += v * vsum;
    }
    const float ang = orb::fast_atan2((float)m01, (float)m10);
    const size_t o = o0 + base + i;
    kp[2 * o + 0] = __fmul_rn((float)x, lv.scale);
    kp[2 * o + 1] = __fmul_rn((float)y, lv.scale);
    angle_out[(size_t)img * L.n * ORB_FINAL_CAP + base + i] = ang;
    if (aux) {
        aux[4 * o + 0] = (float)lev;
        aux[4 * o + 1] = ang;
        aux[4 * o + 2] = fin_resp[f0 + i];
        aux[4 * o + 3] = __fmul_rn(31.0f, lv.scale);
    }
    }
}

__device__ __forceinline__ int reflect101(int i, int n) { return i < 0 ? -i : (i >= n ? 2 * n - 2 - i : i); }

struct GaussK { float k[7]; };

__global__ void orb_blur_row_kernel(OrbLevels L, const uint8_t *__restrict__ pyr, GaussK g, float *__restrict__ tmp_all) {
    int lev, y;
    if (!orb_locate_row(L, blockIdx.y, lev, y)) return;
    const int w = L.l[lev].w;
    const int x = blockIdx.x * blockDim.x + threadIdx.x;
    if (x >= w) return;
    const size_t ofs = orb_img(L.l[lev], blockIdx.z);
    const uint8_t *img = pyr + ofs;
    uint8_t p[7];
#pragma unroll
    for (int i = 0; i < 7; ++i) p[i] = img[(size_t)y * w + reflect101(x + i - 3, w)];
    tmp_all[ofs + (size_t)y * w + x] = orb::blur_row(g.k, p);
}
__global__ void orb_blur_col_kernel(OrbLevels L, const float *__restrict__ tmp_all, GaussK g, uint8_t *__restrict__ blurred) {
    int lev, y;
    if (!orb_locate_row(L, blockIdx.y, lev, y)) return;
    const int w = L.l[lev].w, h = L.l[lev].h;
    const int x = blockIdx.x * blockDim.x + threadIdx.x;
    if (x >= w) return;
    const size_t ofs = orb_img(L.l[lev], blockIdx.z);
    const float *tmp = tmp_all + ofs;
    float c[7];
#pragma unroll
    for (int i = 0; i < 7; ++i) c[i] = tmp[(size_t)reflect101(y + i - 3, h) * w + x];
    blurred[ofs + (size_t)y * w + x] = orb::blur_col(g.k, c);
}

// rBRIEF: one warp per keypoint, lane = descriptor byte (8 point pairs = 16 pattern points).  Rows at or past out_rows
// are dropped, as in orb_finish_kernel.
__global__ void orb_desc_kernel(OrbLevels L, const uint8_t *__restrict__ blurred, const uint32_t *__restrict__ fin_xy,
                                const int32_t *__restrict__ fin_count, const float *__restrict__ angle, int out_rows,
                                uint8_t *__restrict__ desc) {
    const int lev = blockIdx.y, img = blockIdx.z, lane = threadIdx.x & 31;
    const OrbLevel lv = L.l[lev];
    fin_count += 32 * img;
    int base = 0;
    for (int j = 0; j < lev; ++j) base += fin_count[j];
    const int n_lev = min(fin_count[lev], out_rows - base), w = lv.w;
    const size_t f0 = ((size_t)img * L.n + lev) * ORB_FINAL_CAP;
    angle += (size_t)img * L.n * ORB_FINAL_CAP + base;
    desc += ((size_t)img * out_rows + base) * 32;
    for (int i = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5); i < n_lev; i += gridDim.x * (blockDim.x >> 5)) {
    const uint32_t xy = fin_xy[f0 + i];
    const int x = xy & 0xffff, y = xy >> 16;
    const uint8_t *c = blurred + orb_img(lv, img) + (size_t)y * w + x;
    float ca, sb;
    orb::angle_cos_sin(angle[i], ca, sb);
    int val = 0;
#pragma unroll
    for (int b = 0; b < 8; ++b) {
        const int8_t *pp = ORB_PATTERN + (lane * 8 + b) * 4;
        int ix0, iy0, ix1, iy1;
        orb::rotate_pattern_point(pp[0], pp[1], ca, sb, ix0, iy0);
        orb::rotate_pattern_point(pp[2], pp[3], ca, sb, ix1, iy1);
        val |= ((int)c[iy0 * w + ix0] < (int)c[iy1 * w + ix1]) << b;
    }
    desc[(size_t)i * 32 + lane] = (uint8_t)val;
    }
}

}  // namespace
}  // namespace vo

struct vo_orb {
    vo_ctx *ctx;
    int H, W, fast_thr;
    vo::OrbLevels L;
    int S_cap;         // images the scratch buffers hold (the largest batch seen so far)
    uint8_t *pyr, *blurred, *score, *cand_s;
    float *tmp, *resp, *fin_resp, *angle;
    uint32_t *cand_xy, *surv_xy, *fin_xy;
    int32_t *counts;   // per image: cand[8] | surv[8] | fin[8] | overflow | unused[7]
    vo::GaussK g;
};

namespace vo {
namespace {

void orb_free(vo_orb *o) {
    void **ptrs[] = {(void **)&o->pyr, (void **)&o->blurred, (void **)&o->score, (void **)&o->cand_s, (void **)&o->tmp,
                     (void **)&o->resp, (void **)&o->fin_resp, (void **)&o->angle, (void **)&o->cand_xy,
                     (void **)&o->surv_xy, (void **)&o->fin_xy, (void **)&o->counts};
    for (void **p : ptrs) {
        if (*p) cudaFree(*p);
        *p = nullptr;
    }
    o->S_cap = 0;
}

// Scratch for S images: level bases of the level-major pixel buffers follow from S, so they are set here.  Growing
// drains the device first (work queued on any stream may still use the old blocks), as ws_get does.
int orb_reserve(vo_orb *o, int S) {
    if (S <= o->S_cap) return VO_OK;
    cudaSetDevice(o->ctx->device);
    if (o->S_cap) VO_CUDA(cudaDeviceSynchronize());
    orb_free(o);
    OrbLevels &L = o->L;
    size_t img_ofs = 0;
    for (int l = 0; l < L.n; ++l) {
        L.l[l].img_ofs = img_ofs;
        img_ofs += ((size_t)S * L.l[l].w * L.l[l].h + 255) & ~(size_t)255;
    }
    const size_t cand = (size_t)S * L.cand_img, fin = (size_t)S * L.n * ORB_FINAL_CAP;
    cudaError_t e = cudaSuccess;
    auto alloc = [&](void **p, size_t bytes) { if (e == cudaSuccess) e = cudaMalloc(p, bytes ? bytes : 16); };
    alloc((void **)&o->pyr, img_ofs); alloc((void **)&o->blurred, img_ofs); alloc((void **)&o->score, img_ofs);
    alloc((void **)&o->tmp, img_ofs * sizeof(float));
    alloc((void **)&o->cand_xy, cand * 4); alloc((void **)&o->cand_s, cand); alloc((void **)&o->surv_xy, cand * 4);
    alloc((void **)&o->resp, cand * 4);
    alloc((void **)&o->fin_xy, fin * 4); alloc((void **)&o->fin_resp, fin * 4); alloc((void **)&o->angle, fin * 4);
    alloc((void **)&o->counts, sizeof(int32_t) * 32 * S);
    if (e != cudaSuccess) {
        orb_free(o);
        set_error("ORB scratch for %d images: cudaMalloc -> %s", S, cudaGetErrorString(e));
        return VO_ERR_CUDA;
    }
    o->S_cap = S;
    return VO_OK;
}

}  // namespace
}  // namespace vo

extern "C" void vo_orb_destroy(vo_orb *o) {
    if (!o) return;
    cudaSetDevice(o->ctx->device);
    cudaDeviceSynchronize();
    vo::orb_free(o);
    delete o;
}

extern "C" int vo_orb_capacity(const vo_orb *o) { return o ? o->L.n * vo::ORB_FINAL_CAP : 0; }

extern "C" int vo_orb_create(vo_ctx *ctx, const vo_orb_config *cfg, vo_orb **out) {
    using namespace vo;
    VO_REQUIRE(ctx && cfg && out, "vo_orb_create: null argument");
    *out = nullptr;
    VO_REQUIRE(cfg->H >= 2 * ORB_EDGE + 1 && cfg->W >= 2 * ORB_EDGE + 1 && cfg->H < 65536 && cfg->W < 65536,
               "vo_orb_create: image %d x %d out of range", cfg->W, cfg->H);
    VO_REQUIRE(cfg->nfeatures > 0 && cfg->nlevels >= 1 && cfg->nlevels <= ORB_MAX_LEVELS && cfg->fast_threshold > 0 &&
                   cfg->fast_threshold < 255,
               "vo_orb_create: bad configuration");
    vo_orb *o = new vo_orb();
    memset(o, 0, sizeof(*o));
    o->ctx = ctx; o->H = cfg->H; o->W = cfg->W; o->fast_thr = cfg->fast_threshold;
    // level geometry and feature quotas exactly as orb.cpp computes them (fp32 / fp64 mix included)
    const double sf = (double)1.2f;
    const float factor = (float)(1.0 / sf);
    float nd = cfg->nfeatures * (1 - factor) / (1 - (float)pow((double)factor, (double)cfg->nlevels));
    int sum = 0;
    size_t cand_ofs = 0;
    o->L.n = cfg->nlevels;
    for (int l = 0; l < cfg->nlevels; ++l) {
        OrbLevel &lv = o->L.l[l];
        lv.scale = (float)pow(sf, (double)l);
        const float inv = 1.0f / lv.scale;
        lv.w = (int)lrintf(cfg->W * inv);
        lv.h = (int)lrintf(cfg->H * inv);
        if (l < cfg->nlevels - 1) { lv.n_feat = (int)lrintf(nd); sum += lv.n_feat; nd *= factor; }
        else lv.n_feat = cfg->nfeatures - sum > 0 ? cfg->nfeatures - sum : 0;
        lv.cand_cap = lv.w * lv.h / 4 + 1;
        lv.cand_ofs = cand_ofs;
        cand_ofs += ((size_t)lv.cand_cap + 63) & ~(size_t)63;
    }
    for (int l = 0; l < cfg->nlevels; ++l)
        if (o->L.l[l].n_feat > ORB_FINAL_CAP / 2) {   // leave room for ties with the n-th response
            set_error("vo_orb_create: nfeatures %d asks level %d for %d keypoints (at most %d per level)", cfg->nfeatures, l,
                      o->L.l[l].n_feat, ORB_FINAL_CAP / 2);
            delete o;
            return VO_ERR_ARG;
        }
    o->L.cand_img = cand_ofs;
    o->L.total_rows = 0;
    for (int l = 0; l < cfg->nlevels; ++l) o->L.total_rows += o->L.l[l].h;
    orb::gaussian_kernel(o->g.k);
    const int rc = orb_reserve(o, 1);
    if (rc) {
        vo_orb_destroy(o);
        return rc;
    }
    *out = o;
    return VO_OK;
}

// Diagnostic read-back of the extractor's intermediate buffers (tools/orb_bisect.py compares them stage by stage with
// the CPU restatement), of image 0 of the last call.  Synchronises the device.  what: 0 level geometry (int32 {w, h, n_feat, cand_cap} per level),
// 1 pyramid level, 2 FAST score map, 3 blurred level, 4 candidate xy (u32), 5 candidate score (u8), 6 survivor xy (u32),
// 7 survivor Harris response (f32), 8 kept xy (u32), 9 kept response (f32), 10 counts (int32[32]), 11 angles (f32, all levels).
extern "C" int vo_orb_debug_read(vo_orb *o, int what, int level, void *host_dst, size_t cap_bytes, size_t *out_bytes) {
    using namespace vo;
    VO_REQUIRE(o && host_dst && out_bytes, "vo_orb_debug_read: null argument");
    VO_REQUIRE(level >= 0 && level < o->L.n, "vo_orb_debug_read: level %d out of range", level);
    const OrbLevel &lv = o->L.l[level];
    const size_t px = (size_t)lv.w * lv.h;
    const void *src = nullptr;
    size_t bytes = 0;
    int32_t geo[4 * ORB_MAX_LEVELS];
    switch (what) {
    case 0:
        for (int l = 0; l < o->L.n; ++l) { geo[4 * l] = o->L.l[l].w; geo[4 * l + 1] = o->L.l[l].h; geo[4 * l + 2] = o->L.l[l].n_feat; geo[4 * l + 3] = o->L.l[l].cand_cap; }
        bytes = sizeof(int32_t) * 4 * o->L.n;
        VO_REQUIRE(bytes <= cap_bytes, "vo_orb_debug_read: buffer too small");
        memcpy(host_dst, geo, bytes);
        *out_bytes = bytes;
        return VO_OK;
    case 1: src = o->pyr + lv.img_ofs; bytes = px; break;
    case 2: src = o->score + lv.img_ofs; bytes = px; break;
    case 3: src = o->blurred + lv.img_ofs; bytes = px; break;
    case 4: src = o->cand_xy + lv.cand_ofs; bytes = (size_t)lv.cand_cap * 4; break;
    case 5: src = o->cand_s + lv.cand_ofs; bytes = (size_t)lv.cand_cap; break;
    case 6: src = o->surv_xy + lv.cand_ofs; bytes = (size_t)lv.cand_cap * 4; break;
    case 7: src = o->resp + lv.cand_ofs; bytes = (size_t)lv.cand_cap * 4; break;
    case 8: src = o->fin_xy + (size_t)level * ORB_FINAL_CAP; bytes = (size_t)ORB_FINAL_CAP * 4; break;
    case 9: src = o->fin_resp + (size_t)level * ORB_FINAL_CAP; bytes = (size_t)ORB_FINAL_CAP * 4; break;
    case 10: src = o->counts; bytes = sizeof(int32_t) * 32; break;
    case 11: src = o->angle; bytes = (size_t)o->L.n * ORB_FINAL_CAP * 4; break;
    default: set_error("vo_orb_debug_read: unknown buffer %d", what); return VO_ERR_ARG;
    }
    VO_REQUIRE(bytes <= cap_bytes, "vo_orb_debug_read: buffer too small (%zu > %zu)", bytes, cap_bytes);
    cudaSetDevice(o->ctx->device);
    VO_CUDA(cudaDeviceSynchronize());
    VO_CUDA(cudaMemcpy(host_dst, src, bytes, cudaMemcpyDeviceToHost));
    *out_bytes = bytes;
    return VO_OK;
}

namespace vo {
namespace {

// The one launch sequence of the extractor: S images, out_rows output rows per image.  17 launches for BGR, 16 for gray
// (level 0 arrives by one copy), whatever S is.
int orb_run(vo_orb *o, const uint8_t *images, int S, int channels, int out_rows, float *kp, uint8_t *desc, float *aux,
            int32_t *count, void *stream) {
    vo_ctx *ctx = o->ctx;
    cudaStream_t st = (cudaStream_t)stream;
    int rc = orb_reserve(o, S);
    if (rc) return rc;
    const OrbLevels &L = o->L;
    int32_t *cand_count = o->counts, *surv_count = o->counts + 8, *fin_count = o->counts + 16, *overflow = o->counts + 24;
    VO_CUDA(cudaMemsetAsync(o->counts, 0, sizeof(int32_t) * 32 * S, st));
    const int n_px = o->W * o->H;
    if (channels == 3) {
        VO_LAUNCH(orb_gray_kernel, dim3(ceil_div(n_px, 256), S), 256, st, images, o->pyr, n_px);
        VO_LAUNCH_CHECK(ctx);
    } else {   // level 0 of the batch is contiguous (L.l[0].img_ofs == 0)
        VO_CUDA(cudaMemcpyAsync(o->pyr, images, (size_t)S * n_px, cudaMemcpyDefault, st));
    }
    for (int l = 1; l < L.n; ++l) {   // every level is resized from the previous one
        const OrbLevel &lv = L.l[l], &pv = L.l[l - 1];
        VO_LAUNCH(orb_resize_kernel, dim3(ceil_div(lv.w, 128), lv.h, S), 128, st, o->pyr + pv.img_ofs, pv.w, pv.h,
                  o->pyr + lv.img_ofs, lv.w, lv.h);
        VO_LAUNCH_CHECK(ctx);
    }
    // per-pixel work of all levels in one launch each (levels too small for the 31-pixel border yield no candidate)
    const dim3 grid_all(ceil_div(L.l[0].w, 128), L.total_rows, S);
    VO_LAUNCH(orb_fast_kernel, grid_all, 128, st, L, o->pyr, o->fast_thr, o->score);
    VO_LAUNCH_CHECK(ctx);
    VO_LAUNCH(orb_nms_kernel, grid_all, 128, st, L, o->score, o->cand_xy, o->cand_s, cand_count);
    VO_LAUNCH_CHECK(ctx);
    VO_LAUNCH(orb_blur_row_kernel, grid_all, 128, st, L, o->pyr, o->g, o->tmp);
    VO_LAUNCH_CHECK(ctx);
    VO_LAUNCH(orb_blur_col_kernel, grid_all, 128, st, L, o->tmp, o->g, o->blurred);
    VO_LAUNCH_CHECK(ctx);
    VO_LAUNCH_BAR(orb_select_fast_kernel, dim3(L.n, S), 1024, st, L, o->cand_xy, o->cand_s, cand_count, o->surv_xy, surv_count);
    VO_LAUNCH_CHECK(ctx);
    // keypoint-list kernels: a few CTAs per level striding over lists whose lengths only the device knows
    VO_LAUNCH(orb_harris_kernel, dim3(8, L.n, S), 256, st, L, o->pyr, o->surv_xy, surv_count, o->resp);
    VO_LAUNCH_CHECK(ctx);
    VO_LAUNCH_BAR(orb_select_harris_kernel, dim3(L.n, S), 1024, st, L, o->surv_xy, o->resp, surv_count, o->fin_xy, o->fin_resp,
                  fin_count, overflow);
    VO_LAUNCH_CHECK(ctx);
    VO_LAUNCH(orb_finish_kernel, dim3(4, L.n, S), 128, st, L, o->pyr, o->fin_xy, o->fin_resp, fin_count, overflow, out_rows,
              kp, aux, o->angle, count);
    VO_LAUNCH_CHECK(ctx);
    VO_LAUNCH(orb_desc_kernel, dim3(16, L.n, S), 256, st, L, o->blurred, o->fin_xy, fin_count, o->angle, out_rows, desc);
    VO_LAUNCH_CHECK(ctx);
    return VO_OK;
}

}  // namespace
}  // namespace vo

extern "C" int vo_orb_extract(vo_orb *o, const uint8_t *image, int channels, float *kp, uint8_t *desc, float *aux,
                              int32_t *count, void *stream) {
    VO_REQUIRE(o && image && kp && desc && count, "vo_orb_extract: null argument");
    VO_REQUIRE(channels == 1 || channels == 3, "vo_orb_extract: image must have 1 (gray) or 3 (BGR) channels, got %d", channels);
    return vo::orb_run(o, image, 1, channels, vo_orb_capacity(o), kp, desc, aux, count, stream);
}

extern "C" int vo_orb_extract_batch(vo_orb *o, const uint8_t *images, int S, int channels, int out_rows, float *kp,
                                    uint8_t *desc, float *aux, int32_t *count, void *stream) {
    VO_REQUIRE(o && images && kp && desc && count, "vo_orb_extract_batch: null argument");
    VO_REQUIRE(channels == 1 || channels == 3, "vo_orb_extract_batch: images must have 1 (gray) or 3 (BGR) channels, got %d",
               channels);
    VO_REQUIRE(S >= 1 && S <= 65535, "vo_orb_extract_batch: %d images outside [1, 65535]", S);
    VO_REQUIRE(out_rows >= 1, "vo_orb_extract_batch: out_rows %d must be >= 1", out_rows);
    return vo::orb_run(o, images, S, channels, out_rows, kp, desc, aux, count, stream);
}
