// SIFT front-end on the GPU: cv2.SIFT_create().detectAndCompute with the reference's (default) parameters
// (feature_extractors/SIFT.py:10 `cv2.xfeatures2d.SIFT_create()`, :14-23 extract_features_and_desc) — 3 octave layers,
// contrast threshold 0.04, edge threshold 10, sigma 1.6, doubled first octave.  SURVEY 8(f) rank 1.
//
// PARITY BAR: a tolerance, not bit-exactness — OpenCV's own low-order bits depend on the SIMD object the host CPU
// selects (DESIGN 8 item 7): same keypoints to 1e-2 px / 0.25 degrees, descriptor entries within 1.
// STATUS: verified against the CPU restatement under the host emulation of tests/cuda_emu.h (tests/test_sift_emulation.py) and
// on a B200 (tests/test_gpu_sift_frontend.py; 3005 / 3005 keypoints paired with OpenCV's on a KITTI-shaped frame); default
// extractor of feature_extractors/SIFT.py.  640 frames/s on a 1241 x 376 frame (OpenCV: 27 on 16 host threads).
//
// Data layout: per octave six Gaussian layers and five difference-of-Gaussian layers, fp32, back to back.  Octave 0 is
// the x2 bilinear up-sampling of the image; octave o + 1 starts from every second pixel of layer 3 of octave o.
// Candidates (26-neighbour extrema of the DoG stack) are refined and tested by one thread each and given their
// orientations by one warp each; the keypoint list is then sorted exactly as OpenCV's KeyPointsFilter::removeDuplicatedSorted does (rank by
// counting), duplicates are dropped, and one warp per keypoint accumulates the 4 x 4 x 8 descriptor.
//
// Batch (vo_sift_extract_batch): every kernel also runs over S images, the image index being the last grid dimension
// (blockIdx.z of the per-pixel kernels, blockIdx.y of the grid-stride ones), so a call issues the same launches whatever
// S is; vo_sift_extract is the S = 1 call.  Scratch is image-major: image s has its own Gaussian, DoG and blur-temp
// planes, its own candidate / keypoint / sorted / unique lists (max_keypoints entries each) and its own count block.
// Batching changes indexing only: image s's output rows are a prefix of what it alone gives, bit for bit.
#include "common.cuh"
#include "orb_math.cuh"
#include <math.h>
#include <vector>

namespace vo {
namespace {

constexpr int SIFT_MAX_OCT = 12;
constexpr int SIFT_LAYERS = 3;            // nOctaveLayers
constexpr int SIFT_G = SIFT_LAYERS + 3;   // Gaussian images per octave
constexpr int SIFT_D = SIFT_LAYERS + 2;   // DoG images per octave
constexpr int SIFT_BORDER = 5;
constexpr int SIFT_KMAX = 33;             // longest Gaussian kernel (sigma 3.09 -> 25 taps)
// count block of one image: [0] raw keypoint records, [1] unique keypoints, [2 + o] candidates of octave o
constexpr int SIFT_CNT = 16;
static_assert(2 + SIFT_MAX_OCT <= SIFT_CNT, "one candidate counter per octave");

struct SiftOct {
    int w, h;
    size_t g_ofs, d_ofs;   // floats into the Gaussian / DoG buffers (layer stride = w * h)
};
struct SiftGeom {
    SiftOct o[SIFT_MAX_OCT];
    int n_oct;
};
struct SiftKernels {       // [0] = base blur (sig_diff), [1..5] = increments inside an octave
    float k[SIFT_G][SIFT_KMAX];
    int ksize[SIFT_G];
};
struct SiftKp {            // one record per (extremum, orientation peak); coordinates of the doubled image until finalize
    float x, y, size, angle, resp;
    int octave;
};

__device__ __forceinline__ int reflect101i(int i, int n) {
    if (n == 1) return 0;
    while (i < 0 || i >= n) i = i < 0 ? -i : 2 * n - 2 - i;   // kernels longer than the image reflect more than once
    return i;
}

// gray (or BGR) u8 -> fp32, up-sampled x2 (cv2.resize INTER_LINEAR semantics: half-pixel centres, clamped edges).
// blockIdx.z: image (input images back to back, output planes out_img floats apart)
__global__ void sift_upsample_kernel(const uint8_t *__restrict__ img, int channels, int W, int H, float *__restrict__ out,
                                     size_t out_img) {
    const int x = blockIdx.x * blockDim.x + threadIdx.x, y = blockIdx.y;
    if (x >= 2 * W) return;
    img += (size_t)blockIdx.z * W * H * channels;
    out += blockIdx.z * out_img;
    const float fx = (x + 0.5f) * 0.5f - 0.5f, fy = (y + 0.5f) * 0.5f - 0.5f;
    int x0 = (int)floorf(fx), y0 = (int)floorf(fy);
    float wx = fx - x0, wy = fy - y0;
    if (x0 < 0) { x0 = 0; wx = 0.f; }
    if (y0 < 0) { y0 = 0; wy = 0.f; }
    const int x1 = min(x0 + 1, W - 1), y1 = min(y0 + 1, H - 1);
    x0 = min(x0, W - 1); y0 = min(y0, H - 1);
    auto px = [&](int yy, int xx) -> float {
        const uint8_t *p = img + ((size_t)yy * W + xx) * channels;
        return channels == 3 ? (float)orb::bgr_to_gray(p[0], p[1], p[2]) : (float)p[0];
    };
    const float top = px(y0, x0) * (1.f - wx) + px(y0, x1) * wx;
    const float bot = px(y1, x0) * (1.f - wx) + px(y1, x1) * wx;
    out[(size_t)y * (2 * W) + x] = top * (1.f - wy) + bot * wy;
}

// Separable Gaussian, one thread per pixel.  The tap count is a template parameter (the five kernel lengths of the scale space:
// 11, 13, 17, 21, 27): the unrolled loop lets all loads of a pixel issue before the first use, and interior pixels skip the
// border reflection.  The products and the left-to-right sum are rounded one by one as before (-fmad=false): same bits as
// the generic loop, which stays for other lengths.  (Generic loop on a B200: 18-50 us per 2482 x 752 layer, latency-bound;
// the blur passes were 52 % of the front-end after the orientation kernel got its warps.)  blockIdx.z: image (source
// planes src_img floats apart, destination planes dst_img).
template <int N>
__global__ void __launch_bounds__(128)
sift_blur_row_kernel(const float *__restrict__ src, size_t src_img, int w, int h, SiftKernels K, int ki, float *__restrict__ dst,
                     size_t dst_img) {
    const int x = blockIdx.x * blockDim.x + threadIdx.x, y = blockIdx.y;
    if (x >= w) return;
    src += blockIdx.z * src_img;
    dst += blockIdx.z * dst_img;
    const int n = N > 0 ? N : K.ksize[ki], r = n / 2;
    const float *row = src + (size_t)y * w;
    float s = 0.f;
    if (N > 0 && x >= r && x + r < w) {
        float v[N > 0 ? N : 1];
#pragma unroll
        for (int i = 0; i < N; ++i) v[i] = row[x + i - r];
#pragma unroll
        for (int i = 0; i < N; ++i) s += K.k[ki][i] * v[i];
    } else {
        for (int i = 0; i < n; ++i) s += K.k[ki][i] * row[reflect101i(x + i - r, w)];
    }
    dst[(size_t)y * w + x] = s;
}
template <int N>
__global__ void __launch_bounds__(128)
sift_blur_col_kernel(const float *__restrict__ src, size_t src_img, int w, int h, SiftKernels K, int ki, float *__restrict__ dst,
                     size_t dst_img) {
    const int x = blockIdx.x * blockDim.x + threadIdx.x, y = blockIdx.y;
    if (x >= w) return;
    src += blockIdx.z * src_img;
    dst += blockIdx.z * dst_img;
    const int n = N > 0 ? N : K.ksize[ki], r = n / 2;
    float s = 0.f;
    if (N > 0 && y >= r && y + r < h) {
        float v[N > 0 ? N : 1];
        const float *col = src + (size_t)(y - r) * w + x;
#pragma unroll
        for (int i = 0; i < N; ++i) v[i] = col[(size_t)i * w];
#pragma unroll
        for (int i = 0; i < N; ++i) s += K.k[ki][i] * v[i];
    } else {
        for (int i = 0; i < n; ++i) s += K.k[ki][i] * src[(size_t)reflect101i(y + i - r, h) * w + x];
    }
    dst[(size_t)y * w + x] = s;
}
// blockIdx.z: image (src and dst both in the Gaussian buffer, g_img floats per image)
__global__ void sift_decimate_kernel(const float *__restrict__ src, int sw, float *__restrict__ dst, int w, int h, size_t g_img) {
    const int x = blockIdx.x * blockDim.x + threadIdx.x, y = blockIdx.y;
    const size_t o = blockIdx.z * g_img;
    if (x < w) dst[o + (size_t)y * w + x] = src[o + (size_t)(2 * y) * sw + 2 * x];
}
// the five DoG layers of one octave: grid.y = 5 * h, blockIdx.z: image
__global__ void sift_dog_kernel(const float *__restrict__ g, size_t g_img, int w, int h, float *__restrict__ d, size_t d_img) {
    const int x = blockIdx.x * blockDim.x + threadIdx.x;
    if (x >= w) return;
    g += blockIdx.z * g_img;
    d += blockIdx.z * d_img;
    const size_t i = (size_t)blockIdx.y * w + x;       // layer * h * w + y * w + x
    d[i] = g[i + (size_t)w * h] - g[i];
}

struct Dog3 {
    const float *prv, *cur, *nxt;
    int w;
    __device__ __forceinline__ float at(const float *p, int r, int c) const { return p[(size_t)r * w + c]; }
};

__device__ __forceinline__ void sift_solve3(const float a[3][3], const float b[3], float x[3]) {
    const float det = a[0][0] * (a[1][1] * a[2][2] - a[1][2] * a[2][1]) - a[0][1] * (a[1][0] * a[2][2] - a[1][2] * a[2][0]) +
                      a[0][2] * (a[1][0] * a[2][1] - a[1][1] * a[2][0]);
    if (det == 0.f) { x[0] = x[1] = x[2] = 0.f; return; }
    const float d = 1.f / det;
    x[0] = d * (b[0] * (a[1][1] * a[2][2] - a[1][2] * a[2][1]) - a[0][1] * (b[1] * a[2][2] - a[1][2] * b[2]) + a[0][2] * (b[1] * a[2][1] - a[1][1] * b[2]));
    x[1] = d * (a[0][0] * (b[1] * a[2][2] - a[1][2] * b[2]) - b[0] * (a[1][0] * a[2][2] - a[1][2] * a[2][0]) + a[0][2] * (a[1][0] * b[2] - b[1] * a[2][0]));
    x[2] = d * (a[0][0] * (a[1][1] * b[2] - b[1] * a[2][1]) - a[0][1] * (a[1][0] * b[2] - b[1] * a[2][0]) + b[0] * (a[1][0] * a[2][1] - a[1][1] * a[2][0]));
}

// 26-neighbour extremum -> adjustLocalExtrema -> one candidate record.  One thread per pixel of the three inner DoG layers
// of one octave (grid.y = 3 * h).  The orientation histogram of a candidate covers (2 r + 1)^2 = 360 .. 840 pixels with an
// exp, an atan2 and a sqrt each: run in the pixel's own thread it left 31 lanes of the warp idle for ~40 us per keypoint
// (48 % of the whole front-end, ncu launch list r02); sift_orient_kernel now gives every candidate a warp.
struct SiftCand {
    int32_t r, c, layer, octave;
    float xc, xr, contr, size;
};
// blockIdx.z: image (DoG planes d_img floats apart, cap candidates and a SIFT_CNT count block per image)
__global__ void sift_extrema_kernel(const float *__restrict__ dog, size_t d_img, int w, int h, int octv, int threshold,
                                    SiftCand *__restrict__ cands, int32_t *__restrict__ n_cand, int cap) {
    const int c0 = blockIdx.x * blockDim.x + threadIdx.x;
    const int layer0 = 1 + blockIdx.y / h, r0 = blockIdx.y % h;
    if (c0 < SIFT_BORDER || c0 >= w - SIFT_BORDER || r0 < SIFT_BORDER || r0 >= h - SIFT_BORDER) return;
    dog += blockIdx.z * d_img;
    cands += (size_t)blockIdx.z * cap;
    n_cand += SIFT_CNT * blockIdx.z;
    const size_t plane = (size_t)w * h;
    {
        const float *cur = dog + layer0 * plane, *prv = cur - plane, *nxt = cur + plane;
        const float val = cur[(size_t)r0 * w + c0];
        if (!(fabsf(val) > (float)threshold)) return;
        float mx = -INFINITY, mn = INFINITY;
        for (int dy = -1; dy <= 1; ++dy)
            for (int dx = -1; dx <= 1; ++dx) {
                const size_t i = (size_t)(r0 + dy) * w + (c0 + dx);
                mx = fmaxf(mx, fmaxf(prv[i], fmaxf(cur[i], nxt[i])));
                mn = fminf(mn, fminf(prv[i], fminf(cur[i], nxt[i])));
            }
        if (!((val > 0.f && val >= mx) || (val < 0.f && val <= mn))) return;
    }
    // ---- adjustLocalExtrema
    const float img_scale = 1.f / 255.f, ds = img_scale * 0.5f, ss = img_scale, cs = img_scale * 0.25f;
    int r = r0, c = c0, layer = layer0, it = 0;
    float xi = 0.f, xr = 0.f, xc = 0.f;
    Dog3 D;
    D.w = w;
    for (; it < 5; ++it) {
        D.cur = dog + layer * plane; D.prv = D.cur - plane; D.nxt = D.cur + plane;
        const float dD[3] = {(D.at(D.cur, r, c + 1) - D.at(D.cur, r, c - 1)) * ds, (D.at(D.cur, r + 1, c) - D.at(D.cur, r - 1, c)) * ds,
                             (D.at(D.nxt, r, c) - D.at(D.prv, r, c)) * ds};
        const float v2 = D.at(D.cur, r, c) * 2.f;
        const float dxx = (D.at(D.cur, r, c + 1) + D.at(D.cur, r, c - 1) - v2) * ss;
        const float dyy = (D.at(D.cur, r + 1, c) + D.at(D.cur, r - 1, c) - v2) * ss;
        const float dss = (D.at(D.nxt, r, c) + D.at(D.prv, r, c) - v2) * ss;
        const float dxy = (D.at(D.cur, r + 1, c + 1) - D.at(D.cur, r + 1, c - 1) - D.at(D.cur, r - 1, c + 1) + D.at(D.cur, r - 1, c - 1)) * cs;
        const float dxs = (D.at(D.nxt, r, c + 1) - D.at(D.nxt, r, c - 1) - D.at(D.prv, r, c + 1) + D.at(D.prv, r, c - 1)) * cs;
        const float dys = (D.at(D.nxt, r + 1, c) - D.at(D.nxt, r - 1, c) - D.at(D.prv, r + 1, c) + D.at(D.prv, r - 1, c)) * cs;
        const float Hm[3][3] = {{dxx, dxy, dxs}, {dxy, dyy, dys}, {dxs, dys, dss}};
        float X[3];
        sift_solve3(Hm, dD, X);
        xi = -X[2]; xr = -X[1]; xc = -X[0];
        if (fabsf(xi) < 0.5f && fabsf(xr) < 0.5f && fabsf(xc) < 0.5f) break;
        if (fabsf(xi) > 7e8f || fabsf(xr) > 7e8f || fabsf(xc) > 7e8f) return;
        c += __float2int_rn(xc); r += __float2int_rn(xr); layer += __float2int_rn(xi);
        if (layer < 1 || layer > SIFT_LAYERS || c < SIFT_BORDER || c >= w - SIFT_BORDER || r < SIFT_BORDER || r >= h - SIFT_BORDER) return;
    }
    if (it >= 5) return;
    D.cur = dog + layer * plane; D.prv = D.cur - plane; D.nxt = D.cur + plane;
    float contr;
    {
        const float d0 = (D.at(D.cur, r, c + 1) - D.at(D.cur, r, c - 1)) * ds, d1 = (D.at(D.cur, r + 1, c) - D.at(D.cur, r - 1, c)) * ds,
                    d2 = (D.at(D.nxt, r, c) - D.at(D.prv, r, c)) * ds;
        contr = D.at(D.cur, r, c) * img_scale + (d0 * xc + d1 * xr + d2 * xi) * 0.5f;
        if (fabsf(contr) * SIFT_LAYERS < 0.04f) return;
        const float v2 = D.at(D.cur, r, c) * 2.f;
        const float dxx = (D.at(D.cur, r, c + 1) + D.at(D.cur, r, c - 1) - v2) * ss;
        const float dyy = (D.at(D.cur, r + 1, c) + D.at(D.cur, r - 1, c) - v2) * ss;
        const float dxy = (D.at(D.cur, r + 1, c + 1) - D.at(D.cur, r + 1, c - 1) - D.at(D.cur, r - 1, c + 1) + D.at(D.cur, r - 1, c - 1)) * cs;
        const float tr = dxx + dyy, det = dxx * dyy - dxy * dxy;
        if (det <= 0.f || tr * tr * 10.f >= 11.f * 11.f * det) return;
    }
    const float oscale = (float)(1 << octv);
    const float size = 1.6f * powf(2.f, (layer + xi) / SIFT_LAYERS) * oscale * 2.f;
    const int octave = octv + (layer << 8) + (__double2int_rn(((double)xi + 0.5) * 255.0) << 16);
    const int o = atomicAdd(n_cand, 1);
    if (o < cap) {
        SiftCand k;
        k.r = r; k.c = c; k.layer = layer; k.octave = octave; k.xc = xc; k.xr = xr; k.contr = contr; k.size = size;
        cands[o] = k;
    }
}

// calcOrientationHist + the peak loop of findScaleSpaceExtrema, one warp (= one CTA of 32 threads) per candidate: the rows of
// the (2 r + 1)^2 window are dealt to the lanes, every lane accumulates its own 36-bin partial histogram in shared memory
// (bin-major, lane-minor: no bank conflicts, no atomics), the 32 partials of a bin are summed in lane order, and lane 0
// smooths, finds the peaks and appends one keypoint per peak: the result does not depend on scheduling.  blockIdx.y:
// image (Gaussian planes g_img floats apart; cap candidates, cap keypoints and a SIFT_CNT count block per image).
__global__ void __launch_bounds__(32)
sift_orient_kernel(const float *__restrict__ gauss, size_t g_img, int w, int h, int octv, const SiftCand *__restrict__ cands,
                   const int32_t *__restrict__ n_cand, SiftKp *__restrict__ kps, int32_t *__restrict__ count, int cap) {
    __shared__ float part[36 * 32];
    __shared__ float temp[36 + 4];
    gauss += blockIdx.y * g_img;
    cands += (size_t)blockIdx.y * cap;
    kps += (size_t)blockIdx.y * cap;
    n_cand += SIFT_CNT * blockIdx.y;
    count += SIFT_CNT * blockIdx.y;
    const int n = min(n_cand[0], cap), lane = threadIdx.x;
    const size_t plane = (size_t)w * h;
    const float oscale = (float)(1 << octv);
    for (int idx = blockIdx.x; idx < n; idx += gridDim.x) {
        const SiftCand k = cands[idx];
        const int r = k.r, c = k.c;
        const float scl_octv = k.size * 0.5f / oscale;
        const int radius = __float2int_rn(4.5f * scl_octv);
        const float sigma = 1.5f * scl_octv, expf_scale = -1.f / (2.f * sigma * sigma);
        const float *gimg = gauss + k.layer * plane;
        for (int b = 0; b < 36; ++b) part[b * 32 + lane] = 0.f;
        for (int i = -radius + lane; i <= radius; i += 32) {
            const int y = r + i;
            if (y <= 0 || y >= h - 1) continue;
            for (int j = -radius; j <= radius; ++j) {
                const int x = c + j;
                if (x <= 0 || x >= w - 1) continue;
                const float dx = gimg[(size_t)y * w + x + 1] - gimg[(size_t)y * w + x - 1];
                const float dy = gimg[(size_t)(y - 1) * w + x] - gimg[(size_t)(y + 1) * w + x];
                const float wgt = expf((float)(i * i + j * j) * expf_scale);
                int bin = __float2int_rn((36.f / 360.f) * orb::fast_atan2(dy, dx));
                if (bin >= 36) bin -= 36;
                if (bin < 0) bin += 36;
                part[bin * 32 + lane] += wgt * sqrtf(dx * dx + dy * dy);
            }
        }
        __syncthreads();
        for (int b = lane; b < 36; b += 32) {   // the 32 partials of a bin, in lane order
            float sum = 0.f;
            for (int l = 0; l < 32; ++l) sum += part[b * 32 + l];
            temp[2 + b] = sum;
        }
        __syncthreads();
        if (lane == 0) {
            temp[0] = temp[36]; temp[1] = temp[37]; temp[38] = temp[2]; temp[39] = temp[3];
            float hist[36], omax = 0.f;
            for (int i = 0; i < 36; ++i) {
                hist[i] = (temp[i] + temp[i + 4]) * (1.f / 16.f) + (temp[i + 1] + temp[i + 3]) * (4.f / 16.f) + temp[i + 2] * (6.f / 16.f);
                omax = i == 0 ? hist[0] : fmaxf(omax, hist[i]);
            }
            const float mag_thr = omax * 0.8f;
            for (int j = 0; j < 36; ++j) {
                const int l = j > 0 ? j - 1 : 35, r2 = j < 35 ? j + 1 : 0;
                if (hist[j] > hist[l] && hist[j] > hist[r2] && hist[j] >= mag_thr) {
                    float bin = j + 0.5f * (hist[l] - hist[r2]) / (hist[l] - 2.f * hist[j] + hist[r2]);
                    bin = bin < 0.f ? 36.f + bin : (bin >= 36.f ? bin - 36.f : bin);
                    float ang = 360.f - (360.f / 36.f) * bin;
                    if (fabsf(ang - 360.f) < 1.1920929e-07f) ang = 0.f;
                    const int o = atomicAdd(count, 1);
                    if (o < cap) {
                        SiftKp q;
                        q.x = (c + k.xc) * oscale; q.y = (r + k.xr) * oscale; q.size = k.size; q.angle = ang; q.resp = fabsf(k.contr);
                        q.octave = k.octave;
                        kps[o] = q;
                    }
                }
            }
        }
        __syncthreads();   // part[] / temp[] are reused by the next candidate of this CTA
    }
}

// First octave is -1: halve coordinates and size and rewrite the octave byte (SIFT_Impl::detectAndCompute).  blockIdx.y:
// image (also in the rank, unique and descriptor kernels below).
__global__ void sift_rescale_kernel(SiftKp *__restrict__ kps, const int32_t *__restrict__ count, int cap) {
    kps += (size_t)blockIdx.y * cap;
    const int n = min(count[SIFT_CNT * blockIdx.y], cap);
    for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) {
        SiftKp k = kps[i];
        k.x *= 0.5f; k.y *= 0.5f; k.size *= 0.5f;
        k.octave = (k.octave & ~255) | ((k.octave - 1) & 255);
        kps[i] = k;
    }
}

// KeypointGreater-style order of KeyPointsFilter::removeDuplicatedSorted: x, y ascending, then size, angle, response,
// octave descending; ties by the original index (a total order, so ranks are a permutation).
__device__ __forceinline__ bool sift_before(const SiftKp &a, int ia, const SiftKp &b, int ib) {
    if (a.x != b.x) return a.x < b.x;
    if (a.y != b.y) return a.y < b.y;
    if (a.size != b.size) return a.size > b.size;
    if (a.angle != b.angle) return a.angle > b.angle;
    if (a.resp != b.resp) return a.resp > b.resp;
    if (a.octave != b.octave) return a.octave > b.octave;
    return ia < ib;
}
// rank = number of records ordered before this one; the list is streamed through shared-memory tiles (a thread compared its
// record with 3000 others straight from global memory before: 410 us per frame, latency-bound)
constexpr int SIFT_RANK_T = 256;
__global__ void __launch_bounds__(SIFT_RANK_T)
sift_rank_kernel(const SiftKp *__restrict__ kps, const int32_t *__restrict__ count, int cap, SiftKp *__restrict__ sorted) {
    __shared__ SiftKp tile[SIFT_RANK_T];
    kps += (size_t)blockIdx.y * cap;
    sorted += (size_t)blockIdx.y * cap;
    const int n = min(count[SIFT_CNT * blockIdx.y], cap);
    for (int i0 = blockIdx.x * SIFT_RANK_T; i0 < n; i0 += gridDim.x * SIFT_RANK_T) {   // block-uniform loop: barriers inside
        const int i = i0 + threadIdx.x;
        SiftKp k = kps[min(i, n - 1)];
        int rank = 0;
        for (int j0 = 0; j0 < n; j0 += SIFT_RANK_T) {
            const int m = min(SIFT_RANK_T, n - j0);
            if ((int)threadIdx.x < m) tile[threadIdx.x] = kps[j0 + threadIdx.x];
            __syncthreads();
            if (i < n)
                for (int j = 0; j < m; ++j) rank += sift_before(tile[j], j0 + j, k, i);
            __syncthreads();
        }
        if (i < n) sorted[rank] = k;
    }
}
// Drop records that repeat (x, y, size, angle) of their predecessor, keep the order.  One CTA per image; chunks of
// blockDim.  count[1] of the image's block = unique keypoints.
__global__ void __launch_bounds__(1024)
sift_unique_kernel(const SiftKp *__restrict__ sorted, int32_t *__restrict__ count, int cap, SiftKp *__restrict__ out) {
    __shared__ int scan[1024];
    __shared__ int base_s;
    sorted += (size_t)blockIdx.y * cap;
    out += (size_t)blockIdx.y * cap;
    count += SIFT_CNT * blockIdx.y;
    const int n = min(count[0], cap);
    if (threadIdx.x == 0) base_s = 0;
    __syncthreads();
    for (int i0 = 0; i0 < n; i0 += blockDim.x) {
        const int i = i0 + threadIdx.x;
        bool keep = false;
        SiftKp k;
        if (i < n) {
            k = sorted[i];
            keep = true;
            if (i > 0) {
                const SiftKp p = sorted[i - 1];
                keep = !(p.x == k.x && p.y == k.y && p.size == k.size && p.angle == k.angle);
            }
        }
        scan[threadIdx.x] = keep ? 1 : 0;
        __syncthreads();
        for (int s = 1; s < (int)blockDim.x; s <<= 1) {       // inclusive Hillis-Steele scan
            const int v = threadIdx.x >= (unsigned)s ? scan[threadIdx.x - s] : 0;
            __syncthreads();
            scan[threadIdx.x] += v;
            __syncthreads();
        }
        if (keep) out[base_s + scan[threadIdx.x] - 1] = k;
        __syncthreads();
        if (threadIdx.x == 0) base_s += scan[blockDim.x - 1];
        __syncthreads();
    }
    if (threadIdx.x == 0) count[1] = base_s;
}

// calcSIFTDescriptor, one warp (= one CTA of 32 threads) per keypoint.  The (2 r + 1)^2 samples are dealt to the lanes by
// row; every lane accumulates its own 6 x 6 x 10 partial histogram in shared memory (bin-major, lane-minor: no bank
// conflicts, no atomics), the 32 partials are summed in lane order, and lane 0 finishes (circular wrap, clipping,
// normalisation): the result does not depend on scheduling.  Only the first out_rows keypoints of an image are written;
// count_out (optional) [img] = (rows written, flags: 1 = the raw list passed cap, 2 = rows past out_rows were dropped).
constexpr int SIFT_HIST = 6 * 6 * 10;
__global__ void __launch_bounds__(32)
sift_desc_kernel(SiftGeom G, const float *__restrict__ gauss, size_t g_img, const SiftKp *__restrict__ kps,
                 const int32_t *__restrict__ counts, int cap, int out_rows, float *__restrict__ kp_out, float *__restrict__ aux,
                 float *__restrict__ desc, int32_t *__restrict__ count_out) {
    __shared__ float part[SIFT_HIST * 32];
    const int img_i = blockIdx.y, lane = threadIdx.x;
    gauss += img_i * g_img;
    kps += (size_t)img_i * cap;
    counts += SIFT_CNT * img_i;
    kp_out += (size_t)img_i * out_rows * 2;
    desc += (size_t)img_i * out_rows * 128;
    if (aux) aux += (size_t)img_i * out_rows * 4;
    const int n_unique = counts[1], n = min(n_unique, out_rows);
    if (count_out && blockIdx.x == 0 && lane == 0) {
        count_out[2 * img_i] = n;
        count_out[2 * img_i + 1] = (counts[0] > cap ? 1 : 0) | (n_unique > out_rows ? 2 : 0);
    }
    for (int idx = blockIdx.x; idx < n; idx += gridDim.x) {
        const SiftKp k = kps[idx];
        if (lane == 0) {
            kp_out[2 * idx] = k.x; kp_out[2 * idx + 1] = k.y;
            if (aux) { aux[4 * idx] = k.size; aux[4 * idx + 1] = k.angle; aux[4 * idx + 2] = k.resp; aux[4 * idx + 3] = (float)k.octave; }
        }
        int octave = k.octave & 255;
        const int layer = (k.octave >> 8) & 255;
        octave = octave < 128 ? octave : (-128 | octave);
        const float scale = octave >= 0 ? 1.f / (float)(1 << octave) : (float)(1 << -octave);
        const SiftOct oc = G.o[octave + 1];
        const float *img = gauss + oc.g_ofs + (size_t)layer * oc.w * oc.h;
        const int cols = oc.w, rows = oc.h;
        float ori = 360.f - k.angle;
        if (fabsf(ori - 360.f) < 1.1920929e-07f) ori = 0.f;
        const float scl = k.size * scale * 0.5f;
        const int px = __float2int_rn(k.x * scale), py = __float2int_rn(k.y * scale);
        const float rad = ori * (float)(3.14159265358979323846 / 180.0);
        float cos_t = (float)cos((double)rad), sin_t = (float)sin((double)rad);
        const float bins_per_rad = 8.f / 360.f, exp_scale = -1.f / (4 * 4 * 0.5f), hist_width = 3.f * scl;
        int radius = __float2int_rn(hist_width * 1.4142135623730951f * 5.f * 0.5f);
        radius = min(radius, (int)sqrt((double)cols * cols + (double)rows * rows));
        cos_t /= hist_width; sin_t /= hist_width;
        for (int b = 0; b < SIFT_HIST; ++b) part[b * 32 + lane] = 0.f;
        for (int i = -radius + lane; i <= radius; i += 32)
            for (int j = -radius; j <= radius; ++j) {
                const float c_rot = j * cos_t - i * sin_t, r_rot = j * sin_t + i * cos_t;
                float rbin = r_rot + 2 - 0.5f, cbin = c_rot + 2 - 0.5f;
                const int r = py + i, c = px + j;
                if (!(rbin > -1 && rbin < 4 && cbin > -1 && cbin < 4 && r > 0 && r < rows - 1 && c > 0 && c < cols - 1)) continue;
                const float dx = img[(size_t)r * cols + c + 1] - img[(size_t)r * cols + c - 1];
                const float dy = img[(size_t)(r - 1) * cols + c] - img[(size_t)(r + 1) * cols + c];
                const float w = expf((c_rot * c_rot + r_rot * r_rot) * exp_scale);
                float obin = (orb::fast_atan2(dy, dx) - ori) * bins_per_rad;
                const float mag = sqrtf(dx * dx + dy * dy) * w;
                const int r0 = (int)floorf(rbin), c0 = (int)floorf(cbin);
                int o0 = (int)floorf(obin);
                rbin -= r0; cbin -= c0; obin -= o0;
                if (o0 < 0) o0 += 8;
                if (o0 >= 8) o0 -= 8;
                const float v_r1 = mag * rbin, v_r0 = mag - v_r1;
                const float v_rc11 = v_r1 * cbin, v_rc10 = v_r1 - v_rc11, v_rc01 = v_r0 * cbin, v_rc00 = v_r0 - v_rc01;
                const float v111 = v_rc11 * obin, v110 = v_rc11 - v111, v101 = v_rc10 * obin, v100 = v_rc10 - v101;
                const float v011 = v_rc01 * obin, v010 = v_rc01 - v011, v001 = v_rc00 * obin, v000 = v_rc00 - v001;
                float *hp = part + (((r0 + 1) * 6 + c0 + 1) * 10 + o0) * 32 + lane;
                hp[0] += v000; hp[32] += v001; hp[10 * 32] += v010; hp[11 * 32] += v011;
                hp[60 * 32] += v100; hp[61 * 32] += v101; hp[70 * 32] += v110; hp[71 * 32] += v111;
            }
        __syncthreads();
        for (int b = lane; b < SIFT_HIST; b += 32) {   // the 32 partials of a bin, in lane order
            float sum = 0.f;
            for (int l = 0; l < 32; ++l) sum += part[b * 32 + l];
            part[b * 32] = sum;
        }
        __syncthreads();
        if (lane == 0) {
            float *dst = desc + (size_t)idx * 128;
            float nrm2 = 0.f;
            for (int i = 0; i < 4; ++i)
                for (int j = 0; j < 4; ++j) {
                    const int h = ((i + 1) * 6 + (j + 1)) * 10;
                    const float b0 = part[h * 32] + part[(h + 8) * 32], b1 = part[(h + 1) * 32] + part[(h + 9) * 32];
                    for (int b = 0; b < 8; ++b) {
                        const float v = b == 0 ? b0 : (b == 1 ? b1 : part[(h + b) * 32]);
                        dst[(i * 4 + j) * 8 + b] = v;
                        nrm2 += v * v;
                    }
                }
            const float thr = sqrtf(nrm2) * 0.2f;
            nrm2 = 0.f;
            for (int i = 0; i < 128; ++i) { const float v = fminf(dst[i], thr); dst[i] = v; nrm2 += v * v; }
            const float f = 512.f / fmaxf(sqrtf(nrm2), 1.1920929e-07f);
            for (int i = 0; i < 128; ++i) { const int q = __float2int_rn(dst[i] * f); dst[i] = (float)(q < 0 ? 0 : (q > 255 ? 255 : q)); }
        }
        __syncthreads();   // part[] is reused by the next keypoint of this CTA
    }
}

// row pass src -> tmp, column pass tmp -> dst with kernel ki; the unrolled instantiation when the length is one of the scale space's.
// grid.z images: src and dst planes g_img floats apart, tmp planes t_img.
int sift_blur(vo_ctx *ctx, dim3 grid, cudaStream_t st, const float *src, int w, int h, const SiftKernels &K, int ki, float *tmp,
              float *dst, size_t g_img, size_t t_img) {
#define VO_SIFT_BLUR(N)                                                                        \
    VO_LAUNCH(sift_blur_row_kernel<N>, grid, 128, st, src, g_img, w, h, K, ki, tmp, t_img);    \
    VO_LAUNCH_CHECK(ctx);                                                                      \
    VO_LAUNCH(sift_blur_col_kernel<N>, grid, 128, st, tmp, t_img, w, h, K, ki, dst, g_img)
    switch (K.ksize[ki]) {
        case 11: VO_SIFT_BLUR(11); break;
        case 13: VO_SIFT_BLUR(13); break;
        case 17: VO_SIFT_BLUR(17); break;
        case 21: VO_SIFT_BLUR(21); break;
        case 27: VO_SIFT_BLUR(27); break;
        default: VO_SIFT_BLUR(0); break;
    }
#undef VO_SIFT_BLUR
    VO_LAUNCH_CHECK(ctx);
    return VO_OK;
}

}  // namespace
}  // namespace vo

struct vo_sift {
    vo_ctx *ctx;
    int H, W, cap;
    int S_cap;            // images the scratch holds (the largest batch seen so far)
    size_t g_img, d_img;  // floats of one image's Gaussian / DoG planes (all octaves)
    vo::SiftGeom G;
    vo::SiftKernels K;
    float *gauss, *dog, *tmp;
    vo::SiftKp *kps, *sorted, *uniq;
    int32_t *counts;      // per image: SIFT_CNT words ([0] raw count, [1] final count, [2 + o] candidates of octave o)
    vo::SiftCand *cands;
};

namespace vo {
namespace {

void sift_free(vo_sift *s) {
    void **ptrs[] = {(void **)&s->gauss, (void **)&s->dog, (void **)&s->tmp, (void **)&s->kps, (void **)&s->sorted,
                     (void **)&s->uniq, (void **)&s->counts, (void **)&s->cands};
    for (void **p : ptrs) {
        if (*p) cudaFree(*p);
        *p = nullptr;
    }
    s->S_cap = 0;
}

// Scratch for S images (a KITTI-shaped 1241 x 376 image takes ~117 MB, nearly all of it the fp32 planes).  Growing
// drains the device first (work queued on any stream may still use the old blocks), as ws_get does.
int sift_reserve(vo_sift *s, int S) {
    if (S <= s->S_cap) return VO_OK;
    cudaSetDevice(s->ctx->device);
    if (s->S_cap) VO_CUDA(cudaDeviceSynchronize());
    sift_free(s);
    const size_t n = (size_t)S, cap = (size_t)s->cap, t_img = (size_t)s->G.o[0].w * s->G.o[0].h;
    cudaError_t e = cudaSuccess;
    auto alloc = [&](void **p, size_t bytes) { if (e == cudaSuccess) e = cudaMalloc(p, bytes ? bytes : 16); };
    alloc((void **)&s->gauss, n * s->g_img * 4); alloc((void **)&s->dog, n * s->d_img * 4); alloc((void **)&s->tmp, n * t_img * 4);
    alloc((void **)&s->kps, sizeof(SiftKp) * n * cap); alloc((void **)&s->sorted, sizeof(SiftKp) * n * cap);
    alloc((void **)&s->uniq, sizeof(SiftKp) * n * cap); alloc((void **)&s->counts, sizeof(int32_t) * SIFT_CNT * n);
    alloc((void **)&s->cands, sizeof(SiftCand) * n * cap);
    if (e != cudaSuccess) {
        sift_free(s);
        set_error("SIFT scratch for %d images: cudaMalloc -> %s", S, cudaGetErrorString(e));
        return VO_ERR_CUDA;
    }
    s->S_cap = S;
    return VO_OK;
}

}  // namespace
}  // namespace vo

extern "C" void vo_sift_destroy(vo_sift *s) {
    if (!s) return;
    cudaSetDevice(s->ctx->device);
    cudaDeviceSynchronize();
    vo::sift_free(s);
    delete s;
}
extern "C" int vo_sift_capacity(const vo_sift *s) { return s ? s->cap : 0; }

extern "C" int vo_sift_create(vo_ctx *ctx, const vo_sift_config *cfg, vo_sift **out) {
    using namespace vo;
    VO_REQUIRE(ctx && cfg && out, "vo_sift_create: null argument");
    *out = nullptr;
    VO_REQUIRE(cfg->H >= 8 && cfg->W >= 8 && cfg->H <= 8192 && cfg->W <= 8192 && cfg->max_keypoints > 0,
               "vo_sift_create: bad configuration (%d x %d, %d keypoints)", cfg->W, cfg->H, cfg->max_keypoints);
    vo_sift *s = new vo_sift();
    memset(s, 0, sizeof(*s));
    s->ctx = ctx; s->H = cfg->H; s->W = cfg->W; s->cap = cfg->max_keypoints;
    const int bw = 2 * cfg->W, bh = 2 * cfg->H;
    int n_oct = (int)lrint(log((double)(bw < bh ? bw : bh)) / log(2.0) - 2) + 1;
    if (n_oct > SIFT_MAX_OCT) n_oct = SIFT_MAX_OCT;
    if (n_oct < 1) n_oct = 1;
    s->G.n_oct = n_oct;
    size_t g_ofs = 0, d_ofs = 0;
    int w = bw, h = bh;
    for (int o = 0; o < n_oct; ++o) {
        s->G.o[o].w = w; s->G.o[o].h = h; s->G.o[o].g_ofs = g_ofs; s->G.o[o].d_ofs = d_ofs;
        g_ofs += (size_t)SIFT_G * w * h; d_ofs += (size_t)SIFT_D * w * h;
        w /= 2; h /= 2;
        if (w < 1 || h < 1) { s->G.n_oct = o + 1; break; }
    }
    s->g_img = g_ofs; s->d_img = d_ofs;
    // Gaussian kernels: [0] the base blur, [i] the increment from layer i - 1 to layer i
    double sig[SIFT_G];
    sig[0] = sqrt(fmax(1.6 * 1.6 - 0.5 * 0.5 * 4, 0.01));
    const double kf = pow(2.0, 1.0 / SIFT_LAYERS);
    for (int i = 1; i < SIFT_G; ++i) {
        const double prev = pow(kf, (double)(i - 1)) * 1.6, tot = prev * kf;
        sig[i] = sqrt(tot * tot - prev * prev);
    }
    sig[0] = (double)(float)sig[0];   // createInitialImage keeps sig_diff in fp32
    for (int i = 0; i < SIFT_G; ++i) {
        int ks = (int)lrint(sig[i] * 4 * 2 + 1) | 1;
        if (ks > SIFT_KMAX) ks = SIFT_KMAX;
        s->K.ksize[i] = ks;
        double e[SIFT_KMAX], sum = 0.0;
        for (int j = 0; j < ks; ++j) { const double x = j - (ks - 1) * 0.5; e[j] = exp(-(x * x) / (2.0 * sig[i] * sig[i])); sum += e[j]; }
        for (int j = 0; j < ks; ++j) s->K.k[i][j] = (float)(e[j] / sum);
    }
    if (const int rc = sift_reserve(s, 1)) {
        vo_sift_destroy(s);
        return rc;
    }
    *out = s;
    return VO_OK;
}

namespace vo {
namespace {

// CTAs per image of a grid-stride kernel: the one-image grid `one` spread over the batch, at least `least` per image
int sift_ctas(int one, int S, int least) { return ceil_div(one, S) > least ? ceil_div(one, S) : least; }

// The one launch sequence of the extractor: S images, out_rows output rows per image.  The launches depend on the image
// shape only, not on S.  count (optional) [S][2] = (rows written, flags), written by the descriptor kernel.
int sift_run(vo_sift *s, const uint8_t *images, int S, int channels, int out_rows, float *kp, float *desc, float *aux,
             int32_t *count, void *stream) {
    vo_ctx *ctx = s->ctx;
    cudaStream_t st = (cudaStream_t)stream;
    if (int rc = sift_reserve(s, S)) return rc;
    const SiftGeom &G = s->G;
    const size_t g_img = s->g_img, d_img = s->d_img;
    const SiftOct &o0 = G.o[0];
    const size_t t_img = (size_t)o0.w * o0.h;
    // every image's count block, the per-octave candidate counters included, is zeroed here once
    VO_CUDA(cudaMemsetAsync(s->counts, 0, sizeof(int32_t) * SIFT_CNT * S, st));
    float *g00 = s->gauss + o0.g_ofs;
    // base image: up-sample into layer 1's slot (free until it is computed), blur into layer 0
    float *scratch = g00 + (size_t)o0.w * o0.h;
    VO_LAUNCH(sift_upsample_kernel, dim3(ceil_div(o0.w, 128), o0.h, S), 128, st, images, channels, s->W, s->H, scratch, g_img);
    VO_LAUNCH_CHECK(ctx);
    if (int rc = sift_blur(ctx, dim3(ceil_div(o0.w, 128), o0.h, S), st, scratch, o0.w, o0.h, s->K, 0, s->tmp, g00, g_img, t_img))
        return rc;
    const int threshold = (int)floor(0.5 * 0.04 / SIFT_LAYERS * 255);
    const int per_img = sift_ctas(1184, S, 8);   // one-image grid: 8 CTAs per SM, striding
    for (int o = 0; o < G.n_oct; ++o) {
        const SiftOct &oc = G.o[o];
        const size_t plane = (size_t)oc.w * oc.h;
        float *g = s->gauss + oc.g_ofs, *d = s->dog + oc.d_ofs;
        const dim3 grid(ceil_div(oc.w, 128), oc.h, S);
        if (o > 0) {
            const SiftOct &pv = G.o[o - 1];
            VO_LAUNCH(sift_decimate_kernel, grid, 128, st, s->gauss + pv.g_ofs + (size_t)SIFT_LAYERS * pv.w * pv.h, pv.w, g, oc.w,
                      oc.h, g_img);
            VO_LAUNCH_CHECK(ctx);
        }
        for (int i = 1; i < SIFT_G; ++i) {
            if (int rc = sift_blur(ctx, grid, st, g + (i - 1) * plane, oc.w, oc.h, s->K, i, s->tmp, g + i * plane, g_img, t_img))
                return rc;
        }
        VO_LAUNCH(sift_dog_kernel, dim3(ceil_div(oc.w, 128), SIFT_D * oc.h, S), 128, st, g, g_img, oc.w, oc.h, d, d_img);
        VO_LAUNCH_CHECK(ctx);
        if (oc.w > 2 * SIFT_BORDER && oc.h > 2 * SIFT_BORDER) {
            VO_LAUNCH(sift_extrema_kernel, dim3(ceil_div(oc.w, 128), SIFT_LAYERS * oc.h, S), 128, st, d, d_img, oc.w, oc.h, o,
                      threshold, s->cands, s->counts + 2 + o, s->cap);
            VO_LAUNCH_CHECK(ctx);
            VO_LAUNCH_BAR(sift_orient_kernel, dim3(per_img, S), 32, st, g, g_img, oc.w, oc.h, o, s->cands, s->counts + 2 + o,
                          s->kps, s->counts, s->cap);
            VO_LAUNCH_CHECK(ctx);
        }
    }
    VO_LAUNCH(sift_rescale_kernel, dim3(sift_ctas(32, S, 4), S), 256, st, s->kps, s->counts, s->cap);
    VO_LAUNCH_CHECK(ctx);
    VO_LAUNCH_BAR(sift_rank_kernel, dim3(sift_ctas(64, S, 16), S), SIFT_RANK_T, st, s->kps, s->counts, s->cap, s->sorted);
    VO_LAUNCH_CHECK(ctx);
    VO_LAUNCH_BAR(sift_unique_kernel, dim3(1, S), 1024, st, s->sorted, s->counts, s->cap, s->uniq);
    VO_LAUNCH_CHECK(ctx);
    VO_LAUNCH_BAR(sift_desc_kernel, dim3(per_img, S), 32, st, G, s->gauss, g_img, s->uniq, s->counts, s->cap, out_rows, kp, aux,
                  desc, count);
    VO_LAUNCH_CHECK(ctx);
    return VO_OK;
}

}  // namespace
}  // namespace vo

extern "C" int vo_sift_extract(vo_sift *s, const uint8_t *image, int channels, float *kp, float *desc, float *aux,
                               int32_t *count, void *stream) {
    VO_REQUIRE(s && image && kp && desc && count, "vo_sift_extract: null argument");
    VO_REQUIRE(channels == 1 || channels == 3, "vo_sift_extract: image must have 1 (gray) or 3 (BGR) channels, got %d", channels);
    if (int rc = vo::sift_run(s, image, 1, channels, s->cap, kp, desc, aux, nullptr, stream)) return rc;
    // count[0] = keypoints written, count[1] = raw candidates found (> max_keypoints: the list was cut)
    cudaStream_t st = (cudaStream_t)stream;
    VO_CUDA(cudaMemcpyAsync(count, s->counts + 1, sizeof(int32_t), cudaMemcpyDefault, st));
    VO_CUDA(cudaMemcpyAsync(count + 1, s->counts, sizeof(int32_t), cudaMemcpyDefault, st));
    return VO_OK;
}

extern "C" int vo_sift_extract_batch(vo_sift *s, const uint8_t *images, int S, int channels, int out_rows, float *kp, float *desc,
                                     float *aux, int32_t *count, void *stream) {
    VO_REQUIRE(s && images && kp && desc && count, "vo_sift_extract_batch: null argument");
    VO_REQUIRE(channels == 1 || channels == 3, "vo_sift_extract_batch: images must have 1 (gray) or 3 (BGR) channels, got %d",
               channels);
    VO_REQUIRE(S >= 1 && S <= 65535, "vo_sift_extract_batch: %d images outside [1, 65535]", S);
    VO_REQUIRE(out_rows >= 1, "vo_sift_extract_batch: out_rows %d must be >= 1", out_rows);
    return vo::sift_run(s, images, S, channels, out_rows, kp, desc, aux, count, stream);
}
