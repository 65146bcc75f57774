// "Same" 2-D convolution (stride 1, dilation d, k x k taps) on the 5th-generation tensor cores as an implicit GEMM in
// 3xTF32 — the layer type of the R2D2 network (feature_extractors/r2d2/nets/patchnet.py:56-66: every Conv2d of
// Quad_L2Net / Fast_Quad_L2Net keeps the resolution; strides become dilations).
//
// Layout: activations NHWC fp32, already split into tf32 hi / lo parts by the producing layer; weights
// [C_out][tap][C_in] (K-major), split once on the host.  A tile is 128 consecutive pixels of one image row for all
// C_out channels; persistent CTAs (one per SM) walk the tile list:
//   * per (tap, 32-channel block) the producer thread issues four TMA boxes into a 3-stage ring: the activation box
//     {32 c, 128 w, 1 h} at the tap's shifted coordinates (hi and lo) — TMA's out-of-bounds zero fill IS the
//     convolution's zero padding, there is no im2col buffer and no border code — and the weight box {32 k, C_out};
//   * one elected thread issues tcgen05.mma.kind::tf32 M128 x N(C_out) x K8 with both operands from shared memory,
//     three per k-step (a_lo*b_hi, a_hi*b_hi, a_hi*b_lo), accumulating in tensor memory;
//   * four epilogue warps read the accumulator (tcgen05.ld), apply bias + folded batch-norm (+ ReLU) and store the
//     result as fp32 and / or as the hi / lo pair the next layer consumes.
#include "common.cuh"
#include "tc_ptx.cuh"

namespace vo {
namespace {
using namespace tc;

constexpr int CV_PIX = 128;      // pixels per CTA (= TMEM lanes = MMA M)
constexpr int CV_KB = 32;        // channels per box (32 fp32 = one 128 B swizzle row)
constexpr int CV_STAGES = 3;
constexpr int CV_THREADS = 192;  // warps 0..3 epilogue, warp 4 TMA, warp 5 MMA
constexpr int CV_A_BYTES = CV_PIX * 128;

template <int COUT>
struct CvSmem {
    static constexpr int B_BYTES = COUT * 128;
    static constexpr int STAGE_BYTES = 2 * CV_A_BYTES + 2 * B_BYTES;  // A_hi | A_lo | B_hi | B_lo
    static constexpr int OFF_BAR = CV_STAGES * STAGE_BYTES;
    static constexpr int TOTAL = OFF_BAR + 256 + 1024;
};

constexpr uint32_t cv_idesc(int n) {
    return (1u << 4) | (2u << 7) | (2u << 10) | ((uint32_t)(n >> 3) << 17) | ((uint32_t)(CV_PIX >> 4) << 24);
}

struct ConvGeom {
    int H, W, cin, taps_x, taps_y, dil, pad;  // tap (ty, tx) reads pixel (h - pad + ty*dil, w - pad + tx*dil)
    int tiles_x;                              // ceil(W / 128)
    int relu;
};

// Persistent: one CTA per SM walks the tile list (tile = 128 consecutive pixels of one image row).  The producer runs
// ahead across tile boundaries, the MMA thread alternates between two accumulators in tensor memory, and the epilogue
// warps drain one accumulator while the next tile's MMAs fill the other — per-tile set-up (barriers, TMEM allocation)
// and the TMEM -> registers -> global epilogue are off the tensor pipe's critical path.
template <int COUT>
__global__ void __launch_bounds__(CV_THREADS, 1)
conv_tc_kernel(const __grid_constant__ CUtensorMap map_a_hi, const __grid_constant__ CUtensorMap map_a_lo,
               const __grid_constant__ CUtensorMap map_b_hi, const __grid_constant__ CUtensorMap map_b_lo, ConvGeom g,
               const float *__restrict__ scale, const float *__restrict__ shift, float *__restrict__ out_full,
               float *__restrict__ out_hi, float *__restrict__ out_lo) {
    using S = CvSmem<COUT>;
    extern __shared__ uint8_t smem_raw[];
    const uint32_t base = (smem_u32(smem_raw) + 1023u) & ~1023u;
    uint8_t *smem = smem_raw + (base - smem_u32(smem_raw));
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int cblocks = g.cin / CV_KB;
    const int n_items = g.taps_x * g.taps_y * cblocks;
    const int n_tiles = g.H * g.tiles_x;

    const uint32_t s_bar = base + S::OFF_BAR;
    auto bar_full = [&](int s) { return s_bar + 8u * s; };
    auto bar_empty = [&](int s) { return s_bar + 8u * (CV_STAGES + s); };
    auto bar_tfull = [&](int a) { return s_bar + 8u * (2 * CV_STAGES + a); };
    auto bar_tempty = [&](int a) { return s_bar + 8u * (2 * CV_STAGES + 2 + a); };
    uint32_t *tmem_slot = reinterpret_cast<uint32_t *>(smem + S::OFF_BAR + 8 * (2 * CV_STAGES + 4));

    if (threadIdx.x == 0) {
        for (int s = 0; s < CV_STAGES; ++s) { mbar_init(bar_full(s), 1); mbar_init(bar_empty(s), 1); }
        for (int a = 0; a < 2; ++a) { mbar_init(bar_tfull(a), 1); mbar_init(bar_tempty(a), 4); }
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    if (warp == 5) {
        asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(tmem_slot)),
                     "r"((uint32_t)(2 * COUT))
                     : "memory");
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
    }
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem_base = *tmem_slot;

    if (warp == 4) {
        // ===================== TMA producer =====================
        if (lane == 0) {
            int it = 0;
            for (int t = blockIdx.x; t < n_tiles; t += gridDim.x) {
                const int h0 = t / g.tiles_x, w0 = (t % g.tiles_x) * CV_PIX;
                for (int ty = 0; ty < g.taps_y; ++ty)
                    for (int tx = 0; tx < g.taps_x; ++tx) {
                        const int hh = h0 - g.pad + ty * g.dil, ww = w0 - g.pad + tx * g.dil;  // may be out of bounds: zero fill
                        const int krow = (ty * g.taps_x + tx) * g.cin;
                        for (int cb = 0; cb < cblocks; ++cb, ++it) {
                            const int stage = it % CV_STAGES;
                            const uint32_t phase = (uint32_t)(it / CV_STAGES) & 1u;
                            mbar_wait(bar_empty(stage), phase ^ 1u);
                            mbar_expect_tx(bar_full(stage), S::STAGE_BYTES);
                            const uint32_t dst = base + stage * S::STAGE_BYTES;
                            tma_load_3d(dst, &map_a_hi, cb * CV_KB, ww, hh, bar_full(stage));
                            tma_load_3d(dst + CV_A_BYTES, &map_a_lo, cb * CV_KB, ww, hh, bar_full(stage));
                            tma_load_2d(dst + 2 * CV_A_BYTES, &map_b_hi, krow + cb * CV_KB, 0, bar_full(stage));
                            tma_load_2d(dst + 2 * CV_A_BYTES + S::B_BYTES, &map_b_lo, krow + cb * CV_KB, 0, bar_full(stage));
                        }
                    }
            }
        }
    } else if (warp == 5) {
        // ===================== MMA issuer =====================
        constexpr uint32_t IDESC = cv_idesc(COUT);
        uint32_t stage = 0, phase = 0;
        int lt = 0;
        for (int t = blockIdx.x; t < n_tiles; t += gridDim.x, ++lt) {
            const int buf = lt & 1;
            mbar_wait(bar_tempty(buf), (((uint32_t)(lt >> 1)) & 1u) ^ 1u);  // epilogue has drained this accumulator
            tc_fence_after();
            const uint32_t d_tmem = tmem_base + (uint32_t)(buf * COUT);
            for (int it = 0; it < n_items; ++it) {
                mbar_wait(bar_full(stage), phase);
                tc_fence_after();
                if (elect_one()) {
                    const uint32_t sa = base + stage * S::STAGE_BYTES;
                    const uint32_t a_hi = ((sa & 0x3ffffu) >> 4) | (1u << 16);
                    const uint32_t a_lo = (((sa + CV_A_BYTES) & 0x3ffffu) >> 4) | (1u << 16);
                    const uint32_t b_hi = (((sa + 2 * CV_A_BYTES) & 0x3ffffu) >> 4) | (1u << 16);
                    const uint32_t b_lo = (((sa + 2 * CV_A_BYTES + S::B_BYTES) & 0x3ffffu) >> 4) | (1u << 16);
#pragma unroll
                    for (int k8 = 0; k8 < CV_KB / 8; ++k8) {
                        const uint64_t hi = (uint64_t)TC_SDESC_HI << 32;
                        const uint64_t dah = hi | (uint64_t)(a_hi + k8 * 2), dal = hi | (uint64_t)(a_lo + k8 * 2);
                        const uint64_t dbh = hi | (uint64_t)(b_hi + k8 * 2), dbl = hi | (uint64_t)(b_lo + k8 * 2);
                        tc_mma_tf32_ss(d_tmem, dal, dbh, IDESC, (it | k8) ? 1u : 0u);  // small terms first
                        tc_mma_tf32_ss(d_tmem, dah, dbl, IDESC, 1u);
                        tc_mma_tf32_ss(d_tmem, dah, dbh, IDESC, 1u);
                    }
                    tc_commit(bar_empty(stage));
                    if (it == n_items - 1) tc_commit(bar_tfull(buf));
                }
                __syncwarp();
                if (++stage == CV_STAGES) { stage = 0; phase ^= 1u; }
            }
        }
    } else {
        // ===================== epilogue: warp w owns TMEM lanes (= pixels) 32 w .. 32 w + 31 =====================
        int lt = 0;
        for (int t = blockIdx.x; t < n_tiles; t += gridDim.x, ++lt) {
            const int buf = lt & 1;
            const int h0 = t / g.tiles_x, w0 = (t % g.tiles_x) * CV_PIX;
            mbar_wait(bar_tfull(buf), ((uint32_t)(lt >> 1)) & 1u);
            tc_fence_after();
            const int w = w0 + warp * 32 + lane;
            const bool ok = w < g.W;
            const size_t pix = ((size_t)h0 * g.W + (ok ? w : 0)) * COUT;
            const uint32_t taddr = tmem_base + ((uint32_t)(warp * 32) << 16) + (uint32_t)(buf * COUT);
#pragma unroll 1
            for (int c0 = 0; c0 < COUT; c0 += 32) {
                float v[32];
                tc_ld32(taddr + c0, v);
                if (c0 + 32 == COUT) {  // last read of this accumulator: hand it back before the stores
                    tc_fence_before();
                    if (lane == 0) mbar_arrive(bar_tempty(buf));
                }
#pragma unroll
                for (int j = 0; j < 32; ++j) {
                    float y = __fmaf_rn(v[j], __ldg(scale + c0 + j), __ldg(shift + c0 + j));
                    v[j] = g.relu ? fmaxf(y, 0.0f) : y;
                }
                if (ok) {
                    if (out_full) {
#pragma unroll
                        for (int j = 0; j < 32; j += 4)
                            *reinterpret_cast<float4 *>(out_full + pix + c0 + j) = make_float4(v[j], v[j + 1], v[j + 2], v[j + 3]);
                    }
                    if (out_hi) {
#pragma unroll
                        for (int j = 0; j < 32; j += 4) {
                            const float4 hv = make_float4(to_tf32(v[j]), to_tf32(v[j + 1]), to_tf32(v[j + 2]), to_tf32(v[j + 3]));
                            *reinterpret_cast<float4 *>(out_hi + pix + c0 + j) = hv;
                            *reinterpret_cast<float4 *>(out_lo + pix + c0 + j) =
                                make_float4(to_tf32(v[j] - hv.x), to_tf32(v[j + 1] - hv.y), to_tf32(v[j + 2] - hv.z),
                                            to_tf32(v[j + 3] - hv.w));
                        }
                    }
                }
            }
        }
    }
    tc_fence_before();
    __syncthreads();
    if (warp == 5) {
        tc_fence_after();
        asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"((uint32_t)(2 * COUT)) : "memory");
    }
}

__global__ void __launch_bounds__(256)
tf32_split_kernel(const float *__restrict__ x, size_t n4, float *__restrict__ hi, float *__restrict__ lo) {
    const size_t stride = (size_t)gridDim.x * blockDim.x;
    for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < n4; i += stride) {
        const float4 v = reinterpret_cast<const float4 *>(x)[i];
        const float4 h = make_float4(to_tf32(v.x), to_tf32(v.y), to_tf32(v.z), to_tf32(v.w));
        reinterpret_cast<float4 *>(hi)[i] = h;
        reinterpret_cast<float4 *>(lo)[i] = make_float4(to_tf32(v.x - h.x), to_tf32(v.y - h.y), to_tf32(v.z - h.z), to_tf32(v.w - h.w));
    }
}

}  // namespace

// activation map: NHWC [H][W][C] viewed as a 3-D tensor (C, W, H), box {32, 128, 1}
int conv_map_act(vo_ctx *ctx, void *map_out, const float *ptr, int H, int W, int C) {
    int rc = ensure_encode(ctx);
    if (rc) return rc;
    cuuint64_t dims[3] = {(cuuint64_t)C, (cuuint64_t)W, (cuuint64_t)H};
    cuuint64_t strides[2] = {(cuuint64_t)C * 4, (cuuint64_t)W * C * 4};
    cuuint32_t box[3] = {CV_KB, CV_PIX, 1}, estr[3] = {1, 1, 1};
    CUresult r = ((PFN_encodeTiled)ctx->encode_tiled)((CUtensorMap *)map_out, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 3, (void *)ptr, dims,
                                                      strides, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B,
                                                      CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    if (r != CUDA_SUCCESS) { set_error("cuTensorMapEncodeTiled(activation %dx%dx%d) failed (CUresult %d)", H, W, C, (int)r); return VO_ERR_CUDA; }
    return VO_OK;
}

// weight map: [C_out][K] (K = taps * C_in), box {32, C_out}
int conv_map_weight(vo_ctx *ctx, void *map_out, const float *ptr, int cout, int ktot) {
    int rc = ensure_encode(ctx);
    if (rc) return rc;
    cuuint64_t dims[2] = {(cuuint64_t)ktot, (cuuint64_t)cout};
    cuuint64_t strides[1] = {(cuuint64_t)ktot * 4};
    cuuint32_t box[2] = {CV_KB, (cuuint32_t)cout}, estr[2] = {1, 1};
    CUresult r = ((PFN_encodeTiled)ctx->encode_tiled)((CUtensorMap *)map_out, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 2, (void *)ptr, dims,
                                                      strides, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B,
                                                      CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    if (r != CUDA_SUCCESS) { set_error("cuTensorMapEncodeTiled(weights %dx%d) failed (CUresult %d)", cout, ktot, (int)r); return VO_ERR_CUDA; }
    return VO_OK;
}

int conv_tc_launch(vo_ctx *ctx, const void *map_a_hi, const void *map_a_lo, const void *map_b_hi, const void *map_b_lo, int H,
                   int W, int cin, int cout, int k, int dil, int pad, int relu, const float *scale, const float *shift,
                   float *out_full, float *out_hi, float *out_lo, cudaStream_t st) {
    VO_REQUIRE(cin % CV_KB == 0 && cin > 0, "conv: C_in must be a multiple of 32 (got %d)", cin);
    VO_REQUIRE(cout == 32 || cout == 64 || cout == 128, "conv: C_out must be 32, 64 or 128 (got %d)", cout);
    VO_REQUIRE((out_hi == nullptr) == (out_lo == nullptr), "conv: out_hi and out_lo go together");
    ConvGeom g{H, W, cin, k, k, dil, pad, ceil_div(W, CV_PIX), relu};
    const int n_tiles = H * g.tiles_x;
    const int grid = n_tiles < ctx->sm_count ? n_tiles : ctx->sm_count;  // persistent: one CTA per SM
#define CV_LAUNCH(CO)                                                                                                  \
    do {                                                                                                               \
        auto kern = conv_tc_kernel<CO>;                                                                                \
        VO_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, CvSmem<CO>::TOTAL));           \
        kern<<<grid, CV_THREADS, CvSmem<CO>::TOTAL, st>>>(*(const CUtensorMap *)map_a_hi, *(const CUtensorMap *)map_a_lo, \
                                                          *(const CUtensorMap *)map_b_hi, *(const CUtensorMap *)map_b_lo, g, \
                                                          scale, shift, out_full, out_hi, out_lo);                     \
    } while (0)
    if (cout == 32) CV_LAUNCH(32);
    else if (cout == 64) CV_LAUNCH(64);
    else CV_LAUNCH(128);
#undef CV_LAUNCH
    VO_LAUNCH_CHECK(ctx);
    return VO_OK;
}

int tf32_split(vo_ctx *ctx, const float *x, size_t n, float *hi, float *lo, cudaStream_t st) {
    VO_REQUIRE((n & 3) == 0, "tf32_split: element count must be a multiple of 4");
    if (n == 0) return VO_OK;
    size_t blocks = (n / 4 + 255) / 256;
    if (blocks > (size_t)ctx->sm_count * 8) blocks = (size_t)ctx->sm_count * 8;
    tf32_split_kernel<<<(unsigned)blocks, 256, 0, st>>>(x, n / 4, hi, lo);
    VO_LAUNCH_CHECK(ctx);
    return VO_OK;
}

}  // namespace vo

/* Stand-alone convolution entry point (tests, other front-ends): one "same" k x k dilated convolution + per-channel
 * scale / shift (bias and batch-norm folded) + optional ReLU.  x, out: NHWC fp32; w: [C_out][k][k][C_in]. */
extern "C" int vo_conv2d(vo_ctx *ctx, const float *x, int H, int W, int cin, const float *w, int cout, int k, int dil,
                         const float *scale, const float *shift, int relu, float *out, void *stream) {
    using namespace vo;
    VO_REQUIRE(ctx && x && w && scale && shift && out, "vo_conv2d: null argument");
    VO_REQUIRE(H > 0 && W > 0 && k >= 1 && k <= 7 && dil >= 1, "vo_conv2d: bad shape");
    // the channel checks of conv_tc_launch, repeated here so that a refused call enqueues nothing (no split kernels)
    VO_REQUIRE(cin % CV_KB == 0 && cin > 0, "vo_conv2d: C_in must be a multiple of 32 (got %d)", cin);
    VO_REQUIRE(cout == 32 || cout == 64 || cout == 128, "vo_conv2d: C_out must be 32, 64 or 128 (got %d)", cout);
    cudaStream_t st = (cudaStream_t)stream;
    const size_t n_act = (size_t)H * W * cin, n_w = (size_t)cout * k * k * cin;
    float *ws;
    int rc;
    if ((rc = ws_get(ctx, WS_SPLIT_A, sizeof(float) * 2 * (n_act + n_w), (void **)&ws))) return rc;
    float *x_hi = ws, *x_lo = ws + n_act, *w_hi = ws + 2 * n_act, *w_lo = w_hi + n_w;
    if ((rc = tf32_split(ctx, x, n_act, x_hi, x_lo, st))) return rc;
    if ((rc = tf32_split(ctx, w, n_w, w_hi, w_lo, st))) return rc;
    CUtensorMap ma_hi, ma_lo, mb_hi, mb_lo;
    if ((rc = conv_map_act(ctx, &ma_hi, x_hi, H, W, cin))) return rc;
    if ((rc = conv_map_act(ctx, &ma_lo, x_lo, H, W, cin))) return rc;
    if ((rc = conv_map_weight(ctx, &mb_hi, w_hi, cout, k * k * cin))) return rc;
    if ((rc = conv_map_weight(ctx, &mb_lo, w_lo, cout, k * k * cin))) return rc;
    return conv_tc_launch(ctx, &ma_hi, &ma_lo, &mb_hi, &mb_lo, H, W, cin, cout, k, dil, ((k - 1) * dil) / 2, relu, scale, shift, out,
                          nullptr, nullptr, st);
}
