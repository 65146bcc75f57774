// Shared host/device helpers for libvo_b200 (sm_100a only).
#pragma once
#ifdef VO_HOST_EMU          // test builds only: the host emulation of the execution model (tests/cuda_emu.h)
#include VO_HOST_EMU
#else
#include <cuda_runtime.h>
#endif
#include <stdint.h>
#include <stdio.h>
#include <stdarg.h>
#include <string.h>
#include "../../include/vo_b200.h"

#if defined(__CUDA_ARCH__) && (__CUDA_ARCH__ < 1000)
#error "libvo_b200 is written for sm_100a (B200) only"
#endif

namespace vo {

// ---- error plumbing (no exceptions cross the C ABI) ----------------------
void set_error(const char *fmt, ...);
const char *get_error();
void clear_error();

#define VO_CUDA(expr)                                                                          \
    do {                                                                                       \
        cudaError_t _e = (expr);                                                               \
        if (_e != cudaSuccess) {                                                               \
            vo::set_error("%s:%d %s -> %s", __FILE__, __LINE__, #expr, cudaGetErrorString(_e)); \
            return VO_ERR_CUDA;                                                                \
        }                                                                                      \
    } while (0)

#define VO_LAUNCH_CHECK(ctx)                                                                      \
    do {                                                                                          \
        cudaError_t _e = cudaGetLastError();                                                      \
        if (_e != cudaSuccess) {                                                                  \
            vo::set_error("%s:%d kernel launch -> %s", __FILE__, __LINE__, cudaGetErrorString(_e)); \
            return VO_ERR_CUDA;                                                                   \
        }                                                                                         \
        (ctx)->launches++;                                                                        \
    } while (0)

#define VO_REQUIRE(cond, ...)          \
    do {                               \
        if (!(cond)) {                 \
            vo::set_error(__VA_ARGS__); \
            return VO_ERR_ARG;         \
        }                              \
    } while (0)

// Order-preserving float <-> uint32 key (larger float => larger key; NaN sorts high,
// callers squash NaN before keying).
__host__ __device__ inline uint32_t float_to_ordered(float f) {
#ifdef __CUDA_ARCH__
    uint32_t u = __float_as_uint(f);
#else
    uint32_t u;
    memcpy(&u, &f, 4);
#endif
    return (u & 0x80000000u) ? ~u : (u | 0x80000000u);
}
__host__ __device__ inline float ordered_to_float(uint32_t k) {
    uint32_t u = (k & 0x80000000u) ? (k & 0x7fffffffu) : ~k;
#ifdef __CUDA_ARCH__
    return __uint_as_float(u);
#else
    float f;
    memcpy(&f, &u, 4);
    return f;
#endif
}

static inline int ceil_div(int a, int b) { return (a + b - 1) / b; }

// Kernel launch on stream `st` with no dynamic shared memory.  VO_LAUNCH_BAR marks kernels that use __syncthreads: on
// the device the two are the same; the host emulation used by the tests gives those kernels real threads.
#ifdef VO_HOST_EMU
#define VO_LAUNCH(kernel, grid, block, st, ...) vo_emu::launch((grid), (block), false, [&]() { kernel(__VA_ARGS__); })
#define VO_LAUNCH_BAR(kernel, grid, block, st, ...) vo_emu::launch((grid), (block), true, [&]() { kernel(__VA_ARGS__); })
#else
#define VO_LAUNCH(kernel, grid, block, st, ...) kernel<<<(grid), (block), 0, (st)>>>(__VA_ARGS__)
#define VO_LAUNCH_BAR(kernel, grid, block, st, ...) kernel<<<(grid), (block), 0, (st)>>>(__VA_ARGS__)
#endif

}  // namespace vo

// Row partial produced by a matcher CTA for one (row, column-split): best and second
// best "score" (smaller is better) and their column indices.  Scores are stored as
// uint32: integer distance for byte descriptors, ordered-float key for float ones.
struct __align__(16) vo_row_partial {
    uint32_t s1, s2;
    int32_t i1, i2;
};

// ---- context ---------------------------------------------------------------
#define VO_WS_SLOTS 10   /* = vo::WS_SLOTS (static_assert below) */
#define VO_TC_PERSIST_KERNELS 6   /* persistent tensor-core matcher kernels: passes 16, 8, 9 x metric */
struct vo_ctx {
    int device;
    int sm_count;
    long long launches;
    // growable workspace regions (device)
    void *ws[VO_WS_SLOTS];
    size_t ws_bytes[VO_WS_SLOTS];
    void *encode_tiled;  // PFN_encodeTiled, resolved by ensure_encode()
    int tc_max_clusters[VO_TC_PERSIST_KERNELS];  // resident clusters of each persistent matcher kernel (0: not asked yet)
    void *prof;          // vo::Profiler* when profiling was ever enabled
    int prof_on;
    // bumped by every workspace (re)allocation: a CUDA graph that baked in ws pointers is stale once it differs from the
    // value stored at capture
    unsigned long long ws_gen;
};

namespace vo {
enum WsSlot { WS_ROWPART = 0, WS_COLKEY = 1, WS_POSES = 2, WS_BESTKEY = 3, WS_SPLIT_A = 4, WS_SPLIT_B = 5, WS_PIPE = 6, WS_NORMS = 7, WS_FIN = 8, WS_ROWPART2 = 9, WS_SLOTS = 10 };
static_assert(WS_SLOTS == VO_WS_SLOTS, "vo_ctx::ws holds one pointer per workspace slot");
// Returns a device buffer of at least `bytes` for `slot`, reallocating (stream-ordered
// free of the old block) only when it must grow.
int ws_get(vo_ctx *ctx, int slot, size_t bytes, void **out);

// stage timing: record an event on `st` that opens stage `stage` (-1 closes the current one)
void prof_mark(vo_ctx *ctx, cudaStream_t st, int stage);
#define VO_PROF(ctx, st, stage)                       \
    do {                                              \
        if ((ctx)->prof_on) vo::prof_mark((ctx), (st), (stage)); \
    } while (0)

// stages (defined in the .cu files)
int match_finalize(vo_ctx *ctx, const vo_row_partial *part, int n_split, const unsigned long long *colkey, int B,
                   int n_stride, int m_stride, const int32_t *n_ref, const int32_t *n_cur, int score_kind, int mode,
                   double param, const float *row_norm, int32_t *out_pairs, float *out_dist, int32_t *out_count,
                   const vo_knn_out *knn, uint8_t *near_tie, cudaStream_t st);
int match_f32_simt(vo_ctx *ctx, const float *ref, const float *cur, int B, int n_stride, int m_stride, int dim,
                   const int32_t *n_ref, const int32_t *n_cur, int metric, vo_row_partial *part, int n_split,
                   unsigned long long *colkey, cudaStream_t st);
// tcgen05 path: owns its split choice and workspaces; returns the partial buffer, split count and
// (L2 only) the per-row squared norms that finalize adds back.
int match_f32_tc(vo_ctx *ctx, const float *ref, const float *cur, int B, int n_stride, int m_stride,
                 const int32_t *n_ref, const int32_t *n_cur, int metric, int passes, int need_cols,
                 vo_row_partial **part_out, int *n_split_out, unsigned long long *colkey, const float **row_norm_out,
                 cudaStream_t st, int src_u8 = 0);
// tensor-core Hamming (VO_NORM_HAMMING_TC): row partials of the 256-bit descriptors and, if need_cols, the column keys
int match_bits_tc(vo_ctx *ctx, const uint8_t *ref, const uint8_t *cur, int B, int n_stride, int m_stride, const int32_t *n_ref,
                  const int32_t *n_cur, int need_cols, int need_second, vo_row_partial **part_out, int *n_split_out,
                  unsigned long long *colkey, cudaStream_t st);
int pick_split(vo_ctx *ctx, int B, int row_blocks, int col_tiles, int min_tiles_per_split);
// resolves cuTensorMapEncodeTiled into ctx->encode_tiled (once per context) for the TMA descriptors of the tcgen05 kernels
int ensure_encode(vo_ctx *ctx);
// Generator key of one pair: hypotheses and bootstrap rows of pair b are drawn from (keys[b].seed, keys[b].pair).  The
// *_impl entries take an optional device array keys[B]; NULL means (seed, pair0 + b).  The keyframe loop passes one key per
// sequence (its own seed, its history slot - 1), written on the device, so a captured graph replays with fresh keys.
struct vo_pair_key {
    uint64_t seed;
    int64_t pair;
};
int hypotheses_impl(vo_ctx *ctx, const int32_t *n_pts, int B, int H, uint64_t seed, int64_t pair0, const vo_pair_key *keys,
                    int32_t *hyp, void *stream);
int pipeline_impl(vo_ctx *ctx, const vo_pipeline_args *a, void *stream, const vo_pair_key *keys);
int bootstrap_impl(vo_ctx *ctx, const int32_t *n_pts, int B, int restarts, int cap, uint64_t seed, int64_t pair0,
                   const vo_pair_key *keys, int32_t *boot, void *stream);
int pnp_ransac_ref_impl(vo_ctx *ctx, const float *xyz, const float *uv, const int32_t *n_pts, int n_fixed, int B, int cap,
                        const double *K_h, const int32_t *boot_idx, int restarts, int iters, float thr_px, double confidence,
                        int min_inliers, int refine_iters, double *rt, double *rvec_tvec, double *T_rel, int32_t *n_inl,
                        int32_t *best, uint8_t *inlier_mask, int32_t *hyp_counts, double *hyp_poses, int32_t *status,
                        int accumulate_status, void *stream);
int pnp_ransac_impl(vo_ctx *ctx, const float *xyz, const float *uv, const int32_t *n_pts, int B, int cap,
                    const double *K_h, const int32_t *hyp, int H, float thr_px, int min_inliers, int refine_iters,
                    double *rt, double *rvec_tvec, double *T_rel, int32_t *n_inl, int32_t *best_h,
                    uint8_t *inlier_mask, int32_t *hyp_counts, int32_t *status, int accumulate_status,
                    void *stream);
int gather_backproject_impl(vo_ctx *ctx, const int32_t *pairs, const int32_t *n_pairs, int B, int pair_cap,
                            const float *ref_kp, const float *cur_kp, int n_stride, int m_stride, int kp_stride,
                            const float *depth, const float *depth_kp, int H, int W, const double *K_h,
                            float min_flow_px, float z_min, float z_max, float *xyz, float *ref_uv, float *cur_uv,
                            int32_t *src, int32_t *n_out, int32_t *status, void *stream);
int fill_u64(vo_ctx *ctx, unsigned long long *p, size_t n, unsigned long long v, cudaStream_t st);

// score kinds understood by match_finalize
enum ScoreKind {
    SCORE_HAMMING = 0,   // s = integer Hamming distance, dist = (float)s
    SCORE_L2SQ_U32 = 1,  // s = integer squared L2, dist = sqrtf((float)s)
    SCORE_L2SQ_F32 = 2,  // s = ordered key of fp32 squared L2, dist = sqrtf
    SCORE_NEGSIM_F32 = 3, // s = ordered key of -similarity, value = sim, dist = sqrtf(2-2 sim)
    SCORE_HAMMING_F32 = 4, // s = ordered key of -(a.b) over -1 / +1 bit vectors = 2 Hamming - 256 (exact fp32): tensor-core Hamming
    // flag, or-ed into the kind: the partials are 8-byte (s1, i1) pairs (vo_row_best) — written by the matchers when nothing
    // reads a row's second best (mutual / plain-NN rules without k-NN output): half the bytes of the row side
    SCORE_COMPACT_PARTIALS = 0x100
};
struct __align__(8) vo_row_best {
    uint32_t s1;
    int32_t i1;
};
}  // namespace vo
