// Context, error plumbing, float-matcher entry point and the batched whole-path pipeline.
#include "common.cuh"
#include <stdlib.h>
#include <vector>

namespace vo {

static thread_local char g_err[512] = "";

void set_error(const char *fmt, ...) {
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(g_err, sizeof(g_err), fmt, ap);
    va_end(ap);
}
const char *get_error() { return g_err; }
void clear_error() { g_err[0] = 0; }

int ws_get(vo_ctx *ctx, int slot, size_t bytes, void **out) {
    if (bytes == 0) bytes = 16;
    if (ctx->ws_bytes[slot] < bytes) {
        // Growth happens during warm-up only.  The old block may still be in use by work
        // queued on a stream, so drain the device before releasing it.
        if (ctx->ws[slot]) {
            VO_CUDA(cudaDeviceSynchronize());
            VO_CUDA(cudaFree(ctx->ws[slot]));
            ctx->ws[slot] = nullptr;
            ctx->ws_bytes[slot] = 0;
        }
        size_t cap = bytes + bytes / 4;
        cap = (cap + 255) & ~(size_t)255;
        ctx->ws_gen++;
        VO_CUDA(cudaMalloc(&ctx->ws[slot], cap));
        ctx->ws_bytes[slot] = cap;
    }
    *out = ctx->ws[slot];
    return VO_OK;
}

struct Profiler {
    std::vector<cudaEvent_t> pool;
    std::vector<int> stage;  // stage opened by pool[i]
    size_t used = 0;
};

void prof_mark(vo_ctx *ctx, cudaStream_t st, int stage) {
    Profiler *p = (Profiler *)ctx->prof;
    if (!p) return;
    if (p->used == p->pool.size()) {
        cudaEvent_t e;
        if (cudaEventCreate(&e) != cudaSuccess) return;
        p->pool.push_back(e);
        p->stage.push_back(-1);
    }
    p->stage[p->used] = stage;
    cudaEventRecord(p->pool[p->used], st);
    p->used++;
}

int pick_split(vo_ctx *ctx, int B, int row_blocks, int col_tiles, int min_tiles_per_split) {
    int n_split = 1;
    const int want = 2 * ctx->sm_count;
    const int have = B * row_blocks;
    if (have < want) n_split = ceil_div(want, have > 0 ? have : 1);
    int max_split = col_tiles / min_tiles_per_split;
    if (max_split < 1) max_split = 1;
    if (n_split > max_split) n_split = max_split;
    if (n_split > 64) n_split = 64;
    return n_split;
}

int ensure_encode(vo_ctx *ctx) {
    if (ctx->encode_tiled) return VO_OK;
    void *fn = nullptr;
    cudaDriverEntryPointQueryResult qres;
    VO_CUDA(cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &fn, cudaEnableDefault, &qres));
    if (qres != cudaDriverEntryPointSuccess || !fn) {
        set_error("cuTensorMapEncodeTiled is not available from this driver");
        return VO_ERR_UNSUPPORTED;
    }
    ctx->encode_tiled = fn;
    return VO_OK;
}

}  // namespace vo

extern "C" int vo_abi_version(void) { return VO_ABI_VERSION; }
extern "C" const char *vo_last_error(void) { return vo::get_error(); }
extern "C" long long vo_launch_count(const vo_ctx *ctx) { return ctx ? ctx->launches : 0; }
extern "C" unsigned long long vo_workspace_generation(const vo_ctx *ctx) { return ctx ? ctx->ws_gen : 0; }

extern "C" int vo_create(int device, vo_ctx **out) {
    using namespace vo;
    VO_REQUIRE(out, "vo_create: null out");
    *out = nullptr;
    int count = 0;
    VO_CUDA(cudaGetDeviceCount(&count));
    VO_REQUIRE(device >= 0 && device < count, "vo_create: device %d out of range (%d visible)", device, count);
    cudaDeviceProp prop;
    VO_CUDA(cudaGetDeviceProperties(&prop, device));
    if (prop.major != 10) {
        set_error("vo_create: device %d is sm_%d%d; libvo_b200 carries sm_100a code only (no fallback path)", device,
                  prop.major, prop.minor);
        return VO_ERR_UNSUPPORTED;
    }
    VO_CUDA(cudaSetDevice(device));
    vo_ctx *ctx = (vo_ctx *)calloc(1, sizeof(vo_ctx));
    VO_REQUIRE(ctx, "vo_create: out of host memory");
    ctx->device = device;
    ctx->sm_count = prop.multiProcessorCount;
    *out = ctx;
    return VO_OK;
}

extern "C" int vo_profile_enable(vo_ctx *ctx, int on) {
    using namespace vo;
    VO_REQUIRE(ctx, "vo_profile_enable: null ctx");
    if (on && !ctx->prof) ctx->prof = new Profiler();
    ctx->prof_on = on ? 1 : 0;
    return VO_OK;
}

extern "C" int vo_profile_collect(vo_ctx *ctx, double *ms, long long *counts) {
    using namespace vo;
    VO_REQUIRE(ctx && ms && counts, "vo_profile_collect: null argument");
    for (int i = 0; i < VO_STAGE_COUNT; ++i) { ms[i] = 0.0; counts[i] = 0; }
    Profiler *p = (Profiler *)ctx->prof;
    if (!p) return VO_OK;
    VO_CUDA(cudaDeviceSynchronize());
    for (size_t i = 0; i + 1 < p->used; ++i) {
        const int sg = p->stage[i];
        if (sg < 0 || sg >= VO_STAGE_COUNT) continue;
        float t = 0.f;
        if (cudaEventElapsedTime(&t, p->pool[i], p->pool[i + 1]) == cudaSuccess) {
            ms[sg] += t;
            counts[sg] += 1;
        }
    }
    p->used = 0;
    return VO_OK;
}

extern "C" void vo_destroy(vo_ctx *ctx) {
    if (!ctx) return;
    cudaSetDevice(ctx->device);
    cudaDeviceSynchronize();
    if (ctx->prof) {
        vo::Profiler *p = (vo::Profiler *)ctx->prof;
        for (cudaEvent_t e : p->pool) cudaEventDestroy(e);
        delete p;
    }
    for (int i = 0; i < vo::WS_SLOTS; ++i)
        if (ctx->ws[i]) cudaFree(ctx->ws[i]);
    free(ctx);
}

extern "C" int vo_match_f32(vo_ctx *ctx, const float *ref, const float *cur, int B, int n_stride, int m_stride,
                            const int32_t *n_ref, const int32_t *n_cur, int dim, int metric, int mode, double param,
                            int precision, int32_t *out_pairs, float *out_dist, int32_t *out_count,
                            const vo_knn_out *knn, uint8_t *near_tie, void *stream) {
    using namespace vo;
    VO_REQUIRE(ctx && ref && cur, "vo_match_f32: null argument");
    VO_REQUIRE(metric == VO_METRIC_L2 || metric == VO_METRIC_COSINE, "vo_match_f32: bad metric %d", metric);
    VO_REQUIRE(mode >= VO_MODE_RATIO && mode <= VO_MODE_NN, "vo_match_f32: bad mode %d", mode);
    VO_REQUIRE(!((mode == VO_MODE_THRESH || mode == VO_MODE_THRESH_MUTUAL) && metric != VO_METRIC_COSINE),
               "vo_match_f32: similarity-threshold modes need VO_METRIC_COSINE");
    VO_REQUIRE(precision >= VO_PREC_TF32X3 && precision <= VO_PREC_F16X3, "vo_match_f32: bad precision %d", precision);
    VO_REQUIRE(B >= 0 && n_stride >= 0 && m_stride >= 0 && dim > 0, "vo_match_f32: bad size");
    VO_REQUIRE(out_pairs && out_count, "vo_match_f32: null output");
    VO_REQUIRE(((uintptr_t)ref % 16) == 0 && ((uintptr_t)cur % 16) == 0, "vo_match_f32: descriptors must be 16B aligned");
    cudaStream_t st = (cudaStream_t)stream;
    if (B == 0) return VO_OK;
    if (n_stride == 0 || m_stride == 0) {
        VO_CUDA(cudaMemsetAsync(out_count, 0, sizeof(int32_t) * B, st));
        return VO_OK;
    }
    int rc;
    unsigned long long *colkey;
    if ((rc = ws_get(ctx, WS_COLKEY, sizeof(unsigned long long) * (size_t)B * m_stride, (void **)&colkey))) return rc;
    VO_PROF(ctx, st, VO_STAGE_FILL);
    if ((rc = fill_u64(ctx, colkey, (size_t)B * m_stride, ~0ull, st))) return rc;
    vo_row_partial *part;
    const float *row_norm = nullptr;
    int n_split;
    if (precision == VO_PREC_FP32_SIMT) {
        n_split = pick_split(ctx, B, ceil_div(n_stride, 64), ceil_div(m_stride, 64), 4);
        if ((rc = ws_get(ctx, WS_ROWPART, sizeof(vo_row_partial) * (size_t)B * n_split * n_stride, (void **)&part))) return rc;
        VO_PROF(ctx, st, VO_STAGE_MATCH);
        if ((rc = match_f32_simt(ctx, ref, cur, B, n_stride, m_stride, dim, n_ref, n_cur, metric, part, n_split, colkey, st)))
            return rc;
    } else {
        VO_REQUIRE(dim == 128, "vo_match_f32: the tcgen05 path takes 128-d descriptors (got %d); use VO_PREC_FP32_SIMT", dim);
        // the column arg-max feeds the mutual rules and the raw col_idx output only
        const int need_cols = mode == VO_MODE_MUTUAL || mode == VO_MODE_RATIO_MUTUAL || mode == VO_MODE_THRESH_MUTUAL ||
                              (knn && knn->col_idx);
        if ((rc = match_f32_tc(ctx, ref, cur, B, n_stride, m_stride, n_ref, n_cur, metric,
                               precision == VO_PREC_TF32X3 ? 3 : (precision == VO_PREC_F16X1 ? 16 : (precision == VO_PREC_F16X3 ? 48 : 1)), need_cols, &part, &n_split, colkey, &row_norm, st)))
            return rc;
    }
    return match_finalize(ctx, part, n_split, colkey, B, n_stride, m_stride, n_ref, n_cur,
                          metric == VO_METRIC_L2 ? SCORE_L2SQ_F32 : SCORE_NEGSIM_F32, mode, param, row_norm, out_pairs,
                          out_dist, out_count, knn, near_tie, st);
}

// ---------------------------------------------------------------- whole-path pipeline
extern "C" int vo_pipeline(vo_ctx *ctx, const vo_pipeline_args *a, void *stream) { return vo::pipeline_impl(ctx, a, stream, nullptr); }

// keys (optional, device vo_pair_key[B]): the hypothesis / bootstrap generator key of each pair, read on the device instead of
// (a->seed, a->pair0 + b) (vo_seq_*: one key per sequence)
int vo::pipeline_impl(vo_ctx *ctx, const vo_pipeline_args *a, void *stream, const vo_pair_key *keys) {
    using namespace vo;
    VO_REQUIRE(ctx && a, "vo_pipeline: null argument");
    const bool u8 = a->ref_u8 && a->cur_u8, f32 = a->ref_f32 && a->cur_f32;
    VO_REQUIRE(u8 != f32, "vo_pipeline: give exactly one descriptor pair (u8 or f32)");
    VO_REQUIRE(a->pnp_mode == VO_PNP_THROUGHPUT || a->pnp_mode == VO_PNP_REFERENCE, "vo_pipeline: unknown pnp_mode %d", a->pnp_mode);
    const bool ref = a->pnp_mode == VO_PNP_REFERENCE;
    VO_REQUIRE(a->B >= 0 && a->n_stride > 0 && a->m_stride > 0 && (ref || a->n_hyp > 0), "vo_pipeline: bad size");
    VO_REQUIRE(a->ref_restarts >= 0 && a->ref_iters >= 0 && a->ref_confidence >= 0.0, "vo_pipeline: negative Mode R parameter");
    VO_REQUIRE(a->ref_kp && a->cur_kp && (a->depth || a->depth_kp) && a->K_h, "vo_pipeline: null geometry input");
    VO_REQUIRE(a->T_rel && a->n_matches && a->n_corr && a->n_inl && a->status, "vo_pipeline: null output");
    if (a->B == 0) return VO_OK;
    const int B = a->B, cap = a->n_stride, H = a->n_hyp;
    const int restarts = a->ref_restarts ? a->ref_restarts : 3, iters = a->ref_iters ? a->ref_iters : 100;
    const double confidence = a->ref_confidence != 0.0 ? a->ref_confidence : 0.99;
    // scratch: pairs | xyz | ref_uv | cur_uv | hyp (Mode T: [B][H][4]) or bootstrap rows (Mode R: [B][restarts][cap])
    const size_t off_pairs = 0;
    const size_t off_xyz = off_pairs + sizeof(int32_t) * 2 * (size_t)B * cap;
    const size_t off_ruv = off_xyz + sizeof(float) * 3 * (size_t)B * cap;
    const size_t off_cuv = off_ruv + sizeof(float) * 2 * (size_t)B * cap;
    size_t off_hyp = off_cuv + sizeof(float) * 2 * (size_t)B * cap;
    off_hyp = (off_hyp + 255) & ~(size_t)255;
    const size_t total = off_hyp + sizeof(int32_t) * (ref ? (size_t)B * restarts * cap : 4 * (size_t)B * H);
    char *ws;
    int rc;
    if ((rc = ws_get(ctx, WS_PIPE, total, (void **)&ws))) return rc;
    int32_t *pairs = (int32_t *)(ws + off_pairs);
    float *xyz = (float *)(ws + off_xyz), *ruv = (float *)(ws + off_ruv), *cuv = (float *)(ws + off_cuv);
    int32_t *hyp = (int32_t *)(ws + off_hyp);

    if (u8)
        rc = vo_match_u8(ctx, a->ref_u8, a->cur_u8, B, a->n_stride, a->m_stride, a->n_ref, a->n_cur, a->u8_bytes ? a->u8_bytes : 32,
                         a->norm_or_metric, a->mode, a->match_param, pairs, nullptr, a->n_matches, nullptr, stream);
    else
        rc = vo_match_f32(ctx, a->ref_f32, a->cur_f32, B, a->n_stride, a->m_stride, a->n_ref, a->n_cur, 128,
                          a->norm_or_metric, a->mode, a->match_param, a->precision, pairs, nullptr, a->n_matches,
                          nullptr, nullptr, stream);
    if (rc) return rc;
    if ((rc = gather_backproject_impl(ctx, pairs, a->n_matches, B, cap, a->ref_kp, a->cur_kp, a->n_stride, a->m_stride,
                                      a->kp_stride, a->depth_kp ? nullptr : a->depth, a->depth_kp, a->H, a->W, a->K_h,
                                      a->min_flow_px, a->z_min, a->z_max, xyz, ruv, cuv, nullptr, a->n_corr, a->status,
                                      stream)))
        return rc;
    if (ref) {
        if ((rc = bootstrap_impl(ctx, a->n_corr, B, restarts, cap, a->seed, a->pair0, keys, hyp, stream))) return rc;
        return pnp_ransac_ref_impl(ctx, xyz, cuv, a->n_corr, 0, B, cap, a->K_h, hyp, restarts, iters, a->thr_px, confidence,
                                   a->min_inliers, a->refine_iters, a->rt, nullptr, a->T_rel, a->n_inl, nullptr, nullptr, nullptr,
                                   nullptr, a->status, 1, stream);
    }
    if ((rc = hypotheses_impl(ctx, a->n_corr, B, H, a->seed, a->pair0, keys, hyp, stream))) return rc;
    return pnp_ransac_impl(ctx, xyz, cuv, a->n_corr, B, cap, a->K_h, hyp, H, a->thr_px, a->min_inliers,
                           a->refine_iters, a->rt, nullptr, a->T_rel, a->n_inl, nullptr, nullptr, nullptr, a->status,
                           1, stream);
}
