// Device-resident keyframe loop: the control flow of VisualOdometry.process_frame
// (VisualOdometry_Stereo.py:232-297) without a host round trip per frame.
//
// Two frame slots live in HBM (keyframe, current frame).  Per pushed frame the stream carries:
//   copy inputs -> current slot | begin_kernel | vo_pipeline(keyframe slot, current slot, B = 1) | policy_kernel |
//   promote_kernel
// With VO_SEQ_GRAPH=1, from the third frame on everything after begin_kernel is ONE CUDA-graph launch: the pipeline's ~16
// kernels, the policy and the promotion are captured once per loop (all per-frame values they need — keypoint counts, frame
// numbers, the history slot, the hypothesis generator's pair offset — live in device memory, written by begin_kernel) and
// replayed.  Opt-in because it buys nothing (measured on a B200, tools/seq_bench.py, identical poses): the loop is bound by the
// latencies of its small kernels and the 1.87 MB depth upload, not by launches — host enqueue 54-62 us per frame against
// 231 (SIFT 2k) / 291-306 us (ORB 5k) of GPU time; graph replay 233 / 306 us per frame against 231 / 291 us with plain launches.
// policy_kernel is one thread of fp64: the 1.5 m x (frame gap) plausibility gate (:270-274), the bad-PnP counter
// (:273, :279, :282, :295), T_cur = T_key @ T_rel (:283) or T_cur = T_key (:290), the keyframe rule
// common_pts < 200 or inliers < 100 or dist > 1.5 (:285-287) and the history entry (:292-293).  promote_kernel copies
// the current slot over the keyframe slot when the policy said so (:295-296) and exits at once otherwise.
#include "common.cuh"
#include <stdlib.h>

struct vo_seq_state {  // device-resident loop state
    int32_t key_n, cur_n;    // keypoint counts of the two slots (the pipeline's n_ref / n_cur)
    int32_t key_id, cur_id;  // reference frame numbers
    int32_t bad_pnp;
    int32_t promote;         // current frame becomes the keyframe
    int32_t slot;            // history index of the current frame (pose / info row the policy writes)
    int32_t pad_;
    long long pair0;         // pair offset of the hypothesis generator for this frame (= slot - 1)
    double T_key[16];        // global pose of the keyframe
};

struct vo_seq {
    vo_ctx *ctx;
    vo_seq_config cfg;
    size_t desc_row;  // bytes per descriptor
    uint8_t *key_desc, *cur_desc;
    float *key_kp, *cur_kp, *key_depth, *cur_depth;
    vo_seq_state *st;
    double *T_rel, *rt;
    int32_t *out4;  // n_matches, n_corr, n_inl, status
    double *poses;  // [max_frames][16]
    int32_t *info;  // [max_frames][6]
    int pushed;
    cudaGraphExec_t graph;     // pipeline + policy + promotion of one frame, captured at the third push
    int graph_state;           // 0 not tried yet, 1 captured, -1 capture failed / disabled (plain launches)
    long long graph_kernels;   // kernel launches one replay stands for (keeps vo_launch_count meaningful)
};

namespace vo {
namespace {

__global__ void seq_begin_kernel(vo_seq_state *st, int n_kp, int frame_id, int first, int slot, double *poses, int32_t *info) {
    st->cur_n = n_kp;
    st->cur_id = frame_id;
    st->slot = slot;
    st->pair0 = (long long)slot - 1;
    if (first) {  // frame 0: identity pose, becomes the keyframe (:233-239)
        st->bad_pnp = 0;
        st->promote = 1;
        st->key_n = n_kp;
        st->key_id = frame_id;
        for (int j = 0; j < 16; ++j) {
            const double v = (j % 5 == 0) ? 1.0 : 0.0;
            st->T_key[j] = v;
            poses[j] = v;
        }
        info[0] = 0; info[1] = 0; info[2] = 0; info[3] = 0; info[4] = frame_id; info[5] = 1;
    }
}

__global__ void seq_policy_kernel(vo_seq_state *st, const double *__restrict__ T_rel, const int32_t *__restrict__ out4,
                                  double max_step_m, int kf_min_common, int kf_min_inliers, double kf_max_dist,
                                  int bad_pnp_limit, double *poses, int32_t *infos) {
    double *pose_out = poses + 16 * (size_t)st->slot;      // the history row of the current frame
    int32_t *info_out = infos + 6 * (size_t)st->slot;
    const int n_matches = out4[0], n_corr = out4[1], n_inl = out4[2], status = out4[3];
    bool ok = status == 0;
    int bad = st->bad_pnp;
    double dist = 0.0;
    if (ok) {
        const double x = T_rel[3], y = T_rel[7], z = T_rel[11];
        dist = sqrt(x * x + y * y + z * z);
        if (!(dist <= max_step_m * (double)(st->cur_id - st->key_id))) {  // "Inside false PnP condition" (:271-274); written NaN-safe
            ok = false;
            ++bad;
        }
    } else {
        ++bad;  // "NO IT IS A BAD PNP"
    }
    double T[16];
    bool promote = false;
    if (ok) {
        bad = 0;
        for (int i = 0; i < 4; ++i)
            for (int j = 0; j < 4; ++j) {
                double s = 0.0;
                for (int q = 0; q < 4; ++q) s += st->T_key[4 * i + q] * T_rel[4 * q + j];
                T[4 * i + j] = s;
            }
        promote = n_corr < kf_min_common || n_inl < kf_min_inliers || dist > kf_max_dist;
    } else {
        for (int j = 0; j < 16; ++j) T[j] = st->T_key[j];
    }
    promote = promote || bad > bad_pnp_limit;
    for (int j = 0; j < 16; ++j) pose_out[j] = T[j];
    info_out[0] = status; info_out[1] = n_matches; info_out[2] = n_corr; info_out[3] = n_inl;
    info_out[4] = st->key_id; info_out[5] = promote ? 1 : 0;
    st->bad_pnp = bad;
    st->promote = promote ? 1 : 0;
    if (promote) {
        st->key_n = st->cur_n;
        st->key_id = st->cur_id;
        for (int j = 0; j < 16; ++j) st->T_key[j] = T[j];
    }
}

// cur slot -> key slot when st->promote is set (three regions, 16-byte vectors, grid-stride)
__global__ void __launch_bounds__(256)
seq_promote_kernel(const vo_seq_state *__restrict__ st, uint4 *__restrict__ kd, const uint4 *__restrict__ cd, size_t nd,
                   uint4 *__restrict__ kk, const uint4 *__restrict__ ck, size_t nk, uint4 *__restrict__ kz,
                   const uint4 *__restrict__ cz, size_t nz) {
    if (!st->promote) return;
    const size_t stride = (size_t)gridDim.x * blockDim.x;
    const size_t t0 = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    for (size_t i = t0; i < nd; i += stride) kd[i] = cd[i];
    for (size_t i = t0; i < nk; i += stride) kk[i] = ck[i];
    for (size_t i = t0; i < nz; i += stride) kz[i] = cz[i];
}

size_t round16(size_t b) { return (b + 15) & ~(size_t)15; }

}  // namespace
}  // namespace vo

extern "C" int vo_seq_create(vo_ctx *ctx, const vo_seq_config *cfg, vo_seq **out) {
    using namespace vo;
    VO_REQUIRE(ctx && cfg && out, "vo_seq_create: null argument");
    *out = nullptr;
    VO_REQUIRE(cfg->pnp_mode == VO_PNP_THROUGHPUT || cfg->pnp_mode == VO_PNP_REFERENCE, "vo_seq_create: unknown pnp_mode %d",
               cfg->pnp_mode);
    VO_REQUIRE(cfg->n_cap > 0 && cfg->H > 0 && cfg->W > 0 && cfg->kp_stride >= 2 &&
                   (cfg->n_hyp > 0 || cfg->pnp_mode == VO_PNP_REFERENCE) && cfg->max_frames > 0,
               "vo_seq_create: bad size");
    vo_seq *s = (vo_seq *)calloc(1, sizeof(vo_seq));
    VO_REQUIRE(s, "vo_seq_create: out of host memory");
    s->ctx = ctx;
    s->cfg = *cfg;
    s->desc_row = cfg->desc_is_f32 ? 128 * sizeof(float) : 32;
    const size_t nd = round16(s->desc_row * cfg->n_cap), nk = round16(sizeof(float) * cfg->kp_stride * cfg->n_cap);
    const size_t nz = round16(sizeof(float) * (size_t)cfg->H * cfg->W);
    // one allocation: key desc | cur desc | key kp | cur kp | key depth | cur depth | state | outputs | history
    const size_t off_kd = 0, off_cd = off_kd + nd, off_kk = off_cd + nd, off_ck = off_kk + nk, off_kz = off_ck + nk,
                 off_cz = off_kz + nz, off_st = off_cz + nz, off_T = off_st + round16(sizeof(vo_seq_state)),
                 off_rt = off_T + 16 * sizeof(double), off_o4 = off_rt + 16 * sizeof(double),
                 off_poses = off_o4 + 16, off_info = off_poses + sizeof(double) * 16 * (size_t)cfg->max_frames,
                 total = off_info + round16(sizeof(int32_t) * 6 * (size_t)cfg->max_frames);
    char *base = nullptr;
    cudaError_t e = cudaMalloc(&base, total);
    if (e != cudaSuccess) {
        free(s);
        set_error("vo_seq_create: cudaMalloc(%zu) -> %s", total, cudaGetErrorString(e));
        return VO_ERR_CUDA;
    }
    cudaMemset(base, 0, total);
    s->key_desc = (uint8_t *)(base + off_kd); s->cur_desc = (uint8_t *)(base + off_cd);
    s->key_kp = (float *)(base + off_kk); s->cur_kp = (float *)(base + off_ck);
    s->key_depth = (float *)(base + off_kz); s->cur_depth = (float *)(base + off_cz);
    s->st = (vo_seq_state *)(base + off_st);
    s->T_rel = (double *)(base + off_T); s->rt = (double *)(base + off_rt);
    s->out4 = (int32_t *)(base + off_o4);
    s->poses = (double *)(base + off_poses); s->info = (int32_t *)(base + off_info);
    *out = s;
    return VO_OK;
}

extern "C" void vo_seq_destroy(vo_seq *seq) {
    if (!seq) return;
    cudaDeviceSynchronize();
    if (seq->graph) cudaGraphExecDestroy(seq->graph);
    cudaFree(seq->key_desc);  // base of the single allocation
    free(seq);
}

extern "C" int vo_seq_frames(const vo_seq *seq) { return seq ? seq->pushed : 0; }

extern "C" int vo_seq_push(vo_seq *seq, const void *desc, const float *kp, int n_kp, const float *depth, int frame_id,
                           void *stream) {
    using namespace vo;
    VO_REQUIRE(seq && desc && kp && depth, "vo_seq_push: null argument");
    const vo_seq_config &c = seq->cfg;
    VO_REQUIRE(n_kp >= 0 && n_kp <= c.n_cap, "vo_seq_push: %d keypoints exceed the capacity %d", n_kp, c.n_cap);
    VO_REQUIRE(seq->pushed < c.max_frames, "vo_seq_push: history full (%d frames)", c.max_frames);
    cudaStream_t st = (cudaStream_t)stream;
    vo_ctx *ctx = seq->ctx;
    const int slot = seq->pushed;
    const size_t nz = sizeof(float) * (size_t)c.H * c.W;
    if (n_kp > 0) {
        VO_CUDA(cudaMemcpyAsync(seq->cur_desc, desc, seq->desc_row * n_kp, cudaMemcpyDefault, st));
        VO_CUDA(cudaMemcpyAsync(seq->cur_kp, kp, sizeof(float) * c.kp_stride * n_kp, cudaMemcpyDefault, st));
    }
    VO_CUDA(cudaMemcpyAsync(seq->cur_depth, depth, nz, cudaMemcpyDefault, st));
    seq_begin_kernel<<<1, 1, 0, st>>>(seq->st, n_kp, frame_id, slot == 0 ? 1 : 0, slot, seq->poses, seq->info);
    VO_LAUNCH_CHECK(ctx);
    const size_t nd16 = round16(seq->desc_row * c.n_cap) / 16, nk16 = round16(sizeof(float) * c.kp_stride * c.n_cap) / 16,
                 nz16 = round16(nz) / 16;
    // everything after begin_kernel: identical launches for every frame (per-frame values are read from seq->st)
    auto body = [&]() -> int {
        if (slot > 0) {
            vo_pipeline_args a;
            memset(&a, 0, sizeof(a));
            a.B = 1; a.n_stride = c.n_cap; a.m_stride = c.n_cap;
            a.n_ref = &seq->st->key_n; a.n_cur = &seq->st->cur_n;
            if (c.desc_is_f32) { a.ref_f32 = (const float *)seq->key_desc; a.cur_f32 = (const float *)seq->cur_desc; }
            else { a.ref_u8 = seq->key_desc; a.cur_u8 = seq->cur_desc; }
            a.norm_or_metric = c.norm_or_metric; a.mode = c.mode; a.precision = c.precision; a.match_param = c.match_param;
            a.ref_kp = seq->key_kp; a.cur_kp = seq->cur_kp; a.kp_stride = c.kp_stride;
            a.depth = seq->key_depth; a.H = c.H; a.W = c.W; a.K_h = c.K;
            a.min_flow_px = c.min_flow_px; a.z_min = c.z_min; a.z_max = c.z_max;
            a.n_hyp = c.n_hyp; a.seed = c.seed; a.pair0 = slot - 1;
            a.thr_px = c.thr_px; a.min_inliers = c.min_inliers; a.refine_iters = c.refine_iters;
            a.pnp_mode = c.pnp_mode; a.ref_restarts = c.ref_restarts; a.ref_iters = c.ref_iters; a.ref_confidence = c.ref_confidence;
            a.T_rel = seq->T_rel; a.rt = seq->rt;
            a.n_matches = seq->out4 + 0; a.n_corr = seq->out4 + 1; a.n_inl = seq->out4 + 2; a.status = seq->out4 + 3;
            int rc = pipeline_impl(ctx, &a, stream, &seq->st->pair0);
            if (rc) return rc;
            seq_policy_kernel<<<1, 1, 0, st>>>(seq->st, seq->T_rel, seq->out4, c.max_step_m, c.kf_min_common,
                                               c.kf_min_inliers, c.kf_max_dist, c.bad_pnp_limit, seq->poses, seq->info);
            VO_LAUNCH_CHECK(ctx);
        }
        seq_promote_kernel<<<ctx->sm_count * 2, 256, 0, st>>>(seq->st, (uint4 *)seq->key_desc, (const uint4 *)seq->cur_desc, nd16,
                                                             (uint4 *)seq->key_kp, (const uint4 *)seq->cur_kp, nk16,
                                                             (uint4 *)seq->key_depth, (const uint4 *)seq->cur_depth, nz16);
        VO_LAUNCH_CHECK(ctx);
        return VO_OK;
    };
    // frames 0 and 1 run plainly (frame 1 sizes every workspace: nothing may allocate during capture); frame 2 captures.
    // A Mode R loop always runs plainly (its graph is not captured).
    if (slot >= 2 && seq->graph_state == 0 && !ctx->prof_on && c.pnp_mode == VO_PNP_THROUGHPUT && getenv("VO_SEQ_GRAPH")) {
        cudaGraph_t g = nullptr;
        const long long l0 = ctx->launches;
        seq->graph_state = -1;
        if (cudaStreamBeginCapture(st, cudaStreamCaptureModeThreadLocal) == cudaSuccess) {
            const int rc = body();
            const cudaError_t e = cudaStreamEndCapture(st, &g);
            if (rc == VO_OK && e == cudaSuccess && g && cudaGraphInstantiate(&seq->graph, g, 0) == cudaSuccess) {
                seq->graph_state = 1;
                seq->graph_kernels = ctx->launches - l0;
            }
            if (g) cudaGraphDestroy(g);
        }
        (void)cudaGetLastError();          // a failed capture must not poison the next launch check
        ctx->launches = l0;                // (captured launches did not run; the replay below counts them)
    }
    if (seq->graph_state == 1 && slot >= 2 && !ctx->prof_on) {
        VO_CUDA(cudaGraphLaunch(seq->graph, st));
        ctx->launches += seq->graph_kernels;
    } else {
        const int rc = body();
        if (rc) return rc;
    }
    seq->pushed = slot + 1;
    return VO_OK;
}

extern "C" int vo_seq_read(vo_seq *seq, int first, int count, double *poses_h, int32_t *info_h, void *stream) {
    using namespace vo;
    VO_REQUIRE(seq, "vo_seq_read: null sequence");
    VO_REQUIRE(first >= 0 && count >= 0 && first + count <= seq->pushed, "vo_seq_read: range [%d, %d) outside the %d pushed frames",
               first, first + count, seq->pushed);
    cudaStream_t st = (cudaStream_t)stream;
    if (count && poses_h)
        VO_CUDA(cudaMemcpyAsync(poses_h, seq->poses + 16 * (size_t)first, sizeof(double) * 16 * count, cudaMemcpyDeviceToHost, st));
    if (count && info_h)
        VO_CUDA(cudaMemcpyAsync(info_h, seq->info + 6 * (size_t)first, sizeof(int32_t) * 6 * count, cudaMemcpyDeviceToHost, st));
    VO_CUDA(cudaStreamSynchronize(st));
    return VO_OK;
}
