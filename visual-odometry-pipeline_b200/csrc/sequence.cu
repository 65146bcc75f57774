// Device-resident keyframe loop: the control flow of VisualOdometry.process_frame
// (VisualOdometry_Stereo.py:232-297) without a host round trip per frame, for S independent sequences in lock-step.
//
// Each sequence owns two frame slots in HBM (keyframe, current frame), stored sequence-major ([S][n_cap][D] descriptors,
// [S][n_cap][kp_stride] keypoints, [S][H][W] depth), so the S current frames of a step are one vo_pipeline batch against the
// S keyframes.  A keyframe decision depends on the previous frame, so frames of one sequence cannot be batched; frames of
// different sequences at the same step can, and the policy of a sequence does not look at its neighbours.  Per step the
// stream carries:
//   copy inputs -> current slots | begin_kernel | vo_pipeline(keyframe slots, current slots, B = S) | policy_kernel |
//   promote_kernel
// begin_kernel (one thread per sequence) writes the per-sequence state and the counts the pipeline reads: a sequence with no
// frame at this step (n_kp < 0) or at its first frame gets count 0 on both sides, so it costs no matches, and the policy
// skips it.  With device-side counts (vo_seq_push_all_dev) begin_kernel also reads each present sequence's count from the
// extractor's [S][2] (rows, flags) array, clamps it to n_cap and counts the frames that lost rows.  The generator key of sequence q is (seeds[q], slot_q - 1) (common.cuh: vo_pair_key), what a single loop created
// with seed = seeds[q] draws, so each sequence's poses equal that loop's bit for bit.  S = 1 is vo_seq_push's loop.
// With VO_SEQ_GRAPH=1 (Mode T only), once a step has run the pipeline plainly (which sizes every workspace: nothing may
// allocate during capture), everything after begin_kernel is ONE CUDA-graph launch: the pipeline's ~16 kernels, the policy
// and the promotion are captured once (all per-step values they need — counts, frame numbers, history slots, generator keys —
// live in device memory, written by begin_kernel) and replayed.  The graph bakes in the context's workspace pointers; any
// later call that grows a workspace (another loop, a larger ops.* call on the same vo_ctx) frees the old block, so a replay
// first compares vo_ctx::ws_gen with the value stored at capture and re-captures when they differ.  Opt-in because it buys
// nothing at S = 1 (measured on a B200, tools/seq_bench.py, identical poses): the loop is bound by the latencies of its small
// kernels and the 1.87 MB depth upload, not by launches — host enqueue 54-62 us per frame against 231 (SIFT 2k) /
// 291-306 us (ORB 5k) of GPU time; graph replay 233 / 306 us per frame against 231 / 291 us with plain launches.
// policy_kernel is one thread of fp64 per sequence: the 1.5 m x (frame gap) plausibility gate (:270-274), the bad-PnP
// counter (:273, :279, :282, :295), T_cur = T_key @ T_rel (:283) or T_cur = T_key (:290), the keyframe rule
// common_pts < 200 or inliers < 100 or dist > 1.5 (:285-287) and the history entry (:292-293).  promote_kernel copies
// the current slot over the keyframe slot of every sequence whose promote flag is set (:295-296).
#include "common.cuh"
#include <stdlib.h>

struct vo_seq_state {  // device-resident state of one sequence
    int32_t key_n, cur_n;    // keypoint counts of the two slots
    int32_t key_id, cur_id;  // reference frame numbers
    int32_t bad_pnp;
    int32_t promote;         // current frame becomes the keyframe
    int32_t slot;            // history index of the current frame (pose / info row the policy writes)
    int32_t active;          // the current frame is matched against the keyframe at this step (the policy runs)
    double T_key[16];        // global pose of the keyframe
};

struct vo_seq {
    vo_ctx *ctx;
    vo_seq_config cfg;
    int S;            // sequences
    size_t desc_row;  // bytes per descriptor
    size_t nd, nk, nz;  // bytes of one sequence's descriptor / keypoint / depth slot
    uint8_t *key_desc, *cur_desc;
    float *key_kp, *cur_kp, *key_depth, *cur_depth;
    vo_seq_state *st;      // [S]
    int32_t *step_in;      // [3][S]: n_kp (< 0: no frame), frame id, history slot of this step (copied from the host)
    int32_t *n_eff;        // [2][S]: key / current counts the pipeline reads (0 for inactive sequences)
    vo::vo_pair_key *keys; // [S]
    double *T_rel, *rt;    // [S][16], [S][12]
    int32_t *out4;         // [4][S]: n_matches, n_corr, n_inl, status
    int32_t *lost;         // [S]: frames whose device-side count was clamped to n_cap or came with a non-zero flag word
    double *poses;         // [S][max_frames][16]
    int32_t *info;         // [S][max_frames][6]
    int32_t *step_h;       // host [3][S] staging of step_in (pageable: the copy has read it when cudaMemcpyAsync returns)
    int *pushed;           // host [S]: frames pushed per sequence
    int warm;              // a step ran the pipeline plainly: every workspace this loop needs exists
    cudaGraphExec_t graph;     // pipeline + policy + promotion of one step
    int graph_state;           // 0 not captured, 1 captured, -1 capture failed (plain launches)
    int graph_captures;        // successful captures (the first one and every re-capture after a workspace reallocation)
    unsigned long long graph_gen;  // ctx->ws_gen at capture
    long long graph_kernels;   // kernel launches one replay stands for (keeps vo_launch_count meaningful)
};

namespace vo {
namespace {

// n_kp_d: NULL (counts come from step_in) or the device int32 [S][2] (rows, flags) array of vo_seq_push_all_dev, read for
// the present sequences (step_in[q] == 0).
__global__ void seq_begin_kernel(vo_seq_state *sts, int S, const int32_t *__restrict__ step_in, const int32_t *__restrict__ n_kp_d,
                                 int n_cap, int32_t *__restrict__ lost, int32_t *__restrict__ n_eff,
                                 vo_pair_key *__restrict__ keys, double *poses, int32_t *info, int max_frames) {
    const int q = blockIdx.x * blockDim.x + threadIdx.x;
    if (q >= S) return;
    vo_seq_state *st = sts + q;
    int n_kp = step_in[q];
    const int frame_id = step_in[S + q], slot = step_in[2 * S + q];
    st->active = 0;
    n_eff[q] = 0;
    n_eff[S + q] = 0;
    if (n_kp < 0) {  // no frame of this sequence at this step: nothing of it is touched
        st->promote = 0;
        return;
    }
    if (n_kp_d) {
        const int n = n_kp_d[2 * q], flags = n_kp_d[2 * q + 1];
        n_kp = min(max(n, 0), n_cap);
        if (n > n_cap || flags != 0) lost[q]++;
    }
    st->cur_n = n_kp;
    st->cur_id = frame_id;
    st->slot = slot;
    keys[q].pair = (int64_t)slot - 1;
    if (slot == 0) {  // frame 0: identity pose, becomes the keyframe (:233-239)
        st->bad_pnp = 0;
        st->promote = 1;
        st->key_n = n_kp;
        st->key_id = frame_id;
        double *pose = poses + (size_t)q * max_frames * 16;
        int32_t *inf = info + (size_t)q * max_frames * 6;
        for (int j = 0; j < 16; ++j) {
            const double v = (j % 5 == 0) ? 1.0 : 0.0;
            st->T_key[j] = v;
            pose[j] = v;
        }
        inf[0] = 0; inf[1] = 0; inf[2] = 0; inf[3] = 0; inf[4] = frame_id; inf[5] = 1;
    } else {
        st->active = 1;
        n_eff[q] = st->key_n;
        n_eff[S + q] = n_kp;
    }
}

__global__ void seq_policy_kernel(vo_seq_state *sts, int S, const double *__restrict__ T_rels, const int32_t *__restrict__ out4,
                                  double max_step_m, int kf_min_common, int kf_min_inliers, double kf_max_dist,
                                  int bad_pnp_limit, double *poses, int32_t *infos, int max_frames) {
    const int q = blockIdx.x * blockDim.x + threadIdx.x;
    if (q >= S) return;
    vo_seq_state *st = sts + q;
    if (!st->active) return;
    const double *T_rel = T_rels + 16 * (size_t)q;
    double *pose_out = poses + 16 * ((size_t)q * max_frames + st->slot);      // the history row of the current frame
    int32_t *info_out = infos + 6 * ((size_t)q * max_frames + st->slot);
    const int n_matches = out4[q], n_corr = out4[S + q], n_inl = out4[2 * S + q], status = out4[3 * S + q];
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
                for (int k = 0; k < 4; ++k) s += st->T_key[4 * i + k] * T_rel[4 * k + j];
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

// one region of a sequence: 16-byte vectors when the region's size allows (then every sequence's region is 16-byte aligned), else
// 4-byte words (a [n_cap][3] keypoint slot with odd n_cap, an image with H * W odd)
__device__ __forceinline__ void copy_region(void *dst, const void *src, size_t bytes, size_t t0, size_t stride) {
    if ((bytes & 15) == 0) {
        uint4 *d = (uint4 *)dst;
        const uint4 *s = (const uint4 *)src;
        for (size_t i = t0; i < bytes / 16; i += stride) d[i] = s[i];
    } else {
        uint32_t *d = (uint32_t *)dst;
        const uint32_t *s = (const uint32_t *)src;
        for (size_t i = t0; i < bytes / 4; i += stride) d[i] = s[i];
    }
}

// cur slot -> key slot of sequence blockIdx.y when its promote flag is set (three regions, grid-stride over blockIdx.x)
__global__ void __launch_bounds__(256)
seq_promote_kernel(const vo_seq_state *__restrict__ sts, uint8_t *kd, const uint8_t *cd, size_t nd, uint8_t *kk,
                   const uint8_t *ck, size_t nk, uint8_t *kz, const uint8_t *cz, size_t nz) {
    const size_t q = blockIdx.y;
    if (!sts[q].promote) return;
    const size_t stride = (size_t)gridDim.x * blockDim.x;
    const size_t t0 = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    copy_region(kd + q * nd, cd + q * nd, nd, t0, stride);
    copy_region(kk + q * nk, ck + q * nk, nk, t0, stride);
    copy_region(kz + q * nz, cz + q * nz, nz, t0, stride);
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
                   (cfg->n_hyp > 0 || cfg->pnp_mode == VO_PNP_REFERENCE) && cfg->max_frames > 0 && cfg->n_seqs >= 0,
               "vo_seq_create: bad size");
    // seq_promote_kernel runs one grid row per sequence (gridDim.y <= 65535)
    VO_REQUIRE(cfg->n_seqs <= 65535, "vo_seq_create: %d sequences exceed the limit of 65535", cfg->n_seqs);
    const int S = cfg->n_seqs > 1 ? cfg->n_seqs : 1;
    vo_seq *s = (vo_seq *)calloc(1, sizeof(vo_seq));
    VO_REQUIRE(s, "vo_seq_create: out of host memory");
    s->ctx = ctx;
    s->cfg = *cfg;
    s->cfg.seeds = nullptr;  // copied below; the caller's array need not outlive this call
    s->S = S;
    s->desc_row = cfg->desc_is_f32 ? 128 * sizeof(float) : 32;
    s->nd = s->desc_row * cfg->n_cap;
    s->nk = sizeof(float) * cfg->kp_stride * (size_t)cfg->n_cap;
    s->nz = sizeof(float) * (size_t)cfg->H * cfg->W;
    s->step_h = (int32_t *)calloc(3 * (size_t)S, sizeof(int32_t));
    s->pushed = (int *)calloc(S, sizeof(int));
    vo_pair_key *keys_h = (vo_pair_key *)calloc(S, sizeof(vo_pair_key));
    if (!s->step_h || !s->pushed || !keys_h) {
        free(keys_h); free(s->step_h); free(s->pushed); free(s);
        set_error("vo_seq_create: out of host memory");
        return VO_ERR_ARG;
    }
    for (int q = 0; q < S; ++q) keys_h[q].seed = cfg->seeds ? cfg->seeds[q] : cfg->seed + (uint64_t)q;
    const size_t nd = round16(s->nd * S), nk = round16(s->nk * S), nz = round16(s->nz * S);
    const size_t mf = (size_t)cfg->max_frames;
    // one allocation: key desc | cur desc | key kp | cur kp | key depth | cur depth | state | step inputs | counts | keys |
    // outputs | lost-frame counters | history
    const size_t off_kd = 0, off_cd = off_kd + nd, off_kk = off_cd + nd, off_ck = off_kk + nk, off_kz = off_ck + nk,
                 off_cz = off_kz + nz, off_st = off_cz + nz, off_in = off_st + round16(sizeof(vo_seq_state) * S),
                 off_ne = off_in + round16(sizeof(int32_t) * 3 * S), off_keys = off_ne + round16(sizeof(int32_t) * 2 * S),
                 off_T = off_keys + round16(sizeof(vo_pair_key) * S), off_rt = off_T + sizeof(double) * 16 * S,
                 off_o4 = off_rt + sizeof(double) * 12 * S, off_lost = off_o4 + round16(sizeof(int32_t) * 4 * S),
                 off_poses = off_lost + round16(sizeof(int32_t) * S),
                 off_info = off_poses + sizeof(double) * 16 * mf * S, total = off_info + round16(sizeof(int32_t) * 6 * mf * S);
    char *base = nullptr;
    cudaError_t e = cudaMalloc(&base, total);
    if (e == cudaSuccess) e = cudaMemset(base, 0, total);
    if (e == cudaSuccess) e = cudaMemcpy(base + off_keys, keys_h, sizeof(vo_pair_key) * S, cudaMemcpyHostToDevice);
    free(keys_h);
    if (e != cudaSuccess) {
        if (base) cudaFree(base);
        free(s->step_h); free(s->pushed); free(s);
        set_error("vo_seq_create: %zu device bytes -> %s", total, cudaGetErrorString(e));
        return VO_ERR_CUDA;
    }
    s->key_desc = (uint8_t *)(base + off_kd); s->cur_desc = (uint8_t *)(base + off_cd);
    s->key_kp = (float *)(base + off_kk); s->cur_kp = (float *)(base + off_ck);
    s->key_depth = (float *)(base + off_kz); s->cur_depth = (float *)(base + off_cz);
    s->st = (vo_seq_state *)(base + off_st);
    s->step_in = (int32_t *)(base + off_in); s->n_eff = (int32_t *)(base + off_ne);
    s->keys = (vo_pair_key *)(base + off_keys);
    s->T_rel = (double *)(base + off_T); s->rt = (double *)(base + off_rt);
    s->out4 = (int32_t *)(base + off_o4);
    s->lost = (int32_t *)(base + off_lost);
    s->poses = (double *)(base + off_poses); s->info = (int32_t *)(base + off_info);
    *out = s;
    return VO_OK;
}

extern "C" void vo_seq_destroy(vo_seq *seq) {
    if (!seq) return;
    cudaDeviceSynchronize();
    if (seq->graph) cudaGraphExecDestroy(seq->graph);
    cudaFree(seq->key_desc);  // base of the single allocation
    free(seq->step_h);
    free(seq->pushed);
    free(seq);
}

extern "C" int vo_seq_frames_at(const vo_seq *seq, int q) { return seq && q >= 0 && q < seq->S ? seq->pushed[q] : 0; }
extern "C" int vo_seq_frames(const vo_seq *seq) { return vo_seq_frames_at(seq, 0); }
extern "C" int vo_seq_graph_captures(const vo_seq *seq) { return seq ? seq->graph_captures : 0; }

namespace vo {
namespace {

// One step.  desc / kp / depth: `rows` keypoint rows of every sequence's slot, sequence-major with stride n_cap (vo_seq_push
// copies only the n_kp rows of its one sequence).  n_kp_d: NULL, or device counts (then n_kp_h[q] is 0 for a present
// sequence, -1 for an absent one).  All checks come before anything is enqueued.
int seq_step(vo_seq *seq, const void *desc, const float *kp, const int32_t *n_kp_h, const int32_t *n_kp_d, const float *depth,
             const int32_t *frame_id_h, size_t rows, void *stream, const char *who) {
    const vo_seq_config &c = seq->cfg;
    const int S = seq->S;
    bool any_active = false;
    for (int q = 0; q < S; ++q) {
        VO_REQUIRE(n_kp_h[q] <= c.n_cap, "%s: sequence %d: %d keypoints exceed the capacity %d", who, q, n_kp_h[q], c.n_cap);
        if (n_kp_h[q] < 0) continue;
        VO_REQUIRE(seq->pushed[q] < c.max_frames, "%s: sequence %d: history full (%d frames)", who, q, c.max_frames);
        any_active = any_active || seq->pushed[q] > 0;
    }
    cudaStream_t st = (cudaStream_t)stream;
    vo_ctx *ctx = seq->ctx;
    for (int q = 0; q < S; ++q) {
        seq->step_h[q] = n_kp_h[q];
        seq->step_h[S + q] = frame_id_h[q];
        seq->step_h[2 * S + q] = seq->pushed[q];
    }
    if (rows > 0) {
        VO_CUDA(cudaMemcpyAsync(seq->cur_desc, desc, seq->desc_row * rows, cudaMemcpyDefault, st));
        VO_CUDA(cudaMemcpyAsync(seq->cur_kp, kp, sizeof(float) * c.kp_stride * rows, cudaMemcpyDefault, st));
    }
    VO_CUDA(cudaMemcpyAsync(seq->cur_depth, depth, seq->nz * S, cudaMemcpyDefault, st));
    VO_CUDA(cudaMemcpyAsync(seq->step_in, seq->step_h, sizeof(int32_t) * 3 * S, cudaMemcpyHostToDevice, st));
    const int threads = S < 64 ? 32 : 64, blocks = ceil_div(S, threads);
    seq_begin_kernel<<<blocks, threads, 0, st>>>(seq->st, S, seq->step_in, n_kp_d, c.n_cap, seq->lost, seq->n_eff, seq->keys,
                                                 seq->poses, seq->info, c.max_frames);
    VO_LAUNCH_CHECK(ctx);
    // everything after begin_kernel: identical launches for every step (per-step values are read from device memory)
    auto body = [&](bool run_pipeline) -> int {
        if (run_pipeline) {
            vo_pipeline_args a;
            memset(&a, 0, sizeof(a));
            a.B = S; a.n_stride = c.n_cap; a.m_stride = c.n_cap;
            a.n_ref = seq->n_eff; a.n_cur = seq->n_eff + S;
            if (c.desc_is_f32) { a.ref_f32 = (const float *)seq->key_desc; a.cur_f32 = (const float *)seq->cur_desc; }
            else { a.ref_u8 = seq->key_desc; a.cur_u8 = seq->cur_desc; }
            a.norm_or_metric = c.norm_or_metric; a.mode = c.mode; a.precision = c.precision; a.match_param = c.match_param;
            a.ref_kp = seq->key_kp; a.cur_kp = seq->cur_kp; a.kp_stride = c.kp_stride;
            a.depth = seq->key_depth; a.H = c.H; a.W = c.W; a.K_h = c.K;
            a.min_flow_px = c.min_flow_px; a.z_min = c.z_min; a.z_max = c.z_max;
            a.n_hyp = c.n_hyp; a.seed = c.seed;
            a.thr_px = c.thr_px; a.min_inliers = c.min_inliers; a.refine_iters = c.refine_iters;
            a.pnp_mode = c.pnp_mode; a.ref_restarts = c.ref_restarts; a.ref_iters = c.ref_iters; a.ref_confidence = c.ref_confidence;
            a.T_rel = seq->T_rel; a.rt = seq->rt;
            a.n_matches = seq->out4; a.n_corr = seq->out4 + S; a.n_inl = seq->out4 + 2 * S; a.status = seq->out4 + 3 * S;
            int rc = pipeline_impl(ctx, &a, stream, seq->keys);
            if (rc) return rc;
            seq_policy_kernel<<<blocks, threads, 0, st>>>(seq->st, S, seq->T_rel, seq->out4, c.max_step_m, c.kf_min_common,
                                                          c.kf_min_inliers, c.kf_max_dist, c.bad_pnp_limit, seq->poses,
                                                          seq->info, c.max_frames);
            VO_LAUNCH_CHECK(ctx);
        }
        const dim3 grid((unsigned)ceil_div(ctx->sm_count * 2, S), (unsigned)S);
        seq_promote_kernel<<<grid, 256, 0, st>>>(seq->st, seq->key_desc, seq->cur_desc, seq->nd, (uint8_t *)seq->key_kp,
                                                 (const uint8_t *)seq->cur_kp, seq->nk, (uint8_t *)seq->key_depth,
                                                 (const uint8_t *)seq->cur_depth, seq->nz);
        VO_LAUNCH_CHECK(ctx);
        return VO_OK;
    };
    // Mode T with VO_SEQ_GRAPH: capture once a plain step has sized every workspace (no allocation may happen during
    // capture); re-capture when a workspace was reallocated since (the graph holds the old pointers).  A Mode R loop always
    // runs plainly.
    const bool graph = !ctx->prof_on && c.pnp_mode == VO_PNP_THROUGHPUT && seq->warm && getenv("VO_SEQ_GRAPH");
    if (graph && seq->graph_state == 1 && seq->graph_gen != ctx->ws_gen) {
        cudaGraphExecDestroy(seq->graph);
        seq->graph = nullptr;
        seq->graph_state = 0;
    }
    if (graph && seq->graph_state == 0) {
        cudaGraph_t g = nullptr;
        const long long l0 = ctx->launches;
        const unsigned long long gen = ctx->ws_gen;
        seq->graph_state = -1;
        if (cudaStreamBeginCapture(st, cudaStreamCaptureModeThreadLocal) == cudaSuccess) {
            const int rc = body(true);
            const cudaError_t e = cudaStreamEndCapture(st, &g);
            if (rc == VO_OK && e == cudaSuccess && g && ctx->ws_gen == gen &&
                cudaGraphInstantiate(&seq->graph, g, 0) == cudaSuccess) {
                seq->graph_state = 1;
                seq->graph_captures++;
                seq->graph_gen = gen;
                seq->graph_kernels = ctx->launches - l0;
            }
            if (g) cudaGraphDestroy(g);
        }
        (void)cudaGetLastError();          // a failed capture must not poison the next launch check
        ctx->launches = l0;                // (captured launches did not run; the replay below counts them)
    }
    if (graph && seq->graph_state == 1) {
        VO_CUDA(cudaGraphLaunch(seq->graph, st));
        ctx->launches += seq->graph_kernels;
    } else {
        const int rc = body(any_active);
        if (rc) return rc;
        seq->warm = seq->warm || any_active;
    }
    for (int q = 0; q < S; ++q)
        if (n_kp_h[q] >= 0) seq->pushed[q]++;
    return VO_OK;
}

}  // namespace
}  // namespace vo

extern "C" int vo_seq_push(vo_seq *seq, const void *desc, const float *kp, int n_kp, const float *depth, int frame_id,
                           void *stream) {
    using namespace vo;
    VO_REQUIRE(seq && desc && kp && depth, "vo_seq_push: null argument");
    VO_REQUIRE(seq->S == 1, "vo_seq_push: the loop holds %d sequences; push them with vo_seq_push_all", seq->S);
    VO_REQUIRE(n_kp >= 0, "vo_seq_push: negative keypoint count %d", n_kp);
    const int32_t n = n_kp, id = frame_id;
    return seq_step(seq, desc, kp, &n, nullptr, depth, &id, (size_t)n_kp, stream, "vo_seq_push");
}

extern "C" int vo_seq_push_all(vo_seq *seq, const void *desc, const float *kp, const int32_t *n_kp_h, const float *depth,
                               const int32_t *frame_id_h, void *stream) {
    using namespace vo;
    VO_REQUIRE(seq && desc && kp && n_kp_h && depth && frame_id_h, "vo_seq_push_all: null argument");
    return seq_step(seq, desc, kp, n_kp_h, nullptr, depth, frame_id_h, (size_t)seq->S * seq->cfg.n_cap, stream, "vo_seq_push_all");
}

extern "C" int vo_seq_push_all_dev(vo_seq *seq, const void *desc, const float *kp, const int32_t *n_kp_d, const int32_t *present_h,
                                   const float *depth, const int32_t *frame_id_h, void *stream) {
    using namespace vo;
    VO_REQUIRE(seq && desc && kp && n_kp_d && present_h && depth && frame_id_h, "vo_seq_push_all_dev: null argument");
    int32_t *pres = (int32_t *)malloc(sizeof(int32_t) * seq->S);
    VO_REQUIRE(pres, "vo_seq_push_all_dev: out of host memory");
    for (int q = 0; q < seq->S; ++q) pres[q] = present_h[q] ? 0 : -1;
    const int rc = seq_step(seq, desc, kp, pres, n_kp_d, depth, frame_id_h, (size_t)seq->S * seq->cfg.n_cap, stream,
                            "vo_seq_push_all_dev");
    free(pres);
    return rc;
}

extern "C" int vo_seq_lost_frames_at(vo_seq *seq, int q, int32_t *out_h, void *stream) {
    using namespace vo;
    VO_REQUIRE(seq && out_h, "vo_seq_lost_frames_at: null argument");
    VO_REQUIRE(q >= 0 && q < seq->S, "vo_seq_lost_frames_at: sequence %d outside [0, %d)", q, seq->S);
    cudaStream_t st = (cudaStream_t)stream;
    VO_CUDA(cudaMemcpyAsync(out_h, seq->lost + q, sizeof(int32_t), cudaMemcpyDeviceToHost, st));
    VO_CUDA(cudaStreamSynchronize(st));
    return VO_OK;
}

extern "C" int vo_seq_read_at(vo_seq *seq, int q, int first, int count, double *poses_h, int32_t *info_h, void *stream) {
    using namespace vo;
    VO_REQUIRE(seq, "vo_seq_read: null sequence");
    VO_REQUIRE(q >= 0 && q < seq->S, "vo_seq_read: sequence %d outside [0, %d)", q, seq->S);
    const int pushed = seq->pushed[q];
    VO_REQUIRE(first >= 0 && count >= 0 && first + count <= pushed, "vo_seq_read: range [%d, %d) outside the %d pushed frames",
               first, first + count, pushed);
    cudaStream_t st = (cudaStream_t)stream;
    const size_t row = (size_t)q * seq->cfg.max_frames + first;
    if (count && poses_h)
        VO_CUDA(cudaMemcpyAsync(poses_h, seq->poses + 16 * row, sizeof(double) * 16 * count, cudaMemcpyDeviceToHost, st));
    if (count && info_h)
        VO_CUDA(cudaMemcpyAsync(info_h, seq->info + 6 * row, sizeof(int32_t) * 6 * count, cudaMemcpyDeviceToHost, st));
    VO_CUDA(cudaStreamSynchronize(st));
    return VO_OK;
}

extern "C" int vo_seq_read(vo_seq *seq, int first, int count, double *poses_h, int32_t *info_h, void *stream) {
    return vo_seq_read_at(seq, 0, first, count, poses_h, info_h, stream);
}
