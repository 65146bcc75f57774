/*
 * vo_b200.h — C ABI of libvo_b200.so: the B200 (sm_100a) hot path of the RGB-D
 * visual-odometry pipeline: descriptor matching -> keypoint gather / depth
 * back-projection -> PnP-RANSAC -> relative pose.
 *
 * Plain C, no CUDA or torch types in any signature.  Every pointer is a DEVICE
 * pointer unless its name ends in `_h` (host) or the comment says "host".
 * `stream` is a cudaStream_t passed as void* (NULL = legacy default stream).
 * No entry point synchronises the stream; no entry point throws.  Return value:
 * 0 = VO_OK, <0 = hard error (see vo_last_error()), >0 never (soft outcomes such
 * as "no model" are per-pair and written to the `status` output arrays).
 *
 * Each entry point cites the reference interface (file:line under the upstream
 * repository) it replaces.
 *
 * Batch convention: B independent frame pairs are processed per call.  Pair b
 * owns rows [b*n_stride, b*n_stride + n_ref[b]) of the reference-frame arrays and
 * [b*m_stride, b*m_stride + n_cur[b]) of the current-frame arrays.  `n_ref` /
 * `n_cur` are device int32[B]; NULL means "every pair uses the full stride".
 */
#ifndef VO_B200_H
#define VO_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define VO_ABI_VERSION 5   /* 2: vo_pipeline_args.u8_bytes, vo_pnp_ransac_ref, VO_NORM_HAMMING_TC, vo_orb_debug_read
                             3: vo_bootstrap, vo_pnp_ransac_ref_batch, VO_ST_BAD_INPUT, the pnp_mode / ref_* fields of
                                vo_pipeline_args and vo_seq_config
                             4: vo_seq_config.n_seqs / seeds, vo_seq_push_all, vo_seq_read_at, vo_seq_frames_at, vo_seq_graph_captures,
                                vo_workspace_generation
                             5: vo_orb_extract_batch, vo_seq_push_all_dev, vo_seq_lost_frames_at */

#if defined(__GNUC__)
#define VO_API __attribute__((visibility("default")))
#else
#define VO_API
#endif

/* ---- return codes ------------------------------------------------------- */
#define VO_OK 0
#define VO_ERR_ARG (-1)
#define VO_ERR_CUDA (-2)
#define VO_ERR_UNSUPPORTED (-3)

/* ---- per-pair status bits (device int32 status arrays) ------------------ */
#define VO_ST_OK 0
#define VO_ST_NO_MODEL 1        /* no hypothesis reached min_inliers (reference: "NO IT IS A BAD PNP") */
#define VO_ST_TOO_FEW_POINTS 2  /* fewer correspondences than a minimal sample */
#define VO_ST_KP_OUT_OF_IMAGE 4 /* a matched keypoint truncates outside the depth map (reference: IndexError -> bad PnP) */
#define VO_ST_BAD_INPUT 8       /* Mode R: n_pts[b] outside [0, cap] or a bootstrap index outside [0, n_pts[b]); set with
                                   VO_ST_NO_MODEL, and the pair read no point */

/* ---- matcher configuration ---------------------------------------------- */
/* byte descriptors (ORB) */
#define VO_NORM_HAMMING 0 /* popcount(a xor b): cv2.NORM_HAMMING (north-star semantics)          */
#define VO_NORM_L2_U8 1   /* sqrt(sum (a_k-b_k)^2) over byte VALUES: what ORB.py:8 really builds  */
#define VO_NORM_HAMMING_TC 2 /* VO_NORM_HAMMING computed on the tensor cores (bits as e4m3 -1/+1, K = 256 tcgen05 kind::f8f6f4 GEMM, exact integers;
                                a second pass with the roles swapped supplies the column arg-min): bit-identical results, opt-in;
                                VO_NORM_HAMMING itself stays XOR + POPC */
/* float descriptors */
#define VO_METRIC_L2 0     /* d = sqrt(sum (a-b)^2)            : SIFT.py:11,27                    */
#define VO_METRIC_COSINE 1 /* s = a.b, d = sqrt(2-2s)          : R2D2.py:56-59                    */
/* acceptance rule applied to (top-2 of each ref row, top-1 of each cur column) */
#define VO_MODE_RATIO 0         /* d1 <  ratio*d2 (compared in double)      SIFT.py:30 / ORB.py:28 */
#define VO_MODE_MUTUAL 1        /* col_best[nn1[i]] == i                     cv2 crossCheck=True    */
#define VO_MODE_RATIO_MUTUAL 2  /* d1/(d2+1e-8f) <= ratio  AND mutual        R2D2.py:53-66          */
#define VO_MODE_THRESH_MUTUAL 3 /* s1 >= thr AND mutual                      R2D2.py:29-37          */
#define VO_MODE_THRESH 4        /* s1 >= thr                                 R2D2.py:40-51          */
#define VO_MODE_NN 5            /* every row keeps its nearest neighbour                            */
/* float-matcher arithmetic */
#define VO_PREC_TF32X3 0    /* tcgen05 kind::tf32, hi/lo split, 3 MMAs per k-step (fp32-grade)   */
#define VO_PREC_TF32X1 1    /* tcgen05 kind::tf32, 1 MMA per k-step (exact for integer-valued SIFT) */
#define VO_PREC_FP32_SIMT 2 /* CUDA-core FP32, direct (a-b)^2 / dot form (validation kernel)      */
#define VO_PREC_F16X1 3     /* tcgen05 kind::f16, operands rounded to fp16 (11 significant bits, as tf32): exact for
                               integer-valued 128-d descriptors with |x| <= 255 (SIFT; every partial sum < 2^24) at twice
                               the tf32 rate; rules
                               that need the column arg-max run the TF32X1 kernel (identical results there)      */
#define VO_PREC_F16X3 4     /* tcgen05 kind::f16, x * 2^8 = hi + lo in fp16: the 22 operand bits of TF32X3 at twice the
                               MMA rate; for |x| < 255 (unit-norm R2D2 descriptors, SIFT)                         */

/* PnP estimator of vo_pipeline / vo_seq (pnp_mode) */
#define VO_PNP_THROUGHPUT 0 /* Mode T: counter-based P3P hypotheses (vo_hypotheses + vo_pnp_ransac)                      */
#define VO_PNP_REFERENCE 1  /* Mode R: the reference's sampler (vo_bootstrap + vo_pnp_ransac_ref_batch)                 */

typedef struct vo_ctx vo_ctx;

/* Context: one per (process, device).  Owns a growable device workspace and
 * nothing else; all inputs and outputs are caller-owned. */
VO_API int vo_create(int device, vo_ctx **out);
VO_API void vo_destroy(vo_ctx *ctx);
VO_API int vo_abi_version(void);
/* Thread-local text of the last hard error ("" if none). */
VO_API const char *vo_last_error(void);
/* Number of this library's kernels launched through `ctx` since creation. */
VO_API long long vo_launch_count(const vo_ctx *ctx);
/* Number of workspace (re)allocations of `ctx` since creation (VERSION 4).  Each one frees the old block, so work captured
 * before it (a CUDA graph holding workspace pointers) is stale once this value has changed. */
VO_API unsigned long long vo_workspace_generation(const vo_ctx *ctx);

/* Optional raw k-NN outputs shared by both matchers (any pointer may be NULL).
 *   row_idx  int32 [B][n_stride][2]  nearest / second-nearest cur index (-1 if absent)
 *   row_val  float [B][n_stride][2]  their distances (VO_METRIC_COSINE: similarities)
 *   col_idx  int32 [B][m_stride]     nearest ref index of each cur descriptor
 */
typedef struct vo_knn_out {
    int32_t *row_idx;
    float *row_val;
    int32_t *col_idx;
} vo_knn_out;

/*
 * Byte-descriptor matcher.  Replaces cv2.BFMatcher.knnMatch(k=2) + ratio loop
 * (feature_extractors/ORB.py:23-32) and cv2.BFMatcher(NORM_HAMMING, crossCheck).
 *   ref uint8 [B][n_stride][32], cur uint8 [B][m_stride][32]  (bytes must be 32)
 *   out_pairs int32 [B][n_stride][2]  accepted (ref,cur) pairs, ascending ref index
 *   out_dist  float [B][n_stride]     distance of each accepted pair (may be NULL)
 *   out_count int32 [B]
 * Ties resolve to the lowest index (pinned against cv2, SURVEY 8c).
 */
VO_API int vo_match_u8(vo_ctx *ctx, const uint8_t *ref, const uint8_t *cur, int B, int n_stride, int m_stride,
                const int32_t *n_ref, const int32_t *n_cur, int bytes, int norm, int mode, double ratio,
                int32_t *out_pairs, float *out_dist, int32_t *out_count, const vo_knn_out *knn, void *stream);

/*
 * Float-descriptor matcher.  Replaces knnMatch + ratio (feature_extractors/SIFT.py:25-34)
 * and the torch matchers R2D2.py:29-66 (sim = d1 @ d2.T, topk, max, masks).
 *   ref float [B][n_stride][dim], cur float [B][m_stride][dim], dim == 128
 *   param: ratio (RATIO, RATIO_MUTUAL) or similarity threshold (THRESH*); a double because the
 *   reference compares fp32 distances against Python doubles (0.85, 0.90)
 *   near_tie uint8 [B][n_stride] (may be NULL): 1 where the row's best and second best
 *   are within 1e-5 relative in distance terms, !(d2 - d1 > 1e-5f * d2) in fp32 with d the
 *   L2 distance or, for VO_METRIC_COSINE, sqrt(2 - 2 sim), i.e. the arg-min is not robust to
 *   rounding; 0 on rows without a second best and on rows past n_ref[b].
 */
VO_API int vo_match_f32(vo_ctx *ctx, const float *ref, const float *cur, int B, int n_stride, int m_stride,
                 const int32_t *n_ref, const int32_t *n_cur, int dim, int metric, int mode, double param,
                 int precision, int32_t *out_pairs, float *out_dist, int32_t *out_count,
                 const vo_knn_out *knn, uint8_t *near_tie, void *stream);

/*
 * Dense back-projection.  Replaces cv2.rgbd.depthTo3d (VisualOdometry_Stereo.py:96).
 *   depth float [B][H][W] metres; K_h host double[9] row-major; xyz float [B][H][W][3]
 *   X = ((u-cx)*(1/fx))*z, Y = ((v-cy)*(1/fy))*z, Z = z, all in fp32.
 */
VO_API int vo_backproject_dense(vo_ctx *ctx, const float *depth, int B, int H, int W, const double *K_h, float *xyz,
                         void *stream);

/*
 * Fused keypoint gather + min-flow filter + sparse back-projection + range gate +
 * order-preserving compaction.  Replaces VisualOdometry_Stereo.py:257-264 and :96-105.
 *   pairs int32 [B][pair_cap][2], n_pairs int32 [B]
 *   ref_kp float [B][n_stride][kp_stride], cur_kp float [B][m_stride][kp_stride]  (x,y first)
 *   depth float [B][H][W] of the REFERENCE frame
 *   outputs (capacity pair_cap per pair, first n_out[b] valid, order of `pairs` kept):
 *     xyz float [B][pair_cap][3], ref_uv/cur_uv float [B][pair_cap][2],
 *     src int32 [B][pair_cap] index into `pairs` (may be NULL), n_out int32 [B],
 *     status int32 [B] (VO_ST_KP_OUT_OF_IMAGE or 0)
 */
VO_API int vo_gather_backproject(vo_ctx *ctx, const int32_t *pairs, const int32_t *n_pairs, int B, int pair_cap,
                          const float *ref_kp, const float *cur_kp, int n_stride, int m_stride, int kp_stride,
                          const float *depth, int H, int W, const double *K_h, float min_flow_px, float z_min,
                          float z_max, float *xyz, float *ref_uv, float *cur_uv, int32_t *src, int32_t *n_out,
                          int32_t *status, void *stream);

/*
 * Depth at the truncated pixel of every keypoint, depth[int(y), int(x)] (VisualOdometry_Stereo.py:97), written
 * as depth_kp float [B][n_stride] (rows past n_kp[b]: NaN; keypoints outside the image: a reserved NaN that makes
 * the pair fail with VO_ST_KP_OUT_OF_IMAGE if such a keypoint is matched).  `depth` must be device-accessible: a
 * pinned host image works (zero-copy), which moves 32 B per keypoint over PCIe instead of the whole map.
 */
VO_API int vo_sample_depth(vo_ctx *ctx, const float *kp, int B, int n_stride, int kp_stride, const int32_t *n_kp,
                    const float *depth, int H, int W, float *depth_kp, void *stream);

/*
 * Hypothesis table: int32 [B][H][4] of distinct indices in [0, n_pts[b]) drawn from a
 * counter-based generator keyed by (seed, pair0 + b, h, slot).  Rows of pairs with fewer
 * than 4 points are filled with -1.  The CPU oracle implements the same integer recipe.
 */
VO_API int vo_hypotheses(vo_ctx *ctx, const int32_t *n_pts, int B, int H, uint64_t seed, int64_t pair0, int32_t *hyp,
                  void *stream);

/*
 * PnP-RANSAC + refit.  Replaces the 3x cv2.solvePnPRansac loop, cv2.Rodrigues and the
 * pose inversion (VisualOdometry_Stereo.py:120-144).
 *   xyz float [B][cap][3], uv float [B][cap][2], n_pts int32 [B]
 *   K_h host double[9];  hyp int32 [B][H][4] (P3P sample + 1 disambiguation point)
 *   thr_px: inlier iff squared reprojection error <= thr_px^2 (fp32, OpenCV rule)
 *   min_inliers: model accepted iff count > min_inliers (reference: > 20)
 *   outputs: rt double [B][12] (R row-major, t) with X_cur = R X_ref + t, refined;
 *            rvec_tvec double [B][6];  T_rel double [B][16] = inverse of [R|t] (the pose the
 *            reference stores, :141-143);  n_inl, best_h, status int32 [B];
 *            inlier_mask uint8 [B][cap] of the best MINIMAL model (OpenCV semantics);
 *            hyp_counts int32 [B][H] inlier count of every hypothesis (may be NULL; tests use it).
 *   Ties between hypotheses resolve to the lowest hypothesis index.
 */
VO_API int vo_pnp_ransac(vo_ctx *ctx, const float *xyz, const float *uv, const int32_t *n_pts, int B, int cap,
                  const double *K_h, const int32_t *hyp, int H, float thr_px, int min_inliers, int refine_iters,
                  double *rt, double *rvec_tvec, double *T_rel, int32_t *n_inl, int32_t *best_h,
                  uint8_t *inlier_mask, int32_t *hyp_counts, int32_t *status, void *stream);

/*
 * Per-stage device timing (CUDA events recorded on the caller's stream around each kernel launch).
 * Used by bench.py for the per-kernel roofline; off by default (no events recorded).
 * vo_profile_collect synchronises the device, adds up the intervals recorded since the last collect
 * and writes, per stage id, total milliseconds and interval count (arrays of VO_STAGE_COUNT).
 */
#define VO_STAGE_FILL 0     /* column-key reset                  */
#define VO_STAGE_PREP 1     /* tf32 hi/lo split + norms (float)  */
#define VO_STAGE_MATCH 2    /* distance kernel (u8 / f32)        */
#define VO_STAGE_FINALIZE 3 /* merge + acceptance rule + compact */
#define VO_STAGE_GATHER 4   /* gather + back-project + gate      */
#define VO_STAGE_HYP 5      /* hypothesis table                  */
#define VO_STAGE_P3P 6      /* minimal solves                    */
#define VO_STAGE_SCORE 7    /* inlier counting                   */
#define VO_STAGE_REFIT 8    /* winner mask + Gauss-Newton        */
#define VO_STAGE_DENSE 9    /* dense back-projection             */
#define VO_STAGE_COUNT 10
VO_API int vo_profile_enable(vo_ctx *ctx, int on);
VO_API int vo_profile_collect(vo_ctx *ctx, double *ms, long long *counts);

/*
 * Whole hot path for a batch of pairs on one stream (match -> gather/back-project ->
 * hypotheses -> PnP-RANSAC -> pose).  Replaces lines 256-264 + computepose_3D_2D of
 * VisualOdometry.process_frame (VisualOdometry_Stereo.py:223-297) for B pre-declared pairs.
 */
typedef struct vo_pipeline_args {
    int B, n_stride, m_stride;
    const int32_t *n_ref, *n_cur; /* device int32[B] or NULL */
    /* descriptors: exactly one of (ref_u8,cur_u8) / (ref_f32,cur_f32) is non-NULL */
    const uint8_t *ref_u8, *cur_u8;
    const float *ref_f32, *cur_f32;
    int norm_or_metric, mode, precision;
    double match_param;
    /* keypoints + depth */
    const float *ref_kp, *cur_kp;
    int kp_stride;
    const float *depth; /* float [B][H][W] of the reference frames; device memory, or pinned host memory mapped into the
                         * device address space (then only the pixels under matched keypoints cross the bus) */
    int H, W;
    const double *K_h; /* host double[9] */
    float min_flow_px, z_min, z_max;
    /* RANSAC */
    int n_hyp;
    uint64_t seed;
    int64_t pair0;
    float thr_px;
    int min_inliers, refine_iters;
    /* outputs (device) */
    double *T_rel;      /* [B][16] */
    double *rt;         /* [B][12]  (may be NULL) */
    int32_t *n_matches; /* [B] raw matches             */
    int32_t *n_corr;    /* [B] correspondences after gating ("common_pts") */
    int32_t *n_inl;     /* [B] */
    int32_t *status;    /* [B] */
    /* optional: depth already sampled at every reference keypoint (vo_sample_depth), float [B][n_stride];
     * when non-NULL it replaces the dense `depth` lookup */
    const float *depth_kp;
    /* bytes per descriptor of the (ref_u8, cur_u8) pair: 0 or 32 = 256-bit descriptors; 128 = 128-d descriptors whose values are
     * integers 0..255 held as uint8 (OpenCV SIFT: a quarter of the float32 bytes over the bus, same exact results) — with
     * VO_NORM_L2_U8 and a rule without a column side (VO_MODE_RATIO / VO_MODE_NN) only */
    int u8_bytes;
    /* PnP estimator (VERSION 3; zero = Mode T as before).  VO_PNP_REFERENCE runs match -> gather/back-project ->
     * vo_bootstrap(n_corr, ref_restarts, cap = n_stride, seed, pair0) -> vo_pnp_ransac_ref_batch(ref_iters, thr_px,
     * ref_confidence, min_inliers, refine_iters): bit-identical to those calls in sequence; n_hyp is then ignored (any value).
     * ref_restarts 0 = 3, ref_iters 0 = 100, ref_confidence 0 = 0.99 (the reference's values, :121-126). */
    int pnp_mode;
    int ref_restarts, ref_iters;
    double ref_confidence;
} vo_pipeline_args;

VO_API int vo_pipeline(vo_ctx *ctx, const vo_pipeline_args *args, void *stream);

/*
 * Device-resident keyframe loop.  Replaces the host control flow of VisualOdometry.process_frame
 * (VisualOdometry_Stereo.py:232-297) for a stream of frames whose features already exist: keyframe
 * selection (:251, :285-296), the 1.5 m-per-frame plausibility gate (:270-274), the bad-PnP counter
 * (:273, :279, :282, :295) and pose chaining T_cur = T_key @ T_rel (:283, :290) run in a one-thread
 * policy kernel behind vo_pipeline, and a conditional device copy promotes the current frame to
 * keyframe.  No host round trip per frame: vo_seq_push only enqueues work on `stream`.
 *
 *   vo_seq_push: desc (uint8 [n_kp][32] or float [n_kp][128]), kp float [n_kp][kp_stride] (x, y first),
 *   depth float [H][W]; each may be a device pointer or a (pinned) host pointer — they are copied into
 *   the loop's own frame slot with cudaMemcpyAsync on `stream`.  frame_id is the reference's frame_no
 *   (the gate scales with frame_id - keyframe_id).  The first push only installs the keyframe.
 *   vo_seq_read: synchronises `stream` and copies out, for frames [first, first+count):
 *     poses_h  double [count][16]  global pose of each frame (frame 0 = identity), what the
 *                                  reference stores in global_poses (:293)
 *     info_h   int32  [count][6]   status bits | n_matches | n_corr ("common_pts") | n_inl |
 *                                  keyframe id the frame was matched against | 1 if it became the keyframe
 *
 * S independent sequences in lock-step (VERSION 4): n_seqs = S > 1 makes one loop of S sequences whose step is ONE
 * vo_pipeline batch of B = S pairs (sequence q's current frame against its own keyframe); the policy and the promotion
 * run per sequence on the device and never look at a neighbour.  Sequence q draws its hypotheses / bootstrap rows from
 * (seeds[q], its history slot - 1), so its poses and info equal, bit for bit, those of a one-sequence loop created with
 * seed = seeds[q] and fed the same frames.
 *   vo_seq_push_all: desc (uint8 [S][n_cap][32] or float [S][n_cap][128]), kp float [S][n_cap][kp_stride], depth float
 *   [S][H][W], device or (pinned) host memory, each copied with one cudaMemcpyAsync; n_kp_h, frame_id_h host int32 [S],
 *   read before the call returns.  n_kp_h[q] < 0: sequence q has no frame at this step (its state is not touched); a
 *   sequence's first frame installs its keyframe whenever it arrives.  Every check (counts <= n_cap, no pushing sequence's
 *   history full) comes before anything is enqueued: one bad sequence refuses the whole step.
 *   vo_seq_read_at / vo_seq_frames_at: vo_seq_read / vo_seq_frames of sequence q.  vo_seq_push, vo_seq_read and
 *   vo_seq_frames act on sequence 0; vo_seq_push on a loop with S > 1 is an error.
 * VO_SEQ_GRAPH=1 (environment, Mode T only): every step after the first one that ran the pipeline is one CUDA-graph
 * launch.  The graph holds the vo_ctx workspace pointers; when any call on the same vo_ctx has reallocated a workspace
 * since capture, the next step re-captures.  vo_seq_graph_captures: how many times the loop captured its step (0 when
 * it launches plainly; one more for every re-capture).  n_seqs is at most 65535.
 * Device-side counts (VERSION 5), so that S sequences go from images to poses with no host read per step:
 *   vo_seq_push_all_dev: desc / kp / depth as vo_seq_push_all; n_kp_d device int32 [S][2] = (rows, flags), the layout
 *   vo_orb_extract_batch writes; present_h host int32 [S] (non-zero: sequence q has a frame at this step); frame_id_h as
 *   vo_seq_push_all.  The loop reads each present sequence's count on the device and clamps it to n_cap; a frame that was
 *   clamped or whose flag word is non-zero lost rows and is counted per sequence.  Checks (the history of every present
 *   sequence not full) come before anything is enqueued.
 *   vo_seq_lost_frames_at: *out_h = the number of such frames of sequence q so far (synchronises `stream`).
 */
typedef struct vo_seq vo_seq;
typedef struct vo_seq_config {
    int desc_is_f32;            /* 0: 256-bit byte descriptors, 1: 128-d float descriptors */
    int n_cap;                  /* capacity: keypoints per frame */
    int kp_stride;              /* floats per keypoint row (2: SIFT/ORB, 3: R2D2) */
    int H, W;
    double K[9];
    int norm_or_metric, mode, precision;
    double match_param;
    float min_flow_px, z_min, z_max;
    int n_hyp;
    uint64_t seed;
    float thr_px;
    int min_inliers, refine_iters;
    double max_step_m;          /* 1.5  (:271) */
    int kf_min_common;          /* 200  (:286) */
    int kf_min_inliers;         /* 100  (:286) */
    double kf_max_dist;         /* 1.5  (:286) */
    int bad_pnp_limit;          /* 3    (:295) */
    int max_frames;             /* capacity of the pose / info history */
    /* PnP estimator, as in vo_pipeline_args (VERSION 3; zero = Mode T).  A Mode R loop always launches plainly: VO_SEQ_GRAPH
     * is ignored for it (its poses are the same either way); n_hyp is then ignored. */
    int pnp_mode;
    int ref_restarts, ref_iters;
    double ref_confidence;
    /* sequences in lock-step (VERSION 4): 0 or 1 = one sequence */
    int n_seqs;
    const uint64_t *seeds;      /* host uint64 [n_seqs] (copied at create); NULL = seed + q */
} vo_seq_config;
VO_API int vo_seq_create(vo_ctx *ctx, const vo_seq_config *cfg, vo_seq **out);
VO_API void vo_seq_destroy(vo_seq *seq);
VO_API int vo_seq_push(vo_seq *seq, const void *desc, const float *kp, int n_kp, const float *depth, int frame_id,
                void *stream);
VO_API int vo_seq_frames(const vo_seq *seq);
VO_API int vo_seq_read(vo_seq *seq, int first, int count, double *poses_h, int32_t *info_h, void *stream);
VO_API int vo_seq_push_all(vo_seq *seq, const void *desc, const float *kp, const int32_t *n_kp_h, const float *depth,
                    const int32_t *frame_id_h, void *stream);
VO_API int vo_seq_frames_at(const vo_seq *seq, int q);
VO_API int vo_seq_read_at(vo_seq *seq, int q, int first, int count, double *poses_h, int32_t *info_h, void *stream);
VO_API int vo_seq_graph_captures(const vo_seq *seq);
VO_API int vo_seq_push_all_dev(vo_seq *seq, const void *desc, const float *kp, const int32_t *n_kp_d, const int32_t *present_h,
                        const float *depth, const int32_t *frame_id_h, void *stream);
VO_API int vo_seq_lost_frames_at(vo_seq *seq, int q, int32_t *out_h, void *stream);

/*
 * "Same" 2-D convolution on the tensor cores (3xTF32 implicit GEMM; TMA zero fill is the padding): the layer type of
 * the R2D2 network (feature_extractors/r2d2/nets/patchnet.py:56-66, torch.nn.Conv2d with padding = (k-1)*dil/2).
 *   x float [H][W][C_in] (NHWC), w float [C_out][k][k][C_in], out float [H][W][C_out]
 *   out = relu?( conv(x, w) * scale[c] + shift[c] )   — bias and inference batch-norm folded into scale / shift
 *   C_in a multiple of 32, C_out in {32, 64, 128}.
 */
VO_API int vo_conv2d(vo_ctx *ctx, const float *x, int H, int W, int cin, const float *w, int cout, int k, int dil,
              const float *scale, const float *shift, int relu, float *out, void *stream);

/*
 * R2D2 front-end (SURVEY 8(f) rank 1): `extract_features_and_desc` of R2D2.py:202-232 for one image at scale 1 (the
 * reference's extract_multiscale leaves its loop after the first scale, R2D2.py:133-135): network forward
 * (nets/patchnet.py:141-186: a stack of "same" convolutions with inference batch-norm / ReLU, an optional 2x2 max-pool
 * and a final bilinear x2 up-sampling), reliability / repeatability heads on x^2 (:181-186, :16-27), 3x3 non-maximum
 * suppression with both thresholds (R2D2.py:82-101), score = reliability * repeatability > score_thr (:186-188),
 * L2-normalised descriptors of the surviving pixels.
 *   layers[0] must have C_in = 3 (runs on the CUDA cores, with the ImageNet mean / std normalisation of
 *   tools/dataloader.py:norm_RGB folded in); every other layer runs as vo_conv2d.  All weight pointers are HOST
 *   pointers and are copied at creation.  w: [C_out][k][k][C_in].
 *   vo_r2d2_extract: rgb uint8 [H][W][3] (device or pinned host).  Outputs (device): xys float [max_kp][3]
 *   (x, y, 32), desc float [max_kp][128], scores float [max_kp], count int32[1] (total found; at most max_kp are
 *   written, in row-major pixel order like torch.nonzero), rel_map / rep_map float [Ho][Wo] (optional).
 */
typedef struct vo_r2d2_layer {
    int cin, cout, k, dil;
    int bn, relu, pool_after;         /* pool_after: 2 = MaxPool2d(2) follows, 0 = none */
    const float *w, *bias, *bn_mean, *bn_var;
} vo_r2d2_layer;
typedef struct vo_r2d2_config {
    int H, W;
    int n_layers;
    const vo_r2d2_layer *layers;
    int upsample;                     /* 1 or 2 (Fast_Quad_L2Net ends with Upsample(scale_factor=2, bilinear)) */
    const float *clf_w, *clf_b;       /* reliability head  [2][C], [2] */
    const float *sal_w, *sal_b;       /* repeatability head [C], [1]   */
    float bn_eps;
    int max_kp;
} vo_r2d2_config;
typedef struct vo_r2d2 vo_r2d2;
VO_API int vo_r2d2_create(vo_ctx *ctx, const vo_r2d2_config *cfg, vo_r2d2 **out);
VO_API void vo_r2d2_destroy(vo_r2d2 *net);
VO_API int vo_r2d2_out_shape(const vo_r2d2 *net, int *Ho, int *Wo);
VO_API int vo_r2d2_extract(vo_r2d2 *net, const uint8_t *rgb, float rel_thr, float rep_thr, float score_thr, float *xys,
                    float *desc, float *scores, int32_t *count, float *rel_map, float *rep_map, void *stream);

/*
 * Reference-sampler PnP-RANSAC ("Mode R", the drop-in's default): VisualOdometry_Stereo.py:120-135 as the reference runs them.
 * `boot_idx` int32 [restarts][n] (device) are the bootstrap index rows the caller drew with np.random.randint(0, n, n) (:122);
 * every row goes through the inside of cv2.solvePnPRansac(iterationsCount = iters, reprojectionError = thr_px, confidence):
 * OpenCV's own sample table (its RNG is re-seeded per call, so the table is a function of n), EPnP on five points,
 * projectPoints-style fp32 scoring (err <= thr_px^2), the adaptive iteration count, a Gauss-Newton refit on the inliers of the
 * best minimal model (cv2.solvePnP(ITERATIVE)'s fixed point); the best restart by inlier count (strictly more than
 * min_inliers) wins, the first one on ties (:132-135).  One frame pair per call (B = 1): xyz float [>= max idx + 1][3],
 * uv float [..][2] are the gathered / gated correspondences (vo_gather_backproject).
 * Outputs (device, all optional except T_rel / status): rt [12], rvec_tvec [6], T_rel [16] as vo_pnp_ransac; n_inl [1] = inliers
 * of the winning minimal model; best int32 [3] = (restart, iteration, iterations the stopping rule ran); inlier_mask uint8 [n]
 * over the winning restart's resample; hyp_counts int32 [restarts][iters] (-1: no model), hyp_poses double [restarts][iters][12].
 * Parity: sampler, scoring and stopping rule reproduce cv2.solvePnPRansac exactly when driven with OpenCV's minimal solver
 * (tests/test_oracle_pnp_ref.py); OpenCV's five-point EPnP itself depends on an arbitrary null-space basis and is matched
 * statistically (csrc/pnp_ref_math.cuh, DESIGN 3.6).
 * A bootstrap index outside [0, n) gives status VO_ST_NO_MODEL | VO_ST_BAD_INPUT and an identity pose; no point is read.
 * Fewer than 5 points: VO_ST_NO_MODEL.  hyp_poses rows of iterations without a model are zero.  The sample table is built
 * on the host and copied from a host array (not for stream capture: use vo_pnp_ransac_ref_batch there).
 */
VO_API int vo_pnp_ransac_ref(vo_ctx *ctx, const float *xyz, const float *uv, int n, const double *K_h, const int32_t *boot_idx,
                      int restarts, int iters, float thr_px, double confidence, int min_inliers, int refine_iters, double *rt,
                      double *rvec_tvec, double *T_rel, int32_t *n_inl, int32_t *best, uint8_t *inlier_mask, int32_t *hyp_counts,
                      double *hyp_poses, int32_t *status, void *stream);

/*
 * Bootstrap rows for Mode R: boot int32 [B][restarts][cap], entry (b, r, i) uniform in [0, n_pts[b]) for i < n_pts[b] and -1
 * for the padding i >= n_pts[b] (every entry of a pair with n_pts[b] <= 0).  Counter-based, keyed by (seed, pair0 + b, r, i):
 * the pair key, not the batch position, decides a row, so rows do not depend on chunking, lanes or GPU count (as
 * vo_hypotheses).  The restart enters through a domain constant that keeps the row keys apart from the hypothesis keys of the
 * same seed and pair.  Range map: multiply-high of a 32-bit draw, ((uint64) u * n) >> 32, relative bias below n / 2^32.
 * The draw replaces np.random.randint(0, n, n) of :122 by a reproducible stream (a different one: Mode R results with these
 * rows match the reference statistically, not draw for draw).
 */
VO_API int vo_bootstrap(vo_ctx *ctx, const int32_t *n_pts, int B, int restarts, int cap, uint64_t seed, int64_t pair0,
                 int32_t *boot, void *stream);

/*
 * Mode R over B frame pairs in one call, everything on the device (no host read of n_pts, no host-staged copy: capture-safe).
 *   xyz float [B][cap][3], uv float [B][cap][2], n_pts int32 [B] (device); boot_idx int32 [B][restarts][cap]: pair b's rows,
 *   stride cap, first n_pts[b] entries used (vo_bootstrap, or the caller's own rows); restarts <= 8, iters <= 1024.
 *   Outputs: the single-pair entry's with a leading [B]: rt [B][12], rvec_tvec [B][6], T_rel [B][16], n_inl [B], best [B][3],
 *   inlier_mask uint8 [B][cap] (first n_pts[b] entries), hyp_counts int32 [B][restarts][iters],
 *   hyp_poses double [B][restarts][iters][12], status int32 [B]; all optional except T_rel / status.
 *   Per pair: n_pts[b] outside [0, cap] or an index of the first n_pts[b] entries of a row outside [0, n_pts[b]) gives
 *   VO_ST_NO_MODEL | VO_ST_BAD_INPUT, identity pose, zero inliers, a zero mask, and no point of that pair is read; neighbours
 *   are unaffected.  n_pts[b] < 5: VO_ST_NO_MODEL, as the single-pair entry.  The sample table of each pair is OpenCV's
 *   (a function of n_pts[b]), built on the device.
 *   Parity: pair b's outputs are bit-identical to vo_pnp_ransac_ref on xyz[b][:n], uv[b][:n] and boot_idx[b][:, :n], whatever
 *   its position in the batch and its neighbours (tests/test_gpu_pnp_ref_batch.py).
 */
VO_API int vo_pnp_ransac_ref_batch(vo_ctx *ctx, const float *xyz, const float *uv, const int32_t *n_pts, int B, int cap,
                            const double *K_h, const int32_t *boot_idx, int restarts, int iters, float thr_px, double confidence,
                            int min_inliers, int refine_iters, double *rt, double *rvec_tvec, double *T_rel, int32_t *n_inl,
                            int32_t *best, uint8_t *inlier_mask, int32_t *hyp_counts, double *hyp_poses, int32_t *status,
                            void *stream);

/*
 * ORB front-end (SURVEY 8(f) rank 1): `extract_features_and_desc` of feature_extractors/ORB.py:10-21, i.e.
 * cv2.ORB_create() (ORB.py:8, all defaults: scale 1.2f, edge 31, patch 31, Harris score, WTA_K 2) followed by
 * detectAndCompute: gray conversion, INTER_LINEAR_EXACT pyramid, FAST-9/16 + non-maximum suppression, retainBest on
 * the FAST score and on the Harris response (ties kept), intensity-centroid orientation, 7x7 Gaussian, rBRIEF.
 * Bit-identical to the pinned CPU restatement on a B200 (tests/test_gpu_orb_frontend.py).
 *   vo_orb_extract: image uint8 [H][W] (channels = 1) or [H][W][3] BGR (channels = 3), device-accessible.
 *   Outputs (device), vo_orb_capacity() rows each: kp float [cap][2] = KeyPoint.pt; desc uint8 [cap][32];
 *   aux float [cap][4] = (octave, angle in degrees, response, size), optional; count int32[2] = (keypoints written,
 *   overflow flag: a level kept more than its share of ties).  Order: level-major, then row-major (OpenCV's own
 *   order is unspecified: it depends on std::nth_element).
 *   vo_orb_extract_batch (VERSION 5): S images in one call of the same 17 launches (BGR; 16 for gray).  images uint8
 *   [S][H][W] (channels = 1) or [S][H][W][3], device or pinned host memory.  Outputs (device): kp float [S][out_rows][2],
 *   desc uint8 [S][out_rows][32], aux float [S][out_rows][4] (optional), count int32 [S][2] = (rows written, flags): flag
 *   bit 0 = a level kept more tied keypoints than it holds (vo_orb_extract's overflow), bit 1 = rows past out_rows were
 *   dropped.  Image s's rows are a prefix of what vo_orb_extract returns for it, in the same order.  1 <= S <= 65535,
 *   out_rows >= 1.  Scratch grows to the largest S seen (growing synchronises the device).  vo_orb_extract is the S = 1
 *   call with out_rows = vo_orb_capacity().
 */
typedef struct vo_orb_config {
    int H, W;
    int nfeatures;       /* 500 */
    int nlevels;         /* 8 (at most 8) */
    int fast_threshold;  /* 20 */
} vo_orb_config;
typedef struct vo_orb vo_orb;
VO_API int vo_orb_create(vo_ctx *ctx, const vo_orb_config *cfg, vo_orb **out);
VO_API void vo_orb_destroy(vo_orb *orb);
VO_API int vo_orb_capacity(const vo_orb *orb);
VO_API int vo_orb_extract(vo_orb *orb, const uint8_t *image, int channels, float *kp, uint8_t *desc, float *aux,
                   int32_t *count, void *stream);
VO_API int vo_orb_extract_batch(vo_orb *orb, const uint8_t *images, int S, int channels, int out_rows, float *kp, uint8_t *desc,
                         float *aux, int32_t *count, void *stream);
/* Diagnostic: copy one intermediate buffer of the last vo_orb_extract to host memory (synchronises; buffer ids in
 * csrc/orb.cu).  Used by tools/orb_bisect.py to compare the extractor stage by stage with the CPU restatement. */
VO_API int vo_orb_debug_read(vo_orb *orb, int what, int level, void *host_dst, size_t cap_bytes, size_t *out_bytes);

/*
 * SIFT front-end (SURVEY 8(f) rank 1): `extract_features_and_desc` of feature_extractors/SIFT.py:14-23, i.e.
 * cv2.xfeatures2d.SIFT_create() (SIFT.py:10, all defaults) followed by detectAndCompute.  Parity is held to a tolerance
 * (same keypoints to 1e-2 px / 0.25 degrees, descriptor entries within 1): OpenCV's own low-order bits depend on the
 * host CPU.  Verified under the host emulation and on a B200 (tests/test_gpu_sift_frontend.py).
 *   vo_sift_extract: image uint8 [H][W] (channels = 1) or [H][W][3] BGR (channels = 3), device-accessible.
 *   Outputs (device), max_keypoints rows each: kp float [cap][2] = KeyPoint.pt; desc float [cap][128] (values 0..255);
 *   aux float [cap][4] = (size, angle in degrees, response, packed octave word), optional; count int32[2] =
 *   (keypoints written, raw candidates found: more than max_keypoints means the list was cut).  Rows are in OpenCV's
 *   order (sorted by x, y, ...; duplicates removed).
 */
typedef struct vo_sift_config {
    int H, W;
    int max_keypoints;
} vo_sift_config;
typedef struct vo_sift vo_sift;
VO_API int vo_sift_create(vo_ctx *ctx, const vo_sift_config *cfg, vo_sift **out);
VO_API void vo_sift_destroy(vo_sift *sift);
VO_API int vo_sift_capacity(const vo_sift *sift);
VO_API int vo_sift_extract(vo_sift *sift, const uint8_t *image, int channels, float *kp, float *desc, float *aux,
                    int32_t *count, void *stream);

#ifdef __cplusplus
}
#endif
#endif /* VO_B200_H */
