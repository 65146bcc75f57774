"""Tensor-level wrappers over the C ABI.  PyTorch supplies device memory and the stream; every
computation happens inside libvo_b200.so.  All wrappers take and return CUDA tensors and do not
synchronise (callers read results with .cpu() / .item() when they need them).
"""
import ctypes

import numpy as np
import torch

from . import _lib
from ._lib import (KnnOut, PipelineArgs, VO_METRIC_COSINE, VO_METRIC_L2, VO_MODE_MUTUAL, VO_MODE_NN, VO_MODE_RATIO,
                   VO_MODE_RATIO_MUTUAL, VO_MODE_THRESH, VO_MODE_THRESH_MUTUAL, VO_NORM_HAMMING, VO_NORM_HAMMING_TC, VO_NORM_L2_U8,
                   VO_PNP_REFERENCE, VO_PNP_THROUGHPUT, VO_PREC_F16X1, VO_PREC_F16X3, VO_PREC_FP32_SIMT, VO_PREC_TF32X1,
                   VO_PREC_TF32X3, VO_ST_BAD_INPUT, check)

_contexts = {}


def context(device=None, lane=0):
    """Per-device vo_ctx (created on first use).  A vo_ctx owns one workspace, so calls that are to run concurrently on
    different streams of a device use different lanes (lane 0 is the one the profiling / launch counters read)."""
    if not torch.cuda.is_available():
        raise _lib.VoError("no CUDA device: libvo_b200 has no CPU fallback")
    dev = torch.cuda.current_device() if device is None else torch.device(device).index
    dev = 0 if dev is None else dev
    key = dev if lane == 0 else (dev, int(lane))
    if key not in _contexts:
        _contexts[key] = _lib.Context(dev)
    return _contexts[key]


def launch_count(device=None):
    return context(device).launch_count()


def profile_enable(on=True, device=None):
    ctx = context(device)
    check(ctx.lib.vo_profile_enable(ctx.handle, 1 if on else 0), "vo_profile_enable")


def profile_collect(device=None):
    """{stage: (total_ms, intervals)} since the last collect (synchronises the device)."""
    ctx = context(device)
    ms = (ctypes.c_double * len(_lib.STAGES))()
    cnt = (ctypes.c_longlong * len(_lib.STAGES))()
    check(ctx.lib.vo_profile_collect(ctx.handle, ms, cnt), "vo_profile_collect")
    return {name: (ms[i], cnt[i]) for i, name in enumerate(_lib.STAGES)}


def _ptr(t):
    return None if t is None else ctypes.c_void_p(t.data_ptr())


def _stream():
    return ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)


def _dev_of(t):
    return t.device


def _chk(t, dtype, name):
    if t.dtype != dtype or not t.is_cuda or not t.is_contiguous():
        raise ValueError(f"{name}: expected contiguous CUDA {dtype}, got {t.dtype} {t.device} contiguous={t.is_contiguous()}")


def _batchify(t, nd):
    return t if t.dim() == nd else t.unsqueeze(0)


def _k_host(K):
    k = np.ascontiguousarray(np.asarray(K, dtype=np.float64).reshape(9))
    return k, k.ctypes.data_as(ctypes.c_void_p)


class MatchResult:
    """pairs int32 [B, n_stride, 2] (first count[b] rows valid), dist float [B, n_stride], count int32 [B]."""

    def __init__(self, pairs, dist, count, knn_idx=None, knn_val=None, col_idx=None, near_tie=None):
        self.pairs, self.dist, self.count = pairs, dist, count
        self.knn_idx, self.knn_val, self.col_idx, self.near_tie = knn_idx, knn_val, col_idx, near_tie

    def numpy(self, b=0):
        """(K,2) int64 array of pair b — the reference's get_matches return type."""
        k = int(self.count[b].item())
        return self.pairs[b, :k].to(torch.int64).cpu().numpy()


def _match_common(ref, cur, n_ref, n_cur, want_knn, want_dist):
    B, N = ref.shape[0], ref.shape[1]
    M = cur.shape[1]
    dev = ref.device
    pairs = torch.empty((B, max(N, 1), 2), dtype=torch.int32, device=dev)
    dist = torch.empty((B, max(N, 1)), dtype=torch.float32, device=dev) if want_dist else None
    count = torch.zeros((B,), dtype=torch.int32, device=dev)
    knn = None
    kidx = kval = cidx = None
    if want_knn:
        kidx = torch.empty((B, max(N, 1), 2), dtype=torch.int32, device=dev)
        kval = torch.empty((B, max(N, 1), 2), dtype=torch.float32, device=dev)
        if want_knn != "rows":  # "rows": the row top-2 only (no column arg-min: the matcher may skip its column side)
            cidx = torch.empty((B, max(M, 1)), dtype=torch.int32, device=dev)
        knn = KnnOut(kidx.data_ptr(), kval.data_ptr(), cidx.data_ptr() if cidx is not None else None)
    if n_ref is not None:
        _chk(n_ref, torch.int32, "n_ref")
    if n_cur is not None:
        _chk(n_cur, torch.int32, "n_cur")
    return B, N, M, pairs, dist, count, knn, kidx, kval, cidx


def match_u8(ref, cur, norm=VO_NORM_HAMMING, mode=VO_MODE_MUTUAL, ratio=0.85, n_ref=None, n_cur=None,
             want_knn=False, want_dist=True):
    """Byte-descriptor matcher (vo_match_u8).  ref [B,N,32] or [N,32] uint8, cur likewise."""
    ref, cur = _batchify(ref, 3), _batchify(cur, 3)
    _chk(ref, torch.uint8, "ref")
    _chk(cur, torch.uint8, "cur")
    if ref.shape[0] != cur.shape[0] or ref.shape[2] != cur.shape[2]:
        raise ValueError("match_u8: batch / descriptor-size mismatch")
    ctx = context(ref.device)
    B, N, M, pairs, dist, count, knn, kidx, kval, cidx = _match_common(ref, cur, n_ref, n_cur, want_knn, want_dist)
    with torch.cuda.device(ref.device):
        check(ctx.lib.vo_match_u8(ctx.handle, _ptr(ref), _ptr(cur), B, N, M, _ptr(n_ref), _ptr(n_cur),
                                  int(ref.shape[2]), int(norm), int(mode), float(ratio), _ptr(pairs), _ptr(dist),
                                  _ptr(count), ctypes.byref(knn) if knn is not None else None, _stream()),
              "vo_match_u8")
    return MatchResult(pairs, dist, count, kidx, kval, cidx)


def match_f32(ref, cur, metric=VO_METRIC_L2, mode=VO_MODE_RATIO, param=0.85, precision=VO_PREC_TF32X3,
              n_ref=None, n_cur=None, want_knn=False, want_dist=True, want_near_tie=False):
    """Float-descriptor matcher (vo_match_f32).  ref [B,N,D] or [N,D] float32."""
    ref, cur = _batchify(ref, 3), _batchify(cur, 3)
    _chk(ref, torch.float32, "ref")
    _chk(cur, torch.float32, "cur")
    if ref.shape[0] != cur.shape[0] or ref.shape[2] != cur.shape[2]:
        raise ValueError("match_f32: batch / descriptor-size mismatch")
    ctx = context(ref.device)
    B, N, M, pairs, dist, count, knn, kidx, kval, cidx = _match_common(ref, cur, n_ref, n_cur, want_knn, want_dist)
    near = torch.empty((B, max(N, 1)), dtype=torch.uint8, device=ref.device) if want_near_tie else None
    with torch.cuda.device(ref.device):
        check(ctx.lib.vo_match_f32(ctx.handle, _ptr(ref), _ptr(cur), B, N, M, _ptr(n_ref), _ptr(n_cur),
                                   int(ref.shape[2]), int(metric), int(mode), float(param), int(precision),
                                   _ptr(pairs), _ptr(dist), _ptr(count),
                                   ctypes.byref(knn) if knn is not None else None, _ptr(near), _stream()),
              "vo_match_f32")
    return MatchResult(pairs, dist, count, kidx, kval, cidx, near)


def backproject_dense(depth, K):
    """cv2.rgbd.depthTo3d replacement.  depth [B,H,W] or [H,W] float32 -> [..,H,W,3] float32."""
    squeeze = depth.dim() == 2
    d = _batchify(depth, 3)
    _chk(d, torch.float32, "depth")
    B, H, W = d.shape
    out = torch.empty((B, H, W, 3), dtype=torch.float32, device=d.device)
    ctx = context(d.device)
    kh, kp = _k_host(K)
    with torch.cuda.device(d.device):
        check(ctx.lib.vo_backproject_dense(ctx.handle, _ptr(d), B, H, W, kp, _ptr(out), _stream()),
              "vo_backproject_dense")
    return out[0] if squeeze else out


def sample_depth(kp, depth, n_kp=None, out=None):
    """depth[int(y), int(x)] at every keypoint (vo_sample_depth).  kp [B,N,s] CUDA float32; depth [B,H,W] float32 on the
    device OR in pinned host memory (read zero-copy through the mapped pointer).  Returns depth_kp [B,N] CUDA float32."""
    _chk(kp, torch.float32, "kp")
    if depth.dtype != torch.float32 or not depth.is_contiguous() or not (depth.is_cuda or depth.is_pinned()):
        raise ValueError("sample_depth: depth must be contiguous float32 on the device or in pinned host memory")
    B, N, s = kp.shape
    if out is None:
        out = torch.empty((B, N), dtype=torch.float32, device=kp.device)
    ctx = context(kp.device)
    with torch.cuda.device(kp.device):
        check(ctx.lib.vo_sample_depth(ctx.handle, _ptr(kp), B, N, s, _ptr(n_kp), _ptr(depth), int(depth.shape[1]),
                                      int(depth.shape[2]), _ptr(out), _stream()), "vo_sample_depth")
    return out


def conv2d(x, w, scale, shift, k, dil=1, relu=False):
    """vo_conv2d: x [H,W,Cin] NHWC, w [Cout,k,k,Cin], scale/shift [Cout] (all CUDA float32) -> [H,W,Cout]."""
    for t, name in ((x, "x"), (w, "w"), (scale, "scale"), (shift, "shift")):
        _chk(t, torch.float32, name)
    H, W, cin = x.shape
    cout = w.shape[0]
    out = torch.empty((H, W, cout), dtype=torch.float32, device=x.device)
    ctx = context(x.device)
    with torch.cuda.device(x.device):
        check(ctx.lib.vo_conv2d(ctx.handle, _ptr(x), H, W, cin, _ptr(w), cout, int(k), int(dil), _ptr(scale), _ptr(shift),
                                int(bool(relu)), _ptr(out), _stream()), "vo_conv2d")
    return out


class Correspondences:
    def __init__(self, xyz, ref_uv, cur_uv, src, count, status):
        self.xyz, self.ref_uv, self.cur_uv, self.src, self.count, self.status = xyz, ref_uv, cur_uv, src, count, status


def gather_backproject(pairs, n_pairs, ref_kp, cur_kp, depth, K, min_flow_px=3.0, z_min=0.0, z_max=50.0):
    """Fused gather + flow filter + back-projection + Z gate + compaction (vo_gather_backproject).

    pairs int32 [B,cap,2]; n_pairs int32 [B]; ref_kp [B,N,s], cur_kp [B,M,s] float32 (x,y first);
    depth [B,H,W] float32 of the reference frame."""
    _chk(pairs, torch.int32, "pairs")
    _chk(n_pairs, torch.int32, "n_pairs")
    _chk(ref_kp, torch.float32, "ref_kp")
    _chk(cur_kp, torch.float32, "cur_kp")
    _chk(depth, torch.float32, "depth")
    B, cap = pairs.shape[0], pairs.shape[1]
    dev = pairs.device
    xyz = torch.empty((B, cap, 3), dtype=torch.float32, device=dev)
    ruv = torch.empty((B, cap, 2), dtype=torch.float32, device=dev)
    cuv = torch.empty((B, cap, 2), dtype=torch.float32, device=dev)
    src = torch.empty((B, cap), dtype=torch.int32, device=dev)
    n_out = torch.zeros((B,), dtype=torch.int32, device=dev)
    status = torch.zeros((B,), dtype=torch.int32, device=dev)
    ctx = context(dev)
    kh, kp = _k_host(K)
    with torch.cuda.device(dev):
        check(ctx.lib.vo_gather_backproject(ctx.handle, _ptr(pairs), _ptr(n_pairs), B, cap, _ptr(ref_kp), _ptr(cur_kp),
                                            int(ref_kp.shape[1]), int(cur_kp.shape[1]), int(ref_kp.shape[2]),
                                            _ptr(depth), int(depth.shape[1]), int(depth.shape[2]), kp,
                                            float(min_flow_px), float(z_min), float(z_max), _ptr(xyz), _ptr(ruv),
                                            _ptr(cuv), _ptr(src), _ptr(n_out), _ptr(status), _stream()),
              "vo_gather_backproject")
    return Correspondences(xyz, ruv, cuv, src, n_out, status)


def hypotheses(n_pts, H, seed=8214, pair0=0):
    """Counter-based hypothesis table int32 [B,H,4] (vo_hypotheses)."""
    _chk(n_pts, torch.int32, "n_pts")
    B = n_pts.shape[0]
    hyp = torch.empty((B, H, 4), dtype=torch.int32, device=n_pts.device)
    ctx = context(n_pts.device)
    with torch.cuda.device(n_pts.device):
        check(ctx.lib.vo_hypotheses(ctx.handle, _ptr(n_pts), B, int(H), int(seed), int(pair0), _ptr(hyp), _stream()),
              "vo_hypotheses")
    return hyp


class PnpResult:
    def __init__(self, rt, rvec_tvec, T_rel, n_inl, best_h, mask, hyp_counts, status):
        self.rt, self.rvec_tvec, self.T_rel, self.n_inl = rt, rvec_tvec, T_rel, n_inl
        self.best_h, self.mask, self.hyp_counts, self.status = best_h, mask, hyp_counts, status


def pnp_ransac(xyz, uv, n_pts, K, hyp, thr_px=1.5, min_inliers=20, refine_iters=10, want_counts=False):
    """PnP-RANSAC + refit (vo_pnp_ransac).  xyz [B,cap,3], uv [B,cap,2] float32; hyp int32 [B,H,4]."""
    _chk(xyz, torch.float32, "xyz")
    _chk(uv, torch.float32, "uv")
    _chk(n_pts, torch.int32, "n_pts")
    _chk(hyp, torch.int32, "hyp")
    B, cap = xyz.shape[0], xyz.shape[1]
    H = hyp.shape[1]
    dev = xyz.device
    rt = torch.empty((B, 12), dtype=torch.float64, device=dev)
    rv = torch.empty((B, 6), dtype=torch.float64, device=dev)
    T = torch.empty((B, 4, 4), dtype=torch.float64, device=dev)
    n_inl = torch.zeros((B,), dtype=torch.int32, device=dev)
    best_h = torch.zeros((B,), dtype=torch.int32, device=dev)
    mask = torch.zeros((B, cap), dtype=torch.uint8, device=dev)
    counts = torch.zeros((B, H), dtype=torch.int32, device=dev) if want_counts else None
    status = torch.zeros((B,), dtype=torch.int32, device=dev)
    ctx = context(dev)
    kh, kp = _k_host(K)
    with torch.cuda.device(dev):
        check(ctx.lib.vo_pnp_ransac(ctx.handle, _ptr(xyz), _ptr(uv), _ptr(n_pts), B, cap, kp, _ptr(hyp), H,
                                    float(thr_px), int(min_inliers), int(refine_iters), _ptr(rt), _ptr(rv), _ptr(T),
                                    _ptr(n_inl), _ptr(best_h), _ptr(mask), _ptr(counts), _ptr(status), _stream()),
              "vo_pnp_ransac")
    return PnpResult(rt, rv, T, n_inl, best_h, mask, counts, status)


class PnpRefResult:
    def __init__(self, rt, rvec_tvec, T_rel, n_inl, best, mask, hyp_counts, hyp_poses, status):
        self.rt, self.rvec_tvec, self.T_rel, self.n_inl, self.best = rt, rvec_tvec, T_rel, n_inl, best
        self.mask, self.hyp_counts, self.hyp_poses, self.status = mask, hyp_counts, hyp_poses, status


def pnp_ransac_ref(xyz, uv, n, K, boot_idx, iters=100, thr_px=1.5, confidence=0.99, min_inliers=20, refine_iters=20,
                   want_hyp=False):
    """Reference-sampler PnP-RANSAC (vo_pnp_ransac_ref): xyz [cap,3], uv [cap,2] float32 (one pair's correspondences), n of
    them valid; boot_idx int32 [restarts, n] = the bootstrap rows np.random.randint(0, n, n) (VisualOdometry_Stereo.py:122)."""
    xyz, uv = xyz.reshape(-1, 3), uv.reshape(-1, 2)
    _chk(xyz, torch.float32, "xyz")
    _chk(uv, torch.float32, "uv")
    _chk(boot_idx, torch.int32, "boot_idx")
    if boot_idx.dim() != 2 or boot_idx.shape[1] != n:
        raise ValueError(f"pnp_ransac_ref: boot_idx must be [restarts, {n}], got {tuple(boot_idx.shape)}")
    restarts = int(boot_idx.shape[0])
    dev = xyz.device
    rt = torch.empty((12,), dtype=torch.float64, device=dev)
    rv = torch.empty((6,), dtype=torch.float64, device=dev)
    T = torch.empty((4, 4), dtype=torch.float64, device=dev)
    n_inl = torch.zeros((1,), dtype=torch.int32, device=dev)
    best = torch.zeros((3,), dtype=torch.int32, device=dev)
    mask = torch.zeros((max(n, 1),), dtype=torch.uint8, device=dev)
    counts = torch.zeros((restarts, iters), dtype=torch.int32, device=dev) if want_hyp else None
    poses = torch.zeros((restarts, iters, 12), dtype=torch.float64, device=dev) if want_hyp else None
    status = torch.zeros((1,), dtype=torch.int32, device=dev)
    ctx = context(dev)
    kh, kp = _k_host(K)
    with torch.cuda.device(dev):
        check(ctx.lib.vo_pnp_ransac_ref(ctx.handle, _ptr(xyz), _ptr(uv), int(n), kp, _ptr(boot_idx), restarts, int(iters),
                                        float(thr_px), float(confidence), int(min_inliers), int(refine_iters), _ptr(rt), _ptr(rv),
                                        _ptr(T), _ptr(n_inl), _ptr(best), _ptr(mask), _ptr(counts), _ptr(poses), _ptr(status),
                                        _stream()), "vo_pnp_ransac_ref")
    return PnpRefResult(rt, rv, T, n_inl, best, mask, counts, poses, status)


REF_MAX_RESTARTS, REF_MAX_ITERS = 8, 1024


def bootstrap(n_pts, restarts, cap, seed=8214, pair0=0):
    """Mode R bootstrap rows int32 [B, restarts, cap] (vo_bootstrap): entry [b, r, i] uniform in [0, n_pts[b]) for
    i < n_pts[b], -1 past it; keyed by (seed, pair0 + b, r, i), so a pair's rows do not depend on its batch position."""
    _chk(n_pts, torch.int32, "n_pts")
    B = n_pts.shape[0]
    boot = torch.empty((B, int(restarts), int(cap)), dtype=torch.int32, device=n_pts.device)
    ctx = context(n_pts.device)
    with torch.cuda.device(n_pts.device):
        check(ctx.lib.vo_bootstrap(ctx.handle, _ptr(n_pts), B, int(restarts), int(cap), int(seed), int(pair0), _ptr(boot),
                                   _stream()), "vo_bootstrap")
    return boot


def pnp_ransac_ref_batch(xyz, uv, n_pts, K, boot_idx, iters=100, thr_px=1.5, confidence=0.99, min_inliers=20, refine_iters=20,
                         want_hyp=False):
    """Reference-sampler PnP-RANSAC over B pairs (vo_pnp_ransac_ref_batch): xyz [B,cap,3], uv [B,cap,2] float32, n_pts int32 [B]
    (device: no host read), boot_idx int32 [B,restarts,cap] (bootstrap(), or the caller's rows; first n_pts[b] entries used).
    Pair b's outputs equal pnp_ransac_ref on its first n_pts[b] rows bit for bit; a pair with n_pts[b] outside [0, cap] or an
    index outside [0, n_pts[b]) gets status VO_ST_NO_MODEL | VO_ST_BAD_INPUT and reads nothing."""
    _chk(xyz, torch.float32, "xyz")
    _chk(uv, torch.float32, "uv")
    _chk(n_pts, torch.int32, "n_pts")
    _chk(boot_idx, torch.int32, "boot_idx")
    if xyz.dim() != 3 or xyz.shape[2] != 3:
        raise ValueError(f"pnp_ransac_ref_batch: xyz must be [B, cap, 3], got {tuple(xyz.shape)}")
    B, cap = int(xyz.shape[0]), int(xyz.shape[1])
    if tuple(uv.shape) != (B, cap, 2) or tuple(n_pts.shape) != (B,):
        raise ValueError(f"pnp_ransac_ref_batch: uv {tuple(uv.shape)} / n_pts {tuple(n_pts.shape)} do not match xyz {tuple(xyz.shape)}")
    if boot_idx.dim() != 3 or boot_idx.shape[0] != B or boot_idx.shape[2] != cap:
        raise ValueError(f"pnp_ransac_ref_batch: boot_idx must be [{B}, restarts, {cap}], got {tuple(boot_idx.shape)}")
    restarts = int(boot_idx.shape[1])
    if not 1 <= restarts <= REF_MAX_RESTARTS or not 1 <= int(iters) <= REF_MAX_ITERS:
        raise ValueError(f"pnp_ransac_ref_batch: restarts {restarts} must be in 1..{REF_MAX_RESTARTS}, iters {iters} in "
                         f"1..{REF_MAX_ITERS}")
    dev = xyz.device
    rt = torch.empty((B, 12), dtype=torch.float64, device=dev)
    rv = torch.empty((B, 6), dtype=torch.float64, device=dev)
    T = torch.empty((B, 4, 4), dtype=torch.float64, device=dev)
    n_inl = torch.zeros((B,), dtype=torch.int32, device=dev)
    best = torch.zeros((B, 3), dtype=torch.int32, device=dev)
    mask = torch.zeros((B, max(cap, 1)), dtype=torch.uint8, device=dev)
    counts = torch.zeros((B, restarts, int(iters)), dtype=torch.int32, device=dev) if want_hyp else None
    poses = torch.zeros((B, restarts, int(iters), 12), dtype=torch.float64, device=dev) if want_hyp else None
    status = torch.zeros((B,), dtype=torch.int32, device=dev)
    ctx = context(dev)
    kh, kp = _k_host(K)
    with torch.cuda.device(dev):
        check(ctx.lib.vo_pnp_ransac_ref_batch(ctx.handle, _ptr(xyz), _ptr(uv), _ptr(n_pts), B, cap, kp, _ptr(boot_idx), restarts,
                                              int(iters), float(thr_px), float(confidence), int(min_inliers), int(refine_iters),
                                              _ptr(rt), _ptr(rv), _ptr(T), _ptr(n_inl), _ptr(best), _ptr(mask), _ptr(counts),
                                              _ptr(poses), _ptr(status), _stream()), "vo_pnp_ransac_ref_batch")
    return PnpRefResult(rt, rv, T, n_inl, best, mask, counts, poses, status)


_PNP_MODES = {"throughput": VO_PNP_THROUGHPUT, "reference": VO_PNP_REFERENCE}


def pnp_mode_id(pnp_mode):
    """"throughput" (Mode T, the default) or "reference" (Mode R) -> VO_PNP_*."""
    if pnp_mode not in _PNP_MODES:
        raise ValueError(f"pnp_mode must be 'throughput' or 'reference', got {pnp_mode!r}")
    return _PNP_MODES[pnp_mode]


class PipelineResult:
    def __init__(self, T_rel, rt, n_matches, n_corr, n_inl, status):
        self.T_rel, self.rt, self.n_matches, self.n_corr, self.n_inl, self.status = T_rel, rt, n_matches, n_corr, n_inl, status


class PipelineBuffers:
    """Pre-allocated outputs for repeated vo_pipeline calls on a fixed batch size."""

    def __init__(self, B, device):
        self.T_rel = torch.empty((B, 4, 4), dtype=torch.float64, device=device)
        self.rt = torch.empty((B, 12), dtype=torch.float64, device=device)
        self.n_matches = torch.zeros((B,), dtype=torch.int32, device=device)
        self.n_corr = torch.zeros((B,), dtype=torch.int32, device=device)
        self.n_inl = torch.zeros((B,), dtype=torch.int32, device=device)
        self.status = torch.zeros((B,), dtype=torch.int32, device=device)


def pipeline(ref_desc, cur_desc, ref_kp, cur_kp, depth, K, *, norm_or_metric, mode, match_param=0.85,
             precision=VO_PREC_TF32X3, n_ref=None, n_cur=None, n_hyp=1024, seed=8214, pair0=0, thr_px=1.5,
             min_inliers=20, refine_iters=10, min_flow_px=3.0, z_min=0.0, z_max=50.0, out=None, depth_kp=None, hw=None,
             lane=0, pnp_mode="throughput", ref_restarts=3, ref_iters=100, ref_confidence=0.99):
    """match -> gather/back-project -> hypotheses -> PnP-RANSAC -> T_rel for a batch of pairs (vo_pipeline).
    pnp_mode "reference" runs Mode R instead of the hypotheses and P3P RANSAC: bootstrap(n_corr, ref_restarts, N, seed, pair0)
    -> pnp_ransac_ref_batch(ref_iters, thr_px, ref_confidence, min_inliers, refine_iters); n_hyp is then ignored.
    `depth` is the reference frames' dense map [B,H,W], on the device or in pinned host memory (then only the pixels
    under the matched reference keypoints cross the bus, read zero-copy by the gather kernel); alternatively pass
    `depth_kp` [B,N] (sample_depth) and `hw=(H, W)`.  `lane` selects the vo_ctx (see context())."""
    _chk(ref_kp, torch.float32, "ref_kp")
    _chk(cur_kp, torch.float32, "cur_kp")
    if depth_kp is not None:
        _chk(depth_kp, torch.float32, "depth_kp")
        if hw is None and depth is None:
            raise ValueError("pipeline: depth_kp needs hw=(H, W)")
    elif depth.dtype != torch.float32 or not depth.is_contiguous() or not (depth.is_cuda or depth.is_pinned()):
        raise ValueError("pipeline: depth must be contiguous float32 on the device or in pinned host memory")
    if not ref_desc.is_contiguous() or not cur_desc.is_contiguous():
        raise ValueError("pipeline: descriptors must be contiguous")
    B, N, M = ref_desc.shape[0], ref_desc.shape[1], cur_desc.shape[1]
    dev = ref_desc.device
    out = out or PipelineBuffers(B, dev)
    kh, kp = _k_host(K)
    a = PipelineArgs()
    a.B, a.n_stride, a.m_stride = B, N, M
    a.n_ref, a.n_cur = (n_ref.data_ptr() if n_ref is not None else None), (n_cur.data_ptr() if n_cur is not None else None)
    if ref_desc.dtype == torch.uint8:
        a.ref_u8, a.cur_u8 = ref_desc.data_ptr(), cur_desc.data_ptr()
        a.u8_bytes = int(ref_desc.shape[2])          # 32: 256-bit descriptors; 128: SIFT values as uint8 (VO_NORM_L2_U8)
    elif ref_desc.dtype == torch.float32:
        a.ref_f32, a.cur_f32 = ref_desc.data_ptr(), cur_desc.data_ptr()
    else:
        raise ValueError("pipeline: descriptors must be uint8 or float32")
    a.norm_or_metric, a.mode, a.precision, a.match_param = int(norm_or_metric), int(mode), int(precision), float(match_param)
    a.ref_kp, a.cur_kp, a.kp_stride = ref_kp.data_ptr(), cur_kp.data_ptr(), int(ref_kp.shape[2])
    if depth_kp is not None:
        a.depth, a.depth_kp = None, depth_kp.data_ptr()
        a.H, a.W = (int(hw[0]), int(hw[1])) if hw is not None else (int(depth.shape[1]), int(depth.shape[2]))
    else:
        a.depth, a.H, a.W = depth.data_ptr(), int(depth.shape[1]), int(depth.shape[2])
    a.K_h = kp.value
    a.min_flow_px, a.z_min, a.z_max = float(min_flow_px), float(z_min), float(z_max)
    a.n_hyp, a.seed, a.pair0 = int(n_hyp), int(seed), int(pair0)
    a.thr_px, a.min_inliers, a.refine_iters = float(thr_px), int(min_inliers), int(refine_iters)
    a.pnp_mode = pnp_mode_id(pnp_mode)
    if a.pnp_mode == VO_PNP_REFERENCE:
        if not 1 <= int(ref_restarts) <= REF_MAX_RESTARTS or not 1 <= int(ref_iters) <= REF_MAX_ITERS:
            raise ValueError(f"pipeline: ref_restarts {ref_restarts} must be in 1..{REF_MAX_RESTARTS}, ref_iters {ref_iters} in "
                             f"1..{REF_MAX_ITERS}")
        a.ref_restarts, a.ref_iters, a.ref_confidence = int(ref_restarts), int(ref_iters), float(ref_confidence)
    a.T_rel, a.rt = out.T_rel.data_ptr(), out.rt.data_ptr()
    a.n_matches, a.n_corr = out.n_matches.data_ptr(), out.n_corr.data_ptr()
    a.n_inl, a.status = out.n_inl.data_ptr(), out.status.data_ptr()
    ctx = context(dev, lane)
    with torch.cuda.device(dev):
        check(ctx.lib.vo_pipeline(ctx.handle, ctypes.byref(a), _stream()), "vo_pipeline")
    return PipelineResult(out.T_rel, out.rt, out.n_matches, out.n_corr, out.n_inl, out.status)
