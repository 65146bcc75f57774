"""Device-resident keyframe loop (vo_seq_*): the control flow of VisualOdometry.process_frame
(VisualOdometry_Stereo.py:232-297) kept on the GPU.

`DeviceLoop.push(kp, desc, depth, frame_no)` only enqueues work (copies into the loop's frame slot, vo_pipeline
against the keyframe slot, a one-thread policy kernel for the gates / bad-PnP counter / pose chaining / keyframe
rule, a conditional slot promotion).  `poses()` synchronises once and returns what the reference keeps in
`global_poses` (:293).  Features come from the caller (the front-ends stay on the host, SURVEY 8(f) rank 1).
"""
import ctypes

import numpy as np
import torch

from . import _lib, ops
from ._lib import SeqConfig, check


def _seq_config(who, K, wh, n_cap, *, kind="orb", kp_stride=2, norm_or_metric=None, mode=None, match_param=0.85,
                precision=None, allow_inexact=False, n_hyp=512, seed=8214, thr_px=1.5, min_inliers=20, refine_iters=10,
                min_flow_px=3.0, z_range=(0.0, 50.0), max_step_m=1.5, kf_min_common=200, kf_min_inliers=100,
                kf_max_dist=1.5, bad_pnp_limit=3, max_frames=4096, pnp_mode="throughput", ref_restarts=3,
                ref_iters=100, ref_confidence=0.99):
    """Validated vo_seq_config of a loop (one sequence; MultiDeviceLoop sets n_seqs / seeds) and whether its pushes must
    check for integer-valued descriptors."""
    f32 = kind != "orb"
    if norm_or_metric is None:
        norm_or_metric = {"orb": ops.VO_NORM_L2_U8, "sift": ops.VO_METRIC_L2}.get(kind, ops.VO_METRIC_COSINE)
    if mode is None:
        mode = ops.VO_MODE_RATIO_MUTUAL if kind == "r2d2" else ops.VO_MODE_RATIO
    # one 11-bit pass is exact only on integer-valued descriptors in 0..255 (OpenCV SIFT); unit-norm R2D2 descriptors need
    # the split passes to reproduce the reference's fp32 `d1 @ d2.t()` decisions (R2D2.py:56-65).  A SIFT loop left on
    # its default F16X1 pass checks that its descriptors are such integers (push), so RootSIFT or another normalised
    # variant is refused instead of silently matched with 11-bit products.
    check_int = precision is None and kind == "sift"
    if precision is None:
        precision = ops.VO_PREC_F16X1 if kind == "sift" else ops.VO_PREC_TF32X3
    if (f32 and norm_or_metric == ops.VO_METRIC_COSINE and precision in (ops.VO_PREC_TF32X1, ops.VO_PREC_F16X1)
            and not allow_inexact):
        raise ValueError(f"{who}: a single 11-bit pass (TF32X1 / F16X1) on cosine similarities of real-valued "
                         "descriptors changes ratio / mutual decisions (~1e-3 similarity error); use TF32X3 / F16X3 "
                         "or pass allow_inexact=True")
    c = SeqConfig()
    c.desc_is_f32, c.n_cap, c.kp_stride, c.H, c.W = int(f32), int(n_cap), int(kp_stride), int(wh[1]), int(wh[0])
    c.K = (ctypes.c_double * 9)(*np.asarray(K, np.float64).reshape(9))
    c.norm_or_metric, c.mode, c.precision, c.match_param = int(norm_or_metric), int(mode), int(precision), float(match_param)
    c.min_flow_px, c.z_min, c.z_max = float(min_flow_px), float(z_range[0]), float(z_range[1])
    c.n_hyp, c.seed, c.thr_px = int(n_hyp), int(seed), float(thr_px)
    c.min_inliers, c.refine_iters = int(min_inliers), int(refine_iters)
    c.max_step_m, c.kf_min_common, c.kf_min_inliers = float(max_step_m), int(kf_min_common), int(kf_min_inliers)
    c.kf_max_dist, c.bad_pnp_limit, c.max_frames = float(kf_max_dist), int(bad_pnp_limit), int(max_frames)
    c.pnp_mode = ops.pnp_mode_id(pnp_mode)
    if c.pnp_mode == ops.VO_PNP_REFERENCE:
        if not 1 <= int(ref_restarts) <= ops.REF_MAX_RESTARTS or not 1 <= int(ref_iters) <= ops.REF_MAX_ITERS:
            raise ValueError(f"{who}: ref_restarts {ref_restarts} must be in 1..{ops.REF_MAX_RESTARTS}, ref_iters "
                             f"{ref_iters} in 1..{ops.REF_MAX_ITERS}")
        c.ref_restarts, c.ref_iters, c.ref_confidence = int(ref_restarts), int(ref_iters), float(ref_confidence)
    return c, check_int


def _check_integer_descriptors(who, desc):
    """True if `desc` (numpy or torch) holds integers in 0..255; raises otherwise (the default SIFT pass, F16X1, is exact
    only for those)."""
    if isinstance(desc, torch.Tensor):
        ok = bool(((desc == desc.round()) & (desc >= 0) & (desc <= 255)).all().item()) if desc.numel() else True
    else:
        ok = bool(np.all((desc == np.rint(desc)) & (desc >= 0) & (desc <= 255)))
    if not ok:
        raise ValueError(f"{who}: descriptors are not integers in 0..255 (RootSIFT or another normalised "
                         "variant?); the default SIFT pass (F16X1, 11-bit operands) is exact only for those.  Create the "
                         "loop with precision=ops.VO_PREC_TF32X3")


def _ptr(a):
    if isinstance(a, torch.Tensor):
        return ctypes.c_void_p(a.data_ptr())
    return a.ctypes.data_as(ctypes.c_void_p)


class DeviceLoop:
    def __init__(self, K, wh, n_cap, *, device=None, **options):
        """Options (keyword): kind ("orb" / "sift" / "r2d2"), kp_stride, norm_or_metric, mode, match_param, precision,
        allow_inexact, n_hyp, seed, thr_px, min_inliers, refine_iters, min_flow_px, z_range, max_step_m, kf_min_common,
        kf_min_inliers, kf_max_dist, bad_pnp_limit, max_frames, pnp_mode, ref_restarts, ref_iters, ref_confidence.
        pnp_mode "reference": every frame runs Mode R (vo_bootstrap keyed by the frame's history slot - 1, then the batched
        reference-sampler RANSAC with B = 1); such a loop always launches plainly (VO_SEQ_GRAPH does not apply to it)."""
        self.device = torch.device("cuda", torch.cuda.current_device()) if device is None else torch.device(device)
        self.ctx = ops.context(self.device)
        c, self._check_int = _seq_config("DeviceLoop", K, wh, n_cap, **options)
        self.cfg = c
        self.desc_dtype = np.float32 if c.desc_is_f32 else np.uint8
        self.desc_cols = 128 if c.desc_is_f32 else 32
        h = ctypes.c_void_p()
        with torch.cuda.device(self.device):
            check(self.ctx.lib.vo_seq_create(self.ctx.handle, ctypes.byref(c), ctypes.byref(h)), "vo_seq_create")
        self.handle = h
        self._keep = []          # host staging arrays must outlive the asynchronous copies

    _ptr = staticmethod(_ptr)

    def push(self, kp, desc, depth, frame_no):
        """kp (n, >=2) array-like (x, y first), desc (n, 32) uint8 or (n, 128) float32, depth (H, W) float32.
        numpy arrays (copied from host memory) or torch tensors (device or pinned) are accepted."""
        c = self.cfg
        if isinstance(kp, torch.Tensor):
            kp_a = kp[:, :c.kp_stride].to(torch.float32).contiguous()
            n = int(kp_a.shape[0])
        else:
            kp_a = np.ascontiguousarray(np.asarray(kp)[:, :c.kp_stride], dtype=np.float32)
            n = int(kp_a.shape[0])
        if isinstance(desc, torch.Tensor):
            desc_a = desc.contiguous()
        else:
            desc_a = np.ascontiguousarray(desc, dtype=self.desc_dtype)
        if tuple(desc_a.shape) != (n, self.desc_cols):
            raise ValueError(f"DeviceLoop.push: descriptors {tuple(desc_a.shape)} do not match {n} keypoints x {self.desc_cols}")
        if self._check_int:
            self._check_integer_descriptors(desc_a)
        if isinstance(depth, torch.Tensor):
            depth_a = depth.to(torch.float32).contiguous()
        else:
            depth_a = np.ascontiguousarray(depth, dtype=np.float32)
        if tuple(depth_a.shape) != (c.H, c.W):
            raise ValueError(f"DeviceLoop.push: depth {tuple(depth_a.shape)} != ({c.H}, {c.W})")
        self._keep.append((kp_a, desc_a, depth_a))
        with torch.cuda.device(self.device):
            stream = ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)
            check(self.ctx.lib.vo_seq_push(self.handle, self._ptr(desc_a), self._ptr(kp_a), n, self._ptr(depth_a),
                                           int(frame_no), stream), "vo_seq_push")

    def _check_integer_descriptors(self, desc):
        """The default SIFT pass (F16X1) is exact only for integers in 0..255.  Host arrays are checked on every push (no
        device work).  Device tensors are checked on the first non-empty push only: the check needs a host read, which would stall
        the otherwise asynchronous loop on every frame, and a device-side producer emits the same kind of descriptor on
        every frame."""
        if isinstance(desc, torch.Tensor) and desc.is_cuda and desc.numel():
            self._check_int = False
        _check_integer_descriptors("DeviceLoop.push", desc)

    def push_image(self, image, depth, frame_no, nfeatures=500, frontend=None):
        """Extract on the device and push — the image is the only per-frame upload besides the depth map; one host read of
        the keypoint count per frame.  frontend: "orb" (orb_frontend.OrbExtractor, cv2.ORB_create(nfeatures) semantics; the
        default of a byte-descriptor loop) or "sift" (sift_frontend.SiftExtractor; the default of a float-descriptor loop).
        Both extractors are parity-tested on a B200 (tests/test_gpu_orb_frontend.py, tests/test_gpu_sift_frontend.py)."""
        frontend = frontend or ("orb" if self.desc_cols == 32 else "sift")
        if (frontend == "orb") != (self.desc_cols == 32) or frontend not in ("orb", "sift"):
            raise ValueError(f"DeviceLoop.push_image: front-end {frontend!r} does not produce this loop's descriptors")
        if getattr(self, "_extractor", None) is None:
            if frontend == "orb":
                from .orb_frontend import OrbExtractor
                self._extractor = OrbExtractor(self.cfg.H, self.cfg.W, nfeatures=nfeatures, device=self.device)
            else:
                from .sift_frontend import SiftExtractor
                self._extractor = SiftExtractor(self.cfg.H, self.cfg.W, max_keypoints=self.cfg.n_cap, device=self.device)
        kp, desc, _ = self._extractor.extract(image)
        return self.push(kp, desc, depth, frame_no)

    def __len__(self):
        return int(self.ctx.lib.vo_seq_frames(self.handle))

    def poses(self, first=0, count=None):
        """(poses (count,4,4) f64, info (count,6) int32: status, n_matches, n_corr, n_inl, keyframe id, promoted).
        Synchronises the stream."""
        n = len(self)
        count = n - first if count is None else count
        poses = np.empty((count, 4, 4), np.float64)
        info = np.empty((count, 6), np.int32)
        with torch.cuda.device(self.device):
            stream = ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)
            check(self.ctx.lib.vo_seq_read(self.handle, int(first), int(count), self._ptr(poses), self._ptr(info), stream),
                  "vo_seq_read")
        self._keep.clear()
        return poses, info

    def close(self):
        if getattr(self, "handle", None):
            self.ctx.lib.vo_seq_destroy(self.handle)
            self.handle = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


class MultiDeviceLoop:
    """S independent sequences in lock-step: one `push` is one step of every sequence, run as ONE vo_pipeline batch of
    B = S pairs (each sequence's current frame against its own keyframe) followed by the per-sequence policy and promotion on
    the device.  Sequence q draws from (seeds[q], its frame slot - 1), so `poses(q)` equals, bit for bit, what
    `DeviceLoop(seed=seeds[q])` gives for the same frames.  A sequence may start late, end early or skip steps (n_kp < 0).
    `push_images` starts a step from the S camera images instead (batched ORB or SIFT on the device, no host read per step).

    Options are DeviceLoop's (seed is the default seed base: seeds = seed + q when `seeds` is None)."""

    def __init__(self, K, wh, n_cap, n_seqs, *, seeds=None, device=None, **options):
        S = int(n_seqs)
        if S < 1:
            raise ValueError(f"MultiDeviceLoop: n_seqs {n_seqs} must be >= 1")
        self.device = torch.device("cuda", torch.cuda.current_device()) if device is None else torch.device(device)
        self.ctx = ops.context(self.device)
        c, self._check_int = _seq_config("MultiDeviceLoop", K, wh, n_cap, **options)
        if seeds is not None:
            seeds = np.ascontiguousarray(seeds, dtype=np.uint64)
            if seeds.shape != (S,):
                raise ValueError(f"MultiDeviceLoop: seeds {seeds.shape} must hold one seed per sequence ({S},)")
            c.seeds = seeds.ctypes.data_as(ctypes.c_void_p)     # copied by vo_seq_create
        c.n_seqs = S
        self.cfg, self.n_seqs = c, S
        self.desc_dtype = np.float32 if c.desc_is_f32 else np.uint8
        self.desc_cols = 128 if c.desc_is_f32 else 32
        h = ctypes.c_void_p()
        with torch.cuda.device(self.device):
            check(self.ctx.lib.vo_seq_create(self.ctx.handle, ctypes.byref(c), ctypes.byref(h)), "vo_seq_create")
        self.handle = h
        self._keep = []          # host staging arrays must outlive the asynchronous copies

    def push(self, kp, desc, n_kp, depth, frame_no):
        """One step of every sequence, in the loop's slot layout: kp (S, n_cap, >= kp_stride) (x, y first), desc
        (S, n_cap, 32) uint8 or (S, n_cap, 128) float32, n_kp (S,) valid rows per sequence (< 0: no frame at this step),
        depth (S, H, W) float32, frame_no (S,) or one int for all.  numpy arrays or torch tensors (device or pinned)."""
        c, S = self.cfg, self.n_seqs
        n_kp = np.ascontiguousarray(n_kp, dtype=np.int32)
        frame_no = np.ascontiguousarray(np.broadcast_to(np.asarray(frame_no), (S,)), dtype=np.int32)
        if n_kp.shape != (S,):
            raise ValueError(f"MultiDeviceLoop.push: n_kp {n_kp.shape} must be ({S},)")
        if isinstance(kp, torch.Tensor):
            kp_a = kp[:, :, :c.kp_stride].to(torch.float32).contiguous() if kp.dim() == 3 else kp
        else:
            kp = np.asarray(kp)
            kp_a = np.ascontiguousarray(kp[:, :, :c.kp_stride], dtype=np.float32) if kp.ndim == 3 else kp
        desc_a = desc.contiguous() if isinstance(desc, torch.Tensor) else np.ascontiguousarray(desc, dtype=self.desc_dtype)
        if isinstance(depth, torch.Tensor):
            depth_a = depth.to(torch.float32).contiguous()
        else:
            depth_a = np.ascontiguousarray(depth, dtype=np.float32)
        for name, a, want in (("kp", kp_a, (S, c.n_cap, c.kp_stride)), ("desc", desc_a, (S, c.n_cap, self.desc_cols)),
                              ("depth", depth_a, (S, c.H, c.W))):
            if tuple(a.shape) != want:
                raise ValueError(f"MultiDeviceLoop.push: {name} {tuple(a.shape)} != {want}")
        if isinstance(desc_a, torch.Tensor) and desc_a.dtype != (torch.float32 if c.desc_is_f32 else torch.uint8):
            raise ValueError(f"MultiDeviceLoop.push: descriptors of dtype {desc_a.dtype} in a loop of {self.desc_dtype.__name__}")
        if self._check_int:
            rows = np.arange(c.n_cap)[None, :] < np.minimum(n_kp, c.n_cap)[:, None]
            if isinstance(desc_a, torch.Tensor):
                valid = desc_a[torch.from_numpy(rows).to(desc_a.device)]
                if desc_a.is_cuda and valid.numel():
                    self._check_int = False      # device producers: checked on the first non-empty step (a host read)
            else:
                valid = desc_a[rows]
            _check_integer_descriptors("MultiDeviceLoop.push", valid)
        self._keep.append((kp_a, desc_a, depth_a))
        with torch.cuda.device(self.device):
            stream = ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)
            check(self.ctx.lib.vo_seq_push_all(self.handle, _ptr(desc_a), _ptr(kp_a), _ptr(n_kp), _ptr(depth_a),
                                               _ptr(frame_no), stream), "vo_seq_push_all")

    def push_images(self, images, depth, frame_no, present=None, nfeatures=500, max_keypoints=32768):
        """One step of every sequence from its image: images uint8 torch tensor (S, H, W) gray or (S, H, W, 3) BGR, on the
        device or pinned; depth (S, H, W) float32 (torch, device or pinned, or numpy); frame_no (S,) or one int; present
        (S,) truthy where a sequence has a frame at this step (default: all).  The front-end follows the loop's
        descriptors, as in DeviceLoop.push_image: a byte-descriptor loop runs ORB (cv2.ORB_create(nfeatures) semantics,
        OrbExtractor.extract_batch), a float-descriptor loop with kp_stride 2 runs SIFT (cv2.SIFT_create() semantics,
        SiftExtractor.extract_batch), each on all S images in one batched call with rows = n_cap, and the keypoint counts
        reach the loop on the device (vo_seq_push_all_dev): the call only enqueues work.  The images of absent sequences
        are extracted too (the batch has a fixed shape) and their results ignored.  A frame with more keypoints than n_cap
        keeps its first n_cap rows and counts in lost_frames(q): for ORB level-major, then row-major; for SIFT in OpenCV's
        order (sorted by x), so the left of the image is kept.  A SIFT frame whose raw list passes max_keypoints (the raw
        candidate capacity per image) counts too.  SIFT descriptors are integers in 0..255 by construction, so the default
        F16X1 pass gets no integer check here (it would cost a host read per step).  The loop holds the images and depth
        until poses() synchronises; do not write into them before then.  nfeatures (ORB) and max_keypoints (SIFT) are
        read when the extractor is created, at the first call.  R2D2 loops (kp_stride 3) are refused."""
        c, S = self.cfg, self.n_seqs
        if c.kp_stride != 2:
            raise ValueError("MultiDeviceLoop.push_images: images need an ORB (byte-descriptor) or SIFT (float-descriptor) "
                             "loop with kp_stride 2")
        present = np.ones(S, np.int32) if present is None else np.ascontiguousarray(present, dtype=bool).astype(np.int32)
        frame_no = np.ascontiguousarray(np.broadcast_to(np.asarray(frame_no), (S,)), dtype=np.int32)
        if present.shape != (S,):
            raise ValueError(f"MultiDeviceLoop.push_images: present {present.shape} must be ({S},)")
        if not isinstance(images, torch.Tensor) or images.shape[0] != S:
            raise ValueError(f"MultiDeviceLoop.push_images: images must be a torch tensor of {S} images")
        if isinstance(depth, torch.Tensor):
            depth_a = depth.to(torch.float32).contiguous()
        else:
            depth_a = np.ascontiguousarray(depth, dtype=np.float32)
        if tuple(depth_a.shape) != (S, c.H, c.W):
            raise ValueError(f"MultiDeviceLoop.push_images: depth {tuple(depth_a.shape)} != {(S, c.H, c.W)}")
        if getattr(self, "_extractor", None) is None:
            if c.desc_is_f32:
                from .sift_frontend import SiftExtractor
                self._extractor = SiftExtractor(c.H, c.W, max_keypoints=max_keypoints, device=self.device)
            else:
                from .orb_frontend import OrbExtractor
                self._extractor = OrbExtractor(c.H, c.W, nfeatures=nfeatures, device=self.device)
        kp, desc, _, count = self._extractor.extract_batch(images, rows=c.n_cap)
        # the kernels read pinned images and depth asynchronously: hold them (a dropped pinned tensor's block is handed to
        # the next pin_memory() and overwritten) until poses() has synchronised; kp / desc / count are device tensors of
        # this stream, ordered by it
        self._keep.append((images, depth_a))
        with torch.cuda.device(self.device):
            stream = ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)
            check(self.ctx.lib.vo_seq_push_all_dev(self.handle, _ptr(desc), _ptr(kp), _ptr(count), _ptr(present),
                                                   _ptr(depth_a), _ptr(frame_no), stream), "vo_seq_push_all_dev")

    def lost_frames(self, q):
        """Frames of sequence q pushed by push_images (or vo_seq_push_all_dev) that lost keypoint rows: more keypoints than
        n_cap, or an extractor flag (an ORB pyramid level overflowed, a SIFT raw list passed max_keypoints).  Synchronises
        the stream."""
        if not 0 <= int(q) < self.n_seqs:
            raise IndexError(f"MultiDeviceLoop: sequence {q} outside [0, {self.n_seqs})")
        out = np.zeros(1, np.int32)
        with torch.cuda.device(self.device):
            stream = ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)
            check(self.ctx.lib.vo_seq_lost_frames_at(self.handle, int(q), _ptr(out), stream), "vo_seq_lost_frames_at")
        return int(out[0])

    def frames(self, q):
        """Frames pushed to sequence q."""
        if not 0 <= int(q) < self.n_seqs:
            raise IndexError(f"MultiDeviceLoop: sequence {q} outside [0, {self.n_seqs})")
        return int(self.ctx.lib.vo_seq_frames_at(self.handle, int(q)))

    def poses(self, q, first=0, count=None):
        """Sequence q's (poses (count,4,4) f64, info (count,6) int32), as DeviceLoop.poses.  Synchronises the stream."""
        n = self.frames(q)
        count = n - first if count is None else count
        poses = np.empty((count, 4, 4), np.float64)
        info = np.empty((count, 6), np.int32)
        with torch.cuda.device(self.device):
            stream = ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)
            check(self.ctx.lib.vo_seq_read_at(self.handle, int(q), int(first), int(count), _ptr(poses), _ptr(info), stream),
                  "vo_seq_read_at")
        self._keep.clear()
        return poses, info

    def close(self):
        if getattr(self, "handle", None):
            self.ctx.lib.vo_seq_destroy(self.handle)
            self.handle = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass
