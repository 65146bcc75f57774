"""ORB front-end on the GPU (vo_orb_create / vo_orb_extract): cv2.ORB_create().detectAndCompute with the reference's
default parameters (feature_extractors/ORB.py:8-21).

Bit-identical to the CPU restatement pinned on OpenCV (identical keypoint set, pt, angle, response, descriptors) on a B200:
tests/test_gpu_orb_frontend.py; tools/orb_bisect.py compares every stage.  Default extractor of feature_extractors/ORB.py."""
import ctypes

import numpy as np
import torch

from . import ops
from ._lib import OrbConfig, VoError, check


class OrbExtractor:
    """orb = OrbExtractor(H, W); kp, desc, aux = orb.extract(image_uint8)   (image [H,W] gray or [H,W,3] BGR).

    kp [n,2] float32 = KeyPoint.pt, desc [n,32] uint8, aux [n,4] float32 = (octave, angle, response, size); rows in
    level-major, then row-major order (OpenCV's own order is unspecified).  extract_batch runs S images in one call."""

    def __init__(self, H, W, nfeatures=500, nlevels=8, fast_threshold=20, device=None):
        self.device = torch.device("cuda", torch.cuda.current_device()) if device is None else torch.device(device)
        self.ctx = ops.context(self.device)
        self.H, self.W = int(H), int(W)
        cfg = OrbConfig(self.H, self.W, int(nfeatures), int(nlevels), int(fast_threshold))
        h = ctypes.c_void_p()
        with torch.cuda.device(self.device):
            check(self.ctx.lib.vo_orb_create(self.ctx.handle, ctypes.byref(cfg), ctypes.byref(h)), "vo_orb_create")
        self.handle = h
        self.cap = int(self.ctx.lib.vo_orb_capacity(h))
        self.kp = torch.empty((self.cap, 2), dtype=torch.float32, device=self.device)
        self.desc = torch.empty((self.cap, 32), dtype=torch.uint8, device=self.device)
        self.aux = torch.empty((self.cap, 4), dtype=torch.float32, device=self.device)
        self.count = torch.zeros((2,), dtype=torch.int32, device=self.device)

    def extract(self, image):
        if isinstance(image, np.ndarray):
            image = torch.from_numpy(np.ascontiguousarray(image)).to(self.device)
        if image.dtype != torch.uint8 or not image.is_contiguous() or not (image.is_cuda or image.is_pinned()):
            raise ValueError("OrbExtractor.extract: image must be contiguous uint8 on the device or in pinned host memory")
        if tuple(image.shape[:2]) != (self.H, self.W) or (image.dim() == 3 and image.shape[2] != 3) or image.dim() not in (2, 3):
            raise ValueError(f"OrbExtractor.extract: expected [{self.H},{self.W}] or [{self.H},{self.W},3], got {tuple(image.shape)}")
        with torch.cuda.device(self.device):
            check(self.ctx.lib.vo_orb_extract(self.handle, ctypes.c_void_p(image.data_ptr()), 1 if image.dim() == 2 else 3,
                                              ctypes.c_void_p(self.kp.data_ptr()), ctypes.c_void_p(self.desc.data_ptr()),
                                              ctypes.c_void_p(self.aux.data_ptr()), ctypes.c_void_p(self.count.data_ptr()),
                                              ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)), "vo_orb_extract")
        n, overflow = (int(v) for v in self.count.cpu())
        if overflow:
            raise VoError("vo_orb_extract: a pyramid level kept more tied keypoints than the output holds")
        return self.kp[:n], self.desc[:n], self.aux[:n]

    def extract_batch(self, images, rows=None):
        """S images in one call of the same 17 kernels (vo_orb_extract_batch), with no host read: images uint8 torch tensor
        [S,H,W] (gray) or [S,H,W,3] (BGR), contiguous, on this device or in pinned host memory.  Returns device tensors
        kp [S,rows,2], desc [S,rows,32], aux [S,rows,4] and count int32 [S,2] = (rows written, flags); image s's first
        count[s,0] rows are the first rows `extract` gives for it (the rest are unspecified).  Flag bit 0: a level kept more
        tied keypoints than it holds (where `extract` raises); bit 1: rows past `rows` were dropped.  rows defaults to
        vo_orb_capacity (nothing is ever dropped).  Pinned images are read by the kernels after the call returns: keep them
        alive and unchanged until the stream has passed this call."""
        if not isinstance(images, torch.Tensor):
            raise ValueError("OrbExtractor.extract_batch: images must be a torch tensor")
        if images.dtype != torch.uint8 or not images.is_contiguous() or not (images.is_cuda or images.is_pinned()):
            raise ValueError("OrbExtractor.extract_batch: images must be contiguous uint8 on the device or in pinned host memory")
        if images.is_cuda and images.device != self.device:
            raise ValueError(f"OrbExtractor.extract_batch: images on {images.device}, extractor on {self.device}")
        if (images.dim() not in (3, 4) or tuple(images.shape[1:3]) != (self.H, self.W)
                or (images.dim() == 4 and images.shape[3] != 3) or images.shape[0] < 1):
            raise ValueError(f"OrbExtractor.extract_batch: expected [S,{self.H},{self.W}] or [S,{self.H},{self.W},3] with "
                             f"S >= 1, got {tuple(images.shape)}")
        S = int(images.shape[0])
        rows = self.cap if rows is None else int(rows)
        if rows < 1:
            raise ValueError(f"OrbExtractor.extract_batch: rows {rows} must be >= 1")
        kp = torch.empty((S, rows, 2), dtype=torch.float32, device=self.device)
        desc = torch.empty((S, rows, 32), dtype=torch.uint8, device=self.device)
        aux = torch.empty((S, rows, 4), dtype=torch.float32, device=self.device)
        count = torch.empty((S, 2), dtype=torch.int32, device=self.device)
        ptr = lambda t: ctypes.c_void_p(t.data_ptr())  # noqa: E731
        with torch.cuda.device(self.device):
            check(self.ctx.lib.vo_orb_extract_batch(self.handle, ptr(images), S, 1 if images.dim() == 3 else 3, rows, ptr(kp),
                                                    ptr(desc), ptr(aux), ptr(count),
                                                    ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)),
                  "vo_orb_extract_batch")
        return kp, desc, aux, count

    def close(self):
        if self.handle:
            self.ctx.lib.vo_orb_destroy(self.handle)
            self.handle = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass
