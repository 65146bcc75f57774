"""SIFT front-end on the GPU (vo_sift_create / vo_sift_extract): cv2.SIFT_create().detectAndCompute with the reference's
default parameters (feature_extractors/SIFT.py:10-23), held to a tolerance (same keypoints to 1e-2 px / 0.25 degrees,
descriptor entries within 1 — OpenCV's own low-order bits depend on the host CPU).

Verified against the CPU restatement under the host emulation (tests/test_sift_emulation.py) and on a B200
(tests/test_gpu_sift_frontend.py, strict).  Default extractor of the drop-in plug-in feature_extractors/SIFT.py."""
import ctypes

import numpy as np
import torch

from . import ops
from ._lib import SiftConfig, VoError, check


class SiftExtractor:
    """sift = SiftExtractor(H, W); kp, desc, aux = sift.extract(image_uint8)   (image [H,W] gray or [H,W,3] BGR).

    kp [n,2] float32 = KeyPoint.pt, desc [n,128] float32 (0..255), aux [n,4] float32 = (size, angle, response, octave word);
    rows in OpenCV's order (sorted by x, y, ...; duplicates removed).  extract_batch runs S images in one call."""

    def __init__(self, H, W, max_keypoints=32768, device=None):
        self.device = torch.device("cuda", torch.cuda.current_device()) if device is None else torch.device(device)
        self.ctx = ops.context(self.device)
        self.H, self.W, self.cap = int(H), int(W), int(max_keypoints)
        cfg = SiftConfig(self.H, self.W, self.cap)
        h = ctypes.c_void_p()
        with torch.cuda.device(self.device):
            check(self.ctx.lib.vo_sift_create(self.ctx.handle, ctypes.byref(cfg), ctypes.byref(h)), "vo_sift_create")
        self.handle = h
        self.kp = torch.empty((self.cap, 2), dtype=torch.float32, device=self.device)
        self.desc = torch.empty((self.cap, 128), dtype=torch.float32, device=self.device)
        self.aux = torch.empty((self.cap, 4), dtype=torch.float32, device=self.device)
        self.count = torch.zeros((2,), dtype=torch.int32, device=self.device)

    def extract(self, image):
        if isinstance(image, np.ndarray):
            image = torch.from_numpy(np.ascontiguousarray(image)).to(self.device)
        if image.dtype != torch.uint8 or not image.is_contiguous() or not (image.is_cuda or image.is_pinned()):
            raise ValueError("SiftExtractor.extract: image must be contiguous uint8 on the device or in pinned host memory")
        if tuple(image.shape[:2]) != (self.H, self.W) or (image.dim() == 3 and image.shape[2] != 3) or image.dim() not in (2, 3):
            raise ValueError(f"SiftExtractor.extract: expected [{self.H},{self.W}] or [{self.H},{self.W},3], got {tuple(image.shape)}")
        p = lambda t: ctypes.c_void_p(t.data_ptr())  # noqa: E731
        with torch.cuda.device(self.device):
            check(self.ctx.lib.vo_sift_extract(self.handle, p(image), 1 if image.dim() == 2 else 3, p(self.kp), p(self.desc),
                                               p(self.aux), p(self.count),
                                               ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)), "vo_sift_extract")
        n, raw = (int(v) for v in self.count.cpu())
        if raw > self.cap:
            raise VoError(f"vo_sift_extract: {raw} candidates exceed max_keypoints = {self.cap}")
        return self.kp[:n], self.desc[:n], self.aux[:n]

    def extract_batch(self, images, rows=None):
        """S images in one call of the same kernels as `extract` (vo_sift_extract_batch), with no host read: images uint8
        torch tensor [S,H,W] (gray) or [S,H,W,3] (BGR), contiguous, on this device or in pinned host memory.  Returns device
        tensors kp [S,rows,2], desc [S,rows,128], aux [S,rows,4] and count int32 [S,2] = (rows written, flags); image s's
        first count[s,0] rows are, bit for bit, the first rows `extract` gives for it (the rest are unspecified).  Flag bit
        0: the raw list passed max_keypoints (where `extract` raises; which keypoints survive is then unspecified); bit 1:
        rows past `rows` were dropped (the first rows in OpenCV's order, i.e. the left of the image, are kept).  rows
        defaults to max_keypoints.  Scratch grows to the largest S seen (~117 MB per 1241 x 376 image).  Pinned images are
        read by the kernels after the call returns: keep them alive and unchanged until the stream has passed this call."""
        if not isinstance(images, torch.Tensor):
            raise ValueError("SiftExtractor.extract_batch: images must be a torch tensor")
        if images.dtype != torch.uint8 or not images.is_contiguous() or not (images.is_cuda or images.is_pinned()):
            raise ValueError("SiftExtractor.extract_batch: images must be contiguous uint8 on the device or in pinned host memory")
        if images.is_cuda and images.device != self.device:
            raise ValueError(f"SiftExtractor.extract_batch: images on {images.device}, extractor on {self.device}")
        if (images.dim() not in (3, 4) or tuple(images.shape[1:3]) != (self.H, self.W)
                or (images.dim() == 4 and images.shape[3] != 3) or not 1 <= images.shape[0] <= 65535):
            raise ValueError(f"SiftExtractor.extract_batch: expected [S,{self.H},{self.W}] or [S,{self.H},{self.W},3] with "
                             f"1 <= S <= 65535, got {tuple(images.shape)}")
        S = int(images.shape[0])
        rows = self.cap if rows is None else int(rows)
        if rows < 1:
            raise ValueError(f"SiftExtractor.extract_batch: rows {rows} must be >= 1")
        kp = torch.empty((S, rows, 2), dtype=torch.float32, device=self.device)
        desc = torch.empty((S, rows, 128), dtype=torch.float32, device=self.device)
        aux = torch.empty((S, rows, 4), dtype=torch.float32, device=self.device)
        count = torch.empty((S, 2), dtype=torch.int32, device=self.device)
        p = lambda t: ctypes.c_void_p(t.data_ptr())  # noqa: E731
        with torch.cuda.device(self.device):
            check(self.ctx.lib.vo_sift_extract_batch(self.handle, p(images), S, 1 if images.dim() == 3 else 3, rows, p(kp),
                                                     p(desc), p(aux), p(count),
                                                     ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)),
                  "vo_sift_extract_batch")
        return kp, desc, aux, count

    def close(self):
        if self.handle:
            self.ctx.lib.vo_sift_destroy(self.handle)
            self.handle = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass
