"""Tensor-core Hamming pass at the c2 shape (B pairs of N x N 256-bit descriptors): time per call."""
import os
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
import vo_b200  # noqa: E402,F401
from vo_b200 import ops  # noqa: E402

B, N = int(sys.argv[1]) if len(sys.argv) > 1 else 64, int(sys.argv[2]) if len(sys.argv) > 2 else 5000
g = torch.Generator(device="cuda").manual_seed(1)
ref = torch.randint(0, 256, (B, N, 32), dtype=torch.uint8, device="cuda", generator=g)
cur = torch.randint(0, 256, (B, N, 32), dtype=torch.uint8, device="cuda", generator=g)
for norm in (ops.VO_NORM_HAMMING_TC, ops.VO_NORM_HAMMING):
    for _ in range(2):
        ops.match_u8(ref, cur, norm, ops.VO_MODE_MUTUAL, 0.0)
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(10):
        ops.match_u8(ref, cur, norm, ops.VO_MODE_MUTUAL, 0.0)
    e1.record()
    torch.cuda.synchronize()
    ms = e0.elapsed_time(e1) / 10
    print(f"norm={norm} B={B} N={N}: {ms:.3f} ms per call, {B * N * N / ms / 1e9:.3f} T dist/s", flush=True)
