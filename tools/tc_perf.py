"""Tuning helper (GPU box): time the tcgen05 matcher alone on c3-shaped input."""
import os, sys
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch
import vo_b200
from vo_b200 import ops

def run(n, m, B, prec, metric, reps=5):
    g = torch.Generator(device="cuda").manual_seed(0)
    a = torch.nn.functional.normalize(torch.randn(B, n, 128, device="cuda", generator=g), dim=-1).contiguous()
    b = torch.nn.functional.normalize(torch.randn(B, m, 128, device="cuda", generator=g), dim=-1).contiguous()
    mode = ops.VO_MODE_RATIO_MUTUAL if metric == ops.VO_METRIC_COSINE else ops.VO_MODE_RATIO
    for _ in range(2):
        ops.match_f32(a, b, metric, mode, 0.9, precision=prec, want_dist=False)
    torch.cuda.synchronize()
    ops.profile_enable(True); ops.profile_collect()
    for _ in range(reps):
        ops.match_f32(a, b, metric, mode, 0.9, precision=prec, want_dist=False)
    st = ops.profile_collect(); ops.profile_enable(False)
    ms = st["match"][0] / st["match"][1]
    passes = 3 if prec in (ops.VO_PREC_TF32X3, ops.VO_PREC_F16X3) else 1
    tf = 2.0 * n * m * 128 * B * passes / (ms * 1e-3) / 1e12
    kind = "f16" if prec in (ops.VO_PREC_F16X1, ops.VO_PREC_F16X3) else "tf32"
    print(f"n={n} m={m} B={B} passes={passes} {kind}: match {ms:.3f} ms/launch -> {tf:.1f} TFLOP/s issued ({tf/813.3*100:.1f}% of 813 TF); prep {st['prep'][0]/max(st['prep'][1],1):.3f} ms", flush=True)

if __name__ == "__main__":
    B = int(sys.argv[1]) if len(sys.argv) > 1 else 16
    run(10000, 10000, B, ops.VO_PREC_TF32X3, ops.VO_METRIC_COSINE)
    run(10000, 10000, B, ops.VO_PREC_TF32X1, ops.VO_METRIC_COSINE)
    run(10000, 10000, B, ops.VO_PREC_TF32X1, ops.VO_METRIC_L2)
    run(20000, 20000, max(1, B // 2), ops.VO_PREC_TF32X1, ops.VO_METRIC_L2)
    run(2000, 2000, 256, ops.VO_PREC_TF32X1, ops.VO_METRIC_L2)
    run(10000, 10000, B, ops.VO_PREC_F16X3, ops.VO_METRIC_COSINE)
    run(10000, 10000, B, ops.VO_PREC_F16X1, ops.VO_METRIC_L2)
    run(20000, 20000, max(1, B // 2), ops.VO_PREC_F16X1, ops.VO_METRIC_L2)
    run(2000, 2000, 256, ops.VO_PREC_F16X1, ops.VO_METRIC_L2)
