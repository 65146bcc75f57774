"""Mode R (the reference's sampler) on the GPU.  One JSON document.

single-pair latency (default): vo_pnp_ransac_ref against the throughput sampler (vo_pnp_ransac, 512 hypotheses) on one pair's
correspondences, and against the reference's CPU call (3 x cv2.solvePnPRansac).

--resident: batched Mode R against Mode T and against a loop of single-pair calls, on c2-shaped (ORB 5000 keypoints, Hamming
mutual) and c3-shaped (R2D2 10000 keypoints, cosine ratio + mutual, 3xTF32) resident batches:
  mode_r_pairs_per_s / mode_t_pairs_per_s   whole pipeline through sequence.run_resident (match -> gather -> PnP)
  pnp_batch_pairs_per_s                     vo_bootstrap + vo_pnp_ransac_ref_batch on the batch's correspondences
  pnp_single_loop_pairs_per_s               vo_pnp_ransac_ref once per pair on the same correspondences (numpy bootstrap rows,
                                            as the drop-in draws them; no host synchronisation between calls)
CUDA-event timing after a warm-up pass.  The GPU name and power limit are read in the same run."""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

import torch  # noqa: E402
import vo_b200  # noqa: E402,F401
from vo_b200 import ops, sequence, synthetic  # noqa: E402

# c2 / c3 of bench.py (keypoints, Mode T hypotheses, matcher); pair counts here are one resident batch each
WORKLOADS = {
    "c2": dict(kind="orb", n_kp=5000, n_hyp=1024, pairs=250, chunk=250,
               mc=dict(norm_or_metric=ops.VO_NORM_HAMMING, mode=ops.VO_MODE_MUTUAL, match_param=0.0, precision=0)),
    "c3": dict(kind="r2d2", n_kp=10000, n_hyp=4096, pairs=64, chunk=64,
               mc=dict(norm_or_metric=ops.VO_METRIC_COSINE, mode=ops.VO_MODE_RATIO_MUTUAL, match_param=0.90,
                       precision=ops.VO_PREC_TF32X3)),
}


def gpu_info():
    info = {"gpu": torch.cuda.get_device_name(0)}
    try:
        q = subprocess.run(["nvidia-smi", "--id=0", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=30).stdout.strip()
        info["power_limit_and_max_sm_clock"] = q
    except Exception as e:                         # the measurement stands; say why the limit is missing
        info["power_limit_and_max_sm_clock"] = f"unavailable: {e}"
    return info


def event_time(fn, reps):
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    fn()
    torch.cuda.synchronize()
    e0.record()
    for _ in range(reps):
        fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / reps


def single_pair_latency():
    import cv2
    out = {}
    for n in (500, 1500, 4000):
        from test_oracle_pnp_ref import _scene
        X, uv, K = _scene(3, n, 0.3)
        rng = np.random.RandomState(1)
        boot = np.stack([rng.randint(0, n, n) for _ in range(3)]).astype(np.int32)
        gX, gu, gb = (torch.from_numpy(np.ascontiguousarray(a)).cuda() for a in (X, uv, boot))
        cnt = torch.tensor([n], dtype=torch.int32, device="cuda")
        hyp = ops.hypotheses(cnt, 512)
        t_ref = event_time(lambda: ops.pnp_ransac_ref(gX, gu, n, K, gb), 50)
        t_thr = event_time(lambda: ops.pnp_ransac(gX[None], gu[None], cnt, K, hyp), 50)
        cv2.setNumThreads(os.cpu_count() or 1)
        t0 = time.perf_counter()
        for _ in range(5):
            for r in range(3):
                cv2.solvePnPRansac(X[boot[r]], uv[boot[r]].reshape(-1, 1, 2), K, None, iterationsCount=100, reprojectionError=1.5)
        t_cv = (time.perf_counter() - t0) / 5 * 1e3
        out[n] = {"mode_r_ms": t_ref, "mode_t_512hyp_ms": t_thr, "cv2_3x_solvePnPRansac_ms": t_cv}
    return out


def resident(name, wl, reps):
    P, chunk, mc = wl["pairs"], wl["chunk"], wl["mc"]
    chain = synthetic.make_chain(0, P, n_kp=wl["n_kp"], kind=wl["kind"])
    seq = sequence.FrameSequence.from_numpy(chain, "cuda")
    K = chain["K"]
    cfg_t = sequence.PipelineConfig(n_hyp=wl["n_hyp"], **mc)
    cfg_r = sequence.PipelineConfig(pnp_mode="reference", **mc)
    out_t, out_r = ops.PipelineBuffers(P, "cuda"), ops.PipelineBuffers(P, "cuda")
    t_mode_t = event_time(lambda: sequence.run_resident(seq, cfg_t, chunk=chunk, out=out_t), reps)
    t_mode_r = event_time(lambda: sequence.run_resident(seq, cfg_r, chunk=chunk, out=out_r), reps)
    # the correspondences of the whole batch, once (not timed)
    ref, cur = seq.slice(0, P).ref_desc, seq.slice(0, P).cur_desc
    sl = seq.slice(0, P)
    if wl["kind"] == "orb":
        m = ops.match_u8(ref, cur, mc["norm_or_metric"], mc["mode"], mc["match_param"])
    else:
        m = ops.match_f32(ref, cur, mc["norm_or_metric"], mc["mode"], mc["match_param"], mc["precision"])
    c = ops.gather_backproject(m.pairs, m.count, sl.ref_kp, sl.cur_kp, sl.depth, K)
    cap = int(c.xyz.shape[1])

    def batch_pnp():
        boot = ops.bootstrap(c.count, 3, cap)
        return ops.pnp_ransac_ref_batch(c.xyz, c.cur_uv, c.count, K, boot, iters=100, refine_iters=10)
    t_batch = event_time(batch_pnp, reps)
    counts = c.count.cpu().numpy()
    rng = np.random.RandomState(8214)
    rows = [torch.from_numpy(np.stack([rng.randint(0, max(n, 1), n) for _ in range(3)]).astype(np.int32)).cuda() for n in counts]
    live = [b for b in range(P) if counts[b] > 0]

    def loop_pnp():
        for b in live:
            ops.pnp_ransac_ref(c.xyz[b], c.cur_uv[b], int(counts[b]), K, rows[b], iters=100, refine_iters=10)
    t_loop = event_time(loop_pnp, max(1, reps // 2))
    st_r = out_r.status.cpu().numpy()
    return {"pairs": P, "chunk": chunk, "n_kp": wl["n_kp"], "mode_t_hypotheses": wl["n_hyp"],
            "median_correspondences": float(np.median(counts)),
            "mode_r_pairs_per_s": P / t_mode_r * 1e3, "mode_t_pairs_per_s": P / t_mode_t * 1e3,
            "pnp_batch_pairs_per_s": P / t_batch * 1e3, "pnp_single_loop_pairs_per_s": len(live) / t_loop * 1e3,
            "mode_r_ms_per_batch": t_mode_r, "mode_t_ms_per_batch": t_mode_t, "pnp_batch_ms": t_batch,
            "pnp_single_loop_ms": t_loop, "mode_r_ok_pairs": int((st_r == 0).sum()),
            "mode_t_ok_pairs": int((out_t.status.cpu().numpy() == 0).sum())}


def main():
    ap = argparse.ArgumentParser(description=__doc__.splitlines()[0])
    ap.add_argument("--resident", action="store_true", help="batched Mode R vs Mode T vs a single-pair loop (c2, c3)")
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--out", help="also write the JSON document to this file")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("pnp_ref_bench.py measures the GPU: no CUDA device")
    doc = gpu_info()
    if args.resident:
        doc["resident"] = {name: resident(name, wl, args.reps) for name, wl in WORKLOADS.items()}
    else:
        doc["single_pair"] = single_pair_latency()
    text = json.dumps(doc)
    print(text)
    if args.out:
        with open(args.out, "w") as f:
            f.write(text + "\n")


if __name__ == "__main__":
    main()
