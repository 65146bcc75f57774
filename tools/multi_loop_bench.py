#!/usr/bin/env python
"""Aggregate frames/s of the device-resident keyframe loop over S sequences in lock-step (MultiDeviceLoop: one
vo_pipeline(B = S) per step) against S plain DeviceLoops run one after another on the same stream.  Features are
precomputed 60-frame synthetic sequences in pinned host memory (8 distinct ones; every sequence has its own generator
seed).  Prints one JSON line per (workload, S) with the median of 5 timed runs, the plain DeviceLoop rate, the per-stage ms
per step of a separate profiled run and the GPU's name and power limit read in the same call.

  python tools/multi_loop_bench.py [--s 1,4,16,64] [--frames 60] [--out profiles/multi_loop_r04.json]
"""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

# name, kind, keypoints, options: the keyframe loop's c2 semantics (ORB 5k Hamming + mutual), SIFT 2k, and ORB 5k Mode R
WORKLOADS = (
    ("orb5k_hamming_mutual_modeT", "orb", 5000, dict(kind="orb", norm_or_metric=0, mode=1, precision=0)),
    ("sift2k_modeT", "sift", 2000, dict(kind="sift", norm_or_metric=0, mode=0, precision=3)),
    ("orb5k_hamming_mutual_modeR", "orb", 5000, dict(kind="orb", norm_or_metric=0, mode=1, precision=0, pnp_mode="reference")),
)


def gpu_info():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True)
    name, power = (q.stdout.strip().splitlines()[0].split(", ") + ["?"])[:2] if q.returncode == 0 and q.stdout.strip() else ("?", "?")
    return {"gpu": name, "power_limit": power}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--s", default="1,4,16,64")
    ap.add_argument("--frames", type=int, default=60)
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--out", default="")
    args = ap.parse_args()
    import torch
    import vo_b200  # noqa: F401
    from vo_b200 import ops, synthetic, synthetic_sequence
    from vo_b200.device_loop import DeviceLoop, MultiDeviceLoop
    assert torch.cuda.is_available(), "multi_loop_bench needs a CUDA device"
    s_list = [int(x) for x in args.s.split(",")]
    F = args.frames
    results = []
    S_max, n_base = max(s_list), 8
    H, W = synthetic.KITTI_WH[1], synthetic.KITTI_WH[0]
    depth = torch.empty((F, S_max, H, W), dtype=torch.float32, pin_memory=True)      # shared by the workloads (refilled)
    for name, kind, n_kp, opts in WORKLOADS:
        # 8 distinct sequences (seeds 1000 + b); slot q holds sequence q % 8 and draws with its own generator seed 8214 + q.
        # Stacked step-major in the loop's slot layout, pinned.
        bases = [synthetic_sequence.make_sequence(n_frames=F, n_kp=n_kp, kind=kind, seed=1000 + b)[0] for b in range(n_base)]
        cols = bases[0][0]["desc"].shape[1]
        kp = torch.empty((F, S_max, n_kp, 2), dtype=torch.float32, pin_memory=True)
        desc = torch.empty((F, S_max, n_kp, cols), dtype=torch.uint8 if kind == "orb" else torch.float32, pin_memory=True)
        for q in range(S_max):
            for i, f in enumerate(bases[q % n_base]):
                kp[i, q] = torch.from_numpy(np.asarray(f["kp"], np.float32))
                desc[i, q] = torch.from_numpy(f["desc"])
                depth[i, q] = torch.from_numpy(f["depth"])
        n_kps = {S: np.full(S, n_kp, np.int32) for S in s_list}

        def run_multi(S):
            loop = MultiDeviceLoop(synthetic.KITTI_K, synthetic.KITTI_WH, n_kp, S, seeds=np.arange(S) + 8214, **opts)
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            for i in range(F):
                loop.push(kp[i, :S], desc[i, :S], n_kps[S], depth[i, :S], i)
            out = loop.poses(S - 1)
            dt = time.perf_counter() - t0
            loop.close()
            return dt, out

        def run_single(S):
            loops = [DeviceLoop(synthetic.KITTI_K, synthetic.KITTI_WH, n_kp, seed=8214 + q, **opts) for q in range(S)]
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            for q, loop in enumerate(loops):
                for i in range(F):
                    loop.push(kp[i, q], desc[i, q], depth[i, q], i)
            out = loops[-1].poses()
            dt = time.perf_counter() - t0
            for loop in loops:
                loop.close()
            return dt, out

        run_multi(max(s_list)); run_single(1)                      # warm every shape and the workspaces
        t_single1 = float(np.median([run_single(1)[0] for _ in range(args.reps)]))
        for S in s_list:
            run_multi(S)
            times, outs = zip(*[run_multi(S) for _ in range(args.reps)])
            t = float(np.median(times))
            ops.profile_enable(True); ops.profile_collect()
            run_multi(S)
            stages = {k: round(v[0] / F, 4) for k, v in ops.profile_collect().items() if v[1]}
            ops.profile_enable(False)
            # the last sequence inside the batch against its plain DeviceLoop (bit for bit)
            t_s, want = run_single(S) if S <= 4 else (None, None)
            same = None if want is None else bool(np.array_equal(outs[0][0], want[0]) and np.array_equal(outs[0][1], want[1]))
            rec = dict(workload=name, S=S, frames=F, n_kp=n_kp, multi_fps=S * F / t, steps_per_s=F / t,
                       gpu_us_per_step=1e6 * t / F, single_loop_fps=F / t_single1, speedup_vs_single=(S * F / t) / (F / t_single1),
                       sequential_single_fps=None if t_s is None else S * F / t_s, equal_to_single=same,
                       keyframes_last_seq=int(outs[0][1][:, 5].sum()), stage_ms_per_step=stages, **gpu_info())
            print(json.dumps(rec), flush=True)
            results.append(rec)
        del kp, desc
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            json.dump(results, f)


if __name__ == "__main__":
    main()
