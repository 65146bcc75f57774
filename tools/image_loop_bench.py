#!/usr/bin/env python
"""S camera streams from images to poses: the batched front-end (OrbExtractor / SiftExtractor.extract_batch) and the
keyframe loop fed from it (MultiDeviceLoop.push_images: one batched extraction and one vo_pipeline(B = S) per step,
keypoint counts on the device) against the one-stream path (extract per image; DeviceLoop.push_image, S loops run one after
another on the same stream).  KITTI-shaped BGR frames (1241 x 376: a window panning 5 pixels per frame over a seeded
texture, 8 distinct sequences) and depth maps in pinned host memory, Mode T.  --frontend orb: ORB 500 (cv2.ORB_create()
defaults), Hamming + mutual, n_cap 1024.  --frontend sift: cv2.SIFT_create() defaults, L2 + ratio 0.85 on the default
F16X1 pass, n_cap 8192 (above any frame's raw count, so the single loops' extractors never overflow); the record also
gives the device memory the extractor's scratch takes at that S (cudaMemGetInfo before and after, less what torch's
allocator took).  Prints one JSON line per S with medians of --reps timed runs, launches per step, whether the last
sequence equals its single loop bit for bit, and the GPU's name and power limit read in the same call.

One pinned step carries 1.40 MB of BGR image and 1.87 MB of depth per sequence: at S = 64, 209 MB, so the host-to-device
copies alone bound a step from below (DESIGN 5 measured 55.4 GB/s pinned).

  python tools/image_loop_bench.py [--frontend orb|sift] [--s 1,4,16,64] [--frames 20] [--out profiles/image_loop_r05.json]
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

H, W = 376, 1241
N_BASE = 8
FRONTENDS = {
    "orb": dict(opts=dict(kind="orb", norm_or_metric=0, mode=1, precision=0), n_cap=1024, workload="orb500_hamming_mutual_modeT"),
    "sift": dict(opts=dict(kind="sift", norm_or_metric=0, mode=0, match_param=0.85), n_cap=8192,
                 workload="sift_l2_ratio0.85_f16x1_modeT"),
}


def gpu_info():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True)
    name, power = (q.stdout.strip().splitlines()[0].split(", ") + ["?"])[:2] if q.returncode == 0 and q.stdout.strip() else ("?", "?")
    return {"gpu": name, "power_limit": power}


def texture_frames(seed, n):
    """n BGR frames: an H x W window panning 5 pixels per frame over a smooth seeded texture plus noise."""
    rng = np.random.default_rng(seed)
    th, tw = H + 16, W + 5 * n + 16
    coarse = rng.integers(0, 256, (th // 8 + 2, tw // 8 + 2, 3)).astype(np.float32)
    ys, xs = np.arange(th) / 8.0, np.arange(tw) / 8.0
    y0, x0 = ys.astype(int), xs.astype(int)
    fy, fx = (ys - y0)[:, None, None], (xs - x0)[None, :, None]
    tex = (coarse[y0][:, x0] * (1 - fy) * (1 - fx) + coarse[y0 + 1][:, x0] * fy * (1 - fx) +
           coarse[y0][:, x0 + 1] * (1 - fy) * fx + coarse[y0 + 1][:, x0 + 1] * fy * fx)
    tex = np.clip(tex + rng.integers(0, 25, tex.shape), 0, 255).astype(np.uint8)
    return [tex[8:8 + H, 8 + 5 * i:8 + 5 * i + W] for i in range(n)]


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--frontend", choices=sorted(FRONTENDS), default="orb")
    ap.add_argument("--s", default="1,4,16,64")
    ap.add_argument("--frames", type=int, default=20)
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--out", default="")
    args = ap.parse_args()
    import torch
    import vo_b200  # noqa: F401
    from vo_b200 import ops, synthetic
    from vo_b200.device_loop import DeviceLoop, MultiDeviceLoop
    from vo_b200.orb_frontend import OrbExtractor
    from vo_b200.sift_frontend import SiftExtractor
    assert torch.cuda.is_available(), "image_loop_bench needs a CUDA device"
    fe = FRONTENDS[args.frontend]
    OPTS, N_CAP = fe["opts"], fe["n_cap"]
    sift = args.frontend == "sift"
    s_list = [int(x) for x in args.s.split(",")]
    F, S_max = args.frames, max(s_list)
    K = synthetic.KITTI_K
    # step-major pinned stacks: images[i, q] is frame i of sequence q (slot q shows base sequence q % 8)
    bases = [texture_frames(1000 + b, F) for b in range(N_BASE)]
    images = torch.empty((F, S_max, H, W, 3), dtype=torch.uint8, pin_memory=True)
    for i in range(F):
        for q in range(S_max):
            images[i, q] = torch.from_numpy(np.ascontiguousarray(bases[q % N_BASE][i]))
    depth = torch.full((S_max, H, W), 10.0, dtype=torch.float32).pin_memory()
    ext = SiftExtractor(H, W) if sift else OrbExtractor(H, W)
    rows = N_CAP if sift else None                              # SIFT: as push_images asks (max_keypoints rows would be 16 MB each)

    def scratch_mb(S):
        """Device memory a fresh extractor's scratch takes once it has run S images."""
        torch.cuda.synchronize()
        free0, res0 = torch.cuda.mem_get_info()[0], torch.cuda.memory_reserved()
        e = SiftExtractor(H, W) if sift else OrbExtractor(H, W)
        e.extract_batch(images[1, :S], rows=rows)
        torch.cuda.synchronize()
        free1, res1 = torch.cuda.mem_get_info()[0], torch.cuda.memory_reserved()
        e.close()
        return ((free0 - free1) - (res1 - res0)) / 1e6

    def timed(fn, reps):
        out = []
        for _ in range(reps):
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            fn()
            torch.cuda.synchronize()
            out.append(time.perf_counter() - t0)
        return float(np.median(out))

    def run_multi(S):
        loop = MultiDeviceLoop(K, (W, H), N_CAP, S, seeds=np.arange(S) + 8214, **OPTS)
        loop.push_images(images[0, :S], depth[:S], 0)           # extractor scratch and the loop's first keyframes
        torch.cuda.synchronize()
        l0 = ops.launch_count()
        t0 = time.perf_counter()
        for i in range(1, F):
            loop.push_images(images[i, :S], depth[:S], i)
        out = loop.poses(S - 1)
        dt = time.perf_counter() - t0
        launches = (ops.launch_count() - l0) / (F - 1)
        loop.close()
        return dt, out, launches

    def run_single(S):
        loops = [DeviceLoop(K, (W, H), N_CAP, seed=8214 + q, **OPTS) for q in range(S)]
        for q, loop in enumerate(loops):
            loop.push_image(images[0, q], depth[q], 0)
        torch.cuda.synchronize()
        l0 = ops.launch_count()
        t0 = time.perf_counter()
        for q, loop in enumerate(loops):
            for i in range(1, F):
                loop.push_image(images[i, q], depth[q], i)
        out = loops[-1].poses()
        dt = time.perf_counter() - t0
        launches = (ops.launch_count() - l0) / (F - 1)
        for loop in loops:
            loop.close()
        return dt, out, launches

    results = []
    run_multi(S_max)
    run_single(1)                                               # warm every shape and the workspaces
    for S in s_list:
        resident = images[1, :S].cuda()
        ext.extract_batch(images[1, :S], rows=rows); ext.extract_batch(resident, rows=rows)
        t_batch_pinned = timed(lambda: [ext.extract_batch(images[i % F, :S], rows=rows) for i in range(10)], args.reps) / (10 * S)
        t_batch_resident = timed(lambda: [ext.extract_batch(resident, rows=rows) for _ in range(10)], args.reps) / (10 * S)
        t_each_pinned = timed(lambda: [ext.extract(images[1, q]) for q in range(S)], args.reps) / S
        t_each_resident = timed(lambda: [ext.extract(resident[q]) for q in range(S)], args.reps) / S
        l0 = ops.launch_count()
        count = ext.extract_batch(images[1, :S], rows=rows)[3]
        batch_launches = ops.launch_count() - l0
        l0 = ops.launch_count()
        ext.extract(images[1, 0])
        extract_launches = ops.launch_count() - l0
        kp_per_image = float(count[:, 0].float().mean())
        multi = [run_multi(S) for _ in range(args.reps)]
        t_multi = float(np.median([m[0] for m in multi]))
        single = [run_single(S) for _ in range(args.reps if S <= 16 else 1)]
        t_single = float(np.median([s[0] for s in single]))
        same = bool(np.array_equal(multi[0][1][0], single[0][1][0]) and np.array_equal(multi[0][1][1], single[0][1][1]))
        steps = F - 1
        rec = dict(S=S, frames=F, frame="1241x376 BGR", frontend=args.frontend, n_cap=N_CAP, workload=fe["workload"],
                   extract_batch_us_per_image_pinned=1e6 * t_batch_pinned,
                   extract_batch_us_per_image_resident=1e6 * t_batch_resident,
                   extract_us_per_image_pinned=1e6 * t_each_pinned, extract_us_per_image_resident=1e6 * t_each_resident,
                   extract_batch_launches_per_call=batch_launches, extract_launches_per_call=extract_launches,
                   keypoints_per_image=kp_per_image,
                   push_images_fps=S * steps / t_multi, push_images_ms_per_step=1e3 * t_multi / steps,
                   sequential_push_image_fps=S * steps / t_single, speedup=t_single / t_multi,
                   launches_per_step_push_images=multi[0][2], launches_per_step_sequential=single[0][2],
                   h2d_mb_per_step=S * (H * W * 3 + H * W * 4) / 1e6, equal_to_single=same,
                   keyframes_last_seq=int(multi[0][1][1][:, 5].sum()), matches_last_seq=float(multi[0][1][1][1:, 1].mean()),
                   **gpu_info())
        if sift:
            rec["scratch_mb"] = scratch_mb(S)
        else:
            rec["nfeatures"] = 500
        print(json.dumps(rec), flush=True)
        results.append(rec)
        del resident
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            json.dump(results, f, indent=1)


if __name__ == "__main__":
    main()
