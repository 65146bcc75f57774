#!/usr/bin/env python
"""bench.py — frame-pairs/sec of the hot path (match -> gather/back-project -> PnP-RANSAC -> pose).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--workload c1|c2|c2r|c2tc|c3|c4|c5|default]
                    [--dump-outputs DIR]

Input = one synthetic SEQUENCE of P + 1 frames per GPU (synthetic.make_chain): pair i = (frame i, frame i+1), so a frame's
descriptors / keypoints / depth map exist (and, in the e2e leg, cross the bus) once.  A step = R passes of the hot path
over the rank's P consecutive pairs (weak scaling: every rank owns its own block of the pre-declared pair list, SURVEY
D3/8(e)); R is chosen once, before timing, so that the K timed steps last >= ~2.5 s; under N>1 every pass ends with one
NCCL all-gather of the 4x4 relative poses.
Default = BASELINE.json's metric in full: the HEADLINE line is workload c3 (configs[2], the largest single-GPU
configuration: R2D2 10k keypoints, the tcgen05 3xTF32 GEMM-argmin the metric's "matching GEMM % TC peak" names, 4096
hypotheses), and the complete line of c2 (configs[1]: ORB 5k, Hamming mutual-NN, 1024 hypotheses, 1000-pair sequence) rides
in `extra.c2`.  `--workload X` or VO_BENCH_WORKLOAD=X selects a single workload (c4 / c5 for the multi-GPU configs).
Prints ONE JSON line (rank 0).  `--impl reference` times the reference's CPU path (oracle/reference_path.py: the same
OpenCV / torch calls the reference makes) on the host cores instead, on the same workload(s).
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

WORKLOADS = {
    # name: (descriptor kind, keypoints, hypotheses, matcher description, cpu matcher)
    "c1": dict(kind="sift", n_kp=2000, n_hyp=512, pairs=512, chunk=256, shape="kitti", cpu_matcher="knn_ratio",
               desc="SIFT 2k kp, L2 kNN-2 + ratio 0.85, PnP-RANSAC 512 hyp, KITTI 1241x376"),
    "c2": dict(kind="orb", n_kp=5000, n_hyp=1024, pairs=1000, chunk=250, shape="kitti", cpu_matcher="hamming_mutual", e2e_sampled_frac=0.4,
               desc="ORB 5k kp, 256-bit Hamming mutual-NN, PnP-RANSAC 1024 hyp, 1000-pair sequence, KITTI 1241x376"),
    # c2 with the reference's OWN ORB rule (feature_extractors/ORB.py: cv2.BFMatcher() = NORM_L2 over byte values, ratio 0.85;
    # SURVEY D2) instead of the north-star's Hamming / mutual rule: an exact fp16 tensor-core pass
    "c2r": dict(kind="orb", n_kp=5000, n_hyp=1024, pairs=1000, chunk=250, shape="kitti", cpu_matcher="knn_ratio", orb_l2=True, e2e_sampled_frac=0.4,
                desc="ORB 5k kp, reference rule: byte-wise L2 kNN-2 + ratio 0.85, PnP-RANSAC 1024 hyp, 1000-pair sequence, KITTI 1241x376"),
    # c2 with the Hamming distances computed on the tensor cores (VO_NORM_HAMMING_TC: bits as e4m3 -1 / +1, K = 256 tcgen05 kind::f8f6f4
    # GEMM with the fused row top-2 epilogue, run in both directions): bit-identical matches (tests/test_gpu_match_u8.py), opt-in;
    # c2 keeps XOR + POPC
    "c2tc": dict(kind="orb", n_kp=5000, n_hyp=1024, pairs=1000, chunk=250, shape="kitti", cpu_matcher="hamming_mutual", hamming_tc=True,
                 desc="ORB 5k kp, 256-bit Hamming mutual-NN on the tensor cores (opt-in, bit-identical to XOR+POPC), PnP-RANSAC 1024 hyp, 1000-pair sequence, KITTI 1241x376"),
    "c3": dict(kind="r2d2", n_kp=10000, n_hyp=4096, pairs=128, chunk=64, shape="kitti", cpu_matcher="r2d2",
               desc="R2D2 10k kp, cosine GEMM-argmin ratio+mutual, PnP-RANSAC 4096 hyp, KITTI 1241x376"),
    # the two multi-GPU configurations of BASELINE.json (per-GPU block of the sharded sequence; weak scaling)
    "c4": dict(kind="sift", n_kp=20000, n_hyp=16384, pairs=64, chunk=32, shape="kitti", cpu_matcher="knn_ratio", unique=8,
               desc="SIFT 20k kp, L2 kNN-2 + ratio 0.85, PnP-RANSAC 16384 hyp, KITTI 1241x376"),
    "c5": dict(kind="r2d2", n_kp=50000, n_hyp=4096, pairs=8, chunk=8, shape="zed", cpu_matcher="r2d2", unique=4,
               desc="R2D2 50k kp, cosine GEMM-argmin ratio+mutual, PnP-RANSAC 4096 hyp, ZED-Mini-shaped 2208x1242"),
}


def env_rank():
    return int(os.environ.get("RANK", 0)), int(os.environ.get("LOCAL_RANK", 0)), int(os.environ.get("WORLD_SIZE", 1))


def matcher_cfg(kind, ops, wl=None):
    orb_l2 = bool(wl and wl.get("orb_l2"))
    if kind == "orb" and wl and wl.get("hamming_tc"):
        return dict(norm_or_metric=ops.VO_NORM_HAMMING_TC, mode=ops.VO_MODE_MUTUAL, match_param=0.0, precision=0)
    if kind == "orb" and orb_l2:
        return dict(norm_or_metric=ops.VO_NORM_L2_U8, mode=ops.VO_MODE_RATIO, match_param=0.85, precision=0)
    if kind == "orb":
        return dict(norm_or_metric=ops.VO_NORM_HAMMING, mode=ops.VO_MODE_MUTUAL, match_param=0.0, precision=0)
    if kind == "sift":
        return dict(norm_or_metric=ops.VO_METRIC_L2, mode=ops.VO_MODE_RATIO, match_param=0.85, precision=ops.VO_PREC_F16X1)
    return dict(norm_or_metric=ops.VO_METRIC_COSINE, mode=ops.VO_MODE_RATIO_MUTUAL, match_param=0.90, precision=ops.VO_PREC_TF32X3)


def make_host_chain(wl, n_pairs, first_index, pinned=False):
    """P + 1 consecutive synthetic frames (synthetic.make_chain), optionally generated straight into pinned host memory."""
    from vo_b200 import synthetic
    K, wh = (synthetic.KITTI_K, synthetic.KITTI_WH) if wl["shape"] == "kitti" else (synthetic.ZED_K, synthetic.ZED_WH)
    out = None
    if pinned:
        import torch
        F, N = n_pairs + 1, wl["n_kp"]
        ddt, dd = (torch.uint8, 32) if wl["kind"] == "orb" else (torch.float32, 128)
        t = {"desc": torch.empty((F, N, dd), dtype=ddt).pin_memory(), "kp": torch.empty((F, N, 2), dtype=torch.float32).pin_memory(),
             "depth": torch.empty((F, wh[1], wh[0]), dtype=torch.float32).pin_memory()}
        out = {k: v.numpy() for k, v in t.items()}
        out["_pinned"] = t
    ch = synthetic.make_chain(first_index, n_pairs, n_kp=wl["n_kp"], kind=wl["kind"], K=K, wh=wh,
                              out=None if out is None else {k: out[k] for k in ("desc", "kp", "depth")})
    if out is not None:
        ch["_pinned"] = out["_pinned"]
    return ch


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled DURING the timed region (B200_PROFILING.md)."""
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.rows, self.proc, self.index = [], None, index

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--id={self.index}", f"--query-gpu={self.Q}",
                                          "--format=csv,noheader,nounits", "-lms", "25"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._read, daemon=True)
            self.thread.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([x.strip() for x in line.split(",")])

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        names = ("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap")
        for r in self.rows:
            if len(r) < 7:
                continue
            try:
                sm.append(float(r[0])); mx.append(float(r[1]))
            except ValueError:
                continue
            for name, v in zip(names, r[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return d.get("hbm_gbs", 6650.0), d.get("bf16_tflops", 1590.0), "measured"
    return 6650.0, 1590.0, "fallback"


def measure_tf32_peak(dev):
    """cuBLAS TF32 GEMM throughput on this GPU (8192^3, best of 10) — the measuring stick for the matching GEMM,
    taken outside every timed region.  MEASURED_PEAKS.json has no TF32 figure (BASELINE.md section 4)."""
    import torch
    old = torch.backends.cuda.matmul.allow_tf32
    torch.backends.cuda.matmul.allow_tf32 = True
    try:
        n = 8192
        a = torch.randn(n, n, device=dev)
        b = torch.randn(n, n, device=dev)
        for _ in range(3):
            a @ b
        best = float("inf")
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        for _ in range(10):
            e0.record(); a @ b; e1.record(); torch.cuda.synchronize()
            best = min(best, e0.elapsed_time(e1))
        return 2.0 * n ** 3 / (best * 1e-3) / 1e12
    finally:
        torch.backends.cuda.matmul.allow_tf32 = old


def ncu_traffic(kernel_key, pairs_per_launch):
    """DRAM bytes per launch of the dominant kernel from the committed `ncu --set full` capture, scaled to this
    run's pairs per launch (profiles/traffic.json: bytes and pairs of the captured launch)."""
    p = os.path.join(ROOT, "profiles", "traffic.json")
    if not os.path.exists(p):
        return None
    d = json.load(open(p)).get(kernel_key)
    if not d:
        return None
    return d["dram_bytes"] / d["pairs_per_launch"] * pairs_per_launch


# --------------------------------------------------------------------------------------- CPU reference arm
def time_cpu_pairs(wl, n_pairs, first_index=0, warm=1):
    """Runs the reference's CPU path over `n_pairs` synthetic pairs; returns (pairs/s, seconds, threads)."""
    from oracle import reference_path as rp
    from vo_b200 import synthetic
    threads = rp.set_threads(os.cpu_count() or 1)
    chain = make_host_chain(wl, n_pairs + warm, first_index)
    rng = np.random.RandomState(8214)          # vo_stereo_runner.py:20-24
    def run(i):
        p = synthetic.chain_pair(chain, i)
        return rp.process_pair(p["ref_desc"], p["cur_desc"], p["ref_kp"], p["cur_kp"], p["depth"], p["K"],
                               matcher=wl["cpu_matcher"], rng=rng)
    for i in range(warm):
        run(i)
    t0 = time.perf_counter()
    ok = 0
    for i in range(warm, warm + n_pairs):
        ok += bool(run(i)[0])
    dt = time.perf_counter() - t0
    return n_pairs / dt, dt, threads, ok


def run_reference(args, name):
    """--impl reference: the reference's CPU path on the host cores, bounded sample per step (rank 0 only)."""
    wl = WORKLOADS[name]
    sample = args.cpu_pairs or {"c1": 24, "c2": 16, "c2r": 16, "c2tc": 16, "c3": 4, "c4": 2, "c5": 1}[name]
    vals, secs = [], []
    for s in range(args.warmup + args.steps):
        v, dt, threads, ok = time_cpu_pairs(wl, sample, first_index=s)
        if s >= args.warmup:
            vals.append(v); secs.append(dt)
    value = float(np.mean(vals))
    return {
        "impl": "reference", "metric": "frame-pairs/sec (match+PnP)", "value": value, "unit": "pairs/s",
        "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup, "ms_per_step": float(np.mean(secs) * 1e3),
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": dtype_of(wl), "data": "synthetic",
        "config": {"workload": f"{name}: {wl['desc']}", "pairs_per_step": sample,
                   "path": "cv2.BFMatcher / torch matmul+topk + depthTo3d restatement + 3x cv2.solvePnPRansac(100, 1.5) "
                           "(oracle/reference_path.py: the reference's own third-party calls)"},
        "cpu_baseline": {"value": value, "unit": "pairs/s", "cores": threads, "kind": "port",
                         "sample": f"{sample} consecutive pairs/step x {args.steps} steps of the same synthetic workload"},
        "e2e": {"value": value, "unit": "pairs/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }


def measure_api_rate(wl, dev, n_frames=40):
    """Frames/s through the REFERENCE-FACING API on one GPU: the drop-in VisualOdometry.process_frame (host keyframe policy, one
    D2H round trip per frame, the reference's own PnP sampler = pnp_mode: reference) and the device-resident keyframe loop
    (vo_seq_*, throughput sampler), on a short synthetic sequence of the workload's descriptor kind with precomputed features
    (feature extraction is outside the metric, SURVEY 8(d))."""
    import contextlib
    import io
    import tempfile
    import torch
    from vo_b200 import dropin, ops, synthetic, synthetic_sequence
    from vo_b200.device_loop import DeviceLoop
    kind = wl["kind"]
    n_kp = min(wl["n_kp"], 10000)
    frames, gt = synthetic_sequence.make_sequence(n_frames=n_frames, n_kp=n_kp, kind=kind, seed=3)
    if kind == "r2d2":      # the reference's R2D2 keypoints are (x, y, scale) float32 rows, its descriptors CUDA tensors
        for f in frames:
            f["kp"] = np.concatenate([f["kp"], np.full((len(f["kp"]), 1), 32.0)], 1).astype(np.float32)
            f["desc"] = torch.from_numpy(f["desc"]).to(dev)
    cwd = os.getcwd()
    tmp = tempfile.mkdtemp(prefix="vo_api_")
    out = {"frames": n_frames, "keypoints_per_frame": n_kp}
    try:
        extra = "\norb_matcher: hamming_mutual\n" if (kind == "orb" and not wl.get("orb_l2")) else ""
        vos = dropin.load(tmp, kind, extra)
        feed = {}
        vos.extract_features_and_desc = lambda img: feed["cur"]
        img = np.zeros((synthetic.KITTI_WH[1], synthetic.KITTI_WH[0], 3), np.uint8)

        def run_host():
            np.random.seed(8214)
            vo = vos.VisualOdometry(synthetic.KITTI_K, seq=0)
            poses = []
            for i, f in enumerate(frames):
                feed["cur"] = (f["kp"], f["desc"])
                poses.append(vo.process_frame(img, f["depth"], (100, 100), i).pose.copy())
            torch.cuda.synchronize()
            return np.stack(poses), vo
        with contextlib.redirect_stdout(io.StringIO()):
            run_host()
            t_hosts = []
            for _ in range(3):      # a 40-frame run lasts ~0.1 s: one host hiccup would decide a single measurement
                t0 = time.perf_counter()
                poses, vo = run_host()
                t_hosts.append(time.perf_counter() - t0)
            t_host = float(np.median(t_hosts))
        out["dropin_process_frame_fps"] = n_frames / t_host
        out["dropin_pnp_mode"] = vo.pnp_mode
        out["dropin_bad_pnp"] = int(vo.bad_pnp)
        out["dropin_max_pos_err_m"] = float(np.linalg.norm(poses[:, :3, 3] - gt[:, :3, 3], axis=1).max())
    finally:
        os.chdir(cwd)
    mc = matcher_cfg(kind, ops, wl)
    pinned = [(torch.from_numpy(np.ascontiguousarray(f["kp"], dtype=np.float32)).pin_memory(),
               f["desc"] if isinstance(f["desc"], torch.Tensor) else torch.from_numpy(f["desc"]).pin_memory(),
               torch.from_numpy(f["depth"]).pin_memory()) for f in frames]

    def run_dev():
        loop = DeviceLoop(synthetic.KITTI_K, synthetic.KITTI_WH, n_kp, kind=kind, norm_or_metric=mc["norm_or_metric"], mode=mc["mode"],
                          match_param=mc["match_param"] or 0.85, precision=mc["precision"] or None, n_hyp=min(wl["n_hyp"], 1024),
                          kp_stride=3 if kind == "r2d2" else 2)
        for i, (kp, d, z) in enumerate(pinned):
            loop.push(kp, d, z, i)
        res = loop.poses()
        loop.close()
        return res
    run_dev()
    t_devs = []
    for _ in range(5):              # ~25 ms each: median of five
        t0 = time.perf_counter()
        got, info = run_dev()
        t_devs.append(time.perf_counter() - t0)
    out["device_loop_fps"] = n_frames / float(np.median(t_devs))
    out["device_loop_fps_runs"] = [round(n_frames / t, 1) for t in t_devs]
    out["device_loop_max_pos_err_m"] = float(np.linalg.norm(got[:, :3, 3] - gt[:, :3, 3], axis=1).max())
    out["note"] = ("features precomputed; dropin = VisualOdometry.process_frame with the reference's keyframe policy on the host and its own "
                   "PnP sampler on the GPU; device loop = vo_seq_push / vo_seq_read, one synchronisation per sequence; medians of 3 / 5 runs")
    return out


def dtype_of(wl):
    if wl.get("orb_l2"):
        return "u8 -> fp16 (1x, exact on byte values) / f32+f64 PnP"
    if wl.get("hamming_tc"):
        return "256 bits -> e4m3 -1/+1, tcgen05 kind::f8f6f4 K=256 (exact integers) / f32+f64 PnP"
    return {"orb": "u8 (XOR+POPC) / f32+f64 PnP", "sift": "fp16 (1x, exact on integer SIFT) / f32+f64 PnP",
            "r2d2": "tf32x3 / f32+f64 PnP"}[wl["kind"]]


# --------------------------------------------------------------------------------------- our arm
_DIST = {"init": False}


def run_ours(args, name):
    import torch
    import torch.distributed as dist
    import vo_b200  # noqa: F401
    from vo_b200 import ops, sequence, synthetic

    wl = WORKLOADS[name]
    rank, local_rank, world = env_rank()
    numa_cores = sequence.bind_to_gpu_numa(local_rank) if world > 1 else None   # pinned buffers on the GPU's NUMA node
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1 and not _DIST["init"]:
        dist.init_process_group("nccl", device_id=dev)
        _DIST["init"] = True

    P = args.pairs or wl["pairs"]                      # pairs per GPU per pass
    host = make_host_chain(wl, P, first_index=rank, pinned=True)    # P + 1 frames, straight into pinned host memory
    seq = sequence.FrameSequence.from_numpy({**host["_pinned"], "K": host["K"]}, dev)   # every frame resident once: >> L2
    mc = matcher_cfg(wl["kind"], ops, wl)
    if args.precision is not None:
        mc["precision"] = args.precision
    cfg = sequence.PipelineConfig(n_hyp=wl["n_hyp"], **mc)
    chunk = min(args.chunk or wl["chunk"], P)
    out = ops.PipelineBuffers(P, dev)

    def one_pass():
        sequence.run_resident(seq, cfg, pair0=rank * P, chunk=chunk, out=out)
        if world > 1:
            return sequence.all_gather_poses(out.T_rel, out.status, world)
        return out.T_rel, out.status

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)

    def agree_max(x):
        t = torch.tensor([float(x)], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    # passes per step: chosen once, outside the timed region, so that the K timed steps last >= ~2.5 s
    one_pass(); barrier()
    e0.record(); one_pass(); one_pass(); e1.record(); barrier()
    pass_ms = agree_max(e0.elapsed_time(e1) / 2.0)
    R = args.passes or int(min(256, max(1, np.ceil(args.min_timed_ms / (args.steps * pass_ms)))))

    def step():
        for _ in range(R):
            r = one_pass()
        return r

    for _ in range(args.warmup):
        step()
    barrier()
    l0 = ops.launch_count()
    ops.profile_enable(True)
    ops.profile_collect()
    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
    barrier()
    e0.record()
    for _ in range(args.steps):
        T_all, st_all = step()
    e1.record()
    barrier()
    ms = e0.elapsed_time(e1)
    clocks = sampler.stop() if rank == 0 else None
    stages = ops.profile_collect()
    ops.profile_enable(False)
    launches = ops.launch_count() - l0
    ms = agree_max(ms)
    value = world * P * R * args.steps / (ms / 1e3)
    # what run_resident handed back in the last timed step (this rank's block of pairs), read before anything else runs
    outputs = {f: getattr(out, f).cpu().numpy().astype(np.float64)
               for f in ("T_rel", "rt", "n_matches", "n_corr", "n_inl", "status")} if args.dump_outputs else {}

    # ---- matcher variants of the same workload, resident, same pairs, same R (reported beside the headline, never as it):
    # c2: the Hamming distances on the tensor cores (bit-identical matches); c3 / c5: the split-fp16 form of the 3xTF32 GEMM
    variants = {}
    var_cfgs = {"orb": [("hamming_tc", dict(norm_or_metric=ops.VO_NORM_HAMMING_TC))] if not (wl.get("orb_l2") or wl.get("hamming_tc")) else [],
                "r2d2": [("f16x3", dict(precision=ops.VO_PREC_F16X3))] if mc["precision"] == ops.VO_PREC_TF32X3 else []}.get(wl["kind"], [])
    Tn_main = out.T_rel.cpu().numpy().copy()
    for vname, override in ([] if args.no_variants else var_cfgs):
        vcfg = sequence.PipelineConfig(n_hyp=wl["n_hyp"], **{**mc, **override})
        vout = ops.PipelineBuffers(P, dev)

        def vpass():
            sequence.run_resident(seq, vcfg, pair0=rank * P, chunk=chunk, out=vout)
            if world > 1:
                sequence.all_gather_poses(vout.T_rel, vout.status, world)
        for _ in range(2):
            vpass()
        barrier()
        ops.profile_enable(True); ops.profile_collect()
        e0.record()
        for _ in range(args.steps * R):
            vpass()
        e1.record()
        barrier()
        vms = agree_max(e0.elapsed_time(e1))
        vst = ops.profile_collect(); ops.profile_enable(False)
        variants[vname] = {"value": world * P * R * args.steps / (vms / 1e3), "unit": "pairs/s", "timed_region_s": vms / 1e3,
                           "match_ms_per_launch": vst["match"][0] / max(vst["match"][1], 1),
                           "prep_ms_per_launch": vst["prep"][0] / max(vst["prep"][1], 1),
                           "max_abs_pose_diff_vs_headline": float(np.abs(vout.T_rel.cpu().numpy() - Tn_main).max()),
                           "same_status": bool(np.array_equal(vout.status.cpu().numpy(), out.status.cpu().numpy()))}
        del vout

    # sanity of the work done inside the timed region (not a parity test: tests/ does that)
    st = out.status.cpu().numpy()
    ok_frac = float((st == 0).mean())
    n_inl = out.n_inl.cpu().numpy()
    Tn = out.T_rel.cpu().numpy()
    errs = [synthetic.pose_errors(Tn[i], host["T_rel"][i]) for i in range(P)]
    chain = sequence.chain_poses(T_all.cpu().numpy(), sequence.gate_poses(T_all.cpu().numpy(), st_all.cpu().numpy()))

    # ---- e2e: the same sequence from pinned HOST memory through sequence.HostSequenceRunner (the call a user with frames in
    # host memory makes): H2D of every frame, D2H of the poses and the host-side pose chaining inside the timed region.
    # R2D2 workloads: the reference never holds R2D2 descriptors on the host — its network runs on the GPU and Frame.desc stays a
    # CUDA tensor (R2D2.py:224-232, SURVEY a10) — so the reference-facing call gets device descriptors and host keypoints /
    # depth: that is `e2e`; the same run with the descriptors uploaded from host memory too is reported as e2e.all_from_host.
    def measure_e2e(desc_on_device, desc_u8=False):
        src = {**host["_pinned"], "K": host["K"]}
        run_cfg = cfg
        if desc_on_device:
            src["desc"] = seq.desc
        if desc_u8:   # SIFT values (integers 0..255) held as uint8: a quarter of the bytes, the same exact arithmetic on the device
            src["desc"] = host["_pinned"]["desc"].to(torch.uint8).pin_memory()
            run_cfg = sequence.PipelineConfig(n_hyp=wl["n_hyp"], norm_or_metric=ops.VO_NORM_L2_U8, mode=mc["mode"],
                                              match_param=mc["match_param"], precision=0)
        runner = sequence.HostSequenceRunner(src, run_cfg, chunk=min(args.e2e_chunk or max(1, chunk // 2), P), device=dev, depth_mode=args.e2e_depth,
                                             sampled_frac=args.e2e_sampled_frac if args.e2e_sampled_frac is not None else wl.get("e2e_sampled_frac", 0.4))
        tune = {}
        if args.e2e_depth == "hybrid" and args.e2e_sampled_frac is None:
            tune = runner.autotune(sync=barrier)         # untimed: which DMA / zero-copy split suits this host with `world` ranks pulling
            if world > 1:                                # every rank runs the same split (the slowest rank sets the time anyway)
                votes = torch.tensor([tune[f] for f in sorted(tune)], dtype=torch.float64, device=dev)
                dist.all_reduce(votes, op=dist.ReduceOp.MAX)
                runner.frac = sorted(tune)[int(votes.argmin().item())]
                tune = {f: float(v) for f, v in zip(sorted(tune), votes.tolist())}

        def e2e_passes(count):
            """`count` passes, software-pipelined: pass r+1 is submitted (its uploads start at once) before the host waits for,
            reads back and chains the poses of pass r.  Every pass's H2D, compute, D2H and host chaining lie inside the caller's
            timed region; the function returns with the last pass's results read."""
            pending = None
            for _ in range(count):
                t = runner.submit(pair0=rank * P)
                if world > 1:
                    sequence.all_gather_poses(runner.out.T_rel, runner.out.status, world)
                if pending is not None:
                    T_h, st_h, _ = runner.collect(pending)
                    sequence.chain_poses(T_h.numpy(), sequence.gate_poses(T_h.numpy(), st_h.numpy()))
                pending = t
            T_h, st_h, _ = runner.collect(pending)
            sequence.chain_poses(T_h.numpy(), sequence.gate_poses(T_h.numpy(), st_h.numpy()))
            torch.cuda.synchronize()
            return T_h, st_h

        e2e_passes(2); barrier()
        e0.record(); e2e_passes(4); e1.record(); barrier()
        Re = args.passes or int(min(256, max(1, np.ceil(args.min_timed_ms / (args.steps * agree_max(e0.elapsed_time(e1)) / 4.0)))))
        for _ in range(max(1, args.warmup // 2)):
            e2e_passes(Re)
        barrier()
        e0.record()
        T_h, st_h = e2e_passes(args.steps * Re)
        e1.record()
        barrier()
        e2e_ms = agree_max(e0.elapsed_time(e1))
        res = {"value": world * P * Re * args.steps / (e2e_ms / 1e3), "ms": e2e_ms, "Re": Re, "tune": tune, "frac": runner.frac,
               "same": bool(np.array_equal(T_h.numpy(), Tn) and np.array_equal(st_h.numpy(), st)),   # host path == resident path, bit for bit
               "h2d": runner.h2d_bytes, "d2h": runner.d2h_bytes}
        del runner
        return res

    r2d2_like = wl["kind"] == "r2d2"
    em = measure_e2e(desc_on_device=r2d2_like)
    em_host = measure_e2e(desc_on_device=False) if r2d2_like else None
    em_u8 = measure_e2e(desc_on_device=False, desc_u8=True) if wl["kind"] == "sift" else None
    e2e_value, e2e_ms, Re, tune, e2e_same, h2d_pass, d2h_pass = em["value"], em["ms"], em["Re"], em["tune"], em["same"], em["h2d"], em["d2h"]

    if rank != 0:
        return None
    if outputs:
        os.makedirs(args.dump_outputs, exist_ok=True)
        for f, a in outputs.items():
            np.save(os.path.join(args.dump_outputs, f"{name}_{f}.npy"), a)

    # ---- roofline of the dominant kernel, from the per-stage event times of the timed region
    hbm_peak, bf16_peak, peak_kind = peaks()
    N = M = wl["n_kp"]
    stage_ms = {k: v[0] / max(v[1], 1) for k, v in stages.items() if v[1]}
    total_stage = sum(v[0] for v in stages.values())
    share = {k: (v[0] / total_stage if total_stage else 0.0) for k, v in stages.items() if v[1]}
    launches_match = stages["match"][1]                   # profiled intervals of the match stage (one per vo_pipeline call)
    pairs_per_launch = P * R * args.steps / max(launches_match, 1)
    match_s = stage_ms.get("match", float("nan")) / 1e3
    if wl.get("orb_l2"):
        # bytes widened to fp16 and zero-padded to 128 dimensions: the pass SIFT runs (kind::f16, exact integers)
        flops = pairs_per_launch * 2.0 * N * M * 128
        roof = {"kernel": "match_f32_tc_kernel<fp16 single pass> on byte descriptors (tcgen05 kind::f16 fused GEMM + row top-2)",
                "bound": "tensor", "achieved": flops / match_s / 1e12, "peak": bf16_peak, "unit": "TFLOP/s",
                "traffic": None, "peak_source": f"dense bf16 cuBLAS burst peak of MEASURED_PEAKS.json ({peak_kind})",
                "issued_passes": 1, "algorithmic_flops": flops / 4.0,
                "distances_per_s": pairs_per_launch * float(N) * M / match_s,
                "note": "issued FLOPs (128 padded dimensions; 32 carry data).  The pass is bound by its row top-2 epilogue "
                        "(ALU pipe), not by the GEMM, which is why the padding is free: see the c4 line and DESIGN 3.2"}
    elif wl.get("hamming_tc"):
        flops = pairs_per_launch * 2.0 * N * M * 256
        flops *= 2.0      # mutual rule: a second pass with the roles swapped supplies the column arg-min
        roof = {"kernel": "match_f32_tc_kernel<e4m3, K = 256> on 256-bit descriptors as -1 / +1 (tcgen05 kind::f8f6f4, fused row top-2, persistent CTAs; two passes for the mutual rule)",
                "bound": "tensor", "achieved": flops / match_s / 1e12, "peak": 2.0 * bf16_peak, "unit": "TFLOP/s", "traffic": None,
                "peak_source": f"2 x the dense bf16 cuBLAS burst peak of MEASURED_PEAKS.json ({peak_kind}): kind::f8f6f4 issues at twice the kind::f16 rate; "
                               "no fp8 GEMM peak was measured on this pool",
                "issued_passes": 2, "algorithmic_flops": flops / 2.0, "distances_per_s": pairs_per_launch * float(N) * M / match_s,
                "note": "a.b over -1 / +1 bit vectors = 256 - 2 Hamming: 2 x 256 FLOP per distance and pass, exact integers, no norms.  "
                        "achieved counts both passes (the `match` stage covers both launches and the column-key merge).  With e4m3 operands "
                        "the row top-2 fold (ALU pipe), not the tensor pipe, bounds the pass: frac is structurally < 0.5"}
    elif wl["kind"] == "orb":
        alg_bytes = pairs_per_launch * (32.0 * (N + M) + 8.0 * N + 8.0 * M)       # descriptors + row bests (8 B: mutual rule) + column keys
        roof = {"kernel": "match_u8_kernel (XOR+POPC Hamming, fused row/column arg-min)", "bound": "hbm",
                "achieved": alg_bytes / match_s / 1e9, "peak": hbm_peak, "unit": "GB/s",
                "traffic": ncu_traffic("match_u8_kernel", pairs_per_launch), "algorithmic_bytes": alg_bytes,
                "peak_source": f"MEASURED_PEAKS.json ({peak_kind})",
                "note": "structurally << 1: all-pairs Hamming is bound by the integer pipes, not HBM (SURVEY D5); see binding_pipe"}
        # carry-save popcount on prefix-XOR descriptors: 8 XOR + 3 carries + the twos/fours adder = 13 LOP3, + 4 POPC per
        # 256-bit distance, + one 3-input minimum per distance (weights, adds and keys run as IMADs on the FMA pipe).
        # Four POPC per distance is the floor of the formulation (the eight XOR words of a distance hold 9 values per bit
        # column); at 16 POPC lanes/clk/SM that pipe is the binding ceiling, the logic pipe (14 per distance at 64 lanes)
        # sits 10 % below it
        dists = pairs_per_launch * N * M
        sm_mhz = (clocks or {}).get("sm_mhz") or 1965.0
        popc_peak = 16.0 * 148 * sm_mhz * 1e6 / 4.0                                 # distances/s if the POPC pipe never idles
        roof["binding_pipe"] = {"pipe": "xu (POPC)", "achieved": dists / match_s / 1e12, "peak": popc_peak / 1e12,
                                "unit": "Tdist/s", "frac": dists / match_s / popc_peak,
                                "alu_pipe_frac": dists * 14.0 / match_s / (64.0 * 148 * sm_mhz * 1e6),
                                "peak_source": "16 POPC lanes/clk/SM x 148 SM x sampled SM clock / 4 POPC per distance"}
    else:
        passes = 3 if mc["precision"] in (ops.VO_PREC_TF32X3, ops.VO_PREC_F16X3) else 1
        flops = pairs_per_launch * 2.0 * N * M * 128 * (passes if mc["precision"] != ops.VO_PREC_FP32_SIMT else 1)
        tf32_half_bf16 = bf16_peak / 2.0
        if mc["precision"] in (ops.VO_PREC_F16X1, ops.VO_PREC_F16X3):
            # fp16 operands: single pass (exact on integer-valued SIFT descriptors; + one kind::tf32 K-step per tile for the
            # column norm) or the hi/lo split x*2^8 = hi + lo (22 operand bits, as 3xTF32).  The ceiling is the dense
            # 16-bit tensor peak MEASURED_PEAKS.json holds
            single = mc["precision"] == ops.VO_PREC_F16X1
            roof = {"kernel": "match_f32_tc_kernel<fp16 single pass> (tcgen05 kind::f16 fused GEMM + row top-2)" if single else
                              "match_f32_tc_kernel<split fp16, 3 MMAs per 16 k> (tcgen05 kind::f16 fused GEMM + row top-2 / column arg-max)",
                    "bound": "tensor", "achieved": flops / match_s / 1e12, "peak": bf16_peak, "unit": "TFLOP/s",
                    "traffic": ncu_traffic("match_f32_tc_kernel_f16" if single else "match_f32_tc_kernel_f16x3", pairs_per_launch),
                    "peak_source": f"dense bf16 cuBLAS burst peak of MEASURED_PEAKS.json ({peak_kind}); fp16 and bf16 share the rate",
                    "frac_of_tf32_proxy": flops / match_s / 1e12 / tf32_half_bf16,
                    "issued_passes": passes, "algorithmic_flops": flops / passes,
                    "note": "achieved counts ISSUED tensor FLOPs.  The epilogue (row top-2 / column arg-max on the ALU pipe: FMNMX / "
                            "FSETP / SEL / VOTE, 64 lanes/clk/SM), not the tensor pipe, bounds the fp16 passes: ncu "
                            "sm__pipe_tensor_cycles_active 50-54 %, ALU pipe 61-65 % (profiles/r01i_ncu_raw_match_f16*.csv)"}
        else:
            tf32_cublas = measure_tf32_peak(dev)
            sm_mhz_r = (clocks or {}).get("sm_mhz") or 1965.0
            pipe_tf32 = 4055.0 * 148 * sm_mhz_r * 1e6 / 1e12        # tools/probe/mma_issue_probe.cu: tf32 FLOP/clk/SM the pipe retires
            ach = flops / match_s / 1e12
            roof = {"kernel": "match_f32_tc_kernel (tcgen05 kind::tf32 fused GEMM + row top-2 / column arg-max)",
                    "bound": "tensor", "achieved": ach, "peak": pipe_tf32, "unit": "TFLOP/s",
                    "traffic": ncu_traffic("match_f32_tc_kernel", pairs_per_launch),
                    "peak_source": "tensor-pipe tf32 rate measured on this GPU model (tools/probe/mma_issue_probe.cu: 4055 FLOP/clk/SM, "
                                   "half the fp16 rate) x 148 SM x the SM clock sampled in this run.  MEASURED_PEAKS.json has no TF32 "
                                   "entry; the two other yardsticks are printed beside it: cuBLAS TF32 measured in this run "
                                   "(peak_cublas_tf32, power-limited like any long GEMM) and 0.5 x the bf16 burst peak of MEASURED_PEAKS.json",
                    "peak_cublas_tf32": tf32_cublas, "frac_of_cublas_tf32": ach / tf32_cublas,
                    "peak_half_bf16_measured": tf32_half_bf16, "frac_of_half_bf16_measured": ach / tf32_half_bf16,
                    "issued_passes": passes, "algorithmic_flops": flops / passes,
                    "note": "achieved counts ISSUED tensor FLOPs (3 tf32 MMAs per k-step for 3xTF32), as BASELINE.md section 3 specifies"}
    roof["frac"] = roof["achieved"] / roof["peak"]
    roof["avg_launch_ms"] = stage_ms.get("match")
    roof["share_of_step"] = share.get("match")

    # ---- every other kernel of the path against its own ceiling (north-star: HBM GB/s for Hamming, RANSAC and
    # back-projection; the binding pipe is named where HBM is structurally not the limit)
    sm_mhz = (clocks or {}).get("sm_mhz") or 1965.0
    fp32_peak = 148 * 128 * 2 * sm_mhz * 1e6 / 1e12                              # FFMA lanes x 2 FLOP, TFLOP/s
    n_corr = out.n_corr.cpu().numpy().astype(np.float64)
    n_match = out.n_matches.cpu().numpy().astype(np.float64)
    launches_per_step = max(stages["score"][1], 1) / (args.steps * R)      # per pass over the P pairs
    corr_per_launch = float(n_corr.sum()) / launches_per_step
    match_per_launch = float(n_match.sum()) / launches_per_step
    Hh = wl["n_hyp"]
    kernels = []
    if "score" in stage_ms:
        t = stage_ms["score"] / 1e3
        evals = corr_per_launch * Hh                                             # (hypothesis, point) inlier tests
        sc_bytes = corr_per_launch * 20.0 * (Hh / 32.0) + pairs_per_launch * Hh * 52.0   # L2->SM staging per CTA + poses
        entry = {"kernel": "score_kernel (packed FFMA2 inlier tests, 4 hypotheses per warp x 2 points per lane, TMA-staged tiles)",
                 "bound": "fp32", "achieved": evals * 27.0 / t / 1e12, "peak": fp32_peak, "unit": "TFLOP/s",
                 "frac": evals * 27.0 / t / 1e12 / fp32_peak, "avg_launch_ms": stage_ms["score"],
                 "evals_per_s": evals / t, "flop_per_eval": 27, "fp32_lane_ops_per_eval": 15,
                 "hbm_gbs": (corr_per_launch * 40.0 + pairs_per_launch * Hh * 52.0) / t / 1e9,
                 "l2_to_sm_gbs": sc_bytes / t / 1e9,
                 "note": "HBM figure is structurally << peak: every correspondence is re-read from L2 by H/32 CTAs "
                         "and tested against all H hypotheses (SURVEY D5: FP32-pipe bound).  evals = hypotheses x points "
                         "BEFORE the exact pruning (hypotheses that can no longer reach the running best count stop "
                         "being scored), so achieved is an EFFECTIVE rate and may exceed the pipe peak; raw_unpruned is "
                         "the same kernel with pruning off (every test executed)"}
        try:  # raw rate of the same kernel, pruning off, same shape (outside the timed region)
            sys.path.insert(0, os.path.join(os.path.dirname(os.path.abspath(__file__)), "tools"))
            import score_bench
            n_med = int(max(np.median(n_corr), 8))
            rb = score_bench.measure(int(min(max(pairs_per_launch, 1), 64)), Hh, n_med, reps=3, dev=dev)
            raw = rb["unpruned"]["tests_per_s"]
            entry["raw_unpruned"] = {"evals_per_s": raw, "achieved": raw * 27.0 / 1e12, "frac": raw * 27.0 / 1e12 / fp32_peak,
                                     "fp32_lane_frac": raw * 15.0 / (148 * 128 * sm_mhz * 1e6),
                                     "pairs": rb["pairs"], "points": n_med, "score_ms": rb["unpruned"]["score_ms"]}
        except Exception as e:  # the probe is informative only
            entry["raw_unpruned"] = {"error": repr(e)}
        kernels.append(entry)
    if "gather" in stage_ms:
        t = stage_ms["gather"] / 1e3
        gb = match_per_launch * 53.0
        kernels.append({"kernel": "gather_backproject_kernel (fused gather + flow filter + depth lookup + gate + compaction)",
                        "bound": "hbm", "achieved": gb / t / 1e9, "peak": hbm_peak, "unit": "GB/s",
                        "frac": gb / t / 1e9 / hbm_peak, "avg_launch_ms": stage_ms["gather"],
                        "note": "53 B per match incl. one 32 B sector per depth pixel; latency-bound at this size"})
    # dense back-projection (cv2.rgbd.depthTo3d replacement): not on the fused pipeline's critical path, timed here on
    # the same depth maps, L2-cold (every launch reads / writes frames no earlier launch of the loop touched)
    try:
        nfr = int(min(seq.depth.shape[0], max(8, (2 << 30) // (seq.depth[0].numel() * 16))))
        frames = seq.depth[:nfr]
        ops.backproject_dense(frames[:2], seq.K)
        torch.cuda.synchronize()
        ops.profile_enable(True); ops.profile_collect()
        xyz_dense = ops.backproject_dense(frames, seq.K)
        st_d = ops.profile_collect(); ops.profile_enable(False)
        t = st_d["dense"][0] / max(st_d["dense"][1], 1) / 1e3
        db = float(frames.numel()) * 16.0
        del xyz_dense
        kernels.append({"kernel": "backproject_dense_kernel (depthTo3d)", "bound": "hbm", "achieved": db / t / 1e9,
                        "peak": hbm_peak, "unit": "GB/s", "frac": db / t / 1e9 / hbm_peak, "avg_launch_ms": t * 1e3,
                        "frames": nfr, "algorithmic_bytes": db,
                        "note": "16 B per pixel (4 read + 12 written); single launch over frames >> L2"})
    except Exception as e:  # never lose the headline line to the side measurement
        kernels.append({"kernel": "backproject_dense_kernel", "error": str(e)[:200]})

    # ---- CPU baseline on a bounded sample (rank 0, N=1 only)
    cpu = None
    if world == 1 and not args.no_cpu:
        sample = args.cpu_pairs or {"c1": 48, "c2": 24, "c2r": 24, "c2tc": 24, "c3": 6, "c4": 2, "c5": 1}[name]
        v, dt, threads, okc = time_cpu_pairs(wl, sample, first_index=0)
        cpu = {"value": v, "unit": "pairs/s", "cores": threads, "kind": "port",
               "sample": f"first {sample} consecutive pairs of the same synthetic workload, {dt:.1f} s, reference CPU path "
                         f"(cv2 {wl['cpu_matcher']} + 3x solvePnPRansac), {okc}/{sample} poses found"}

    if clocks is not None and not clocks.get("samples") and not args.allow_no_clocks:
        raise SystemExit("bench.py: no nvidia-smi clock sample fell inside the timed region; the line would be unverifiable "
                         "(--allow-no-clocks to print it anyway)")
    api = None
    if world == 1 and not args.no_api_rate:
        try:
            api = measure_api_rate(wl, dev)
        except Exception as e:  # informative block: never lose the headline line to it
            api = {"error": repr(e)[:300]}
    line = {
        "metric": "frame-pairs/sec (match+PnP)", "value": value, "unit": "pairs/s", "n_gpus": world,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms / args.steps, "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": dtype_of(wl), "data": "synthetic",
        "config": {"workload": f"{name}: {wl['desc']}", "pairs_per_gpu_per_step": P * R, "passes_per_step": R,
                   "pairs_per_pass": P, "frames_per_gpu": P + 1, "chunk": chunk, "timed_region_s": ms / 1e3,
                   "sequence": "consecutive pairs of one synthetic sequence per GPU: frame i+1 is the current frame of pair i and "
                               "the reference frame of pair i+1 (synthetic.make_chain; no pair or frame is repeated inside a pass)",
                   "l2": f"inputs larger than L2: {seq.nbytes() / 1e6:.0f} MB of frames per GPU are streamed from HBM in every pass",
                   "parallelism": f"pairs sharded over {world} GPU(s), 1 NCCL all-gather of 4x4 poses per pass" if world > 1 else "single GPU",
                   "host_numa_binding": (f"rank 0 bound to {len(numa_cores)} GPU-local cores" if numa_cores else "none")},
        "e2e": {"value": e2e_value, "unit": "pairs/s", "h2d_bytes_per_step": int(h2d_pass * Re),
                "d2h_bytes_per_step": int(d2h_pass * Re), "ms_per_step": e2e_ms / args.steps, "passes_per_step": Re,
                "timed_region_s": e2e_ms / 1e3, "frac_of_resident": e2e_value / value,
                "depth": args.e2e_depth, "sampled_frac": em["frac"],
                "sampled_frac_autotune_ms_per_pass": tune or None, "equals_resident_bitwise": e2e_same,
                "precondition": ("keypoints and depth maps are in PINNED host memory when the timed region starts; the R2D2 descriptors are "
                                 "device-resident, as the reference holds them (its network runs on the GPU and Frame.desc stays a CUDA "
                                 "tensor, R2D2.py:224-232); all_from_host = the same run with the descriptors uploaded from pinned host "
                                 "memory as well" if r2d2_like else
                                 "frames (descriptors, keypoints, depth maps) are in PINNED host memory when the timed region starts") +
                                "; every frame crosses the bus once per pass, poses / status / inlier counts come back, host-side gating + "
                                "pose chaining included",
                "u8_descriptors": (None if em_u8 is None else
                                   {"value": em_u8["value"], "frac_of_resident": em_u8["value"] / value, "h2d_bytes_per_step": int(em_u8["h2d"] * em_u8["Re"]),
                                    "h2d_gbs_per_gpu": em_u8["h2d"] * em_u8["Re"] * args.steps / (em_u8["ms"] / 1e3) / 1e9,
                                    "sampled_frac": em_u8["frac"], "equals_resident_bitwise": em_u8["same"],
                                    "precondition": "as e2e, but the SIFT descriptors are held as uint8 in pinned host memory (OpenCV's SIFT "
                                                    "descriptors are integers 0..255 stored as float32; vo_match_u8 with 128-byte rows / "
                                                    "vo_pipeline_args.u8_bytes = 128 widens them on the device: identical matches and poses)"}),
                "all_from_host": (None if em_host is None else
                                  {"value": em_host["value"], "frac_of_resident": em_host["value"] / value, "h2d_bytes_per_step": int(em_host["h2d"] * em_host["Re"]),
                                   "h2d_gbs_per_gpu": em_host["h2d"] * em_host["Re"] * args.steps / (em_host["ms"] / 1e3) / 1e9,
                                   "sampled_frac": em_host["frac"], "equals_resident_bitwise": em_host["same"]}),
                "h2d_gbs_per_gpu": h2d_pass * Re * args.steps / (e2e_ms / 1e3) / 1e9},
        "gpu_launches": int(launches),
        "clocks": clocks,
        "variants": variants or None,
        "api_rate": api,
        "roofline": roof,
        "kernels": kernels,
        "cpu_baseline": cpu,
        "stages_ms_per_launch": stage_ms,
        "stage_share": share,
        "check": {"pairs_ok_frac": ok_frac, "median_inliers": float(np.median(n_inl)),
                  "median_rot_err_rad": float(np.median([e[0] for e in errs])),
                  "median_trans_err_m": float(np.median([e[1] for e in errs])),
                  "chained_poses": int(chain.shape[0])},
    }
    del seq, out
    torch.cuda.empty_cache()
    return line


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default=os.environ.get("VO_BENCH_WORKLOAD", "default"), choices=sorted(WORKLOADS) + ["default"],
                    help="default = headline c3 (the tcgen05 GEMM of BASELINE.json's metric) with the c2 line in extra.c2; "
                         "VO_BENCH_WORKLOAD sets it for driver-launched runs")
    ap.add_argument("--pairs", type=int, default=0, help="pairs per GPU per pass (default: workload's)")
    ap.add_argument("--passes", type=int, default=0, help="passes over the sequence per step (default: sized for --min-timed-ms)")
    ap.add_argument("--min-timed-ms", type=float, default=2500.0, help="lower bound of the timed region the pass count is sized for")
    ap.add_argument("--chunk", type=int, default=0, help="pairs per vo_pipeline call (default: workload's)")
    ap.add_argument("--e2e-chunk", type=int, default=0, help="pairs per H2D/compute chunk of the e2e run (default: chunk/2)")
    ap.add_argument("--e2e-sampled-frac", type=float, default=None, help="hybrid: fraction of each chunk's maps sampled zero-copy "
                    "(default: autotuned before timing over 0.2 / 0.4 / 0.6 / 0.8 / 1.0)")
    ap.add_argument("--e2e-depth", default="hybrid", choices=["sampled", "dense", "hybrid"],
                    help="e2e leg: copy whole depth maps (dense), read depth at the reference keypoints zero-copy from pinned "
                         "host memory (sampled), or both concurrently (hybrid, default)")
    ap.add_argument("--precision", type=int, default=None)
    ap.add_argument("--cpu-pairs", type=int, default=0)
    ap.add_argument("--no-cpu", action="store_true")
    ap.add_argument("--no-api-rate", action="store_true", help="skip the frames/s measurement through process_frame / the device loop")
    ap.add_argument("--no-variants", action="store_true", help="skip the matcher variants measured beside the headline (hamming_tc, f16x3)")
    ap.add_argument("--allow-no-clocks", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the last timed step's pipeline outputs (poses, rt, match / correspondence / inlier counts, status; "
                         "float64) as DIR/<workload>_<name>.npy, so that two builds can be compared on identical seeded inputs")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs applies to --impl ours")
    rank, _, world = env_rank()
    names = ["c2", "c3"] if args.workload == "default" else [args.workload]     # headline last
    if args.impl == "reference":
        if rank != 0:
            return                                                             # N > 1: rank 0 alone runs and prints it
        lines = [run_reference(args, n) for n in names]
    else:
        lines = [run_ours(args, n) for n in names]
        if world > 1:
            import torch.distributed as dist
            dist.barrier()
            dist.destroy_process_group()
        if rank != 0:
            return
    line = lines[-1]
    if len(lines) > 1:
        line["extra"] = {n: l for n, l in zip(names[:-1], lines[:-1])}
        line["config"]["also_measured"] = "extra.c2 = the complete line of workload c2 (BASELINE.json configs[1]) from the same run"
    print(json.dumps(line), flush=True)


if __name__ == "__main__":
    main()
