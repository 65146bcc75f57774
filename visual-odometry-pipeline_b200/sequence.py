"""Throughput mode: a pre-declared list of frame pairs, sharded across GPUs (SURVEY D3, 8(e)).

Each rank runs vo_pipeline over its contiguous block of pairs; one all-gather of the 4x4 relative poses
(+ status) follows; the host chains them with a prefix product in which failed or implausible pairs
contribute the identity, mirroring VisualOdometry.process_frame (VisualOdometry_Stereo.py:270-274, 283, 290).
There is no other collective: pairs are independent.
"""
import numpy as np
import torch

from . import ops


def bind_to_gpu_numa(device_index):
    """Pin this process to the CPU cores NVML reports as local to the GPU, BEFORE host buffers are allocated, so that
    pinned staging memory lands on the GPU's NUMA node (first touch).  With one process per GPU on an 8-GPU box the
    host-to-device legs otherwise all pull from whichever node the ranks happened to start on.  Returns the core
    list, or None when NVML / affinity is unavailable (nothing is changed then)."""
    import os
    try:
        import pynvml
        pynvml.nvmlInit()
        visible = os.environ.get("CUDA_VISIBLE_DEVICES")
        idx = int(visible.split(",")[device_index]) if visible and visible.split(",")[device_index].isdigit() else device_index
        h = pynvml.nvmlDeviceGetHandleByIndex(idx)
        n_cpu = os.cpu_count() or 1
        words = pynvml.nvmlDeviceGetCpuAffinity(h, (n_cpu + 63) // 64)
        cores = [64 * w + b for w, mask in enumerate(words) for b in range(64) if (mask >> b) & 1 and 64 * w + b < n_cpu]
        allowed = sorted(set(cores) & set(os.sched_getaffinity(0)))
        if allowed:
            os.sched_setaffinity(0, allowed)
            return allowed
    except Exception:
        pass
    return None


def shard_range(n_pairs, rank, world):
    """Contiguous block [lo, hi) of the pair list owned by `rank`."""
    base, rem = divmod(int(n_pairs), int(world))
    lo = rank * base + min(rank, rem)
    return lo, lo + base + (1 if rank < rem else 0)


def gate_poses(T_rel, status, max_step_m=1.5):
    """Host-side a9 gate: a pair is used iff PnP succeeded and ||t|| <= 1.5 m (consecutive frames)."""
    T_rel = np.asarray(T_rel, np.float64).reshape(-1, 4, 4)
    ok = (np.asarray(status).reshape(-1) == 0) & (np.linalg.norm(T_rel[:, :3, 3], axis=1) <= max_step_m)
    return ok


def chain_poses(T_rel, ok=None):
    """Global poses G_0 = I, G_k = prod_{i<k} T_i (failed pairs -> identity).  Vectorised log-depth scan:
    ceil(log2 P) batched 4x4 products instead of P sequential ones.  Returns (P+1, 4, 4) f64."""
    T = np.array(T_rel, np.float64).reshape(-1, 4, 4)
    P = T.shape[0]
    if ok is not None:
        T[~np.asarray(ok, bool)] = np.eye(4)
    acc = T.copy()
    shift = 1
    while shift < P:
        nxt = acc.copy()
        nxt[shift:] = acc[:-shift] @ acc[shift:]     # inclusive scan, left-to-right products
        acc = nxt
        shift *= 2
    out = np.empty((P + 1, 4, 4), np.float64)
    out[0] = np.eye(4)
    out[1:] = acc
    return out


def all_gather_poses(T_rel, status, world=None):
    """One all-gather of [T_rel | status] over the default process group (NCCL on GPUs, gloo in CPU tests).
    T_rel [P_local,4,4] f64, status [P_local] int32 -> concatenated over ranks in rank order.  Every rank
    must contribute the same P_local (pad the tail rank)."""
    import torch.distributed as dist
    if world is None:
        world = dist.get_world_size() if dist.is_initialized() else 1
    packed = torch.cat([T_rel.reshape(T_rel.shape[0], 16), status.to(torch.float64).reshape(-1, 1)], dim=1).contiguous()
    if world == 1:
        return T_rel.reshape(-1, 4, 4), status
    out = torch.empty((world * packed.shape[0], 17), dtype=torch.float64, device=packed.device)
    dist.all_gather_into_tensor(out, packed)
    return out[:, :16].reshape(-1, 4, 4), out[:, 16].to(torch.int32)


class PairBatch:
    """Device-resident inputs of a block of frame pairs (what a front-end would have produced)."""

    def __init__(self, ref_desc, cur_desc, ref_kp, cur_kp, depth, K):
        self.ref_desc, self.cur_desc, self.ref_kp, self.cur_kp, self.depth = ref_desc, cur_desc, ref_kp, cur_kp, depth
        self.K = np.asarray(K, np.float64)
        self.B = ref_desc.shape[0]

    @staticmethod
    def from_numpy(batch, device="cuda", repeat=1):
        def up(a):
            t = torch.from_numpy(np.ascontiguousarray(a)).to(device)
            return t.repeat((repeat,) + (1,) * (t.dim() - 1)) if repeat > 1 else t
        return PairBatch(up(batch["ref_desc"]), up(batch["cur_desc"]), up(batch["ref_kp"]), up(batch["cur_kp"]),
                         up(batch["depth"]), batch["K"])

    def slice(self, lo, hi):
        return PairBatch(self.ref_desc[lo:hi], self.cur_desc[lo:hi], self.ref_kp[lo:hi], self.cur_kp[lo:hi],
                         self.depth[lo:hi], self.K)

    def nbytes(self):
        return sum(t.numel() * t.element_size() for t in (self.ref_desc, self.cur_desc, self.ref_kp, self.cur_kp, self.depth))


class FrameSequence:
    """Device-resident frames of one sequence: desc [F,N,..], kp [F,N,s], depth [F,H,W].  Pair i = (frame i, frame i+1):
    frame i+1 is the current frame of pair i and the reference frame of pair i+1 (as in VisualOdometry.process_frame when
    every frame becomes the keyframe), so every frame is resident once and the two sides of a pair batch are views of the
    same arrays shifted by one frame."""

    def __init__(self, desc, kp, depth, K):
        self.desc, self.kp, self.depth = desc, kp, depth
        self.K = np.asarray(K, np.float64)
        self.B = desc.shape[0] - 1

    @staticmethod
    def from_numpy(chain, device="cuda"):
        up = lambda a: (a if isinstance(a, torch.Tensor) else torch.from_numpy(np.ascontiguousarray(a))).to(device)  # noqa: E731
        return FrameSequence(up(chain["desc"]), up(chain["kp"]), up(chain["depth"]), chain["K"])

    def slice(self, lo, hi):
        return PairBatch(self.desc[lo:hi], self.desc[lo + 1:hi + 1], self.kp[lo:hi], self.kp[lo + 1:hi + 1],
                         self.depth[lo:hi], self.K)

    def nbytes(self):
        return sum(t.numel() * t.element_size() for t in (self.desc, self.kp, self.depth))


class PipelineConfig:
    """Keyword arguments of ops.pipeline shared by every chunk.  pnp_mode "reference" selects Mode R (the reference's sampler,
    bootstrap rows keyed by the pair like the hypotheses: results do not depend on chunk or lanes); the default is Mode T."""
    def __init__(self, norm_or_metric, mode, match_param=0.85, precision=ops.VO_PREC_TF32X3, n_hyp=1024, seed=8214,
                 thr_px=1.5, min_inliers=20, refine_iters=10, pnp_mode="throughput", ref_restarts=3, ref_iters=100,
                 ref_confidence=0.99):
        ops.pnp_mode_id(pnp_mode)
        self.kw = dict(norm_or_metric=norm_or_metric, mode=mode, match_param=match_param, precision=precision,
                       n_hyp=n_hyp, seed=seed, thr_px=thr_px, min_inliers=min_inliers, refine_iters=refine_iters)
        if pnp_mode != "throughput":
            self.kw.update(pnp_mode=pnp_mode, ref_restarts=ref_restarts, ref_iters=ref_iters, ref_confidence=ref_confidence)


_LANE_STREAMS = {}


def _lane_streams(device, lanes):
    key = (torch.device(device).index, lanes)
    if key not in _LANE_STREAMS:
        _LANE_STREAMS[key] = [torch.cuda.Stream(device=device) for _ in range(lanes)]
    return _LANE_STREAMS[key]


def run_resident(batch, cfg, pair0=0, chunk=None, out=None, lanes=1):
    """vo_pipeline over device-resident pairs, in chunks; returns a PipelineBuffers covering the whole block.
    `lanes` > 1 issues the chunks round-robin on that many streams (one vo_ctx, i.e. one workspace, each), forked from and
    joined to the current stream: the small-grid tail of one chunk (gather, P3P, score, refit — one CTA per pair) then
    overlaps the next chunk's matcher instead of leaving most SMs idle.  Results do not depend on `lanes`."""
    B = batch.B
    chunk = chunk or B
    dev = batch.slice(0, 1).ref_desc.device
    out = out or ops.PipelineBuffers(B, dev)
    cur = torch.cuda.current_stream(dev)
    streams = _lane_streams(dev, lanes) if lanes > 1 else [cur]
    if lanes > 1:
        for ls in streams:
            ls.wait_stream(cur)
    for i, lo in enumerate(range(0, B, chunk)):
        hi = min(B, lo + chunk)
        sub = batch.slice(lo, hi)
        view = ops.PipelineBuffers.__new__(ops.PipelineBuffers)
        view.T_rel, view.rt = out.T_rel[lo:hi], out.rt[lo:hi]
        view.n_matches, view.n_corr = out.n_matches[lo:hi], out.n_corr[lo:hi]
        view.n_inl, view.status = out.n_inl[lo:hi], out.status[lo:hi]
        with torch.cuda.stream(streams[i % lanes]):
            ops.pipeline(sub.ref_desc, sub.cur_desc, sub.ref_kp, sub.cur_kp, sub.depth, batch.K, pair0=pair0 + lo,
                         out=view, lane=i % lanes, **cfg.kw)
    if lanes > 1:
        for ls in streams:
            cur.wait_stream(ls)
    return out


def chunk_schedule(B, chunk):
    """[(lo, hi)] covering B pairs.  The copy engine is the bottleneck of the host path, so nothing is gained at the
    front, but the compute of the LAST chunk overlaps no copy: the tail is cut into chunk/2 and chunk/4 pieces (drain
    time 4.1 -> 1 ms per 1000 ORB pairs at chunk 125) and the remaining full chunks are equalised."""
    tail = [max(1, chunk // 2), max(1, chunk // 4)]
    body = B - sum(tail)
    if body < chunk:
        sizes = [min(chunk, B - lo) for lo in range(0, B, chunk)]
    else:
        n_body = -(-body // chunk)
        base, rem = divmod(body, n_body)
        sizes = [base + (1 if i < rem else 0) for i in range(n_body)] + tail
    out, lo = [], 0
    for n in sizes:
        out.append((lo, lo + n))
        lo += n
    assert lo == B and all(hi - lo_ <= chunk for lo_, hi in out)
    return out


class HostPairRunner:
    """End-to-end path for HOST inputs: pinned host buffers -> H2D on a copy stream, double-buffered against
    vo_pipeline on the compute stream -> D2H of poses / status.  This is the call a user with frames in host
    memory makes; bench.py times it as `e2e`.

    Depth maps are 82 % of the bytes of an ORB pair (1.87 MB of 2.27 MB at 1241x376) although only the pixels under the
    reference keypoints are read, and the bulk copy alone saturates PCIe.  depth_mode selects how they travel:
      "dense"    whole maps by DMA (copy engine);
      "sampled"  maps stay in pinned host memory; vo_sample_depth reads depth[int(y), int(x)] of every reference
                 keypoint through the mapped pointer (one 32 B sector per keypoint, ~125 M reads/s measured);
      "hybrid"   both at once: the first (1 - sampled_frac) of each chunk's maps go by DMA on the copy stream while the
                 SMs pull the samples of the rest zero-copy on a third stream — the two paths are limited by different
                 things (link bandwidth vs outstanding small reads), so together they move a chunk faster than either.
      "matched"  maps stay in pinned host memory and vo_pipeline gets the mapped pointer: the gather kernel reads only
                 the pixels under the MATCHED reference keypoints that pass the flow filter (~3.6 k of 5 k at ORB 5k).
                 Those reads sit inside the pipeline (after the matcher), so consecutive chunks alternate between two
                 lanes (stream + vo_ctx each): one chunk's reads are in flight while the next chunk's matcher runs.
    In "sampled" / "hybrid" vo_pipeline consumes the compact depth_kp array (sampled on the device for DMA'd maps)."""

    def __init__(self, host_batch, cfg, chunk, device="cuda", depth_mode="dense", sampled_frac=0.2):
        if depth_mode not in ("dense", "sampled", "hybrid", "matched"):
            raise ValueError(depth_mode)
        self.depth_mode = depth_mode
        self.cfg, self.chunk, self.device = cfg, chunk, torch.device(device)
        self.K = np.asarray(host_batch["K"], np.float64)
        keys = ("ref_desc", "cur_desc", "ref_kp", "cur_kp", "depth")
        self.host = {k: torch.from_numpy(np.ascontiguousarray(host_batch[k])).pin_memory() for k in keys}
        self.B = self.host["ref_desc"].shape[0]
        # pairs [0, n_dma) of a chunk send their map by DMA, pairs [n_dma, chunk) are sampled from host memory
        self.frac = {"dense": 0.0, "sampled": 1.0, "hybrid": float(sampled_frac), "matched": 1.0}[depth_mode]
        self.n_dma = chunk - int(round(chunk * self.frac))
        self.schedule = chunk_schedule(self.B, chunk)
        self.hw = tuple(self.host["depth"].shape[1:])
        N = self.host["ref_kp"].shape[1]
        self.stage = []
        self.n_stage = 4 if depth_mode == "matched" else 2   # matched: two chunks computing + one copying
        for _ in range(self.n_stage):
            st = {k: torch.empty((chunk,) + tuple(self.host[k].shape[1:]), dtype=self.host[k].dtype, device=self.device)
                  for k in keys if k != "depth"}
            if self.n_dma and depth_mode != "matched":
                st["depth"] = torch.empty((self.n_dma,) + self.hw, dtype=torch.float32, device=self.device)
            if depth_mode in ("sampled", "hybrid"):
                st["depth_kp"] = torch.empty((chunk, N), dtype=torch.float32, device=self.device)
            self.stage.append(st)
        self.lanes = [torch.cuda.Stream(device=self.device) for _ in range(2)] if depth_mode == "matched" else []
        self.copy_stream = torch.cuda.Stream(device=self.device)
        self.sample_stream = torch.cuda.Stream(device=self.device)
        self.copied = [torch.cuda.Event() for _ in range(self.n_stage)]
        self.kp_ready = [torch.cuda.Event() for _ in range(self.n_stage)]
        self.sampled = [torch.cuda.Event() for _ in range(self.n_stage)]
        self.consumed = [torch.cuda.Event() for _ in range(self.n_stage)]
        self.out = ops.PipelineBuffers(self.B, self.device)
        self.host_T = torch.empty((self.B, 4, 4), dtype=torch.float64).pin_memory()
        self.host_status = torch.empty((self.B,), dtype=torch.int32).pin_memory()
        self.host_inl = torch.empty((self.B,), dtype=torch.int32).pin_memory()
        per_pair = {k: v[0].numel() * v.element_size() for k, v in self.host.items()}
        dma_pairs = sum(self._n_dma(hi - lo) for lo, hi in self.schedule)
        self.h2d_bytes = self.B * sum(b for k, b in per_pair.items() if k != "depth") + dma_pairs * per_pair["depth"] \
            + (self.B - dma_pairs) * N * 32          # one 32-byte sector per zero-copy sample
        self.d2h_bytes = self.host_T.numel() * 8 + self.host_status.numel() * 4 + self.host_inl.numel() * 4
        self._base_bytes = self.B * sum(b for k, b in per_pair.items() if k != "depth")

    def count_matched_bytes(self):
        """matched mode, after a run: h2d_bytes = descriptors / keypoints + one 32-byte sector per match (every match
        reads at most one depth pixel; those under the flow filter read none, so this is an upper bound)."""
        if self.depth_mode == "matched":
            self.h2d_bytes = self._base_bytes + int(self.out.n_matches.sum().item()) * 32
        return self.h2d_bytes

    def _view(self, lo, hi):
        view = ops.PipelineBuffers.__new__(ops.PipelineBuffers)
        view.T_rel, view.rt = self.out.T_rel[lo:hi], self.out.rt[lo:hi]
        view.n_matches, view.n_corr = self.out.n_matches[lo:hi], self.out.n_corr[lo:hi]
        view.n_inl, view.status = self.out.n_inl[lo:hi], self.out.status[lo:hi]
        return view

    def _run_matched(self, pair0):
        compute = torch.cuda.current_stream(self.device)
        for ls in self.lanes:
            ls.wait_stream(compute)
        for c, (lo, hi) in enumerate(self.schedule):
            n, buf, lane = hi - lo, c % self.n_stage, c % 2
            st = self.stage[buf]
            with torch.cuda.stream(self.copy_stream):
                if c >= self.n_stage:
                    self.copy_stream.wait_event(self.consumed[buf])
                for k in ("ref_kp", "cur_kp", "ref_desc", "cur_desc"):
                    st[k][:n].copy_(self.host[k][lo:hi], non_blocking=True)
                self.copied[buf].record(self.copy_stream)
            with torch.cuda.stream(self.lanes[lane]):
                self.lanes[lane].wait_event(self.copied[buf])
                ops.pipeline(st["ref_desc"][:n], st["cur_desc"][:n], st["ref_kp"][:n], st["cur_kp"][:n],
                             self.host["depth"][lo:hi], self.K, pair0=pair0 + lo, out=self._view(lo, hi), lane=lane,
                             **self.cfg.kw)
                self.consumed[buf].record(self.lanes[lane])
        for ls in self.lanes:
            compute.wait_stream(ls)
        self.host_T.copy_(self.out.T_rel, non_blocking=True)
        self.host_status.copy_(self.out.status, non_blocking=True)
        self.host_inl.copy_(self.out.n_inl, non_blocking=True)
        return self.host_T, self.host_status, self.host_inl

    def _n_dma(self, n):
        """pairs of an n-pair chunk whose depth map travels by DMA (the rest is sampled zero-copy)"""
        return n - int(round(n * self.frac))

    def run(self, pair0=0):
        """One pass over all pairs.  Returns after the D2H copies were enqueued; caller synchronises."""
        if self.depth_mode == "matched":
            return self._run_matched(pair0)
        compute = torch.cuda.current_stream(self.device)
        for c, (lo, hi) in enumerate(self.schedule):
            n, buf = hi - lo, c % 2
            st = self.stage[buf]
            n_dma = self._n_dma(n)
            with torch.cuda.stream(self.copy_stream):
                if c >= 2:
                    self.copy_stream.wait_event(self.consumed[buf])
                st["ref_kp"][:n].copy_(self.host["ref_kp"][lo:hi], non_blocking=True)
                self.kp_ready[buf].record(self.copy_stream)
                for k in ("cur_kp", "ref_desc", "cur_desc"):   # one copy stream: a second one for the descriptors measured slower
                    st[k][:n].copy_(self.host[k][lo:hi], non_blocking=True)
                if n_dma:
                    st["depth"][:n_dma].copy_(self.host["depth"][lo:lo + n_dma], non_blocking=True)
                    if self.depth_mode != "dense":   # maps that came by DMA are sampled from HBM
                        ops.sample_depth(st["ref_kp"][:n_dma], st["depth"][:n_dma], out=st["depth_kp"][:n_dma])
                self.copied[buf].record(self.copy_stream)
            if n > n_dma:
                with torch.cuda.stream(self.sample_stream):   # zero-copy samples, concurrent with the DMA above
                    self.sample_stream.wait_event(self.kp_ready[buf])
                    ops.sample_depth(st["ref_kp"][n_dma:n], self.host["depth"][lo + n_dma:hi], out=st["depth_kp"][n_dma:n])
                    self.sampled[buf].record(self.sample_stream)
                compute.wait_event(self.sampled[buf])
            compute.wait_event(self.copied[buf])
            view = ops.PipelineBuffers.__new__(ops.PipelineBuffers)
            view.T_rel, view.rt = self.out.T_rel[lo:hi], self.out.rt[lo:hi]
            view.n_matches, view.n_corr = self.out.n_matches[lo:hi], self.out.n_corr[lo:hi]
            view.n_inl, view.status = self.out.n_inl[lo:hi], self.out.status[lo:hi]
            if self.depth_mode == "dense":
                ops.pipeline(st["ref_desc"][:n], st["cur_desc"][:n], st["ref_kp"][:n], st["cur_kp"][:n], st["depth"][:n],
                             self.K, pair0=pair0 + lo, out=view, **self.cfg.kw)
            else:
                ops.pipeline(st["ref_desc"][:n], st["cur_desc"][:n], st["ref_kp"][:n], st["cur_kp"][:n], None, self.K,
                             pair0=pair0 + lo, out=view, depth_kp=st["depth_kp"][:n], hw=self.hw, **self.cfg.kw)
            self.consumed[buf].record(compute)
        self.host_T.copy_(self.out.T_rel, non_blocking=True)
        self.host_status.copy_(self.out.status, non_blocking=True)
        self.host_inl.copy_(self.out.n_inl, non_blocking=True)
        return self.host_T, self.host_status, self.host_inl


class HostSequenceRunner:
    """End-to-end path for a SEQUENCE held in pinned host memory: frames desc [F,N,..], kp [F,N,s], depth [F,H,W]; pair i =
    (frame i, frame i+1).  Every frame crosses the bus once: a chunk of n pairs uploads its n+1 frames' descriptors and
    keypoints (the first frame of a chunk is copied device-to-device from the previous chunk's last one) on a copy
    stream, double-buffered against vo_pipeline on the compute stream; poses, status and inlier counts come back with one
    D2H copy per pass.  Depth maps are needed for reference frames only, and only under their keypoints:
      "dense"    whole maps by DMA;
      "sampled"  maps stay in pinned host memory, vo_sample_depth reads depth[int(y), int(x)] of every reference keypoint
                 zero-copy through the mapped pointer (one 32 B sector per keypoint);
      "hybrid"   the first (1 - sampled_frac) of a chunk's maps by DMA while the SMs pull the samples of the rest on a
                 third stream.  `autotune()` picks sampled_frac by timing whole passes (the best split depends on how many
                 GPUs share the host's memory system).
    Precondition: the frames are already in pinned host memory (numpy inputs are pinned here, outside any timed region).
    `host_seq["desc"]` may be a CUDA tensor instead: descriptors that never left the device — how the reference holds R2D2
    descriptors (R2D2.py:224-232 keeps them CUDA tensors, the network runs on the GPU) — are used in place; only keypoints and
    depth then cross the bus."""

    def __init__(self, host_seq, cfg, chunk, device="cuda", depth_mode="hybrid", sampled_frac=0.4):
        if depth_mode not in ("dense", "sampled", "hybrid"):
            raise ValueError(depth_mode)
        self.depth_mode = depth_mode
        self.cfg, self.chunk, self.device = cfg, int(chunk), torch.device(device)
        self.K = np.asarray(host_seq["K"], np.float64)

        def pinned(a):
            t = a if isinstance(a, torch.Tensor) else torch.from_numpy(np.ascontiguousarray(a))
            return t if t.is_pinned() else t.pin_memory()
        self.dev_desc = host_seq["desc"] if isinstance(host_seq["desc"], torch.Tensor) and host_seq["desc"].is_cuda else None
        self.host = {k: pinned(host_seq[k]) for k in (("kp", "depth") if self.dev_desc is not None else ("desc", "kp", "depth"))}
        self.B = self.host["kp"].shape[0] - 1
        self.hw = tuple(self.host["depth"].shape[1:])
        self.N = self.host["kp"].shape[1]
        self.frac = {"dense": 0.0, "sampled": 1.0, "hybrid": float(sampled_frac)}[depth_mode]
        self.schedule = chunk_schedule(self.B, self.chunk)
        c = self.chunk
        self.stage = []
        for _ in range(2):
            st = {k: torch.empty((c + 1,) + tuple(self.host[k].shape[1:]), dtype=self.host[k].dtype, device=self.device)
                  for k in ("desc", "kp") if k in self.host}
            if depth_mode != "sampled":
                st["depth"] = torch.empty((c,) + self.hw, dtype=torch.float32, device=self.device)
            if depth_mode != "dense":
                st["depth_kp"] = torch.empty((c, self.N), dtype=torch.float32, device=self.device)
            self.stage.append(st)
        self.copy_stream = torch.cuda.Stream(device=self.device)
        self.sample_stream = torch.cuda.Stream(device=self.device, priority=-1)   # its thin CTAs go ahead of pending matcher CTAs
        self.copied = [torch.cuda.Event() for _ in range(2)]
        self.kp_ready = [torch.cuda.Event() for _ in range(2)]
        self.sampled = [torch.cuda.Event() for _ in range(2)]
        self.consumed = [torch.cuda.Event() for _ in range(2)]
        self.out = ops.PipelineBuffers(self.B, self.device)
        self.host_out = [(torch.empty((self.B, 4, 4), dtype=torch.float64).pin_memory(),
                          torch.empty((self.B,), dtype=torch.int32).pin_memory(),
                          torch.empty((self.B,), dtype=torch.int32).pin_memory(), torch.cuda.Event()) for _ in range(2)]
        self.d2h_bytes = self.B * (128 + 4 + 4)
        self._issued = 0                                   # chunks submitted so far (stage buffers alternate across passes too)
        self._passes = 0

    def _n_dma(self, n):
        return n - int(round(n * self.frac))

    @property
    def h2d_bytes(self):
        """bytes that cross the bus per pass: every frame's descriptors + keypoints once (+ the first frame of the pass),
        whole maps for the DMA share, one 32-byte sector per reference keypoint for the sampled share."""
        per = {k: v[0].numel() * v.element_size() for k, v in self.host.items()}
        dma = sum(self._n_dma(hi - lo) for lo, hi in self.schedule)
        return (self.B + 1) * (per.get("desc", 0) + per["kp"]) + dma * per["depth"] + (self.B - dma) * self.N * 32

    def _view(self, lo, hi):
        view = ops.PipelineBuffers.__new__(ops.PipelineBuffers)
        view.T_rel, view.rt = self.out.T_rel[lo:hi], self.out.rt[lo:hi]
        view.n_matches, view.n_corr = self.out.n_matches[lo:hi], self.out.n_corr[lo:hi]
        view.n_inl, view.status = self.out.n_inl[lo:hi], self.out.status[lo:hi]
        return view

    def submit(self, pair0=0):
        """Enqueue one pass over all pairs (copies, sampling, vo_pipeline per chunk, D2H of the results) and return a ticket
        for `collect`.  Nothing here waits for the GPU: the next pass can be submitted while this one runs, its first
        chunks' copies then overlap this pass's last chunks (two passes' results may be in flight: ping-pong host buffers)."""
        compute = torch.cuda.current_stream(self.device)
        prev = None                                        # (stage index, pairs) of the previous chunk of THIS pass
        for lo, hi in self.schedule:
            n, buf = hi - lo, self._issued % 2
            reuse = self._issued >= 2                      # the stage buffer was used by an earlier chunk (of this or the last pass)
            self._issued += 1
            st = self.stage[buf]
            n_dma = self._n_dma(n)
            with torch.cuda.stream(self.copy_stream):
                if reuse:
                    self.copy_stream.wait_event(self.consumed[buf])
                first = 0
                if prev is not None:                       # frame lo is already on the device: last frame of the previous chunk
                    pst, pn = self.stage[prev[0]], prev[1]
                    st["kp"][0].copy_(pst["kp"][pn], non_blocking=True)
                    if self.dev_desc is None:
                        st["desc"][0].copy_(pst["desc"][pn], non_blocking=True)
                    first = 1
                st["kp"][first:n + 1].copy_(self.host["kp"][lo + first:hi + 1], non_blocking=True)
                self.kp_ready[buf].record(self.copy_stream)
                if self.dev_desc is None:
                    st["desc"][first:n + 1].copy_(self.host["desc"][lo + first:hi + 1], non_blocking=True)
                if n_dma:
                    st["depth"][:n_dma].copy_(self.host["depth"][lo:lo + n_dma], non_blocking=True)
                    if self.depth_mode != "dense":         # maps that came by DMA are sampled from HBM
                        ops.sample_depth(st["kp"][:n_dma], st["depth"][:n_dma], out=st["depth_kp"][:n_dma])
                self.copied[buf].record(self.copy_stream)
            if n > n_dma:
                with torch.cuda.stream(self.sample_stream):   # zero-copy samples, concurrent with the DMA above and the matcher
                    self.sample_stream.wait_event(self.kp_ready[buf])
                    ops.sample_depth(st["kp"][n_dma:n], self.host["depth"][lo + n_dma:hi], out=st["depth_kp"][n_dma:n])
                    self.sampled[buf].record(self.sample_stream)
                compute.wait_event(self.sampled[buf])
            compute.wait_event(self.copied[buf])
            d_ref, d_cur = (st["desc"][:n], st["desc"][1:n + 1]) if self.dev_desc is None else \
                (self.dev_desc[lo:hi], self.dev_desc[lo + 1:hi + 1])
            if self.depth_mode == "dense":
                ops.pipeline(d_ref, d_cur, st["kp"][:n], st["kp"][1:n + 1], st["depth"][:n], self.K,
                             pair0=pair0 + lo, out=self._view(lo, hi), **self.cfg.kw)
            else:
                ops.pipeline(d_ref, d_cur, st["kp"][:n], st["kp"][1:n + 1], None, self.K,
                             pair0=pair0 + lo, out=self._view(lo, hi), depth_kp=st["depth_kp"][:n], hw=self.hw, **self.cfg.kw)
            self.consumed[buf].record(compute)
            prev = (buf, n)
        slot = self._passes % 2
        self._passes += 1
        T_h, st_h, inl_h, done = self.host_out[slot]
        T_h.copy_(self.out.T_rel, non_blocking=True)
        st_h.copy_(self.out.status, non_blocking=True)
        inl_h.copy_(self.out.n_inl, non_blocking=True)
        done.record(compute)
        return slot

    def collect(self, ticket):
        """Wait for a submitted pass; returns its pinned host results (T_rel [B,4,4] f64, status, n_inl), valid until the
        pass after the next one is submitted."""
        T_h, st_h, inl_h, done = self.host_out[ticket]
        done.synchronize()
        return T_h, st_h, inl_h

    def run(self, pair0=0):
        """One pass over all pairs.  Returns after the D2H copies were enqueued; the caller synchronises."""
        T_h, st_h, inl_h, _ = self.host_out[self.submit(pair0)]
        return T_h, st_h, inl_h

    def autotune(self, fracs=(0.2, 0.4, 0.6, 0.8, 1.0), sync=None):
        """hybrid only: time one pass per candidate sampled_frac (after one warm pass) and keep the fastest.  `sync` is
        called before every timed pass (a barrier under torch.distributed, so that all ranks load the host together).
        Returns {frac: ms}."""
        if self.depth_mode != "hybrid":
            return {}
        res = {}
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        self.run()
        torch.cuda.synchronize(self.device)
        for f in fracs:
            self.frac = float(f)
            if sync:
                sync()
            e0.record()
            self.run()
            e1.record()
            torch.cuda.synchronize(self.device)
            res[float(f)] = e0.elapsed_time(e1)
        self.frac = min(res, key=res.get)
        return res
