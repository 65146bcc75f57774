"""S sequences from camera images (MultiDeviceLoop.push_images: batched ORB, then vo_seq_push_all_dev with the keypoint counts
on the device).  Each sequence's poses and info equal, bit for bit, a single DeviceLoop fed the same images through
push_image; a frame with more keypoints than n_cap keeps its first n_cap rows and is counted; no step synchronises."""
import ctypes

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

H, W = 320, 640
K = np.array([[500.0, 0.0, 320.0], [0.0, 500.0, 160.0], [0.0, 0.0, 1.0]])
DEPTH = 10.0
LENGTHS = (10, 12, 8, 11)
STARTS = (0, 2, 0, 4)                         # the step of each sequence's first frame
SKIPS = (set(), {5}, {3, 4}, set())           # steps (after its start) at which a sequence has no frame
SEEDS = (8214, 77, 2 ** 40 + 3, 5)
CONFIGS = {
    "orb_l2_ratio_T": dict(norm_or_metric=1, mode=0, pnp_mode="throughput"),
    "orb_hamming_mutual_T": dict(norm_or_metric=0, mode=1, pnp_mode="throughput"),
    "orb_hamming_mutual_R": dict(norm_or_metric=0, mode=1, pnp_mode="reference"),
}


def _frames(q, n):
    """n BGR frames of sequence q: an H x W window panning 5 pixels per frame over the sequence's own seeded texture
    (smooth random field plus noise, per channel)."""
    rng = np.random.default_rng(500 + q)
    th, tw = H + 16, W + 5 * n + 16
    coarse = rng.integers(0, 256, (th // 10 + 2, tw // 10 + 2, 3)).astype(np.float32)
    ys, xs = np.arange(th) / 10.0, np.arange(tw) / 10.0
    y0, x0 = ys.astype(int), xs.astype(int)
    fy, fx = (ys - y0)[:, None, None], (xs - x0)[None, :, None]
    tex = (coarse[y0][:, x0] * (1 - fy) * (1 - fx) + coarse[y0 + 1][:, x0] * fy * (1 - fx) +
           coarse[y0][:, x0 + 1] * (1 - fy) * fx + coarse[y0 + 1][:, x0 + 1] * fy * fx)
    tex = np.clip(tex + rng.integers(0, 25, tex.shape), 0, 255).astype(np.uint8)
    return [np.ascontiguousarray(tex[8:8 + H, 8 + 5 * i:8 + 5 * i + W]) for i in range(n)]


def _schedule(lengths, starts, skips):
    nxt, steps, t = [0] * len(lengths), [], 0
    while any(nxt[q] < lengths[q] for q in range(len(lengths))):
        row = []
        for q in range(len(lengths)):
            if t >= starts[q] and t not in skips[q] and nxt[q] < lengths[q]:
                row.append(nxt[q])
                nxt[q] += 1
            else:
                row.append(None)
        steps.append(row)
        t += 1
    return steps


def _run_images(seqs, opts, n_cap, starts, skips, hook=None):
    """MultiDeviceLoop.push_images over the schedule; an absent sequence's slot holds a noise image (extracted, ignored)."""
    import torch
    from vo_b200.device_loop import MultiDeviceLoop
    S = len(seqs)
    loop = MultiDeviceLoop(K, (W, H), n_cap, S, seeds=list(SEEDS[:S]), kind="orb", n_hyp=256, **opts)
    noise = np.random.default_rng(1).integers(0, 256, (H, W, 3), dtype=np.uint8)
    depth = torch.full((S, H, W), DEPTH, dtype=torch.float32).pin_memory()
    for t, row in enumerate(_schedule([len(s) for s in seqs], starts, skips)):
        images = torch.from_numpy(np.stack([seqs[q][i] if i is not None else noise for q, i in enumerate(row)])).pin_memory()
        loop.push_images(images, depth, [i or 0 for i in row], present=[i is not None for i in row])
        if hook:
            hook(t, loop)
    out = [loop.poses(q) for q in range(S)]
    lost = [loop.lost_frames(q) for q in range(S)]
    assert [loop.frames(q) for q in range(S)] == [len(s) for s in seqs]
    loop.close()
    return out, lost


def _same(a, b):
    return np.array_equal(a[0], b[0]) and np.array_equal(a[1], b[1])


@pytest.mark.parametrize("name", list(CONFIGS))
def test_each_sequence_equals_a_single_loop_from_images(name):
    import vo_b200  # noqa: F401
    from vo_b200.device_loop import DeviceLoop
    opts = CONFIGS[name]
    seqs = [_frames(q, n) for q, n in enumerate(LENGTHS)]
    got, lost = _run_images(seqs, opts, 1024, STARTS, SKIPS)
    assert lost == [0] * len(seqs)
    depth = np.full((H, W), DEPTH, np.float32)
    for q, frames in enumerate(seqs):
        single = DeviceLoop(K, (W, H), 1024, kind="orb", seed=SEEDS[q], n_hyp=256, **opts)
        for i, f in enumerate(frames):
            single.push_image(f, depth, i)
        want = single.poses()
        single.close()
        assert _same(got[q], want), (name, q)
        info = got[q][1]
        assert info[1:, 1].mean() > 50, info[:, 1]                       # the panned frames do match
        assert (info[1:, 0] == 0).mean() > 0.5, info[:, 0]


def test_n_cap_below_the_extracted_count_keeps_the_prefix_and_counts_the_frames():
    import vo_b200  # noqa: F401
    from vo_b200.device_loop import DeviceLoop
    from vo_b200.orb_frontend import OrbExtractor
    opts = CONFIGS["orb_hamming_mutual_T"]
    cap = 300
    seqs = [_frames(q, n) for q, n in enumerate(LENGTHS[:2])]
    got, lost = _run_images(seqs, opts, cap, STARTS[:2], SKIPS[:2])
    orb = OrbExtractor(H, W)
    depth = np.full((H, W), DEPTH, np.float32)
    for q, frames in enumerate(seqs):
        single = DeviceLoop(K, (W, H), cap, kind="orb", seed=SEEDS[q], n_hyp=256, **opts)
        n_over = 0
        for i, f in enumerate(frames):
            kp, desc, _ = orb.extract(f)
            n_over += len(kp) > cap
            single.push(kp[:cap].clone(), desc[:cap].clone(), depth, i)
        want = single.poses()
        single.close()
        assert n_over == len(frames)
        assert _same(got[q], want), q
        assert lost[q] == n_over, (q, lost[q], n_over)
    orb.close()


def test_graph_replay_gives_the_same_poses(monkeypatch):
    import torch
    import vo_b200  # noqa: F401
    from vo_b200 import ops
    opts = CONFIGS["orb_hamming_mutual_T"]
    seqs = [_frames(q, n) for q, n in enumerate(LENGTHS)]
    ctx = ops.context()
    captures = []
    side = torch.cuda.Stream()                         # the legacy default stream cannot be captured
    with torch.cuda.stream(side):
        monkeypatch.delenv("VO_SEQ_GRAPH", raising=False)
        plain, _ = _run_images(seqs, opts, 1024, STARTS, SKIPS)
        monkeypatch.setenv("VO_SEQ_GRAPH", "1")
        graphed, _ = _run_images(seqs, opts, 1024, STARTS, SKIPS,
                                 hook=lambda t, loop: captures.append(int(ctx.lib.vo_seq_graph_captures(loop.handle))))
    assert captures[-1] >= 1, captures
    for q in range(len(seqs)):
        assert _same(graphed[q], plain[q]), q


def test_device_counts_equal_host_counts():
    """vo_seq_push_all_dev fed a hand-made device (rows, flags) array equals vo_seq_push_all with the same counts: a count
    above n_cap is clamped, a non-zero flag word changes nothing but the lost-frame counter."""
    import torch
    import vo_b200  # noqa: F401
    from vo_b200 import _lib, ops, synthetic, synthetic_sequence
    from vo_b200.device_loop import MultiDeviceLoop
    cap, n_kp, S = 1000, (900, 1000, 700), 3
    seqs = [synthetic_sequence.make_sequence(n_frames=8, n_kp=n_kp[q], kind="orb", seed=300 + q)[0] for q in range(S)]
    opts = dict(kind="orb", norm_or_metric=0, mode=1, n_hyp=256)
    host = MultiDeviceLoop(synthetic.KITTI_K, synthetic.KITTI_WH, cap, S, seeds=list(SEEDS[:S]), **opts)
    dev = MultiDeviceLoop(synthetic.KITTI_K, synthetic.KITTI_WH, cap, S, seeds=list(SEEDS[:S]), **opts)
    ctx = ops.context()
    stream = ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)
    p = lambda a: ctypes.c_void_p(a.data_ptr()) if isinstance(a, torch.Tensor) else a.ctypes.data_as(ctypes.c_void_p)  # noqa: E731
    want_lost = [0] * S
    for t in range(9):
        # sequence 0: steps 0-7; sequence 1 starts one step late; sequence 2 skips step 3
        rows = [t if t < 8 else None, t - 1 if t >= 1 else None, t if t < 3 else (None if t == 3 else t - 1)]
        kp = np.zeros((S, cap, 2), np.float32)
        desc = np.zeros((S, cap, 32), np.uint8)
        depth = np.zeros((S,) + seqs[0][0]["depth"].shape, np.float32)
        n = np.full(S, -1, np.int32)
        fno = np.zeros(S, np.int32)
        cnt = np.zeros((S, 2), np.int32)
        for q, i in enumerate(rows):
            if i is None:
                continue
            f = seqs[q][i]
            m = len(f["kp"])
            kp[q, :m], desc[q, :m], depth[q], n[q], fno[q] = f["kp"][:, :2], f["desc"], f["depth"], m, i
            cnt[q] = (m, 0)
        if rows[1] is not None:                       # sequence 1 (full slots): a count above n_cap every step
            cnt[1, 0] = cap + 50
            want_lost[1] += 1
        if t == 5:                                    # sequence 0: a flag word alone
            cnt[0, 1] = 1
            want_lost[0] += 1
        host.push(kp, desc, n, depth, fno)
        present = (n >= 0).astype(np.int32)
        cnt_d, kp_d, desc_d = (torch.from_numpy(a).cuda() for a in (cnt, kp, desc))
        _lib.check(ctx.lib.vo_seq_push_all_dev(dev.handle, p(desc_d), p(kp_d), p(cnt_d), p(present), p(depth), p(fno), stream),
                   "vo_seq_push_all_dev")
        torch.cuda.synchronize()
    for q in range(S):
        assert host.frames(q) == dev.frames(q) == 8
        assert _same(host.poses(q), dev.poses(q)), q
        assert dev.lost_frames(q) == want_lost[q] and host.lost_frames(q) == 0, (q, dev.lost_frames(q), want_lost[q])
    host.close()
    dev.close()


def test_push_images_does_not_synchronise():
    """A ~50 ms sleep kernel queued ahead of several warm push_images steps is still running when they return: no step
    waits for the device."""
    import torch
    import vo_b200  # noqa: F401
    from vo_b200.device_loop import MultiDeviceLoop
    S = 4
    seqs = [_frames(q, 8) for q in range(S)]
    loop = MultiDeviceLoop(K, (W, H), 1024, S, seeds=list(SEEDS[:S]), kind="orb", norm_or_metric=0, mode=1, n_hyp=256)
    depth = torch.full((S, H, W), DEPTH, dtype=torch.float32).pin_memory()
    images = [torch.from_numpy(np.stack([seqs[q][i] for q in range(S)])).pin_memory() for i in range(8)]
    for i in range(3):                                # warm-up: extractor scratch and pipeline workspaces exist
        loop.push_images(images[i], depth, i)
    torch.cuda.synchronize()
    done = torch.cuda.Event()
    torch.cuda._sleep(100_000_000)                    # ~50 ms at B200 clocks
    for i in range(3, 8):
        loop.push_images(images[i], depth, i)
    done.record()
    assert not done.query(), "a push_images step waited for the device"
    torch.cuda.synchronize()
    poses, info = loop.poses(0)
    assert len(poses) == 8
    loop.close()
