"""S SIFT sequences from camera images (MultiDeviceLoop.push_images on a float-descriptor loop: batched SIFT, then
vo_seq_push_all_dev with the keypoint counts on the device).  Each sequence's poses and info equal, bit for bit, a single
DeviceLoop(kind="sift") fed the same images through push_image; a frame with more keypoints than n_cap keeps its first
n_cap rows in OpenCV's order and is counted; graph replay gives the same poses; no step synchronises; an R2D2 loop is
refused."""
import numpy as np
import pytest

from test_gpu_multi_loop_images import DEPTH, H, K, LENGTHS, SEEDS, SKIPS, STARTS, W, _frames, _same, _schedule

pytestmark = pytest.mark.gpu

N_CAP = 4096
CONFIGS = {
    "sift_l2_ratio_F16X1_T": dict(norm_or_metric=0, mode=0, pnp_mode="throughput"),
    "sift_l2_ratio_F16X1_R": dict(norm_or_metric=0, mode=0, pnp_mode="reference"),
    "sift_l2_ratio_TF32X3_T": dict(norm_or_metric=0, mode=0, precision=0, pnp_mode="throughput"),
}


def _run_images(seqs, opts, n_cap, starts, skips, hook=None):
    """MultiDeviceLoop.push_images over the schedule; an absent sequence's slot holds a noise image (extracted, ignored)."""
    import torch
    from vo_b200.device_loop import MultiDeviceLoop
    S = len(seqs)
    loop = MultiDeviceLoop(K, (W, H), n_cap, S, seeds=list(SEEDS[:S]), kind="sift", n_hyp=256, **opts)
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


@pytest.mark.parametrize("name", list(CONFIGS))
def test_each_sequence_equals_a_single_sift_loop_from_images(name):
    import vo_b200  # noqa: F401
    from vo_b200.device_loop import DeviceLoop
    opts = CONFIGS[name]
    seqs = [_frames(q, n) for q, n in enumerate(LENGTHS)]
    got, lost = _run_images(seqs, opts, N_CAP, STARTS, SKIPS)
    assert lost == [0] * len(seqs)
    depth = np.full((H, W), DEPTH, np.float32)
    for q, frames in enumerate(seqs):
        single = DeviceLoop(K, (W, H), N_CAP, kind="sift", seed=SEEDS[q], n_hyp=256, **opts)
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
    from vo_b200.sift_frontend import SiftExtractor
    opts = CONFIGS["sift_l2_ratio_F16X1_T"]
    cap = 300
    seqs = [_frames(q, n) for q, n in enumerate(LENGTHS[:2])]
    got, lost = _run_images(seqs, opts, cap, STARTS[:2], SKIPS[:2])
    sift = SiftExtractor(H, W, max_keypoints=32768)
    depth = np.full((H, W), DEPTH, np.float32)
    for q, frames in enumerate(seqs):
        single = DeviceLoop(K, (W, H), cap, kind="sift", seed=SEEDS[q], n_hyp=256, **opts)
        n_over = 0
        for i, f in enumerate(frames):
            kp, desc, _ = sift.extract(f)
            n_over += len(kp) > cap
            single.push(kp[:cap].clone(), desc[:cap].clone(), depth, i)
        want = single.poses()
        single.close()
        assert n_over == len(frames)
        assert _same(got[q], want), q
        assert lost[q] == n_over, (q, lost[q], n_over)
    sift.close()


def test_graph_replay_gives_the_same_poses(monkeypatch):
    import torch
    import vo_b200  # noqa: F401
    from vo_b200 import ops
    opts = CONFIGS["sift_l2_ratio_F16X1_T"]
    seqs = [_frames(q, n) for q, n in enumerate(LENGTHS)]
    ctx = ops.context()
    captures = []
    side = torch.cuda.Stream()                         # the legacy default stream cannot be captured
    with torch.cuda.stream(side):
        monkeypatch.delenv("VO_SEQ_GRAPH", raising=False)
        plain, _ = _run_images(seqs, opts, N_CAP, STARTS, SKIPS)
        monkeypatch.setenv("VO_SEQ_GRAPH", "1")
        graphed, _ = _run_images(seqs, opts, N_CAP, STARTS, SKIPS,
                                 hook=lambda t, loop: captures.append(int(ctx.lib.vo_seq_graph_captures(loop.handle))))
    assert captures[-1] >= 1, captures
    for q in range(len(seqs)):
        assert _same(graphed[q], plain[q]), q


def test_push_images_does_not_synchronise():
    """A ~50 ms sleep kernel queued ahead of several warm push_images steps of a SIFT loop is still running when they
    return: no step waits for the device."""
    import torch
    import vo_b200  # noqa: F401
    from vo_b200.device_loop import MultiDeviceLoop
    S = 4
    seqs = [_frames(q, 8) for q in range(S)]
    loop = MultiDeviceLoop(K, (W, H), N_CAP, S, seeds=list(SEEDS[:S]), kind="sift", n_hyp=256)
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


def test_r2d2_loop_is_refused_and_enqueues_nothing():
    import torch
    import vo_b200  # noqa: F401
    from vo_b200 import ops
    from vo_b200.device_loop import MultiDeviceLoop
    S = 2
    loop = MultiDeviceLoop(K, (W, H), 1024, S, kind="r2d2", kp_stride=3, n_hyp=256)
    images = torch.zeros((S, H, W, 3), dtype=torch.uint8, device="cuda")
    depth = torch.full((S, H, W), DEPTH, dtype=torch.float32, device="cuda")
    torch.cuda.synchronize()
    l0 = ops.launch_count()
    with pytest.raises(ValueError):
        loop.push_images(images, depth, 0)
    torch.cuda.synchronize()
    assert ops.launch_count() == l0 and loop.frames(0) == 0
    loop.close()
