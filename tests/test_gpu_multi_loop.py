"""S sequences in one device-resident keyframe loop (MultiDeviceLoop, vo_seq_push_all): each sequence's poses and info equal a
single DeviceLoop's bit for bit, whatever its neighbours do, when it starts or which steps it skips."""
import ctypes
import functools

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

# per-kind options of tests/test_gpu_device_loop.py
KINDS = {
    "orb_l2_ratio": dict(kind="orb", norm_or_metric=1, mode=0, precision=0),
    "orb_hamming_mutual": dict(kind="orb", norm_or_metric=0, mode=1, precision=0),
    "sift": dict(kind="sift", norm_or_metric=0, mode=0, precision=1),
    "r2d2": dict(kind="r2d2", norm_or_metric=1, mode=2, precision=0, match_param=0.90, kp_stride=3),
}
N_KP = (900, 1000, 700, 1000, 800)            # keypoints per frame of each sequence (ragged batch)
LENGTHS = (12, 20, 9, 15, 11)
STARTS = (0, 0, 3, 1, 5)                      # the step at which each sequence pushes its first frame
SKIPS = ({}, {4, 9}, {6}, set(), {7, 8})      # steps a sequence has no frame (after its start)
SEEDS = (8214, 77, 123456789, 5, 2 ** 40 + 3)
CAP = 1000


@functools.lru_cache(maxsize=None)
def _frames(kind, q, n_frames=None, n_kp=None):
    from vo_b200 import synthetic_sequence
    frames, _ = synthetic_sequence.make_sequence(n_frames=n_frames or LENGTHS[q], n_kp=n_kp or N_KP[q], kind=kind, seed=300 + q)
    if kind == "r2d2":          # the reference's R2D2 keypoints are (x, y, scale) float32 rows (R2D2.py:160-166)
        for f in frames:
            f["kp"] = np.concatenate([f["kp"], np.full((len(f["kp"]), 1), 32.0)], 1).astype(np.float32)
    return frames


def _schedule(seqs, starts, skips):
    """steps[t] = [(q, frame index) or None per sequence]: sequence q pushes its frames in order from step starts[q] on,
    nothing at the steps in skips[q]."""
    nxt, steps, t = [0] * len(seqs), [], 0
    while any(nxt[q] < len(seqs[q]) for q in range(len(seqs))):
        row = []
        for q in range(len(seqs)):
            if t >= starts[q] and t not in skips[q] and nxt[q] < len(seqs[q]):
                row.append(nxt[q])
                nxt[q] += 1
            else:
                row.append(None)
        steps.append(row)
        t += 1
    return steps


def _stack_step(seqs, row, opts, cap):
    S = len(seqs)
    ks = opts.get("kp_stride", 2)
    f0 = seqs[0][0]
    H, W = f0["depth"].shape
    cols, dt = f0["desc"].shape[1], f0["desc"].dtype
    kp = np.zeros((S, cap, ks), np.float32)
    desc = np.zeros((S, cap, cols), dt)
    depth = np.zeros((S, H, W), np.float32)
    n_kp = np.full(S, -1, np.int32)
    frame_no = np.zeros(S, np.int32)
    for q, i in enumerate(row):
        if i is None:
            continue
        f = seqs[q][i]
        n = len(f["kp"])
        kp[q, :n] = f["kp"][:, :ks]
        desc[q, :n] = f["desc"]
        depth[q] = f["depth"]
        n_kp[q] = n
        frame_no[q] = i
    return kp, desc, n_kp, depth, frame_no


def _run_multi(seqs, seeds, opts, starts=None, skips=None, cap=CAP, hook=None, **extra):
    from vo_b200 import synthetic
    from vo_b200.device_loop import MultiDeviceLoop
    S = len(seqs)
    loop = MultiDeviceLoop(synthetic.KITTI_K, synthetic.KITTI_WH, cap, S, seeds=list(seeds), **opts, **extra)
    steps = _schedule(seqs, starts or (0,) * S, skips or ({},) * S)
    for t, row in enumerate(steps):
        loop.push(*_stack_step(seqs, row, opts, cap))
        if hook:
            hook(t, loop)
    out = [loop.poses(q) for q in range(S)]
    assert [loop.frames(q) for q in range(S)] == [len(s) for s in seqs]
    loop.close()
    return out


def _run_single(frames, seed, opts, cap=CAP, **extra):
    from vo_b200 import synthetic
    from vo_b200.device_loop import DeviceLoop
    loop = DeviceLoop(synthetic.KITTI_K, synthetic.KITTI_WH, cap, seed=seed, **opts, **extra)
    for i, f in enumerate(frames):
        loop.push(f["kp"], f["desc"], f["depth"], i)
    out = loop.poses()
    loop.close()
    return out


def _same(a, b):
    return np.array_equal(a[0], b[0]) and np.array_equal(a[1], b[1])


@pytest.mark.parametrize("name,pnp_mode", [
    ("orb_l2_ratio", "throughput"), ("orb_hamming_mutual", "throughput"), ("sift", "throughput"), ("r2d2", "throughput"),
    ("orb_hamming_mutual", "reference"), ("r2d2", "reference"),
])
def test_each_sequence_equals_a_single_loop(name, pnp_mode):
    import vo_b200  # noqa: F401
    opts = KINDS[name]
    seqs = [_frames(opts["kind"], q) for q in range(5)]
    got = _run_multi(seqs, SEEDS, opts, STARTS, SKIPS, pnp_mode=pnp_mode)
    for q in range(5):
        want = _run_single(seqs[q], SEEDS[q], opts, pnp_mode=pnp_mode)
        assert _same(got[q], want), (name, pnp_mode, q)
        poses, info = got[q]
        assert poses.shape == (LENGTHS[q], 4, 4)
        assert info[:, 5].sum() >= 3, (q, info[:, 5])                 # the keyframe rule fired
        assert (info[1:, 0] == 0).mean() > 0.8, info[:, 0]


def test_permuting_sequences_permutes_outputs_and_s1_equals_s5():
    import vo_b200  # noqa: F401
    opts = KINDS["orb_hamming_mutual"]
    seqs = [_frames("orb", q) for q in range(5)]
    base = _run_multi(seqs, SEEDS, opts, STARTS, SKIPS)
    perm = [3, 0, 4, 2, 1]
    got = _run_multi([seqs[p] for p in perm], [SEEDS[p] for p in perm], opts, [STARTS[p] for p in perm],
                     [SKIPS[p] for p in perm])
    for i, p in enumerate(perm):
        assert _same(got[i], base[p]), (i, p)
    for q in (1, 4):
        alone = _run_multi([seqs[q]], [SEEDS[q]], opts, [STARTS[q]], [SKIPS[q]])[0]
        assert _same(alone, base[q]), q


def test_failures_stay_in_their_sequence():
    """Sequence 1 gets junk descriptors on frames 3-7 and an empty frame 11: its bad-PnP counter and forced promotion behave
    as a single loop's (test_device_loop_failures_and_bad_pnp_counter); the other sequences are bit-identical to a clean run."""
    import vo_b200  # noqa: F401
    from vo_b200 import synthetic_sequence
    opts = dict(kind="orb", norm_or_metric=0, mode=1, n_hyp=256)
    frames, _ = synthetic_sequence.make_sequence(n_frames=12, n_kp=800, kind="orb", seed=5)
    rng = np.random.default_rng(0)
    bad = [dict(f) for f in frames]
    for i in range(3, 8):
        bad[i]["desc"] = rng.integers(0, 256, (800, 32), dtype=np.uint8)      # descriptors that match nothing consistently
    bad[11]["kp"], bad[11]["desc"] = np.zeros((0, 2)), np.zeros((0, 32), np.uint8)
    others = [_frames("orb", q, 12, 800) for q in (0, 2, 3)]
    clean = _run_multi([others[0], frames] + others[1:], SEEDS[:4], opts, cap=800)
    got = _run_multi([others[0], bad] + others[1:], SEEDS[:4], opts, cap=800)
    for q in (0, 2, 3):
        assert _same(got[q], clean[q]), q
    poses, info = got[1]
    assert np.all(info[3:7, 0] != 0)                                   # bad PnP on the junk frames
    for i in (3, 4, 5):
        assert np.array_equal(poses[i], poses[info[i, 4]]) and info[i, 5] == 0
    assert info[6, 5] == 1                                             # 4th consecutive failure: promoted (:295)
    assert info[7, 4] == 6
    assert info[10, 0] == 0                                            # recovered once real descriptors return
    assert info[11, 0] != 0 and np.array_equal(poses[11], poses[info[11, 4]])   # the empty frame: bad PnP, keyframe pose
    assert _same(got[1], _run_single(bad, SEEDS[1], opts, cap=800))


def test_loud_errors_enqueue_nothing():
    import torch
    import vo_b200  # noqa: F401
    from vo_b200 import _lib, ops, synthetic
    from vo_b200.device_loop import MultiDeviceLoop
    opts = dict(kind="orb", norm_or_metric=0, mode=1, n_hyp=128)
    seqs = [_frames("orb", q, 4, 700) for q in range(3)]
    with pytest.raises(ValueError, match="seeds"):
        MultiDeviceLoop(synthetic.KITTI_K, synthetic.KITTI_WH, 700, 3, seeds=[1, 2], **opts)
    loop = MultiDeviceLoop(synthetic.KITTI_K, synthetic.KITTI_WH, 700, 3, seeds=SEEDS[:3], max_frames=3, **opts)
    rows = [[0, 0, None], [1, None, 0], [2, 1, 1]]                     # sequence 0's history is then full
    for row in rows:
        loop.push(*_stack_step(seqs, row, opts, 700))
    torch.cuda.synchronize()
    ctx = ops.context()
    before = (ctx.launch_count(), [loop.frames(q) for q in range(3)], [loop.poses(q) for q in range(3)])

    def refused(exc, *args):
        with pytest.raises(exc):
            loop.push(*args)
        torch.cuda.synchronize()
        assert ctx.launch_count() == before[0]
        assert [loop.frames(q) for q in range(3)] == before[1]

    kp, desc, n_kp, depth, fno = _stack_step(seqs, [None, 2, 2], opts, 700)
    big = n_kp.copy()
    big[2] = 701
    refused(_lib.VoError, kp, desc, big, depth, fno)                   # n_kp > n_cap
    full = n_kp.copy()
    full[0] = 700
    refused(_lib.VoError, kp, desc, full, depth, fno)                  # sequence 0's history is full
    refused(ValueError, kp[:2], desc[:2], n_kp[:2], depth[:2], fno[:2])    # S = 2 arrays for a 3-sequence loop
    refused(ValueError, kp, desc[:, :, :16], n_kp, depth, fno)
    refused(ValueError, kp, desc, n_kp, depth[:, :100], fno)
    refused(ValueError, kp, desc, n_kp[:2], depth, fno)
    # vo_seq_push addresses a one-sequence loop only
    f = seqs[0][0]
    kp0 = np.ascontiguousarray(f["kp"], np.float32)
    rc = ctx.lib.vo_seq_push(loop.handle, f["desc"].ctypes.data_as(ctypes.c_void_p), kp0.ctypes.data_as(ctypes.c_void_p),
                             len(kp0), f["depth"].ctypes.data_as(ctypes.c_void_p), 0, None)
    assert rc == _lib.VO_ERR_ARG and b"vo_seq_push_all" in ctx.lib.vo_last_error()
    torch.cuda.synchronize()
    assert ctx.launch_count() == before[0]
    for q in range(3):
        assert _same(loop.poses(q), before[2][q])
    loop.push(kp, desc, n_kp, depth, fno)                              # the step itself was fine: it still runs
    assert [loop.frames(q) for q in range(3)] == [3, 3, 3]
    loop.close()


def test_graph_recaptures_after_workspace_growth(monkeypatch):
    """VO_SEQ_GRAPH=1: the loop captures its step once the pipeline has run plainly (step 2).  After step 4 an ops call on the
    same context reallocates a workspace (the request doubles until vo_workspace_generation moves, so it grows whatever
    earlier calls left behind).  The next step must see the stale graph and capture again: two captures in all, and poses
    equal to a plain run's.  Runs on a side stream: the legacy default stream cannot be captured."""
    import torch
    import vo_b200  # noqa: F401
    from vo_b200 import ops
    opts = KINDS["orb_hamming_mutual"]
    seqs = [_frames("orb", q) for q in range(3)]
    ctx = ops.context()
    gen = lambda: int(ctx.lib.vo_workspace_generation(ctx.handle))  # noqa: E731
    captures, grown = [], []

    def grow(t, loop):
        captures.append(int(ctx.lib.vo_seq_graph_captures(loop.handle)))
        if t == 4:
            g0, m = gen(), 1 << 16
            ref = torch.zeros((1, 64, 32), dtype=torch.uint8, device="cuda")
            while gen() == g0 and m <= 1 << 27:       # column keys: 8 bytes per current-frame row
                ops.match_u8(ref, torch.zeros((1, m, 32), dtype=torch.uint8, device="cuda"))
                m *= 2
            grown.append(gen() != g0)

    side = torch.cuda.Stream()
    with torch.cuda.stream(side):
        monkeypatch.delenv("VO_SEQ_GRAPH", raising=False)
        plain = _run_multi(seqs, SEEDS[:3], opts)
        monkeypatch.setenv("VO_SEQ_GRAPH", "1")
        graphed = _run_multi(seqs, SEEDS[:3], opts, hook=grow)
    assert grown == [True]
    assert captures[:5] == [0, 0, 1, 1, 1] and captures[5:] == [2] * (len(captures) - 5), captures
    for q in range(3):
        assert _same(graphed[q], plain[q]), q
