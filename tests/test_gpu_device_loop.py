"""Device-resident keyframe loop (vo_seq_*, SURVEY 8(f) rank 2) against the drop-in VisualOdometry.process_frame,
whose host-side control flow is the reference's (VisualOdometry_Stereo.py:232-297): same keyframe decisions, same
poses, no host round trip per frame."""
import os
import sys

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "tests"))


def _run_dropin(tmp_path, kind, frames, extra=""):
    from test_gpu_dropin import _load_dropin
    from vo_b200 import synthetic
    vos = _load_dropin(tmp_path, kind, extra + "\npnp_mode: throughput\n")   # the device loop runs the throughput sampler
    feed = {}
    vos.extract_features_and_desc = lambda img: feed["cur"]
    vo = vos.VisualOdometry(synthetic.KITTI_K, seq=0)
    img = np.zeros((synthetic.KITTI_WH[1], synthetic.KITTI_WH[0], 3), np.uint8)
    poses, keys = [], []
    for i, f in enumerate(frames):
        feed["cur"] = (f["kp"], f["desc"])
        keys.append(vo.ref_data[-1].id if i else 0)
        poses.append(vo.process_frame(img, f["depth"], (100, 100), i).pose.copy())
    return np.stack(poses), np.asarray(keys), vo


@pytest.mark.parametrize("kind,extra,norm,mode,prec", [
    ("orb", "", 1, 0, 0),                                        # reference ORB semantics: byte-L2 + ratio
    ("orb", "\norb_matcher: hamming_mutual\n", 0, 1, 0),         # north-star semantics
    ("sift", "", 0, 0, 1),
    ("r2d2", "", 1, 2, 0),                                       # cosine ratio+mutual 0.90, 3xTF32, (x, y, scale) keypoints
])
def test_device_loop_equals_host_policy(tmp_path, kind, extra, norm, mode, prec):
    import vo_b200  # noqa: F401
    from vo_b200 import synthetic, synthetic_sequence
    from vo_b200.device_loop import DeviceLoop
    cwd = os.getcwd()
    try:
        frames, gt = synthetic_sequence.make_sequence(n_frames=20, n_kp=1500, kind=kind, seed=91)
        if kind == "r2d2":      # the reference's R2D2 keypoints are (x, y, scale) float32 rows (R2D2.py:160-166)
            for f in frames:
                f["kp"] = np.concatenate([f["kp"], np.full((len(f["kp"]), 1), 32.0)], 1).astype(np.float32)
        want, keys, vo = _run_dropin(tmp_path, kind, frames, extra)
        loop = DeviceLoop(synthetic.KITTI_K, synthetic.KITTI_WH, 1500, kind=kind, norm_or_metric=norm, mode=mode,
                          match_param=0.90 if kind == "r2d2" else 0.85, precision=prec, n_hyp=vo.n_hyp, seed=vo.seed,
                          kp_stride=3 if kind == "r2d2" else 2)
        for i, f in enumerate(frames):
            loop.push(f["kp"], f["desc"], f["depth"], i)        # enqueue only
        got, info = loop.poses()                                 # the one synchronisation
        assert got.shape == want.shape and len(loop) == len(frames)
        assert np.array_equal(info[:, 4], keys)                  # matched against the same keyframes
        assert len(set(keys.tolist())) > 3                       # the keyframe rule did fire
        assert np.all(info[1:, 0] == 0)
        assert np.abs(got - want).max() < 1e-9
        # and the trajectory is right in absolute terms
        assert np.linalg.norm(got[:, :3, 3] - gt[:, :3, 3], axis=1).max() < 0.15
        # the keyframe decisions against the REFERENCE's loop (oracle/reference_vo.py: pinned pose for pose to the reference's own
        # class, cv2 matcher + 3 x cv2.solvePnPRansac): the same frames become keyframes, up to one decision that sits on a
        # threshold (inliers < 100 / common points < 200 / 1.5 m) and flips with the sampler
        from oracle.reference_vo import ReferenceVO
        matcher = {"orb": "hamming_mutual" if "hamming" in extra else "knn_ratio", "sift": "knn_ratio", "r2d2": "r2d2"}[kind]
        ref = ReferenceVO(synthetic.KITTI_K, matcher=matcher)
        ref_keys, ref_poses = [], []
        for i, f in enumerate(frames):
            ref_keys.append(ref.key[0] if i else 0)
            ref_poses.append(ref.process_frame(f["kp"][:, :2] if kind == "r2d2" else f["kp"], f["desc"], f["depth"], i).copy())
        assert (np.asarray(ref_keys) != info[:, 4]).sum() <= 1, (ref_keys, info[:, 4].tolist())
        assert np.linalg.norm(got[:, :3, 3] - np.stack(ref_poses)[:, :3, 3], axis=1).max() < 0.05
    finally:
        os.chdir(cwd)


def test_device_loop_failures_and_bad_pnp_counter():
    """A frame with no usable matches is a bad PnP: pose = keyframe pose (:290); after more than 3 in a row the
    current frame is promoted anyway (:295)."""
    import vo_b200  # noqa: F401
    from vo_b200 import synthetic, synthetic_sequence
    from vo_b200.device_loop import DeviceLoop
    frames, gt = synthetic_sequence.make_sequence(n_frames=12, n_kp=800, kind="orb", seed=5)
    rng = np.random.default_rng(0)
    junk = lambda: rng.integers(0, 256, (800, 32), dtype=np.uint8)     # descriptors that match nothing consistently
    loop = DeviceLoop(synthetic.KITTI_K, synthetic.KITTI_WH, 800, kind="orb", norm_or_metric=0, mode=1, n_hyp=256)
    for i, f in enumerate(frames):
        loop.push(f["kp"], junk() if 3 <= i <= 7 else f["desc"], f["depth"], i)
    poses, info = loop.poses()
    assert np.all(info[3:7, 0] != 0)                                   # bad PnP on the junk frames
    for i in (3, 4, 5):
        assert np.array_equal(poses[i], poses[info[i, 4]]) and info[i, 5] == 0
    assert info[6, 5] == 1                                             # 4th consecutive failure: promoted (:295)
    assert info[7, 4] == 6
    assert info[10, 0] == 0                                            # recovered once real descriptors return
    # capacity and argument errors are loud
    from vo_b200 import _lib
    with pytest.raises(_lib.VoError):
        loop.push(np.zeros((900, 2)), np.zeros((900, 32), np.uint8), frames[0]["depth"], 99)


def test_device_loop_empty_frames_and_history_limit():
    import vo_b200  # noqa: F401
    from vo_b200 import _lib, synthetic, synthetic_sequence
    from vo_b200.device_loop import DeviceLoop
    frames, _ = synthetic_sequence.make_sequence(n_frames=4, n_kp=300, kind="orb", seed=2)
    loop = DeviceLoop(synthetic.KITTI_K, synthetic.KITTI_WH, 300, kind="orb", norm_or_metric=0, mode=1, n_hyp=128, max_frames=4)
    loop.push(frames[0]["kp"], frames[0]["desc"], frames[0]["depth"], 0)
    loop.push(np.zeros((0, 2)), np.zeros((0, 32), np.uint8), frames[1]["depth"], 1)      # a frame without keypoints
    loop.push(frames[2]["kp"], frames[2]["desc"], frames[2]["depth"], 2)
    loop.push(frames[3]["kp"], frames[3]["desc"], frames[3]["depth"], 3)
    poses, info = loop.poses()
    assert info[1, 0] != 0 and np.array_equal(poses[1], poses[0])       # bad PnP: pose of the keyframe (:290)
    assert info[2, 0] == 0 and info[2, 4] == 0                          # still matched against keyframe 0
    with pytest.raises(_lib.VoError):
        loop.push(frames[0]["kp"], frames[0]["desc"], frames[0]["depth"], 4)               # history full
    p2, i2 = loop.poses(first=2, count=2)
    assert np.array_equal(p2, poses[2:]) and np.array_equal(i2, info[2:])


def test_default_sift_loop_refuses_non_integer_descriptors():
    """The default SIFT pass (F16X1) is exact for integers in 0..255 only: RootSIFT frames are refused, on the host and as
    device tensors, and an explicit TF32X3 loop takes them and gives the poses of an explicit TF32X3 loop on the device
    copies."""
    import torch
    import vo_b200  # noqa: F401
    from vo_b200 import ops, synthetic, synthetic_sequence
    from vo_b200.device_loop import DeviceLoop
    frames, _ = synthetic_sequence.make_sequence(n_frames=4, n_kp=400, kind="sift", seed=5)
    root = [np.sqrt(f["desc"] / np.maximum(f["desc"].sum(1, keepdims=True), 1)).astype(np.float32) for f in frames]
    loop = DeviceLoop(synthetic.KITTI_K, synthetic.KITTI_WH, 512, kind="sift", n_hyp=128)
    loop.push(frames[0]["kp"], frames[0]["desc"], frames[0]["depth"], 0)             # integer SIFT: accepted
    with pytest.raises(ValueError, match="not integers"):
        loop.push(frames[1]["kp"], root[1], frames[1]["depth"], 1)
    loop.close()
    loop = DeviceLoop(synthetic.KITTI_K, synthetic.KITTI_WH, 512, kind="sift", n_hyp=128)
    with pytest.raises(ValueError, match="not integers"):
        loop.push(frames[0]["kp"], torch.from_numpy(root[0]).cuda(), frames[0]["depth"], 0)
    loop.close()
    out = []
    for dev in (False, True):
        loop = DeviceLoop(synthetic.KITTI_K, synthetic.KITTI_WH, 512, kind="sift", n_hyp=128, precision=ops.VO_PREC_TF32X3)
        for i, f in enumerate(frames):
            loop.push(f["kp"], torch.from_numpy(root[i]).cuda() if dev else root[i], f["depth"], i)
        out.append(loop.poses())
        loop.close()
    assert np.array_equal(out[0][0], out[1][0]) and np.array_equal(out[0][1], out[1][1])
    assert (out[0][1][1:, 0] == 0).all(), out[0][1]                                   # the RootSIFT frames do match
