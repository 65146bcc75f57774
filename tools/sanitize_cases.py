"""Every kernel family of libvo_b200.so at small shapes, the case list that tests/test_gpu_small_shapes.py runs:
all matcher precisions x acceptance rules (float and byte), raw k-NN output, ragged counts, the whole pipeline with
pruned / sorted / unpruned scoring, dense back-projection, the device-resident keyframe loop, the ORB / SIFT front-ends.
Usage: python tools/sanitize_cases.py [group ...]   groups: match_f32 match_u8 pipeline geometry seq orb sift conv"""
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import torch  # noqa: E402
import vo_b200  # noqa: E402,F401
from vo_b200 import ops, synthetic  # noqa: E402

g = lambda a: torch.from_numpy(np.ascontiguousarray(a)).cuda()  # noqa: E731


def match_f32():
    for kind, metric in (("sift", ops.VO_METRIC_L2), ("r2d2", ops.VO_METRIC_COSINE)):
        b = synthetic.make_batch(0, 2, n_kp=300, kind=kind, n_cur=333)
        ref, cur = g(b["ref_desc"]), g(b["cur_desc"])
        n_ref = torch.tensor([300, 257], dtype=torch.int32, device="cuda")
        n_cur = torch.tensor([333, 129], dtype=torch.int32, device="cuda")
        for prec in (ops.VO_PREC_TF32X3, ops.VO_PREC_TF32X1, ops.VO_PREC_F16X1, ops.VO_PREC_F16X3, ops.VO_PREC_FP32_SIMT):
            for mode, param in ((ops.VO_MODE_RATIO, 0.85), (ops.VO_MODE_MUTUAL, 0.0), (ops.VO_MODE_RATIO_MUTUAL, 0.9),
                                (ops.VO_MODE_THRESH_MUTUAL, 0.9), (ops.VO_MODE_THRESH, 0.9), (ops.VO_MODE_NN, 0.0)):
                if metric == ops.VO_METRIC_L2 and mode in (ops.VO_MODE_THRESH_MUTUAL, ops.VO_MODE_THRESH):
                    continue                       # similarity thresholds are defined on cosine similarities only
                for ragged in (False, True):
                    r = ops.match_f32(ref, cur, metric, mode, param, precision=prec, n_ref=n_ref if ragged else None,
                                      n_cur=n_cur if ragged else None, want_knn=(mode == ops.VO_MODE_MUTUAL))
                    torch.cuda.synchronize()
                    assert int(r.count.sum()) >= 0
    print("match_f32 ok")


def match_u8():
    b = synthetic.make_batch(0, 2, n_kp=300, kind="orb", n_cur=333)
    ref, cur = g(b["ref_desc"]), g(b["cur_desc"])
    n_ref = torch.tensor([300, 131], dtype=torch.int32, device="cuda")
    n_cur = torch.tensor([333, 200], dtype=torch.int32, device="cuda")
    for norm in (ops.VO_NORM_HAMMING, ops.VO_NORM_HAMMING_TC, ops.VO_NORM_L2_U8):
        for mode, param in ((ops.VO_MODE_RATIO, 0.85), (ops.VO_MODE_MUTUAL, 0.0), (ops.VO_MODE_NN, 0.0)):
            for ragged in (False, True):
                for knn in (False, True, "rows"):
                    ops.match_u8(ref, cur, norm, mode, param, n_ref=n_ref if ragged else None, n_cur=n_cur if ragged else None,
                                 want_knn=knn)
                    torch.cuda.synchronize()
    print("match_u8 ok")


def pipeline():
    for kind, nm, mode, param, prec, n_kp, n_hyp in (
            ("orb", ops.VO_NORM_HAMMING, ops.VO_MODE_MUTUAL, 0.0, 0, 300, 128),
            ("orb", ops.VO_NORM_L2_U8, ops.VO_MODE_RATIO, 0.85, 0, 300, 128),
            ("sift", ops.VO_METRIC_L2, ops.VO_MODE_RATIO, 0.85, ops.VO_PREC_F16X1, 300, 128),
            ("r2d2", ops.VO_METRIC_COSINE, ops.VO_MODE_RATIO_MUTUAL, 0.90, ops.VO_PREC_TF32X3, 300, 128),
            ("sift", ops.VO_METRIC_L2, ops.VO_MODE_RATIO, 0.85, ops.VO_PREC_F16X1, 9000, 256)):   # > 6 tiles: sorted scoring
        b = synthetic.make_batch(0, 2, n_kp=n_kp, kind=kind)
        res = ops.pipeline(g(b["ref_desc"]), g(b["cur_desc"]), g(b["ref_kp"]), g(b["cur_kp"]), g(b["depth"]), b["K"],
                           norm_or_metric=nm, mode=mode, match_param=param, precision=prec, n_hyp=n_hyp, seed=8214, pair0=0)
        torch.cuda.synchronize()
        assert int(res.n_inl.min()) > 20, (kind, res.n_inl)
    # stand-alone RANSAC with per-hypothesis counts (unpruned path)
    b = synthetic.make_batch(0, 2, n_kp=300, kind="orb")
    m = ops.match_u8(g(b["ref_desc"]), g(b["cur_desc"]))
    c = ops.gather_backproject(m.pairs, m.count, g(b["ref_kp"]), g(b["cur_kp"]), g(b["depth"]), b["K"])
    hyp = ops.hypotheses(c.count, 96)
    ops.pnp_ransac(c.xyz, c.cur_uv, c.count, b["K"], hyp, want_counts=True)
    torch.cuda.synchronize()
    print("pipeline ok")


def geometry():
    b = synthetic.make_batch(0, 2, n_kp=300, kind="orb")
    ops.backproject_dense(g(b["depth"]), b["K"])
    ops.sample_depth(g(b["ref_kp"]), g(b["depth"]))
    torch.cuda.synchronize()
    print("geometry ok")


def seq():
    from vo_b200 import synthetic_sequence
    from vo_b200.device_loop import DeviceLoop
    for kind in ("orb", "sift"):
        frames, _ = synthetic_sequence.make_sequence(n_frames=4, n_kp=400, kind=kind, seed=91)
        loop = DeviceLoop(synthetic.KITTI_K, synthetic.KITTI_WH, 512, kind=kind, n_hyp=64)
        for i, f in enumerate(frames):
            loop.push(f["kp"], f["desc"], f["depth"], i)
        loop.poses()
        loop.close()
    print("seq ok")


def orb():
    from vo_b200.orb_frontend import OrbExtractor
    rng = np.random.default_rng(1)
    img = rng.integers(0, 256, (150, 260), dtype=np.uint8)
    o = OrbExtractor(*img.shape)
    kp, _, _ = o.extract(img)
    torch.cuda.synchronize()
    o.close()
    print("orb ok", len(kp))


def sift():
    from vo_b200.sift_frontend import SiftExtractor
    rng = np.random.default_rng(1)
    img = np.kron(rng.integers(0, 256, (20, 32), dtype=np.uint8), np.ones((6, 6), np.uint8))
    s = SiftExtractor(*img.shape)
    kp, _, _ = s.extract(img)
    torch.cuda.synchronize()
    s.close()
    print("sift ok", len(kp))


def conv():
    x = torch.randn(40, 136, 32, device="cuda")
    w = torch.randn(64, 3, 3, 32, device="cuda")
    ops.conv2d(x, w, torch.ones(64, device="cuda"), torch.zeros(64, device="cuda"), 3, 1, True)
    torch.cuda.synchronize()
    print("conv ok")


GROUPS = {"match_f32": match_f32, "match_u8": match_u8, "pipeline": pipeline, "geometry": geometry, "seq": seq, "orb": orb,
          "sift": sift, "conv": conv}

if __name__ == "__main__":
    for name in (sys.argv[1:] or list(GROUPS)):
        GROUPS[name]()
    print("SANITIZE CASES DONE")
