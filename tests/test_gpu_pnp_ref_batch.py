"""Mode R over B frame pairs (vo_pnp_ransac_ref_batch, vo_bootstrap, vo_pipeline / vo_seq with pnp_mode = reference).

The batched entry launches the kernels of the single-pair one (vo_pnp_ransac_ref) with a pair index, so every output of a
pair must equal a single-pair call on that pair's rows bit for bit, wherever the pair sits in the batch; bad input is
confined to its pair; the device bootstrap equals its numpy restatement; the pipeline, the resident runner and the device
loop compose those calls without changing a bit."""
import os

import numpy as np
import pytest

from test_oracle_bootstrap import bootstrap_ref

pytestmark = pytest.mark.gpu

CAP = 2048
BIG = 1 << 30          # bootstrap padding: an index that would fault if anything read past n


def _gpu(a):
    import torch
    return torch.from_numpy(np.ascontiguousarray(a)).cuda()


def _bits(a):
    a = np.ascontiguousarray(a)
    return a.view(np.uint64) if a.dtype == np.float64 else a


def _scenes():
    """(n, X, uv) of a ragged batch: tiny counts, ordinary scenes, a coplanar wall and an all-outlier set."""
    from test_oracle_pnp_ref import _scene
    out = []
    for k, n in enumerate((0, 3, 4, 5, 6, 60, 300, 900, 1500, 2000)):
        X, uv, _ = _scene(100 + k, n, 0.3)
        out.append((n, X, uv))
    X, uv, _ = _scene(120, 800, 0.2, planar=True)
    out.append((800, X, uv))
    X, uv, _ = _scene(121, 40, 1.0)
    out.append((40, X, uv))
    return out


def _pack(scenes, restarts, seed):
    """Padded batch arrays: NaN past n in xyz / uv, a huge index past n in the bootstrap rows (numpy-drawn, like the drop-in)."""
    rng = np.random.RandomState(seed)
    B = len(scenes)
    xyz = np.full((B, CAP, 3), np.nan, np.float32)
    uv = np.full((B, CAP, 2), np.nan, np.float32)
    boot = np.full((B, restarts, CAP), BIG, np.int32)
    n_pts = np.zeros(B, np.int32)
    for b, (n, X, u) in enumerate(scenes):
        xyz[b, :n], uv[b, :n], n_pts[b] = X, u, n
        for r in range(restarts):
            boot[b, r, :n] = rng.randint(0, n, n) if n else []
    return xyz, uv, boot, n_pts


def _batch(xyz, uv, boot, n_pts, iters):
    import torch
    from vo_b200 import synthetic, ops
    res = ops.pnp_ransac_ref_batch(_gpu(xyz), _gpu(uv), _gpu(n_pts), synthetic.KITTI_K, _gpu(boot), iters=iters, want_hyp=True)
    torch.cuda.synchronize()
    return {k: getattr(res, k).cpu().numpy() for k in ("rt", "rvec_tvec", "T_rel", "n_inl", "best", "mask", "hyp_counts",
                                                      "hyp_poses", "status")}


def _single(xyz, uv, boot, n, iters):
    import torch
    from vo_b200 import synthetic, ops
    res = ops.pnp_ransac_ref(_gpu(xyz[:n]), _gpu(uv[:n]), n, synthetic.KITTI_K, _gpu(boot[:, :n]), iters=iters, want_hyp=True)
    torch.cuda.synchronize()
    return {k: getattr(res, k).cpu().numpy() for k in ("rt", "rvec_tvec", "T_rel", "n_inl", "best", "mask", "hyp_counts",
                                                      "hyp_poses", "status")}


def _pair_equal(got, b, want, n, what=""):
    for k in ("rt", "rvec_tvec", "T_rel", "hyp_counts", "hyp_poses", "best"):
        assert np.array_equal(_bits(got[k][b]), _bits(want[k].reshape(got[k][b].shape))), (what, b, k)
    assert int(got["n_inl"][b]) == int(want["n_inl"][0]) and int(got["status"][b]) == int(want["status"][0]), (what, b)
    assert np.array_equal(got["mask"][b, :n], want["mask"][:n]), (what, b)


def _no_model(got, b, restarts, iters, bad=False):
    from vo_b200 import _lib
    assert int(got["status"][b]) == _lib.VO_ST_NO_MODEL | (_lib.VO_ST_BAD_INPUT if bad else 0), (b, got["status"][b])
    assert np.array_equal(got["T_rel"][b], np.eye(4)) and int(got["n_inl"][b]) == 0
    assert got["best"][b].tolist() == [-1, -1, 0]
    assert np.all(got["hyp_counts"][b] == -1) and not np.any(got["hyp_poses"][b])


@pytest.mark.parametrize("restarts,iters", [(1, 1), (1, 100), (3, 1), (3, 100), (3, 1024), (8, 100), (8, 1024), (1, 1024),
                                            (8, 1)])
def test_batch_equals_single_pair_calls(restarts, iters):
    scenes = _scenes()
    xyz, uv, boot, n_pts = _pack(scenes, restarts, 8214 + restarts * 7 + iters)
    got = _batch(xyz, uv, boot, n_pts, iters)
    for b, (n, _, _) in enumerate(scenes):
        if n == 0:                 # the single-pair entry needs a non-empty resample; the batched one gives "no model"
            _no_model(got, b, restarts, iters)
            continue
        want = _single(xyz[b], uv[b], boot[b], n, iters)
        _pair_equal(got, b, want, n, (restarts, iters))
        if n < 5:
            _no_model(got, b, restarts, iters)
    if restarts == 3 and iters == 100:            # the ordinary scenes do find their model
        ok = [b for b, (n, _, _) in enumerate(scenes) if n >= 60 and b != len(scenes) - 1]
        assert np.all(got["status"][ok] == 0) and np.all(got["n_inl"][ok] > 20)
        assert got["status"][-1] != 0              # all outliers


def test_outputs_do_not_depend_on_batch_position_or_neighbours():
    scenes = _scenes()
    xyz, uv, boot, n_pts = _pack(scenes, 3, 99)
    base = _batch(xyz, uv, boot, n_pts, 100)
    B = len(scenes)
    k = 7                                          # n = 900
    for order in (np.r_[k, np.delete(np.arange(B), k)], np.r_[np.arange(B)[::-1][np.arange(B)[::-1] != k], k],
                  np.array([3, k, 11, 2]), np.array([k])):
        got = _batch(xyz[order], uv[order], boot[order], n_pts[order], 100)
        pos = int(np.flatnonzero(order == k)[0])
        for key in base:
            assert np.array_equal(_bits(got[key][pos]), _bits(base[key][k])), (order.tolist(), key)


def test_bad_input_is_confined_to_its_pair():
    from vo_b200 import _lib
    scenes = _scenes()
    xyz, uv, boot, n_pts = _pack(scenes, 3, 4242)
    base = _batch(xyz, uv, boot, n_pts, 100)
    boot2, n2 = boot.copy(), n_pts.copy()
    boot2[6, 1, 17] = -1                           # n = 300: a negative index
    boot2[8, 2, 1499] = 1500                       # n = 1500: the last entry one past the end
    n2[9] = CAP + 1                                # n_pts > cap
    got = _batch(xyz, uv, boot2, n2, 100)
    for b in range(len(scenes)):
        if b in (6, 8, 9):
            _no_model(got, b, 3, 100, bad=True)
            assert not got["mask"][b].any()
        else:
            for key in base:
                assert np.array_equal(_bits(got[key][b]), _bits(base[key][b])), (b, key)
    assert int(base["status"][6]) == 0 and int(base["status"][8]) == 0
    # the single-pair entry checks its rows the same way
    bad = _single(xyz[6], uv[6], boot2[6], 300, 100)
    assert int(bad["status"][0]) == _lib.VO_ST_NO_MODEL | _lib.VO_ST_BAD_INPUT and np.array_equal(bad["T_rel"], np.eye(4))


def test_device_bootstrap_equals_restatement():
    import torch
    from vo_b200 import ops
    n = np.array([0, 1, 5, 37, 1000, CAP, 2047, 64, -3], np.int32)
    for restarts, seed, pair0 in ((3, 8214, 0), (8, 12345, 777), (1, 2 ** 63 + 5, -4)):
        got = ops.bootstrap(_gpu(n), restarts, CAP, seed=seed, pair0=pair0)
        torch.cuda.synchronize()
        got = got.cpu().numpy()
        for b in range(len(n)):
            assert np.array_equal(got[b], bootstrap_ref(int(n[b]), restarts, seed=seed, pair=pair0 + b, cap=CAP)), (seed, b)


def _mc(kind):
    from vo_b200 import ops
    if kind == "orb":
        return dict(norm_or_metric=ops.VO_NORM_HAMMING, mode=ops.VO_MODE_MUTUAL, match_param=0.0, precision=0)
    return dict(norm_or_metric=ops.VO_METRIC_COSINE, mode=ops.VO_MODE_RATIO_MUTUAL, match_param=0.90,
                precision=ops.VO_PREC_TF32X3)


@pytest.mark.parametrize("kind", ["orb", "r2d2"])
def test_pipeline_is_the_composition_of_its_calls(kind):
    import torch
    from vo_b200 import ops, sequence, synthetic
    B, N, P0 = 9, 1500, 300
    batch = synthetic.make_batch(40, B, n_kp=N, kind=kind)
    mc = _mc(kind)
    g = {k: _gpu(batch[k]) for k in ("ref_desc", "cur_desc", "ref_kp", "cur_kp", "depth")}
    res = ops.pipeline(g["ref_desc"], g["cur_desc"], g["ref_kp"], g["cur_kp"], g["depth"], batch["K"], seed=8214, pair0=P0,
                       n_hyp=0, pnp_mode="reference", **mc)
    if kind == "orb":
        m = ops.match_u8(g["ref_desc"], g["cur_desc"], mc["norm_or_metric"], mc["mode"], mc["match_param"])
    else:
        m = ops.match_f32(g["ref_desc"], g["cur_desc"], mc["norm_or_metric"], mc["mode"], mc["match_param"], mc["precision"])
    c = ops.gather_backproject(m.pairs, m.count, g["ref_kp"], g["cur_kp"], g["depth"], batch["K"])
    boot = ops.bootstrap(c.count, 3, c.xyz.shape[1], seed=8214, pair0=P0)
    r = ops.pnp_ransac_ref_batch(c.xyz, c.cur_uv, c.count, batch["K"], boot, iters=100, refine_iters=10)
    torch.cuda.synchronize()
    assert np.array_equal(res.n_matches.cpu().numpy(), m.count.cpu().numpy())
    assert np.array_equal(res.n_corr.cpu().numpy(), c.count.cpu().numpy())
    assert np.array_equal(res.n_inl.cpu().numpy(), r.n_inl.cpu().numpy())
    assert np.array_equal(res.status.cpu().numpy(), c.status.cpu().numpy() | r.status.cpu().numpy())
    assert np.array_equal(_bits(res.T_rel.cpu().numpy()), _bits(r.T_rel.cpu().numpy()))
    assert np.array_equal(_bits(res.rt.cpu().numpy()), _bits(r.rt.cpu().numpy()))
    T = res.T_rel.cpu().numpy()
    ok = res.status.cpu().numpy() == 0
    assert ok.sum() >= B - 1
    for b in np.flatnonzero(ok):
        ang, dt = synthetic.pose_errors(T[b], batch["T_rel"][b])
        assert ang < 5e-3 and dt < 5e-2, (b, ang, dt)
    # the resident runner: chunking and stream lanes never show in the result (the bootstrap is keyed by the pair)
    pb = sequence.PairBatch.from_numpy(batch)
    cfg = sequence.PipelineConfig(pnp_mode="reference", **mc)
    want = None
    for chunk, lanes in ((B, 1), (-(-B // 3), 1), (B, 2), (-(-B // 3), 2)):
        out = sequence.run_resident(pb, cfg, pair0=P0, chunk=chunk, lanes=lanes)
        torch.cuda.synchronize()
        got = (_bits(out.T_rel.cpu().numpy()), out.n_inl.cpu().numpy(), out.status.cpu().numpy())
        if want is None:
            want = got
            assert np.array_equal(got[0], _bits(T)) and np.array_equal(got[2], res.status.cpu().numpy())
        for a, b_ in zip(want, got):
            assert np.array_equal(a, b_), (chunk, lanes)


def test_batched_mode_r_matches_the_dropin_estimator_in_distribution():
    """Mode R through vo_pipeline (device bootstrap) against the drop-in path (numpy bootstrap rows, single-pair calls) on the
    same correspondences of synthetic pairs with known motion.  The two bootstrap streams differ, so poses differ pair by
    pair; their error distributions must not.  Measured on a B200: median rotation-error ratio (batched / drop-in) 1.02,
    translation 0.80 (40 ORB pairs; medians 5.2e-5 / 5.1e-5 rad, 0.76 / 0.96 mm)."""
    import torch
    from vo_b200 import ops, synthetic
    B, N = 40, 1500
    batch = synthetic.make_batch(900, B, n_kp=N, kind="orb")
    mc = _mc("orb")
    g = {k: _gpu(batch[k]) for k in ("ref_desc", "cur_desc", "ref_kp", "cur_kp", "depth")}
    res = ops.pipeline(g["ref_desc"], g["cur_desc"], g["ref_kp"], g["cur_kp"], g["depth"], batch["K"], seed=8214, pair0=0,
                       pnp_mode="reference", refine_iters=20, **mc)
    m = ops.match_u8(g["ref_desc"], g["cur_desc"], mc["norm_or_metric"], mc["mode"], mc["match_param"])
    c = ops.gather_backproject(m.pairs, m.count, g["ref_kp"], g["cur_kp"], g["depth"], batch["K"])
    torch.cuda.synchronize()
    T_b = res.T_rel.cpu().numpy()
    counts = c.count.cpu().numpy()
    rng = np.random.RandomState(8214)
    err_b, err_d = [], []
    for b in range(B):
        n = int(counts[b])
        boot = np.stack([rng.randint(0, n, n) for _ in range(3)]).astype(np.int32)
        r = ops.pnp_ransac_ref(c.xyz[b], c.cur_uv[b], n, batch["K"], _gpu(boot))
        assert int(r.status.item()) == 0 and int(res.status[b].item()) == 0
        err_b.append(synthetic.pose_errors(T_b[b], batch["T_rel"][b]))
        err_d.append(synthetic.pose_errors(r.T_rel.cpu().numpy(), batch["T_rel"][b]))
    err_b, err_d = np.array(err_b), np.array(err_d)
    ratio = np.median(err_b, 0) / np.median(err_d, 0)
    print("median error ratio (rotation, translation):", ratio.tolist(), "medians", np.median(err_b, 0), np.median(err_d, 0))
    assert np.all(ratio > 0.5) and np.all(ratio < 2.0), ratio
    assert np.all(err_b.max(0) < 10 * err_d.max(0) + 1e-3)


def test_device_loop_reference_mode_equals_per_frame_replay():
    import torch
    from vo_b200 import ops, synthetic, synthetic_sequence
    from vo_b200.device_loop import DeviceLoop
    frames, gt = synthetic_sequence.make_sequence(n_frames=16, n_kp=1500, kind="orb", seed=91)
    cap = 1500
    runs = []
    for graph in (None, "1"):
        old = os.environ.pop("VO_SEQ_GRAPH", None)
        if graph:
            os.environ["VO_SEQ_GRAPH"] = graph
        try:
            loop = DeviceLoop(synthetic.KITTI_K, synthetic.KITTI_WH, cap, kind="orb", norm_or_metric=0, mode=1, n_hyp=0,
                              pnp_mode="reference")
            for i, f in enumerate(frames):
                loop.push(f["kp"], f["desc"], f["depth"], i)
            runs.append(loop.poses())
            loop.close()
        finally:
            os.environ.pop("VO_SEQ_GRAPH", None)
            if old is not None:
                os.environ["VO_SEQ_GRAPH"] = old
    (got, info), (got_g, info_g) = runs
    assert np.array_equal(_bits(got), _bits(got_g)) and np.array_equal(info, info_g)      # VO_SEQ_GRAPH changes nothing

    def pad(a, n):
        out = np.zeros((1, cap) + a.shape[1:], a.dtype)
        out[0, :n] = a
        return _gpu(out)
    for i in range(1, len(frames)):
        key = int(info[i, 4])
        fk, fc = frames[key], frames[i]
        nk, nc = len(fk["kp"]), len(fc["kp"])
        res = ops.pipeline(pad(fk["desc"], nk), pad(fc["desc"], nc), pad(fk["kp"].astype(np.float32), nk),
                           pad(fc["kp"].astype(np.float32), nc), _gpu(fk["depth"][None].astype(np.float32)), synthetic.KITTI_K,
                           norm_or_metric=0, mode=1, match_param=0.85, n_ref=_gpu(np.array([nk], np.int32)),
                           n_cur=_gpu(np.array([nc], np.int32)), n_hyp=0, seed=8214, pair0=i - 1, pnp_mode="reference")
        torch.cuda.synchronize()
        st = int(res.status.item())
        assert info[i, :4].tolist() == [st, int(res.n_matches.item()), int(res.n_corr.item()), int(res.n_inl.item())], i
        T_rel = res.T_rel[0].cpu().numpy()
        ok = st == 0 and np.linalg.norm(T_rel[:3, 3]) <= 1.5 * (i - key)
        want = got[key] @ T_rel if ok else got[key]
        assert np.abs(got[i] - want).max() < 1e-9, i
    assert len(set(info[:, 4].tolist())) > 1 and np.all(info[1:, 0] == 0)
    assert np.linalg.norm(got[:, :3, 3] - gt[:, :3, 3], axis=1).max() < 0.15
