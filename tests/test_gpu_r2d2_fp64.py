"""The R2D2 front-end (vo_r2d2_*) at the shapes it runs on, against torch fp64 on the GPU and against a numpy
restatement of its keypoint rule:
  * the Fast architecture with the shipped faster2d2_WASF_N16 weights on a KITTI-shaped image (376 x 1241 -> 376 x 1240
    maps): maps and descriptors within 2e-4 of fp64, keypoint sets equal except on decision boundaries;
  * odd image sizes with random weights: MaxPool2d(2) floors, the bilinear heads clamp at the last row / column, tiles
    end mid-row at both resolutions, and a 3-row image leaves a single pooled row;
  * NMS and ordering exactly: the keypoints are the pixels the rule selects on the library's own fp32 maps, in
    row-major order, with scores equal to the fp32 product rel * rep, including past 2048 rows, where the row scan
    carries its offset across 1024-row chunks;
  * a capped keypoint buffer reports the full count and holds the prefix of the uncapped output.
Measured on a B200 at 376 x 1241 with the shipped weights: max |rel - fp64| = 2.6e-5, max |rep - fp64| = 4.3e-5,
max descriptor error 1.4e-5; 2504 keypoints, none differing from the fp64 reference's set.  With random weights at
377 x 1241 the map errors are 1.1e-5 and the descriptor error 4.8e-6."""
import os
import sys

import numpy as np
import pytest

sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
from test_r2d2_frontend import _torch_net, _weights  # noqa: E402

pytestmark = pytest.mark.gpu

FAST = "Fast_Quad_L2Net_ConfCFS"
QUAD = "Quad_L2Net_ConfCFS"
KITTI = (376, 1241)


def _random_sd(name, seed):
    """random weights for either architecture (channel counts of the shipped models)"""
    from vo_b200 import r2d2_frontend as rf
    rng = np.random.default_rng(seed)
    chans = [3, 32, 32, 64, 64, 128, 128, 128, 128, 128]
    sd, idx = {}, 0
    for li, (k, dil, bn, relu, pool) in enumerate(rf.ARCH[name]["layers"]):
        cin, cout = chans[li], chans[li + 1]
        sd[f"ops.{idx}.weight"] = (rng.standard_normal((cout, cin, k, k)) / np.sqrt(cin * k * k)).astype(np.float32)
        sd[f"ops.{idx}.bias"] = (0.1 * rng.standard_normal(cout)).astype(np.float32)
        if bn:
            sd[f"ops.{idx + 1}.running_mean"] = (0.1 * rng.standard_normal(cout)).astype(np.float32)
            sd[f"ops.{idx + 1}.running_var"] = rng.uniform(0.5, 1.5, cout).astype(np.float32)
        idx += 1 + bn + relu
    sd["clf.weight"] = (rng.standard_normal((2, 128, 1, 1)) * 0.3).astype(np.float32)
    sd["clf.bias"] = rng.standard_normal(2).astype(np.float32) * 0.1
    sd["sal.weight"] = (rng.standard_normal((1, 128, 1, 1)) * 0.3).astype(np.float32)
    sd["sal.bias"] = rng.standard_normal(1).astype(np.float32) * 0.1
    return sd


def _textured(H, W, seed):
    """blocks of several sizes plus per-pixel noise: corners and texture at every scale"""
    rng = np.random.default_rng(seed)
    img = np.zeros((H, W, 3), np.float64)
    for b, a in ((16, 0.4), (6, 0.35), (2, 0.15)):
        img += a * np.kron(rng.uniform(0, 255, (H // b + 1, W // b + 1, 3)), np.ones((b, b, 1)))[:H, :W]
    img += rng.normal(0, 8, (H, W, 3))
    return np.clip(img, 0, 255).astype(np.uint8)


def _torch_fp64(name, sd, img):
    """rel, rep [Ho,Wo] and L2-normalised descriptors [C,Ho,Wo] of the reference network in fp64 on the GPU"""
    import torch
    import torch.nn.functional as F
    dev = torch.device("cuda")
    body = _torch_net(name, sd, dev)
    mean = torch.tensor([0.485, 0.456, 0.406], device=dev).view(1, 3, 1, 1)
    std = torch.tensor([0.229, 0.224, 0.225], device=dev).view(1, 3, 1, 1)
    x = ((torch.from_numpy(img).to(dev).permute(2, 0, 1)[None].float() / 255 - mean) / std).double()
    t = lambda a: torch.from_numpy(np.asarray(a)).double().to(dev)  # noqa: E731
    with torch.no_grad():
        f = body(x)
        u = F.conv2d(f ** 2, t(sd["clf.weight"]), t(sd["clf.bias"]))
        rel = F.softmax(u, dim=1)[0, 1]
        s = F.softplus(F.conv2d(f ** 2, t(sd["sal.weight"]), t(sd["sal.bias"])))
        rep = (s / (1 + s))[0, 0]
        d = F.normalize(f, p=2, dim=1)[0]
    return rel, rep, d


def _nms_np(rel, rep, rel_thr, rep_thr, score_thr):
    """is_keypoint (r2d2_net.cu) over fp32 maps: both thresholds, the fp32 product rel * rep > score_thr, and rep equal to
    the 3x3 maximum over neighbours inside the map -> (x, y, score) in row-major order"""
    rel = np.asarray(rel, np.float32)
    rep = np.asarray(rep, np.float32)
    Ho, Wo = rep.shape
    pad = np.full((Ho + 2, Wo + 2), -np.inf, np.float32)
    pad[1:-1, 1:-1] = rep
    m = rep.copy()
    for dy in range(3):
        for dx in range(3):
            m = np.maximum(m, pad[dy:dy + Ho, dx:dx + Wo])
    prod = rel * rep
    keep = (rep >= np.float32(rep_thr)) & (rel >= np.float32(rel_thr)) & (prod > np.float32(score_thr)) & (rep == m)
    ys, xs = np.nonzero(keep)
    return xs, ys, prod[keep]


def _check_nms_exact(net, out, thr):
    xys, desc, scores, rel, rep = out
    xs, ys, sc = _nms_np(rel.cpu().numpy(), rep.cpu().numpy(), *thr)
    assert int(net.count.item()) == len(xs)
    assert len(xs) <= net.max_kp
    g = xys.cpu().numpy()
    assert np.array_equal(g[:, 0], xs.astype(np.float32)) and np.array_equal(g[:, 1], ys.astype(np.float32))
    assert np.all(g[:, 2] == 32.0)
    assert np.array_equal(scores.cpu().numpy().view(np.uint32), sc.view(np.uint32))
    return xs, ys


def _near_boundary(rel_t, rep_t, x, y, thr, tol=3e-4):
    """the rule of test_r2d2_frontend: a keypoint present in one set only must sit within tol of a threshold or a tie"""
    c, q = float(rel_t[y, x]), float(rep_t[y, x])
    nb = rep_t[max(0, y - 1):y + 2, max(0, x - 1):x + 2]
    second = np.sort(nb.reshape(-1))[-2] if nb.size > 1 else -1
    return (abs(c - thr[0]) < tol or abs(q - thr[1]) < tol or abs(c * q - thr[2]) < tol
            or abs(q - nb.max()) < tol and abs(q - second) < tol)


@pytest.fixture(scope="module")
def production(golden):
    """the Fast net with the shipped weights at 376 x 1241, capacity for every pixel"""
    from vo_b200 import r2d2_frontend as rf
    name, sd = _weights(golden("r2d2_net.npz"))
    img = _textured(*KITTI, seed=21)
    net = rf.R2D2Net(name, sd, *KITTI, max_kp=KITTI[0] * (KITTI[1] - 1))
    assert (net.Ho, net.Wo) == (376, 1240)
    return name, sd, img, net


def _maps_and_desc_vs_fp64(name, sd, img, out):
    import torch
    xys, desc, scores, rel, rep = out
    rel_t, rep_t, d_t = _torch_fp64(name, sd, img)
    assert rel.shape == rel_t.shape and rep.shape == rep_t.shape
    e_rel = float((rel.double() - rel_t).abs().max())
    e_rep = float((rep.double() - rep_t).abs().max())
    xi, yi = xys[:, 0].long(), xys[:, 1].long()
    e_desc = float((desc.double() - d_t[:, yi, xi].t()).abs().max()) if len(xys) else 0.0
    assert e_rel < 2e-4 and e_rep < 2e-4, (e_rel, e_rep)
    assert e_desc < 2e-4, e_desc
    if len(xys):
        assert float((desc.double().norm(dim=1) - 1).abs().max()) < 1e-5
    assert bool(torch.isfinite(rel).all()) and bool(torch.isfinite(rep).all())
    return rel_t.cpu().numpy(), rep_t.cpu().numpy()


def test_production_shape_against_torch_fp64(production):
    name, sd, img, net = production
    thr = (0.7, 0.7, 0.85)
    out = net.extract(img, *thr, want_maps=True)
    rel_t, rep_t = _maps_and_desc_vs_fp64(name, sd, img, out)
    xys = out[0].cpu().numpy()
    got = {(int(x), int(y)) for x, y in xys[:, :2]}
    # the fp64 reference's own set, decided in fp64
    keep = (rep_t >= thr[1]) & (rel_t >= thr[0]) & (rel_t * rep_t > thr[2])
    pad = np.full((rep_t.shape[0] + 2, rep_t.shape[1] + 2), -np.inf)
    pad[1:-1, 1:-1] = rep_t
    mx = np.max(np.stack([pad[dy:dy + rep_t.shape[0], dx:dx + rep_t.shape[1]] for dy in range(3) for dx in range(3)]), 0)
    ys, xs = np.nonzero(keep & (rep_t == mx))
    want = {(int(x), int(y)) for x, y in zip(xs, ys)}
    assert len(got) > 100
    diff = got ^ want
    for (x, y) in diff:
        assert _near_boundary(rel_t, rep_t, x, y, thr), (x, y, rel_t[y, x], rep_t[y, x])
    assert len(diff) <= max(2, len(want) // 200)


@pytest.mark.parametrize("thr", [(0.0, 0.0, -1.0), (0.7, 0.7, 0.85)], ids=["thresholds_off", "defaults"])
def test_production_shape_nms_is_exact_on_the_returned_maps(production, thr):
    name, sd, img, net = production
    xs, ys = _check_nms_exact(net, net.extract(img, *thr, want_maps=True), thr)
    assert len(xs) > 100
    assert xs.max() >= 1024 and ys.max() >= 300          # keypoints in the last 256-pixel chunk of a row


def test_production_shape_capacity_keeps_the_prefix(production):
    import torch
    from vo_b200 import r2d2_frontend as rf
    name, sd, img, net = production
    thr = (0.5, 0.5, 0.3)
    xa, da, sa = (t.clone() for t in net.extract(img, *thr))
    n = len(xa)
    assert n > 1000 and int(net.count.item()) == n
    small = rf.R2D2Net(name, sd, *KITTI, max_kp=n // 3)
    xb, db, sb = small.extract(img, *thr)
    assert len(xb) == n // 3 and int(small.count.item()) == n
    assert torch.equal(xb, xa[:n // 3]) and torch.equal(db, da[:n // 3]) and torch.equal(sb, sa[:n // 3])


@pytest.mark.parametrize("H,W", [(377, 1241), (101, 259), (97, 163), (3, 40)])
def test_fast_architecture_odd_shapes_against_torch_fp64(H, W):
    from vo_b200 import r2d2_frontend as rf
    sd = _random_sd(FAST, seed=H + W)
    img = _textured(H, W, seed=H * W)
    net = rf.R2D2Net(FAST, sd, H, W, max_kp=max(64, (H // 2 * 2) * (W // 2 * 2)))
    assert (net.Ho, net.Wo) == (H // 2 * 2, W // 2 * 2)
    thr = (0.0, 0.0, -1.0)
    out = net.extract(img, *thr, want_maps=True)
    _maps_and_desc_vs_fp64(FAST, sd, img, out)
    xs, _ = _check_nms_exact(net, out, thr)
    assert len(xs) > 0


@pytest.mark.parametrize("name", [FAST, QUAD])
def test_row_scan_carries_past_2048_rows(name, golden):
    """2100 output rows: the exclusive scan of the per-row counts runs three 1024-row chunks"""
    from vo_b200 import r2d2_frontend as rf
    sd = _weights(golden("r2d2_net.npz"))[1] if name == FAST else _random_sd(QUAD, seed=4)
    H, W = 2100, 40
    img = _textured(H, W, seed=5)
    net = rf.R2D2Net(name, sd, H, W, max_kp=H * W)
    assert net.Ho == 2100
    thr = (0.0, 0.0, -1.0)
    xs, ys = _check_nms_exact(net, net.extract(img, *thr, want_maps=True), thr)
    assert (ys < 1024).sum() > 0 and ((ys >= 1024) & (ys < 2048)).sum() > 0 and (ys >= 2048).sum() > 0
