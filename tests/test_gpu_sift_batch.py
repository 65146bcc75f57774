"""Batched SIFT front-end on a B200 (SiftExtractor.extract_batch, vo_sift_extract_batch): image s of a batch gives, bit for
bit, what SiftExtractor.extract gives for it alone (kp, desc, aux, count), for BGR and gray, from device and from pinned
memory, at S in {1, 3, 8} and on a KITTI-shaped pair; a short output keeps the prefix and sets flag bit 1; a raw list past
max_keypoints sets flag bit 0; the launch count does not depend on S; malformed input raises before anything is
enqueued."""
import numpy as np
import pytest

pytestmark = pytest.mark.gpu


def _texture(rng, H, W):
    coarse = rng.integers(0, 256, (H // 8 + 2, W // 8 + 2, 3)).astype(np.float32)
    ys, xs = np.arange(H) / 8.0, np.arange(W) / 8.0
    y0, x0 = ys.astype(int), xs.astype(int)
    fy, fx = (ys - y0)[:, None, None], (xs - x0)[None, :, None]
    img = (coarse[y0][:, x0] * (1 - fy) * (1 - fx) + coarse[y0 + 1][:, x0] * fy * (1 - fx) +
           coarse[y0][:, x0 + 1] * (1 - fy) * fx + coarse[y0 + 1][:, x0 + 1] * fy * fx)
    return np.clip(img + rng.integers(0, 20, img.shape), 0, 255).astype(np.uint8)


def _contents(H, W, S, seed):
    """S images H x W x 3 cycling through smooth texture / noise / flat / gradient."""
    rng = np.random.default_rng(seed)
    out = []
    for s in range(S):
        k = s % 4
        if k == 0:
            img = _texture(rng, H, W)
        elif k == 1:
            img = rng.integers(0, 256, (H, W, 3), dtype=np.uint8)
        elif k == 2:
            img = np.full((H, W, 3), 77 + s, np.uint8)
        else:
            yy, xx = np.mgrid[:H, :W]
            img = np.repeat(((xx * 3 + yy * 2 + rng.integers(0, 40, (H, W))) % 256).astype(np.uint8)[:, :, None], 3, 2)
        out.append(np.ascontiguousarray(img))
    return np.stack(out)


def _gray(bgr):
    from oracle import orb_frontend as of
    return np.stack([of.bgr_to_gray(im) for im in bgr])


def _per_image(sift, images):
    """extract() on each image: (kp, desc, aux, count) numpy, count = (written, raw)."""
    out = []
    for im in images:
        kp, desc, aux = sift.extract(im)
        out.append((kp.cpu().numpy(), desc.cpu().numpy(), aux.cpu().numpy(), sift.count.cpu().numpy()))
    return out


def _check_batch(sift, images, want):
    import torch
    S = len(images)
    for where in ("cuda", "pinned"):
        t = torch.from_numpy(images)
        t = t.cuda() if where == "cuda" else t.pin_memory()
        kp, desc, aux, count = sift.extract_batch(t)
        assert kp.shape == (S, sift.cap, 2) and desc.shape == (S, sift.cap, 128) and count.shape == (S, 2)
        kp, desc, aux, count = (x.cpu().numpy() for x in (kp, desc, aux, count))
        for s in range(S):
            n = int(want[s][3][0])
            assert want[s][3][1] <= sift.cap
            assert count[s, 0] == n and count[s, 1] == 0, (where, s, count[s], want[s][3])
            assert np.array_equal(kp[s, :n], want[s][0]), (where, s)
            assert np.array_equal(desc[s, :n], want[s][1]), (where, s)
            assert np.array_equal(aux[s, :n], want[s][2]), (where, s)


@pytest.mark.parametrize("shape", [(240, 416), (97, 163)])      # (97, 163): the top octaves are smaller than the border
@pytest.mark.parametrize("S", [1, 3, 8])
def test_batch_equals_extract_image_by_image(shape, S):
    import vo_b200  # noqa: F401
    from vo_b200.sift_frontend import SiftExtractor
    H, W = shape
    bgr = _contents(H, W, S, seed=S * 100 + H)
    sift = SiftExtractor(H, W)
    for images in (bgr, _gray(bgr)):
        want = _per_image(sift, images)
        assert sum(int(w[3][0]) for w in want) > 0
        _check_batch(sift, images, want)
    sift.close()


def test_kitti_shaped_pair():
    import vo_b200  # noqa: F401
    from vo_b200.sift_frontend import SiftExtractor
    bgr = _contents(376, 1241, 2, seed=5)
    sift = SiftExtractor(376, 1241)
    want = _per_image(sift, bgr)
    assert int(want[0][3][0]) > 1000
    _check_batch(sift, bgr, want)
    sift.close()


def test_short_rows_set_flag_bit_1_and_small_max_keypoints_flag_bit_0():
    import torch
    import vo_b200  # noqa: F401
    from vo_b200._lib import VoError
    from vo_b200.sift_frontend import SiftExtractor
    bgr = _contents(240, 416, 4, seed=7)
    sift = SiftExtractor(240, 416)
    want = _per_image(sift, bgr)
    rows = 200
    kp, desc, aux, count = (x.cpu().numpy() for x in sift.extract_batch(torch.from_numpy(bgr).cuda(), rows=rows))
    assert kp.shape == (4, rows, 2)
    n_cut = 0
    for s in range(4):
        n = int(want[s][3][0])
        m = min(n, rows)
        n_cut += n > rows
        assert count[s, 0] == m and count[s, 1] == (2 if n > rows else 0), (s, count[s], n)
        assert np.array_equal(kp[s, :m], want[s][0][:m]) and np.array_equal(desc[s, :m], want[s][1][:m])
        assert np.array_equal(aux[s, :m], want[s][2][:m])
    assert n_cut >= 2
    sift.close()
    small = SiftExtractor(240, 416, max_keypoints=50)
    with pytest.raises(VoError):
        small.extract(bgr[0])
    count = small.extract_batch(torch.from_numpy(bgr).cuda())[3].cpu().numpy()
    assert count[0, 1] & 1 and count[1, 1] & 1 and count[2].tolist() == [0, 0], count
    small.close()


def test_launches_per_call_do_not_depend_on_S():
    import torch
    import vo_b200  # noqa: F401
    from vo_b200 import ops
    from vo_b200.sift_frontend import SiftExtractor
    bgr = torch.from_numpy(_contents(240, 416, 8, seed=3)).cuda()
    sift = SiftExtractor(240, 416)
    l0 = ops.launch_count()
    sift.extract(bgr[0])
    one = ops.launch_count() - l0
    n = {}
    for S in (1, 8, 1):
        for images in (bgr[:S], bgr[:S, :, :, 1].contiguous()):
            l0 = ops.launch_count()
            sift.extract_batch(images)
            n[(S, images.dim())] = ops.launch_count() - l0
    assert set(n.values()) == {one}, (n, one)
    sift.close()


def test_malformed_input_raises_and_enqueues_nothing():
    import torch
    import vo_b200  # noqa: F401
    from vo_b200 import ops
    from vo_b200.sift_frontend import SiftExtractor
    sift = SiftExtractor(120, 200)
    good = torch.zeros((2, 120, 200, 3), dtype=torch.uint8, device="cuda")
    torch.cuda.synchronize()
    l0 = ops.launch_count()
    bad = [good.float(),                                          # wrong dtype
           torch.zeros((2, 120, 200, 4), dtype=torch.uint8, device="cuda"),     # wrong channel count
           torch.zeros((2, 121, 200), dtype=torch.uint8, device="cuda"),        # wrong size
           torch.zeros((120, 200), dtype=torch.uint8, device="cuda"),           # no batch dimension
           good.transpose(1, 2),                                  # non-contiguous
           torch.zeros((2, 120, 200, 6), dtype=torch.uint8, device="cuda")[..., :3],
           good[:0],                                              # S = 0
           good.cpu(),                                            # pageable host memory
           good.cpu().numpy()]
    for images in bad:
        with pytest.raises(ValueError):
            sift.extract_batch(images)
    with pytest.raises(ValueError):
        sift.extract_batch(good, rows=0)
    torch.cuda.synchronize()
    assert ops.launch_count() == l0
    sift.extract_batch(good)
    assert ops.launch_count() > l0
    sift.close()
