"""Batched ORB front-end on a B200 (OrbExtractor.extract_batch, vo_orb_extract_batch): image s of a batch gives, bit for bit,
what OrbExtractor.extract gives for it alone (kp, desc, aux, count), for BGR and gray, from device and from pinned memory, at
S in {1, 3, 8}; a short output keeps the prefix and sets flag bit 1; the launch count does not depend on S; malformed
input raises before anything is enqueued."""
import numpy as np
import pytest

pytestmark = pytest.mark.gpu


def _contents(H, W, S, seed):
    """S images H x W x 3 cycling through golden crop / noise / flat / blocky texture (tie-heavy) / smooth gradient."""
    import os
    rng = np.random.default_rng(seed)
    here = os.path.dirname(os.path.abspath(__file__))
    gold = np.load(os.path.join(here, "golden", "orb_golden.npz"))["image"]
    out = []
    for s in range(S):
        k = s % 5
        if k == 0 and gold.shape[0] >= H and gold.shape[1] >= W:
            img = gold[:H, :W]
        elif k in (0, 1):
            img = rng.integers(0, 256, (H, W, 3), dtype=np.uint8)
        elif k == 2:
            img = np.full((H, W, 3), 77 + s, np.uint8)
        elif k == 3:
            img = np.kron(rng.integers(0, 256, (H // 8 + 1, W // 8 + 1, 3), dtype=np.uint8), np.ones((8, 8, 1), np.uint8))[:H, :W]
        else:
            yy, xx = np.mgrid[:H, :W]
            img = np.repeat(((xx * 3 + yy * 2 + rng.integers(0, 40, (H, W))) % 256).astype(np.uint8)[:, :, None], 3, 2)
        out.append(np.ascontiguousarray(img))
    return np.stack(out)


def _gray(bgr):
    from oracle import orb_frontend as of
    return np.stack([of.bgr_to_gray(im) for im in bgr])


def _per_image(orb, images):
    """extract() on each image: (kp, desc, aux, count) numpy."""
    out = []
    for im in images:
        kp, desc, aux = orb.extract(im)
        out.append((kp.cpu().numpy(), desc.cpu().numpy(), aux.cpu().numpy(), orb.count.cpu().numpy()))
    return out


@pytest.mark.parametrize("shape", [(240, 416), (97, 163)])      # (97, 163): the top levels are smaller than the border
@pytest.mark.parametrize("S", [1, 3, 8])
def test_batch_equals_extract_image_by_image(shape, S):
    import torch
    import vo_b200  # noqa: F401
    from vo_b200.orb_frontend import OrbExtractor
    H, W = shape
    bgr = _contents(H, W, S, seed=S * 100 + H)
    orb = OrbExtractor(H, W)
    for images in (bgr, _gray(bgr)):
        want = _per_image(orb, images)
        assert sum(int(w[3][0]) for w in want) > 0
        for where in ("cuda", "pinned"):
            t = torch.from_numpy(images)
            t = t.cuda() if where == "cuda" else t.pin_memory()
            kp, desc, aux, count = orb.extract_batch(t)
            assert kp.shape == (S, orb.cap, 2) and desc.shape == (S, orb.cap, 32) and count.shape == (S, 2)
            kp, desc, aux, count = (x.cpu().numpy() for x in (kp, desc, aux, count))
            for s in range(S):
                n = int(want[s][3][0])
                assert np.array_equal(count[s], want[s][3]), (where, s, count[s], want[s][3])
                assert np.array_equal(kp[s, :n], want[s][0]), (where, s)
                assert np.array_equal(desc[s, :n], want[s][1]), (where, s)
                assert np.array_equal(aux[s, :n], want[s][2]), (where, s)
    orb.close()


def test_short_output_is_a_prefix_with_flag_bit_1():
    import torch
    import vo_b200  # noqa: F401
    from vo_b200.orb_frontend import OrbExtractor
    bgr = _contents(240, 416, 5, seed=7)
    orb = OrbExtractor(240, 416)
    want = _per_image(orb, bgr)
    rows = 150
    kp, desc, aux, count = (x.cpu().numpy() for x in orb.extract_batch(torch.from_numpy(bgr).cuda(), rows=rows))
    assert kp.shape == (5, rows, 2)
    n_cut = 0
    for s in range(5):
        n = int(want[s][3][0])
        m = min(n, rows)
        n_cut += n > rows
        assert count[s, 0] == m and count[s, 1] == (2 if n > rows else 0), (s, count[s], n)
        assert np.array_equal(kp[s, :m], want[s][0][:m]) and np.array_equal(desc[s, :m], want[s][1][:m])
        assert np.array_equal(aux[s, :m], want[s][2][:m])
    assert n_cut >= 2
    orb.close()


def test_launches_per_call_do_not_depend_on_S():
    import torch
    import vo_b200  # noqa: F401
    from vo_b200 import ops
    from vo_b200.orb_frontend import OrbExtractor
    bgr = torch.from_numpy(_contents(240, 416, 8, seed=3)).cuda()
    orb = OrbExtractor(240, 416)
    n = {}
    for S in (1, 8, 1):
        for images in (bgr[:S], bgr[:S, :, :, 1].contiguous()):
            l0 = ops.launch_count()
            orb.extract_batch(images)
            n[(S, images.dim())] = ops.launch_count() - l0
    assert n == {(1, 4): 17, (8, 4): 17, (1, 3): 16, (8, 3): 16}, n
    orb.close()


def test_malformed_input_raises_and_enqueues_nothing():
    import torch
    import vo_b200  # noqa: F401
    from vo_b200 import ops
    from vo_b200.orb_frontend import OrbExtractor
    orb = OrbExtractor(120, 200)
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
            orb.extract_batch(images)
    with pytest.raises(ValueError):
        orb.extract_batch(good, rows=0)
    torch.cuda.synchronize()
    assert ops.launch_count() == l0
    orb.extract_batch(good)
    assert ops.launch_count() == l0 + 17
    orb.close()
