"""vo_conv2d (ops.conv2d) against the fp64 reference of tests/conv64.py, element by element, on a grid of shapes chosen
relative to the SM count: the persistent CTAs run 1, 2, 3 and >= 5 tiles each, so both tensor-memory accumulators,
the phase wraps of their barriers and a ring that carries over between tiles are compared with the reference, not
only the first tile of every CTA.  Integer data must be exact (bit for bit, whatever the accumulation order);
real-valued data must lie within eps = 2^-18 * sigma of fp64 at every element (see conv64.py for the derivation).
Also: impulse images that pin tap addressing and zero padding exactly, determinism, and refused calls that enqueue
nothing.

Measured on a B200 (148 SMs, 1000 W power limit): the integer class is exact at every shape; the worst |err| / eps of
the real-valued classes is 0.74 (k5_w129, K = 5*5*96 = 2400, activations * 1e3), 0.48 on tiles_5sm_ring (K = 864) and
0.36 or less elsewhere.  The numpy model of conv64.emulate_3xtf32 (round-to-nearest fp32 additions, one product at a
time) stays below 0.25 at the same shapes, so the tensor core accumulates less accurately than that model; the share
of the 2^-18 budget left for accumulation still covers it at K = 2400."""
import os
import sys

import numpy as np
import pytest

sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
import conv64 as c64  # noqa: E402

pytestmark = pytest.mark.gpu

FAMILIES = sorted(c64.shape_grid(148))


def _sm():
    import torch
    return torch.cuda.get_device_properties(0).multi_processor_count


def _cuda(*arrays):
    import torch
    return [torch.from_numpy(np.ascontiguousarray(a)).cuda() for a in arrays]


@pytest.mark.parametrize("family", FAMILIES)
@pytest.mark.parametrize("cls", c64.CLASSES)
def test_conv_certifies_against_fp64(family, cls):
    from vo_b200 import ops
    shape = c64.shape_grid(_sm())[family]
    H, W, cin, cout, k, dil = shape
    x, w, scale, shift, relu = c64.make_case(cls, shape, seed=100 + 10 * FAMILIES.index(family) + c64.CLASSES.index(cls))
    xd, wd, sd, hd = _cuda(x, w, scale, shift)
    got = ops.conv2d(xd, wd, sd, hd, k, dil, relu)
    worst, at = c64.certify(got, xd, wd, sd, hd, k, dil, relu, gamma=0.0 if cls == "int" else c64.GAMMA)
    assert cls != "int" or worst == 0.0, (worst, at)


def _impulse(H, W, cin, seed):
    """zero image with integer pixels only at the four corners, at columns 127 and 128 and along the last row"""
    rng = np.random.default_rng(seed)
    x = np.zeros((H, W, cin), np.float32)
    pts = [(0, 0), (0, W - 1), (H - 1, 0), (H - 1, W - 1), (H // 2, 127), (H // 2, 128), (0, 127), (H - 1, 128)]
    pts += [(H - 1, c) for c in range(0, W, 37)]
    for (h, c) in pts:
        if c < W:
            x[h, c] = rng.integers(-15, 16, cin)
    return x


@pytest.mark.parametrize("H,W,cin,cout,k,dil", [
    (5, 130, 32, 64, 3, 2),
    (6, 200, 32, 32, 4, 1),      # even k, odd dilation: one more pixel of padding after than before
    (5, 129, 96, 128, 2, 3),
    (5, 256, 32, 32, 7, 1),
    (3, 1241, 32, 32, 5, 3),
])
def test_impulse_images_are_exact(H, W, cin, cout, k, dil):
    from vo_b200 import ops
    rng = np.random.default_rng(H * W + k)
    x = _impulse(H, W, cin, seed=k * 10 + dil)
    w = rng.integers(-15, 16, (cout, k, k, cin)).astype(np.float32)
    scale = np.ones(cout, np.float32)
    shift = np.zeros(cout, np.float32)
    xd, wd, sd, hd = _cuda(x, w, scale, shift)
    got = ops.conv2d(xd, wd, sd, hd, k, dil, False)
    ref = c64.conv64(xd, wd, sd, hd, k, dil, False)
    assert bool((ref != 0).any())
    diff = got.double() != ref
    assert not bool(diff.any()), [tuple(int(v) for v in p) for p in np.argwhere(diff.cpu().numpy())[:8]]


def test_two_calls_are_bit_identical_at_the_largest_multi_tile_shape():
    import torch
    from vo_b200 import ops
    shape = c64.shape_grid(_sm())["tiles_25sm_k1"]
    H, W, cin, cout, k, dil = shape
    x, w, scale, shift, relu = c64.make_case("randn", shape, seed=7)
    xd, wd, sd, hd = _cuda(x, w, scale, shift)
    a = ops.conv2d(xd, wd, sd, hd, k, dil, relu)
    b = ops.conv2d(xd, wd, sd, hd, k, dil, relu)
    assert torch.equal(a, b)
    shape = c64.shape_grid(_sm())["tiles_5sm_ring"]
    H, W, cin, cout, k, dil = shape
    x, w, scale, shift, relu = c64.make_case("relu_pos", shape, seed=8)
    xd, wd, sd, hd = _cuda(x, w, scale, shift)
    assert torch.equal(ops.conv2d(xd, wd, sd, hd, k, dil, relu), ops.conv2d(xd, wd, sd, hd, k, dil, relu))


def test_malformed_calls_raise_before_any_launch():
    """Every tensor passed is at least as large as the call claims, so even a build without the checks reads in
    bounds; what is asserted is that the call raises and enqueues no kernel."""
    import torch
    from vo_b200 import _lib, ops

    def t(*shape):
        return torch.randn(*shape, device="cuda")
    cases = [
        ("C_in 48", (t(8, 130, 48), t(32, 3, 3, 48), t(32), t(32), 3, 1)),
        ("C_out 96", (t(8, 130, 32), t(96, 3, 3, 32), t(96), t(96), 3, 1)),
        ("k 8", (t(8, 130, 32), t(32, 8, 8, 32), t(32), t(32), 8, 1)),
        ("dilation 0", (t(8, 130, 32), t(32, 3, 3, 32), t(32), t(32), 3, 0)),
        ("k=3 weights passed as k=2", (t(8, 130, 32), t(32, 3, 3, 32), t(32), t(32), 2, 1)),
        ("scale shorter than C_out", (t(8, 130, 32), t(64, 3, 3, 32), t(32), t(64), 3, 1)),
        ("shift shorter than C_out", (t(8, 130, 32), t(64, 3, 3, 32), t(64), t(32), 3, 1)),
        ("w C_in differs from x", (t(8, 130, 32), t(32, 3, 3, 64), t(32), t(32), 3, 1)),
        ("x not [H,W,C]", (t(1, 8, 130, 32), t(32, 3, 3, 32), t(32), t(32), 3, 1)),
    ]
    torch.cuda.synchronize()
    for name, args in cases:
        n0 = ops.launch_count()
        with pytest.raises((ValueError, _lib.VoError)):
            ops.conv2d(*args)
        assert ops.launch_count() == n0, name
    # a well-formed call after the refusals still runs and counts its launches
    x, w, scale, shift = t(8, 130, 32), t(32, 3, 3, 32), t(32), t(32)
    n0 = ops.launch_count()
    ops.conv2d(x, w, scale, shift, 3, 1)
    assert ops.launch_count() > n0
