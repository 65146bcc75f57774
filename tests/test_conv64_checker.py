"""The fp64 convolution reference and certifier (tests/conv64.py) on the CPU: the numpy model of the 3xTF32 kernel
certifies at every shape of the GPU grid with room to spare (the error budget is not tight on the arithmetic it was
derived from), integer data is exact, and every planted defect is rejected, so GPU output that certifies cannot
carry it."""
import os
import sys

import numpy as np
import pytest

sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
import conv64 as c64  # noqa: E402

SM = 148          # B200; the GPU tests build the same grid from the device's own SM count
GRID = c64.shape_grid(SM)


def test_reference_padding_is_the_kernels_rule():
    """left padding floor((k-1)*dil / 2), the rest after the last pixel: checked against a direct sum over taps"""
    rng = np.random.default_rng(0)
    for k, dil in ((2, 1), (2, 3), (4, 1), (3, 2), (1, 1), (5, 1)):
        H, W, cin, cout = 6, 7, 3, 2
        x = rng.standard_normal((H, W, cin))
        w = rng.standard_normal((cout, k, k, cin))
        pad = ((k - 1) * dil) // 2
        want = np.zeros((H, W, cout))
        for h in range(H):
            for ww in range(W):
                for ty in range(k):
                    for tx in range(k):
                        hh, xx = h - pad + ty * dil, ww - pad + tx * dil
                        if 0 <= hh < H and 0 <= xx < W:
                            want[h, ww] += w[:, ty, tx, :] @ x[hh, xx]
        got = c64.conv_fp64(x, w, k, dil).numpy()
        assert got.shape == want.shape and np.abs(got - want).max() < 1e-12


def test_tf32_rna_rounds_to_nearest_ties_away():
    one = np.float32(1.0)
    ulp = np.float32(2.0 ** -10)
    x = np.array([1 + 2.0 ** -11, -(1 + 2.0 ** -11), 1 + 2.0 ** -11 - 2.0 ** -23, 1 + 3 * 2.0 ** -11, 3.0, 0.0], np.float32)
    got = c64.tf32_rna(x)
    assert got.tolist() == [one + ulp, -(one + ulp), one, one + 2 * ulp, 3.0, 0.0]
    v = np.random.default_rng(1).standard_normal(10000).astype(np.float32)
    h = c64.tf32_rna(v)
    assert np.all(np.abs(v.astype(np.float64) - h) <= 2.0 ** -11 * np.abs(v))
    assert np.all((h.view(np.uint32) & 0x1fff) == 0)
    r = v.astype(np.float64) - h - c64.tf32_rna(v - h)
    assert np.all(np.abs(r) <= 2.0 ** -22 * np.abs(v))


@pytest.mark.parametrize("family", sorted(GRID))
@pytest.mark.parametrize("cls", c64.CLASSES)
def test_emulated_kernel_certifies_on_the_gpu_grid(family, cls):
    shape = GRID[family]
    H, W, cin, cout, k, dil = shape
    x, w, scale, shift, relu = c64.make_case(cls, shape, seed=10 * sorted(GRID).index(family) + c64.CLASSES.index(cls))
    got = c64.emulate_3xtf32(x, w, scale, shift, k, dil, relu)
    if cls == "int":
        worst, _ = c64.certify(got, x, w, scale, shift, k, dil, relu, gamma=0.0)
        assert worst == 0.0
    else:
        worst, at = c64.certify(got, x, w, scale, shift, k, dil, relu)
        assert worst <= 0.25, (worst, at)


def _seam_case(k=2, dil=1, cls="randn"):
    shape = (6, 131, 32, 32, k, dil)        # second tile starts at w = 128
    x, w, scale, shift, relu = c64.make_case(cls, shape, seed=11)
    return shape, x, w, scale, shift, relu


def _affine(acc, scale, shift, relu):
    y = acc * scale.astype(np.float64) + shift.astype(np.float64)
    return np.maximum(y, 0.0) if relu else y


def test_certify_rejects_a_tap_shifted_by_one_pixel():
    (H, W, cin, cout, k, dil), x, w, scale, shift, relu = _seam_case(k=3)
    w0 = np.zeros_like(w)
    w0[:, 1, 2] = w[:, 1, 2]
    xs = np.zeros_like(x)
    xs[:, :-1] = x[:, 1:]                               # tap (1, 2) reads one pixel further right
    acc = (c64.conv_fp64(x, w - w0, k, dil) + c64.conv_fp64(xs, w0, k, dil)).numpy()
    with pytest.raises(AssertionError):
        c64.certify(_affine(acc, scale, shift, relu), x, w, scale, shift, k, dil, relu)


@pytest.mark.parametrize("k,dil", [(2, 1), (2, 3), (4, 1)])
def test_certify_rejects_symmetric_padding_for_even_k(k, dil):
    (H, W, cin, cout, _, _), x, w, scale, shift, relu = _seam_case(k, dil)
    tot = (k - 1) * dil
    acc = c64.conv_fp64(x, w, k, dil, left=tot - tot // 2).numpy()     # the odd pixel of padding before, not after
    with pytest.raises(AssertionError):
        c64.certify(_affine(acc, scale, shift, relu), x, w, scale, shift, k, dil, relu)


def test_certify_rejects_two_swapped_input_channels():
    (H, W, cin, cout, k, dil), x, w, scale, shift, relu = _seam_case(k=3)
    xs = x[:, :, [1, 0] + list(range(2, cin))]
    got = c64.emulate_3xtf32(xs, w, scale, shift, k, dil, relu)
    with pytest.raises(AssertionError):
        c64.certify(got, x, w, scale, shift, k, dil, relu)


@pytest.mark.parametrize("cls", ["randn", "randn_1e3", "relu_pos"])
def test_certify_rejects_2xtf32_without_the_lo_hi_product(cls):
    """activations already rounded to tf32 have lo = 0: the emulation then issues a_hi*b_lo and a_hi*b_hi only"""
    (H, W, cin, cout, k, dil), x, w, scale, shift, relu = _seam_case(k=3, cls=cls)
    got = c64.emulate_3xtf32(c64.tf32_rna(x), w, scale, shift, k, dil, relu)
    with pytest.raises(AssertionError):
        c64.certify(got, x, w, scale, shift, k, dil, relu)


def test_certify_rejects_shift_applied_twice():
    (H, W, cin, cout, k, dil), x, w, scale, shift, relu = _seam_case(k=3)
    got = c64.emulate_3xtf32(x, w, scale, shift, k, dil, relu) + shift
    with pytest.raises(AssertionError):
        c64.certify(got, x, w, scale, shift, k, dil, relu)


def test_certify_rejects_relu_before_scale():
    (H, W, cin, cout, k, dil), x, w, scale, shift, _ = _seam_case(k=3)
    acc = c64.conv_fp64(x, w, k, dil).numpy()
    got = np.maximum(acc, 0.0) * scale + shift
    with pytest.raises(AssertionError):
        c64.certify(got, x, w, scale, shift, k, dil, True)


@pytest.mark.parametrize("px", [127, 128])
def test_certify_rejects_one_pixel_off_by_4eps_at_a_tile_seam(px):
    (H, W, cin, cout, k, dil), x, w, scale, shift, relu = _seam_case(k=3)
    got = c64.emulate_3xtf32(x, w, scale, shift, k, dil, relu).astype(np.float64)
    worst, _ = c64.certify(got, x, w, scale, shift, k, dil, relu)
    assert worst <= 0.25
    eps = c64.GAMMA * c64.sigma64(x, w, scale, k, dil, shift).numpy()
    got[H - 1, px, 5] += 4 * eps[H - 1, px, 5]
    with pytest.raises(AssertionError, match=rf"output \({H - 1},{px},5\)"):
        c64.certify(got, x, w, scale, shift, k, dil, relu)


def test_integer_class_is_exact_and_a_unit_error_is_rejected():
    shape = GRID["h2_k4_w129"]
    H, W, cin, cout, k, dil = shape
    x, w, scale, shift, relu = c64.make_case("int", shape, seed=3)
    got = c64.emulate_3xtf32(x, w, scale, shift, k, dil, relu)
    assert c64.certify(got, x, w, scale, shift, k, dil, relu, gamma=0.0)[0] == 0.0
    assert np.abs(got).max() < 2 ** 24
    got = got.copy()
    got[1, 128, 0] = np.nextafter(got[1, 128, 0], np.float32(np.inf))
    with pytest.raises(AssertionError):
        c64.certify(got, x, w, scale, shift, k, dil, relu, gamma=0.0)
