"""fp64 reference, error model and certifier for the tensor-core convolution (vo_conv2d / ops.conv2d), plus a numpy
emulation of what the kernel computes.  Test infrastructure: nothing here needs a GPU.

The convolution is the "same" one of conv_tc.cu: stride 1, dilation d, k x k taps, total padding (k-1)*d of which
floor((k-1)*d / 2) goes before the first pixel (vo_conv2d's pad = ((k-1)*dil)/2; the rest falls after the last pixel,
where TMA's out-of-bounds zero fill supplies it).  For odd (k-1)*d the padding is asymmetric.  Layouts: x [H,W,Cin],
w [Cout,k,k,Cin], scale / shift [Cout], output [H,W,Cout]; y = conv * scale + shift, then ReLU if asked.

Error model.  eps = GAMMA * sigma with sigma = |scale| * conv(|x|, |w|) + |shift| (fp64), per output element.
GAMMA = 2^-18 is derived as follows:
  * the producing layer (here tf32_split_kernel) splits every operand with round-to-nearest-away:
    a_hi = rna_tf32(a), a_lo = rna_tf32(a - a_hi).  tf32 keeps 10 fraction bits, so |a - a_hi| <= 2^-11 |a| and the
    remainder r = a - a_hi - a_lo satisfies |r| <= 2^-11 |a - a_hi| <= 2^-22 |a|;
  * the kernel issues three MMAs per k-step (a_lo*b_hi, a_hi*b_lo, a_hi*b_hi).  Against the exact product a*b they
    drop a_lo*b_lo (<= 2^-22 |a||b|), r_a*b and a_hi*r_b (each <= 2^-22 |a||b| to first order): about 3 * 2^-22 of
    sigma in total, i.e. 3/16 of the budget;
  * products of two tf32 values have at most 22 significant bits and are exact in fp32;
  * the remaining 13 * 2^-22 covers the fp32 accumulation in tensor memory (3 * K / 8 accumulator updates for
    K = k*k*Cin) and the epilogue FMA (one rounding, 2^-24 relative).  Rounding errors of an fp32 sum of terms with
    mixed signs grow like sqrt(#updates), so at the largest K here (2304) this is a few units of 2^-24 of sigma.
    The tensor core's internal summation order and rounding are not documented: that this share of the budget
    suffices is an assumption, which the GPU tests check at every shape; it is not derived from a specification.
On integer data (|x|, |w| <= 15, scale a power of two, shift an integer, every partial sum below 2^24) all split
remainders are 0 and every partial sum is exact, so the kernel must agree with the reference bit for bit: GAMMA = 0.
"""
import numpy as np
import torch
import torch.nn.functional as F

GAMMA = 2.0 ** -18


def shape_grid(sm):
    """{family: (H, W, Cin, Cout, k, dil)} relative to the SM count `sm` (one persistent CTA per SM; a tile is 128
    pixels of one row, n_tiles = H * ceil(W / 128)).  Kept small enough in H*W*Cout*K for the numpy emulation."""
    return {
        "tiles_sm-1":      (sm - 1, 128, 32, 32, 3, 1),        # every CTA one tile except one idle SM; W = 128 exactly
        "tiles_sm":        (sm, 9, 64, 64, 2, 1),              # one tile per SM; even k, odd dilation (asymmetric pad)
        "tiles_sm+1":      (sm + 1, 1, 256, 128, 3, 3),        # CTA 0 runs two tiles: accumulator 1; W = 1; C_in 256
        "tiles_2sm+1":     (2 * sm + 1, 127, 32, 32, 2, 3),    # three tiles on CTA 0: accumulator 0 reused after a wrap
        "tiles_5sm_ring":  (5 * sm + 20, 9, 96, 64, 3, 2),     # >= 5 tiles per CTA, 27 ring items per tile
        "tiles_25sm_k1":   (376, 1241, 32, 32, 1, 1),          # KITTI width, 3760 tiles of one ring item each
        "h1_k7":           (1, 1241, 32, 32, 7, 2),            # one row: all but the middle row of taps is padding
        "h2_k4_w129":      (2, 129, 96, 64, 4, 1),             # even k, odd dilation; a 1-pixel second tile
        "h5_k3_dil8":      (5, 128, 32, 128, 3, 8),            # taps entirely outside a 5-row image
        "h5_k2_dil8":      (5, 130, 32, 128, 2, 8),
        "k5_w129":         (17, 129, 96, 32, 5, 1),
    }


CLASSES = ("int", "randn", "randn_1e3", "relu_pos")


def make_case(cls, shape, seed):
    """(x, w, scale, shift, relu) as float32 numpy arrays for one data class:
    int        integers in [-15, 15], scale a power of two, integer shift: exact in tf32 and in every fp32 partial sum
    randn      standard normal activations, weights randn / sqrt(K), scale of either sign
    randn_1e3  the same with activations * 1e3: the lo parts carry more than the shift
    relu_pos   non-negative activations (a ReLU layer's output) and ReLU on the output"""
    H, W, cin, cout, k, dil = shape
    rng = np.random.default_rng(seed)
    K = k * k * cin
    if cls == "int":
        x = rng.integers(-15, 16, (H, W, cin)).astype(np.float32)
        w = rng.integers(-15, 16, (cout, k, k, cin)).astype(np.float32)
        scale = (2.0 ** rng.integers(-2, 3, cout)).astype(np.float32)
        shift = rng.integers(-100, 101, cout).astype(np.float32)
        return x, w, scale, shift, False
    x = rng.standard_normal((H, W, cin), dtype=np.float32)
    w = (rng.standard_normal((cout, k, k, cin), dtype=np.float32) / np.float32(np.sqrt(K))).astype(np.float32)
    scale = (rng.uniform(0.5, 1.5, cout) * rng.choice([-1.0, 1.0], cout)).astype(np.float32)
    shift = rng.standard_normal(cout).astype(np.float32)
    if cls == "randn":
        return x, w, scale, shift, False
    if cls == "randn_1e3":
        return (x * np.float32(1e3)).astype(np.float32), w, scale, shift, False
    if cls == "relu_pos":
        return np.abs(x), w, np.abs(scale), (0.5 * shift).astype(np.float32), True
    raise ValueError(cls)


def _t64(a, dev):
    if isinstance(a, torch.Tensor):
        return a.detach().to(dev, torch.float64)
    return torch.as_tensor(np.asarray(a), dtype=torch.float64, device=dev)


def conv_fp64(x, w, k, dil, left=None, device=None):
    """sum over taps and channels in fp64: x [H,W,Cin], w [Cout,k,k,Cin] -> [H,W,Cout] (no scale / shift).
    `left`: padding before the first pixel (default floor((k-1)*dil / 2), the kernel's rule)."""
    dev = device if device is not None else (x.device if isinstance(x, torch.Tensor) else "cpu")
    x, w = _t64(x, dev), _t64(w, dev)
    tot = (k - 1) * dil
    lo = tot // 2 if left is None else left
    xp = F.pad(x.permute(2, 0, 1)[None], (lo, tot - lo, lo, tot - lo))
    return F.conv2d(xp, w.permute(0, 3, 1, 2), dilation=dil)[0].permute(1, 2, 0)


def conv64(x, w, scale, shift, k, dil, relu):
    """the reference: fp64 'same' convolution, * scale + shift, ReLU if asked -> fp64 [H,W,Cout] on x's device"""
    dev = x.device if isinstance(x, torch.Tensor) else "cpu"
    y = conv_fp64(x, w, k, dil, device=dev) * _t64(scale, dev) + _t64(shift, dev)
    return y.clamp_min(0) if relu else y


def sigma64(x, w, scale, k, dil, shift):
    """|scale| * conv(|x|, |w|) + |shift| in fp64 (the magnitude the error bound scales with)"""
    dev = x.device if isinstance(x, torch.Tensor) else "cpu"
    return conv_fp64(_t64(x, dev).abs(), _t64(w, dev).abs(), k, dil, device=dev) * _t64(scale, dev).abs() + _t64(shift, dev).abs()


def certify(got, x, w, scale, shift, k, dil, relu, gamma=GAMMA):
    """Raise AssertionError on the first output element (row-major h, w, c) with |got - ref| > gamma * sigma; return
    (worst |err| / eps, (h, w, c) of the worst).  gamma = 0 demands bit equality with the fp64 reference."""
    dev = got.device if isinstance(got, torch.Tensor) else "cpu"
    g = _t64(got, dev)
    ref = conv64(_t64(x, dev), w, scale, shift, k, dil, relu)
    assert g.shape == ref.shape, (tuple(g.shape), tuple(ref.shape))
    assert bool(torch.isfinite(g).all()), "non-finite output"
    eps = gamma * sigma64(_t64(x, dev), w, scale, k, dil, shift)
    err = (g - ref).abs()
    bad = err > eps
    if bool(bad.any()):
        h, ww, c = (int(v) for v in torch.nonzero(bad)[0])
        raise AssertionError(f"output ({h},{ww},{c}): got {float(g[h, ww, c])!r}, fp64 {float(ref[h, ww, c])!r}, "
                             f"|err| {float(err[h, ww, c]):.3e} > eps {float(eps[h, ww, c]):.3e} "
                             f"({int(bad.sum())} elements outside the bound)")
    ratio = torch.where(eps > 0, err / torch.where(eps > 0, eps, torch.ones_like(eps)), torch.zeros_like(err))
    i = int(torch.argmax(ratio))
    H, W, C = ratio.shape
    return float(ratio.reshape(-1)[i]), (i // (W * C), (i // C) % W, i % C)


def tf32_rna(a):
    """round fp32 to tf32, nearest with ties away from zero: the bit rule of tf32_rna_host (r2d2_net.cu) and of
    cvt.rna.tf32.f32 for finite inputs"""
    u = np.ascontiguousarray(a, dtype=np.float32).view(np.uint32)
    return ((u + np.uint32(0x1000)) & np.uint32(0xffffe000)).view(np.float32)


def emulate_3xtf32(x, w, scale, shift, k, dil, relu):
    """numpy model of conv_tc_kernel: operands split into tf32 hi / lo, per tap (row-major) and input channel the three
    exact products a_lo*b_hi, a_hi*b_lo, a_hi*b_hi added one by one to an fp32 accumulator, then fp32
    fma(acc, scale, shift) and ReLU.  x [H,W,Cin], w [Cout,k,k,Cin] float32 -> [H,W,Cout] float32."""
    x = np.asarray(x, np.float32)
    w = np.asarray(w, np.float32)
    H, W, cin = x.shape
    cout = w.shape[0]
    tot = (k - 1) * dil
    lo = tot // 2
    xh = tf32_rna(x)
    xl = tf32_rna(x - xh)
    wh = tf32_rna(w)
    wl = tf32_rna(w - wh)
    ph = np.zeros((H + tot, W + tot, cin), np.float32)
    pl = np.zeros_like(ph)
    ph[lo:lo + H, lo:lo + W] = xh
    pl[lo:lo + H, lo:lo + W] = xl
    acc = np.zeros((H, W, cout), np.float32)
    p = np.empty_like(acc)
    for ty in range(k):
        for tx in range(k):
            sh = ph[ty * dil:ty * dil + H, tx * dil:tx * dil + W]
            sl = pl[ty * dil:ty * dil + H, tx * dil:tx * dil + W]
            for c in range(cin):
                ah, al = sh[:, :, c:c + 1], sl[:, :, c:c + 1]
                np.multiply(al, wh[:, ty, tx, c], out=p)
                acc += p
                np.multiply(ah, wl[:, ty, tx, c], out=p)
                acc += p
                np.multiply(ah, wh[:, ty, tx, c], out=p)
                acc += p
    # fp32 FMA: the fp64 product of two fp32 values is exact; one rounding of the sum (double rounding is negligible)
    y = (acc.astype(np.float64) * np.asarray(scale, np.float64) + np.asarray(shift, np.float64)).astype(np.float32)
    return np.maximum(y, np.float32(0)) if relu else y
