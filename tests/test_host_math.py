"""csrc/pnp_math.cuh compiled for the host (g++ -ffp-contract=off) must equal the oracle bit for bit: same
hypothesis table, same P3P poses, same fp32 errors.  This is the CPU-side half of the "inlier sets bit-exact
under a shared hypothesis set" claim; tests/test_gpu_pnp.py is the device half."""
import ctypes
import os
import subprocess

import numpy as np
import pytest

HERE = os.path.dirname(os.path.abspath(__file__))


@pytest.fixture(scope="module")
def hm(tmp_path_factory):
    so = str(tmp_path_factory.mktemp("shim") / "libvo_host_math_test.so")
    subprocess.check_call(["g++", "-O2", "-ffp-contract=off", "-shared", "-fPIC", "-o", so,
                           os.path.join(HERE, "host_math_shim.cpp")])
    lib = ctypes.CDLL(so)
    lib.hm_is_inlier.restype = ctypes.c_int
    lib.hm_orb_harris.restype = ctypes.c_float
    lib.hm_orb_atan2.restype = ctypes.c_float
    lib.hm_orb_atan2.argtypes = [ctypes.c_float, ctypes.c_float]
    return lib


def _p(a):
    return a.ctypes.data_as(ctypes.c_void_p)


def test_hypothesis_generator_equals_oracle(hm, orc):
    for n, pair in ((4, 0), (57, 3), (5000, 999)):
        want = orc.hypotheses(n, 256, 8214, pair)
        got = np.zeros((256, 4), np.int32)
        for h in range(256):
            hm.hm_draw(ctypes.c_ulonglong(8214), ctypes.c_longlong(pair), h, n, _p(got[h]))
        assert np.array_equal(got, want)


def test_p3p_and_scoring_bit_exact(hm, orc, golden):
    g = golden("pnp.npz")
    xyz, uv, K = g["xyz"], g["uv"], g["K"]
    hyp = orc.hypotheses(len(xyz), 128, 8214, 0)
    poses, counts = orc.solve_and_score(xyz, uv, K, hyp)
    kv = np.array([K[0, 0], K[1, 1], K[0, 2], K[1, 2]])
    kf = kv.astype(np.float32)
    nvalid = 0
    for h in range(128):
        P = np.ascontiguousarray(xyz[hyp[h]].astype(np.float64))
        q = np.ascontiguousarray(uv[hyp[h]].astype(np.float64))
        out = np.zeros(12)
        ok = hm.hm_p3p4(_p(P), _p(q), _p(kv), _p(out))
        if not ok:
            assert np.isnan(poses[h]).all()
            continue
        nvalid += 1
        assert np.array_equal(out.astype(np.float32), poses[h])          # identical bits after the fp32 cast
        p32 = np.ascontiguousarray(poses[h])
        cnt = 0
        for i in range(0, len(xyz), 7):
            cnt += hm.hm_is_inlier(_p(p32), _p(kf), ctypes.c_float(1.5),
                                   *(ctypes.c_float(float(x)) for x in (*xyz[i], *uv[i])))
        m = orc.inlier_mask(xyz, uv, K, poses[h])
        assert cnt == int(m[::7].sum())
    assert nvalid > 100


def test_prefix_xor_hamming_tree_equals_popcount(hm):
    """csrc/hamming_math.cuh (prefix-XOR descriptors, carries from two inputs and the sum, 4 weighted popcounts) must
    give the plain 256-bit Hamming distance for every input: random words, sparse and dense differences, the extremes
    (0 and 256) and single-bit differences in every position."""
    rng = np.random.default_rng(8214)
    n = 20000
    a = rng.integers(0, 2 ** 32, (n, 8), dtype=np.uint64).astype(np.uint32)
    b = rng.integers(0, 2 ** 32, (n, 8), dtype=np.uint64).astype(np.uint32)
    sparse = (rng.integers(0, 2 ** 32, (n, 8), dtype=np.uint64) & rng.integers(0, 2 ** 32, (n, 8), dtype=np.uint64)
              & rng.integers(0, 2 ** 32, (n, 8), dtype=np.uint64)).astype(np.uint32)
    b[: n // 3] = a[: n // 3] ^ sparse[: n // 3]                       # matches: few differing bits
    b[n // 3: n // 2] = ~(a[n // 3: n // 2] ^ sparse[n // 3: n // 2])  # nearly all bits differ (carries into the fours)
    b[n // 2] = a[n // 2]                                              # distance 0
    b[n // 2 + 1] = ~a[n // 2 + 1]                                     # distance 256: every bit column counts 8
    for bit in range(256):                                             # one differing bit, every position
        b[n // 2 + 2 + bit] = a[n // 2 + 2 + bit]
        b[n // 2 + 2 + bit, bit // 32] ^= np.uint32(1 << (bit % 32))
    a, b = np.ascontiguousarray(a), np.ascontiguousarray(b)
    got = np.zeros(n, np.int32)
    hm.hm_hamming256_many(_p(a), _p(b), n, _p(got))
    want = np.unpackbits((a ^ b).view(np.uint8), axis=1).sum(1)
    assert np.array_equal(got, want)
    assert got[n // 2] == 0 and got[n // 2 + 1] == 256 and (got[n // 2 + 2: n // 2 + 258] == 1).all()


def test_orb_math_header_equals_oracle(hm):
    """csrc/orb_math.cuh (the arithmetic the ORB front-end kernels will run) against oracle/orb_frontend.py, which is
    pinned against OpenCV: gray weights, INTER_LINEAR_EXACT, FAST corner score, Harris response, fastAtan2, the float
    Gaussian, the rotated rBRIEF pattern, the circular-patch table."""
    from oracle import orb_frontend as of
    rng = np.random.default_rng(8214)
    assert [hm.hm_orb_umax(v) for v in range(16)] == [int(u) for u in of.umax_table(15)[:16]]
    bgr = rng.integers(0, 256, (64, 3), dtype=np.uint8)
    assert [hm.hm_orb_gray(int(b), int(g), int(r)) for b, g, r in bgr] == [int(v) for v in of.bgr_to_gray(bgr[None])[0]]
    # resize cascade of a KITTI-wide strip
    img = rng.integers(0, 256, (60, 1241), dtype=np.uint8)
    for dw, dh in ((1034, 50), (862, 42), (97, 7), (1241, 60), (2000, 90)):
        out = np.zeros((dh, dw), np.uint8)
        hm.hm_orb_resize(_p(img), 1241, 60, _p(out), dw, dh)
        assert np.array_equal(out, of.resize_linear_exact(img, dw, dh)), (dw, dh)
    # FAST score map: noise (dense corners) and a smooth image with flat rectangles (ties, non-corners)
    smooth = np.kron(rng.integers(0, 256, (12, 20), dtype=np.uint8), np.ones((8, 8), np.uint8))
    for im in (rng.integers(0, 256, (70, 90), dtype=np.uint8), np.ascontiguousarray(smooth)):
        got = np.zeros(im.shape, np.int32)
        hm.hm_orb_fast_map(_p(im), im.shape[1], im.shape[0], 20, _p(got))
        want = of.fast_scores(im, 20)
        assert np.array_equal(got, want) and (want > 0).any()
    # Harris response from integer sums (incl. the magnitudes a 7x7 block of extreme gradients reaches)
    for a, b, c in np.concatenate([rng.integers(0, 49 * 1020 * 1020, (200, 3)), [[0, 0, 0], [49 * 1020 * 1020] * 3]]):
        c = int(c) - 20_000_000
        fa, fb, fc = np.float32(int(a)), np.float32(int(b)), np.float32(c)
        scale = np.float32(1.0) / np.float32(28 * np.float32(255.0))
        want = (fa * fb - fc * fc - np.float32(0.04) * (fa + fb) * (fa + fb)) * (scale * scale * scale * scale)
        assert np.float32(hm.hm_orb_harris(int(a), int(b), c)) == want
    for y, x in np.concatenate([rng.integers(-60000, 60000, (400, 2)), [[0, 0], [0, 5], [5, 0], [-5, 0], [0, -5], [7, 7], [-7, 7]]]):
        assert np.float32(hm.hm_orb_atan2(float(y), float(x))) == of.fast_atan2(y, x), (y, x)
    tex = rng.integers(0, 256, (40, 57), dtype=np.uint8)
    out = np.zeros_like(tex)
    hm.hm_orb_blur(_p(tex), 57, 40, _p(out))
    assert np.array_equal(out, of.blur_7x7(tex))
    pat = np.ascontiguousarray(of.pattern().astype(np.int32))
    for ang in np.concatenate([rng.uniform(0, 360, 100).astype(np.float32), np.float32([0, 90, 180, 270, 359.99])]):
        ix, iy = np.zeros(512, np.int32), np.zeros(512, np.int32)
        hm.hm_orb_rotate(ctypes.c_float(float(ang)), _p(pat), 512, _p(ix), _p(iy))
        wx, wy = of.rotated_pattern(ang, pat)
        assert np.array_equal(ix, wx) and np.array_equal(iy, wy), ang
