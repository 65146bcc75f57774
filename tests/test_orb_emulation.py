"""csrc/orb.cu — kernels AND launch sequence — executed on the host through tests/cuda_emu.h (blocks one after another,
barrier kernels on real threads) and compared with the pinned CPU restatement (oracle/orb_frontend.py): the CPU-side
half of the ORB front-end's parity claim; tests/test_gpu_orb_frontend.py is the device half."""
import ctypes
import os
import subprocess

import numpy as np
import pytest

from oracle import orb_frontend as of

HERE = os.path.dirname(os.path.abspath(__file__))
CAP = 8 * 4096


@pytest.fixture(scope="module")
def emu(tmp_path_factory):
    so = str(tmp_path_factory.mktemp("shim") / "libvo_orb_emu_test.so")
    subprocess.check_call(["g++", "-x", "c++", "-std=c++17", "-O2", "-ffp-contract=off", "-pthread", "-Wno-unknown-pragmas",
                           "-Wno-subobject-linkage", "-shared", "-fPIC", '-DVO_HOST_EMU="cuda_emu.h"', "-I", HERE, "-o", so,
                           os.path.join(HERE, "orb_emu_shim.cpp")])
    lib = ctypes.CDLL(so)
    lib.emu_last_error.restype = ctypes.c_char_p
    lib.emu_launches.restype = ctypes.c_longlong
    return lib


def _run(emu, image, nfeatures=500, nlevels=8, thr=20):
    image = np.ascontiguousarray(image)
    H, W = image.shape[:2]
    kp = np.zeros((CAP, 2), np.float32)
    desc = np.zeros((CAP, 32), np.uint8)
    aux = np.zeros((CAP, 4), np.float32)
    cnt = np.zeros(2, np.int32)
    p = lambda a: a.ctypes.data_as(ctypes.c_void_p)
    n = emu.emu_orb_run(p(image), H, W, 1 if image.ndim == 2 else 3, nfeatures, nlevels, thr, p(kp), p(desc), p(aux), p(cnt))
    assert n >= 0, (n, emu.emu_last_error())
    assert cnt[1] == 0
    return kp[:n], desc[:n], aux[:n]


def _sets(level, x, y, *fields):
    return {(int(l), int(a), int(b)): tuple(np.asarray(f[i]) for f in fields) for i, (l, a, b) in enumerate(zip(level, x, y))}


def _check(emu, image, gray, **kw):
    want = of.detect_and_compute(gray, **{k: v for k, v in kw.items() if k in ("nfeatures", "nlevels")})
    kp, desc, aux = _run(emu, image, **kw)
    assert len(kp) == len(want["level"])
    if not len(kp):
        return 0
    scales = of.level_scales()
    lev = aux[:, 0].astype(int)
    s = np.array([scales[l] for l in lev], np.float32)
    gx, gy = np.rint(kp[:, 0] / s).astype(int), np.rint(kp[:, 1] / s).astype(int)
    got = _sets(lev, gx, gy, kp, aux[:, 1], aux[:, 2], aux[:, 3], desc)
    ref = _sets(want["level"], want["xl"], want["yl"], want["pt"], want["angle"], want["response"], want["size"], want["desc"])
    assert set(got) == set(ref)
    for key, fields in ref.items():
        for a, b in zip(fields, got[key]):
            assert np.array_equal(a, b), key
    assert np.array_equal(np.lexsort((gx, gy, lev)), np.arange(len(kp)))       # level-major, then row-major
    return len(kp)


def test_emulated_kernels_equal_the_reference_plugin_output(emu, golden):
    g = golden("orb_golden.npz")
    n = _check(emu, g["image"], of.bgr_to_gray(g["image"]))                     # BGR in: gray conversion in a kernel
    assert n == len(g["kp"])
    assert emu.emu_launches() == 17          # gray + 7 resizes + 4 all-level pixel kernels + 5 keypoint kernels


def test_emulated_kernels_edge_cases(emu):
    rng = np.random.default_rng(8214)
    blocky = np.kron(rng.integers(0, 256, (20, 33), dtype=np.uint8), np.ones((8, 8), np.uint8))[:150, :260]
    assert _check(emu, blocky, np.ascontiguousarray(blocky)) > 0                # flat blocks: tie-heavy scores
    assert _check(emu, *(2 * [rng.integers(0, 256, (150, 260), dtype=np.uint8)])) > 300   # noise: dense corners
    assert _check(emu, *(2 * [np.full((120, 200), 77, np.uint8)])) == 0         # flat: nothing found
    assert _check(emu, *(2 * [rng.integers(0, 256, (97, 163), dtype=np.uint8)])) > 0      # top levels below the border
    noise = rng.integers(0, 256, (130, 170), dtype=np.uint8)
    assert _check(emu, noise, noise, nfeatures=40) > 0                          # small quotas: both retainBest cuts bite
    assert _check(emu, noise, noise, nfeatures=300, nlevels=3) > 0              # fewer pyramid levels


def test_emulated_kernels_kitti_shaped_frame(emu):
    """1241 x 376, smooth texture + noise: 500 keypoints over all eight levels."""
    rng = np.random.default_rng(3)
    coarse = rng.integers(0, 256, (48, 156)).astype(np.float32)
    ys, xs = np.linspace(0, 46.999, 376), np.linspace(0, 154.999, 1241)
    y0, x0 = ys.astype(int), xs.astype(int)
    fy, fx = (ys - y0)[:, None], (xs - x0)[None, :]
    smooth = (coarse[y0][:, x0] * (1 - fy) * (1 - fx) + coarse[y0 + 1][:, x0] * fy * (1 - fx) +
              coarse[y0][:, x0 + 1] * (1 - fy) * fx + coarse[y0 + 1][:, x0 + 1] * fy * fx)
    img = np.clip(smooth + rng.integers(0, 25, smooth.shape), 0, 255).astype(np.uint8)
    assert _check(emu, img, img) >= 450
    assert _check(emu, img, img, nfeatures=5000) >= 3000        # the bench's ORB-5k setting: ~1100 keypoints on level 0
