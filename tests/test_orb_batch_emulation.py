"""vo_orb_extract_batch — kernels and launch sequence of csrc/orb.cu — executed on the host through tests/cuda_emu.h: S images
in one call equal the per-image call (vo_orb_extract) on each image and the pinned CPU restatement (oracle/orb_frontend.py),
bit for bit; a short output keeps the prefix and raises flag bit 1; the launch count does not depend on S.  The device half
is tests/test_gpu_orb_batch.py."""
import ctypes
import os
import subprocess

import numpy as np
import pytest

from oracle import orb_frontend as of

HERE = os.path.dirname(os.path.abspath(__file__))


@pytest.fixture(scope="module")
def emu(tmp_path_factory):
    so = str(tmp_path_factory.mktemp("shim") / "libvo_orb_batch_emu_test.so")
    # -fno-gnu-unique: the emulator's inline launch counter must not be merged with that of tests/orb_emu_shim.cpp's
    # library when both are loaded in one process (tests/test_orb_emulation.py counts launches from zero)
    subprocess.check_call(["g++", "-x", "c++", "-std=c++17", "-O2", "-ffp-contract=off", "-fno-gnu-unique", "-pthread", "-Wno-unknown-pragmas",
                           "-Wno-subobject-linkage", "-shared", "-fPIC", '-DVO_HOST_EMU="cuda_emu.h"', "-I", HERE, "-o", so,
                           os.path.join(HERE, "orb_batch_emu_shim.cpp")])
    lib = ctypes.CDLL(so)
    lib.emu_last_error.restype = ctypes.c_char_p
    lib.emu_launches.restype = ctypes.c_longlong
    lib.emu_orb_create.restype = ctypes.c_void_p
    lib.emu_orb_create.argtypes = [ctypes.c_int] * 5
    return lib


def _p(a):
    return a.ctypes.data_as(ctypes.c_void_p)


class Orb:
    def __init__(self, emu, H, W):
        self.emu = emu
        self.h = ctypes.c_void_p(emu.emu_orb_create(H, W, 500, 8, 20))
        assert self.h.value, emu.emu_last_error()
        self.cap = emu.emu_orb_capacity(self.h)

    def extract(self, image):
        image = np.ascontiguousarray(image)
        kp, desc = np.zeros((self.cap, 2), np.float32), np.zeros((self.cap, 32), np.uint8)
        aux, cnt = np.zeros((self.cap, 4), np.float32), np.zeros(2, np.int32)
        rc = self.emu.emu_orb_extract(self.h, _p(image), 1 if image.ndim == 2 else 3, _p(kp), _p(desc), _p(aux), _p(cnt))
        assert rc == 0, self.emu.emu_last_error()
        n = int(cnt[0])
        return kp[:n], desc[:n], aux[:n], cnt

    def batch(self, images, rows=None, expect_rc=0):
        images = np.ascontiguousarray(images)
        S, rows = images.shape[0], self.cap if rows is None else rows
        # sentinel fill: rows past the count must stay untouched
        kp = np.full((max(S, 1), max(rows, 1), 2), -7, np.float32)
        desc = np.full((max(S, 1), max(rows, 1), 32), 0xA5, np.uint8)
        aux = np.full((max(S, 1), max(rows, 1), 4), -7, np.float32)
        cnt = np.full((max(S, 1), 2), -1, np.int32)
        l0 = self.emu.emu_launches()
        rc = self.emu.emu_orb_extract_batch(self.h, _p(images), S, 3 if images.ndim == 4 else 1, rows, _p(kp), _p(desc),
                                            _p(aux), _p(cnt))
        assert rc == expect_rc, (rc, self.emu.emu_last_error())
        return kp, desc, aux, cnt, self.emu.emu_launches() - l0

    def close(self):
        self.emu.emu_orb_destroy(self.h)


def _images(H, W):
    """BGR golden image, blocky texture (tie-heavy), flat: all H x W x 3."""
    img = np.load(os.path.join(HERE, "golden", "orb_golden.npz"))["image"][:H, :W]
    rng = np.random.default_rng(8214)
    blocky = np.kron(rng.integers(0, 256, (H // 8 + 1, W // 8 + 1, 3), dtype=np.uint8), np.ones((8, 8, 1), np.uint8))[:H, :W]
    flat = np.full((H, W, 3), 77, np.uint8)
    return np.stack([img, blocky, flat])


def _equals_oracle(gray, kp, desc, aux):
    want = of.detect_and_compute(gray)
    assert len(kp) == len(want["level"])
    if not len(kp):
        return
    scales = of.level_scales()
    lev = aux[:, 0].astype(int)
    s = np.array([scales[l] for l in lev], np.float32)
    gx, gy = np.rint(kp[:, 0] / s).astype(int), np.rint(kp[:, 1] / s).astype(int)
    got = {(l, a, b): (kp[i], aux[i, 1], aux[i, 2], aux[i, 3], desc[i]) for i, (l, a, b) in enumerate(zip(lev, gx, gy))}
    ref = {(int(l), int(a), int(b)): (want["pt"][i], want["angle"][i], want["response"][i], want["size"][i], want["desc"][i])
           for i, (l, a, b) in enumerate(zip(want["level"], want["xl"], want["yl"]))}
    assert set(got) == set(ref)
    for key, fields in ref.items():
        for a, b in zip(fields, got[key]):
            assert np.array_equal(np.asarray(a), np.asarray(b)), key
    assert np.array_equal(np.lexsort((gx, gy, lev)), np.arange(len(kp)))


@pytest.mark.parametrize("gray_in", [False, True])
def test_batch_equals_per_image_extract_and_the_oracle(emu, gray_in):
    bgr = _images(240, 416)
    grays = np.stack([of.bgr_to_gray(im) for im in bgr])
    images = grays if gray_in else bgr
    orb = Orb(emu, 240, 416)
    kp, desc, aux, cnt, launches = orb.batch(images)             # the first call grows the scratch from 1 image to 3
    assert launches == (16 if gray_in else 17)
    assert cnt[0, 0] > 300 and cnt[1, 0] > 0 and cnt[2, 0] == 0
    for s in range(3):
        k1, d1, a1, c1 = orb.extract(images[s])                   # per-image call on the grown scratch
        n = int(cnt[s, 0])
        assert np.array_equal(cnt[s], c1) and cnt[s, 1] == 0
        assert np.array_equal(kp[s, :n], k1) and np.array_equal(desc[s, :n], d1) and np.array_equal(aux[s, :n], a1)
        assert np.all(kp[s, n:] == -7) and np.all(desc[s, n:] == 0xA5) and np.all(aux[s, n:] == -7)
        _equals_oracle(grays[s], k1, d1, a1)
    one = orb.batch(images[1:2])                                  # S = 1: the same launches, the same rows
    assert one[4] == launches and np.array_equal(one[3][0], cnt[1])
    assert np.array_equal(one[1][0, :cnt[1, 0]], desc[1, :cnt[1, 0]])
    orb.close()


def test_short_output_keeps_the_prefix_and_flags_it(emu):
    images = _images(240, 416)
    orb = Orb(emu, 240, 416)
    full = orb.batch(images)
    rows = 200
    kp, desc, aux, cnt, launches = orb.batch(images, rows=rows)
    assert launches == 17
    for s in range(3):
        n = int(full[3][s, 0])
        assert cnt[s, 0] == min(n, rows) and cnt[s, 1] == (2 if n > rows else 0), (s, cnt[s], n)
        m = int(cnt[s, 0])
        assert np.array_equal(kp[s, :m], full[0][s, :m]) and np.array_equal(desc[s, :m], full[1][s, :m])
        assert np.array_equal(aux[s, :m], full[2][s, :m])
    assert cnt[0, 1] == 2 and cnt[2, 1] == 0
    orb.close()


def test_bad_arguments_enqueue_nothing(emu):
    images = _images(240, 416)
    orb = Orb(emu, 240, 416)
    for imgs, rows in ((images[:0], None), (images, 0)):
        assert orb.batch(imgs, rows=rows, expect_rc=-1)[4] == 0
    kp, cnt = np.zeros((1, 8, 2), np.float32), np.zeros((1, 2), np.int32)
    desc, aux = np.zeros((1, 8, 32), np.uint8), np.zeros((1, 8, 4), np.float32)
    for S, ch in ((65536, 3), (1, 2)):
        l0 = emu.emu_launches()
        assert emu.emu_orb_extract_batch(orb.h, _p(images), S, ch, 8, _p(kp), _p(desc), _p(aux), _p(cnt)) == -1
        assert emu.emu_launches() == l0
    orb.close()
