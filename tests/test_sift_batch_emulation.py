"""vo_sift_extract_batch — kernels and launch sequence of csrc/sift.cu — executed on the host through tests/cuda_emu.h: S
images in one call equal the per-image call (vo_sift_extract) on each image, bit for bit; a short output keeps the prefix
and sets flag bit 1; a raw list past max_keypoints sets flag bit 0; the launch count does not depend on S, also after the
scratch has grown; bad arguments launch nothing.  The emulator spends seconds per small image, so the file makes few
calls.  The device half is tests/test_gpu_sift_batch.py."""
import ctypes
import os
import subprocess

import numpy as np
import pytest

from oracle import orb_frontend as of

HERE = os.path.dirname(os.path.abspath(__file__))
H, W = 72, 96


@pytest.fixture(scope="module")
def emu(tmp_path_factory):
    so = str(tmp_path_factory.mktemp("shim") / "libvo_sift_batch_emu_test.so")
    # -fno-gnu-unique: the emulator's inline launch counter must not be merged with that of another shim's library when
    # both are loaded in one process
    subprocess.check_call(["g++", "-x", "c++", "-std=c++17", "-O2", "-ffp-contract=off", "-fno-gnu-unique", "-pthread",
                           "-Wno-unknown-pragmas", "-Wno-subobject-linkage", "-shared", "-fPIC", '-DVO_HOST_EMU="cuda_emu.h"',
                           "-I", HERE, "-o", so, os.path.join(HERE, "sift_batch_emu_shim.cpp")])
    lib = ctypes.CDLL(so)
    lib.emu_last_error.restype = ctypes.c_char_p
    lib.emu_launches.restype = ctypes.c_longlong
    lib.emu_sift_create.restype = ctypes.c_void_p
    lib.emu_sift_create.argtypes = [ctypes.c_int] * 3
    return lib


def _p(a):
    return a.ctypes.data_as(ctypes.c_void_p)


class Sift:
    def __init__(self, emu, cap):
        self.emu, self.cap = emu, cap
        self.h = ctypes.c_void_p(emu.emu_sift_create(H, W, cap))
        assert self.h.value, emu.emu_last_error()

    def extract(self, image):
        image = np.ascontiguousarray(image)
        kp, desc = np.zeros((self.cap, 2), np.float32), np.zeros((self.cap, 128), np.float32)
        aux, cnt = np.zeros((self.cap, 4), np.float32), np.zeros(2, np.int32)
        l0 = self.emu.emu_launches()
        rc = self.emu.emu_sift_extract(self.h, _p(image), 1 if image.ndim == 2 else 3, _p(kp), _p(desc), _p(aux), _p(cnt))
        assert rc == 0, self.emu.emu_last_error()
        n = int(cnt[0])
        return kp[:n], desc[:n], aux[:n], cnt, self.emu.emu_launches() - l0

    def batch(self, images, rows=None, expect_rc=0):
        images = np.ascontiguousarray(images)
        S, rows = images.shape[0], self.cap if rows is None else rows
        # sentinel fill: rows past the count must stay untouched
        kp = np.full((max(S, 1), max(rows, 1), 2), -7, np.float32)
        desc = np.full((max(S, 1), max(rows, 1), 128), -7, np.float32)
        aux = np.full((max(S, 1), max(rows, 1), 4), -7, np.float32)
        cnt = np.full((max(S, 1), 2), -1, np.int32)
        l0 = self.emu.emu_launches()
        rc = self.emu.emu_sift_extract_batch(self.h, _p(images), S, 3 if images.ndim == 4 else 1, rows, _p(kp), _p(desc),
                                             _p(aux), _p(cnt))
        assert rc == expect_rc, (rc, self.emu.emu_last_error())
        return kp, desc, aux, cnt, self.emu.emu_launches() - l0

    def close(self):
        self.emu.emu_sift_destroy(self.h)


def _images():
    """BGR: noise, flat, smooth gradient with a little noise (H x W x 3 each)."""
    rng = np.random.default_rng(11)
    noise = rng.integers(0, 256, (H, W, 3), dtype=np.uint8)
    flat = np.full((H, W, 3), 77, np.uint8)
    yy, xx = np.mgrid[:H, :W]
    grad = np.repeat(((xx * 2 + yy + rng.integers(0, 30, (H, W))) % 256).astype(np.uint8)[:, :, None], 3, 2)
    return np.stack([noise, flat, grad])


def test_batch_equals_per_image_extract_and_short_rows_keep_the_prefix(emu):
    bgr = _images()
    sift = Sift(emu, 4000)
    kp, desc, aux, cnt, launches = sift.batch(bgr)              # the first call grows the scratch from 1 image to 3
    assert cnt[0, 0] > 20 and cnt[1, 0] == 0, cnt
    one = []
    for s in range(3):
        k1, d1, a1, c1, l1 = sift.extract(bgr[s])               # per-image call on the grown scratch
        assert l1 == launches
        n = int(cnt[s, 0])
        assert n == c1[0] and cnt[s, 1] == 0 and c1[1] <= sift.cap, (s, cnt[s], c1)
        assert np.array_equal(kp[s, :n], k1) and np.array_equal(desc[s, :n], d1) and np.array_equal(aux[s, :n], a1), s
        assert np.all(kp[s, n:] == -7) and np.all(desc[s, n:] == -7) and np.all(aux[s, n:] == -7)
        one.append((k1, d1, a1))
    # back to S = 1, gray in: the gray conversion is the kernels' own, so the rows are those of the BGR image
    rows = int(cnt[0, 0]) // 2
    kp, desc, aux, c, l1 = sift.batch(of.bgr_to_gray(bgr[0])[None], rows=rows)
    assert l1 == launches
    assert c[0, 0] == rows and c[0, 1] == 2, c
    assert np.array_equal(kp[0], one[0][0][:rows]) and np.array_equal(desc[0], one[0][1][:rows])
    assert np.array_equal(aux[0], one[0][2][:rows])
    sift.close()


def test_raw_list_past_max_keypoints_sets_flag_bit_0(emu):
    sift = Sift(emu, 8)
    noise = _images()[0]
    _, _, _, c1, _ = sift.extract(noise)
    assert c1[1] > sift.cap and c1[0] <= sift.cap, c1           # where SiftExtractor.extract raises
    kp, desc, aux, cnt, _ = sift.batch(noise[None], rows=4)
    assert cnt[0, 0] == min(int(c1[0]), 4) and cnt[0, 1] == (1 | (2 if c1[0] > 4 else 0)), (cnt, c1)
    assert np.all(kp[0, :cnt[0, 0]] >= 0) and np.all((desc[0, :cnt[0, 0]] >= 0) & (desc[0, :cnt[0, 0]] <= 255))
    sift.close()


def test_bad_arguments_launch_nothing(emu):
    images = _images()
    sift = Sift(emu, 64)
    for imgs, rows in ((images[:0], None), (images, 0)):
        assert sift.batch(imgs, rows=rows, expect_rc=-1)[4] == 0
    kp, cnt = np.zeros((1, 8, 2), np.float32), np.zeros((1, 2), np.int32)
    desc, aux = np.zeros((1, 8, 128), np.float32), np.zeros((1, 8, 4), np.float32)
    for S, ch, p_img in ((65536, 3, _p(images)), (1, 2, _p(images)), (1, 3, None)):
        l0 = emu.emu_launches()
        assert emu.emu_sift_extract_batch(sift.h, p_img, S, ch, 8, _p(kp), _p(desc), _p(aux), _p(cnt)) == -1
        assert emu.emu_launches() == l0
    sift.close()
