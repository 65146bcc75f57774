"""csrc/sift.cu — kernels and launch sequence — executed on the host through tests/cuda_emu.h and compared with the CPU
restatement (oracle/sift_frontend.py, itself pinned to OpenCV within a tolerance).  Same tolerance as there: the
kernels use plain fp32 (device expf / powf / atan polynomial), not OpenCV's operation order."""
import ctypes
import os
import subprocess

import numpy as np
import pytest

from oracle import sift_frontend as sf
from test_oracle_sift import _check

HERE = os.path.dirname(os.path.abspath(__file__))
CAP = 20000


@pytest.fixture(scope="module")
def emu(tmp_path_factory):
    so = str(tmp_path_factory.mktemp("shim") / "libvo_sift_emu_test.so")
    subprocess.check_call(["g++", "-x", "c++", "-std=c++17", "-O2", "-ffp-contract=off", "-pthread", "-Wno-unknown-pragmas",
                           "-Wno-subobject-linkage", "-shared", "-fPIC", '-DVO_HOST_EMU="cuda_emu.h"', "-I", HERE, "-o", so,
                           os.path.join(HERE, "sift_emu_shim.cpp")])
    lib = ctypes.CDLL(so)
    lib.emu_last_error.restype = ctypes.c_char_p
    return lib


def _run(emu, image):
    image = np.ascontiguousarray(image)
    H, W = image.shape[:2]
    kp = np.zeros((CAP, 2), np.float32)
    desc = np.zeros((CAP, 128), np.float32)
    aux = np.zeros((CAP, 4), np.float32)
    cnt = np.zeros(2, np.int32)
    p = lambda a: a.ctypes.data_as(ctypes.c_void_p)
    n = emu.emu_sift_run(p(image), H, W, 1 if image.ndim == 2 else 3, CAP, p(kp), p(desc), p(aux), p(cnt))
    assert n >= 0, (n, emu.emu_last_error())
    assert cnt[1] <= CAP
    return {"pt": kp[:n], "size": aux[:n, 0], "angle": aux[:n, 1], "response": aux[:n, 2], "octave": aux[:n, 3].astype(np.int64),
            "desc": desc[:n]}


def test_emulated_sift_matches_the_oracle_and_the_reference_plugin(emu, golden):
    g = golden("sift_golden.npz")
    got = _run(emu, g["image"])                                             # BGR in
    want = sf.detect_and_compute(sf.bgr_to_gray(g["image"]))
    assert _check(want, got) >= 480                                         # kernels vs restatement
    ref = {"pt": g["kp"].astype(np.float32), "size": g["size"], "angle": g["angle"], "desc": g["desc"]}
    assert _check(ref, got) >= 480                                          # kernels vs the reference's own plug-in
    assert np.all(np.diff(got["pt"][:, 0]) >= 0)                            # OpenCV's order: sorted by x first
    assert np.array_equal(got["octave"], want["octave"][:len(got["octave"])]) or len(got["octave"]) != len(want["octave"])


def test_emulated_sift_edge_cases(emu):
    rng = np.random.default_rng(5)
    assert _check(sf.detect_and_compute(n := rng.integers(0, 256, (120, 160), dtype=np.uint8)), _run(emu, n)) > 50
    flat = np.full((64, 80), 77, np.uint8)
    assert len(_run(emu, flat)["size"]) == 0 == len(sf.detect_and_compute(flat)["size"])
    tiny = rng.integers(0, 256, (17, 23), dtype=np.uint8)                   # fewer octaves, every layer near the border
    assert abs(len(_run(emu, tiny)["size"]) - len(sf.detect_and_compute(tiny)["size"])) <= 1


def test_emulated_sift_kitti_shaped_frame(emu):
    from test_gpu_sift_frontend import _kitti_like
    img = _kitti_like()
    assert _check(sf.detect_and_compute(img), _run(emu, img)) > 500
