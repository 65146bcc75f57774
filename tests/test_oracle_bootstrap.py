"""Mode R bootstrap rows (vo_bootstrap; vo::draw_bootstrap in csrc/pnp_math.cuh): the integer recipe restated in numpy
(`bootstrap_ref`, which tests/test_gpu_pnp_ref_batch.py holds the device to bit for bit), the header built for the host against
it, and the properties of the stream it defines."""
import ctypes
import os
import subprocess

import numpy as np
import pytest

HEADER = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "visual-odometry-pipeline_b200", "csrc",
                      "pnp_math.cuh")

M64 = (1 << 64) - 1
GOLDEN_GAMMA = 0x9E3779B97F4A7C15      # pair key step, shared with the hypothesis generator (csrc/pnp_math.cuh draw_hypothesis)
DRAW_STEP = 0xD1B54A32D192ED03
BOOT_DOMAIN = 0xB0075742A9B5D0E1       # keeps the row keys apart from the hypothesis keys of the same (seed, pair)


def _mix64(z):
    """splitmix64's finaliser on uint64 numpy arrays (wrapping arithmetic)."""
    z = np.asarray(z, dtype=np.uint64)
    with np.errstate(over="ignore"):
        z = (z ^ (z >> np.uint64(30))) * np.uint64(0xBF58476D1CE4E5B9)
        z = (z ^ (z >> np.uint64(27))) * np.uint64(0x94D049BB133111EB)
        return z ^ (z >> np.uint64(31))


def bootstrap_ref(n, restarts, seed=8214, pair=0, cap=None):
    """int32 [restarts, cap] (cap defaults to n): entry (r, i) uniform in [0, n) for i < n, -1 for i >= n.
    key = mix64(seed + G (pair + 1)); row key = mix64(key ^ D ^ r); draw i: u = high word of mix64(row key + i C),
    value = (u * n) >> 32 (multiply-high: relative bias below n / 2^32)."""
    cap = max(int(n), 0) if cap is None else int(cap)
    out = np.full((int(restarts), cap), -1, np.int32)
    m = min(max(int(n), 0), cap)
    if m == 0:
        return out
    key = int(_mix64(np.uint64((int(seed) + GOLDEN_GAMMA * ((int(pair) + 1) & M64)) & M64)))
    i = np.arange(m, dtype=np.uint64)
    for r in range(int(restarts)):
        rk = int(_mix64(np.uint64(key ^ BOOT_DOMAIN ^ r)))
        with np.errstate(over="ignore"):
            z = _mix64(np.uint64(rk) + i * np.uint64(DRAW_STEP))
        u = z >> np.uint64(32)
        out[r, :m] = ((u * np.uint64(n)) >> np.uint64(32)).astype(np.int32)
    return out


def test_padding_is_minus_one_exactly_past_n():
    for n, cap in ((0, 16), (1, 16), (5, 5), (37, 64), (1000, 1024)):
        b = bootstrap_ref(n, 3, seed=5, pair=9, cap=cap)
        assert b.shape == (3, cap)
        assert np.all(b[:, n:] == -1)
        assert np.all(b[:, :n] >= 0)
    assert np.all(bootstrap_ref(-4, 2, cap=8) == -1)


@pytest.mark.parametrize("n", [1, 2, 5, 1000, 65536])
def test_values_stay_in_range(n):
    b = bootstrap_ref(n, 8, seed=8214, pair=3)
    assert b.min() >= 0 and b.max() < n
    if n == 1:
        assert np.all(b == 0)
    if n >= 1000:                                   # the draws reach both ends of the range
        assert b.min() < n // 100 and b.max() >= n - n // 100


def test_rows_depend_on_seed_pair_and_restart_only():
    a = bootstrap_ref(300, 3, seed=11, pair=40)
    assert np.array_equal(a, bootstrap_ref(300, 3, seed=11, pair=40))                 # deterministic
    assert np.array_equal(a, bootstrap_ref(300, 8, seed=11, pair=40)[:3])             # restart count does not matter
    assert np.array_equal(a, bootstrap_ref(300, 3, seed=11, pair=40, cap=512)[:, :300])  # nor does the row stride
    assert len({a[r].tobytes() for r in range(3)}) == 3                               # rows of one pair differ
    for other in (bootstrap_ref(300, 3, seed=12, pair=40), bootstrap_ref(300, 3, seed=11, pair=41),
                  bootstrap_ref(300, 3, seed=11, pair=-1)):
        assert (a != other).mean() > 0.9
    # the same 32-bit words at every n: a longer row extends a shorter one's word stream (values are rescaled, not redrawn)
    w1, w2 = bootstrap_ref(1 << 16, 1, cap=64), bootstrap_ref(1 << 8, 1, cap=64)
    assert np.array_equal(w1 >> 8, w2)


def test_uniform_at_n_1000():
    from scipy import stats
    n = 1000
    counts = np.zeros(n, np.int64)
    for pair in range(50):
        counts += np.bincount(bootstrap_ref(n, 8, seed=8214, pair=pair).ravel(), minlength=n)
    assert counts.sum() == 50 * 8 * n
    chi2 = float(((counts - 400.0) ** 2 / 400.0).sum())
    assert stats.chi2.sf(chi2, n - 1) > 1e-4, chi2
    assert stats.chi2.cdf(chi2, n - 1) > 1e-4, chi2      # not suspiciously flat either


@pytest.fixture(scope="module")
def header_rows(tmp_path_factory):
    """vo::draw_bootstrap of csrc/pnp_math.cuh (what bootstrap_kernel runs) built for the host."""
    d = tmp_path_factory.mktemp("boot_shim")
    src, so = d / "boot_shim.cpp", str(d / "libboot_shim.so")
    src.write_text(f'''#include "{HEADER}"
extern "C" void boot_rows(unsigned long long seed, long long pair, int restarts, int n, int cap, int *out) {{
    for (int r = 0; r < restarts; ++r)
        for (int i = 0; i < cap; ++i) out[r * cap + i] = i < n ? vo::draw_bootstrap(seed, pair, r, i, n) : -1;
}}
''')
    subprocess.check_call(["g++", "-O2", "-shared", "-fPIC", "-o", so, str(src)])
    lib = ctypes.CDLL(so)
    lib.boot_rows.argtypes = [ctypes.c_uint64, ctypes.c_int64, ctypes.c_int, ctypes.c_int, ctypes.c_int, ctypes.c_void_p]

    def rows(n, restarts, seed, pair, cap):
        out = np.empty((restarts, cap), np.int32)
        lib.boot_rows(seed, pair, restarts, n, cap, out.ctypes.data_as(ctypes.c_void_p))
        return out
    return rows


def test_device_header_equals_restatement(header_rows):
    for n, restarts, seed, pair, cap in ((1, 3, 8214, 0, 4), (5, 8, 8214, 7, 8), (1000, 3, 12345, 777, 1024),
                                         (65536, 2, 2 ** 63 + 5, -4, 65536), (2048, 1, 1, 2 ** 40, 2048), (0, 2, 3, 3, 16)):
        assert np.array_equal(header_rows(n, restarts, seed, pair, cap), bootstrap_ref(n, restarts, seed=seed, pair=pair, cap=cap))
