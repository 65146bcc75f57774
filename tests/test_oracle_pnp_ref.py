"""Reference-sampler PnP-RANSAC ("Mode R"): the CPU side of the parity chain.

1. oracle/pnp_ref.ransac_replica with cv2's own minimal solver reproduces cv2.solvePnPRansac — the call the reference makes
   (VisualOdometry_Stereo.py:129) — bit for bit: same inlier indices, same rvec / tvec.  This pins the sample table
   (OpenCV's MWC generator), the scoring arithmetic, the adaptive stopping rule and the refit.
2. csrc/pnp_ref_math.cuh, compiled for the host, equals the numpy restatement: identical tables, identical fp32 errors,
   identical scan decisions, EPnP poses to 1e-7 (two eigen-solvers: cyclic Jacobi vs LAPACK).
3. The restated EPnP and OpenCV's binary agree only statistically: OpenCV's five-point models hang on the arbitrary null-space
   basis of its SVD (documented by the numbers this test prints)."""
import ctypes
import os
import subprocess

import numpy as np
import pytest

HERE = os.path.dirname(os.path.abspath(__file__))


@pytest.fixture(scope="module")
def hm(tmp_path_factory):
    so = str(tmp_path_factory.mktemp("shim") / "libvo_host_math_ref_test.so")
    subprocess.check_call(["g++", "-O2", "-ffp-contract=off", "-shared", "-fPIC", "-o", so, os.path.join(HERE, "host_math_shim.cpp")])
    lib = ctypes.CDLL(so)
    lib.hm_ref_scan.argtypes = [ctypes.c_void_p, ctypes.c_int, ctypes.c_int, ctypes.c_double, ctypes.c_void_p, ctypes.c_void_p]
    return lib


def _p(a):
    return a.ctypes.data_as(ctypes.c_void_p)


def _scene(seed, n=900, outliers=0.35, noise=0.3, planar=False):
    import cv2
    from vo_b200 import synthetic
    rng = np.random.default_rng(seed)
    K = synthetic.KITTI_K
    X = np.stack([rng.uniform(-12, 12, n), rng.uniform(-3, 3, n), rng.uniform(4, 45, n)], 1).astype(np.float32)
    if planar:                                   # a fronto-parallel wall: the third principal direction vanishes exactly
        X[:, 0] *= 0.3
        X[:, 2] = 5.0
    R = cv2.Rodrigues(rng.normal(0, 0.01, 3))[0]
    t = np.array([rng.normal(0, 0.02), rng.normal(0, 0.01), -0.67])
    Xc = X.astype(np.float64) @ R.T + t
    uv = (Xc[:, :2] / Xc[:, 2:]) * [K[0, 0], K[1, 1]] + [K[0, 2], K[1, 2]] + rng.normal(0, noise, (n, 2))
    bad = rng.random(n) < outliers
    uv[bad] = np.stack([rng.uniform(0, 1241, bad.sum()), rng.uniform(0, 376, bad.sum())], 1)
    return X, uv.astype(np.float32), K


@pytest.mark.parametrize("seed,n,outliers,planar", [(1, 900, 0.35, False), (2, 300, 0.2, False), (3, 2000, 0.5, False), (4, 60, 0.1, False),
                                                    (5, 800, 0.2, True)])
def test_replica_with_cv_minimal_solver_equals_solvepnpransac(seed, n, outliers, planar):
    import cv2
    from oracle import pnp_ref
    X, uv, K = _scene(seed, n, outliers, planar=planar)
    ok, rv, tv, inl = cv2.solvePnPRansac(objectPoints=X, imagePoints=np.ascontiguousarray(uv).reshape(-1, 1, 2), cameraMatrix=K,
                                         distCoeffs=None, iterationsCount=100, reprojectionError=1.5)
    ok2, rv2, tv2, inl2, counts, poses, best, iters_run = pnp_ref.ransac_replica(X, uv, K, solver="cv")
    assert ok and ok2
    assert np.array_equal(inl.ravel(), inl2.ravel())
    assert np.abs(rv.ravel() - rv2.ravel()).max() < 1e-9 and np.abs(tv.ravel() - tv2.ravel()).max() < 1e-9
    assert 0 <= best < iters_run <= 100


def test_header_equals_numpy_restatement(hm):
    from oracle import pnp_ref
    for n in (5, 7, 60, 1500, 20000):
        got = np.zeros((100, 5), np.int32)
        hm.hm_ref_table(n, 100, _p(got))
        assert np.array_equal(got, pnp_ref.mwc_table(n, 100))
        assert all(len(set(r.tolist())) == 5 for r in got) and got.max() < n
    _header_vs_numpy_on_scene(hm, pnp_ref, *_scene(11, 1200, 0.3), tol=1e-6)
    # coplanar points (three effective control points): the weakest direction of the 9 x 9 block is poorly conditioned, the two
    # eigen-solvers agree to millimetres only — the same models for RANSAC's purposes (counts within a few percent)
    _header_vs_numpy_on_scene(hm, pnp_ref, *_scene(11, 1200, 0.3, planar=True), tol=2e-2)


def _header_vs_numpy_on_scene(hm, pnp_ref, X, uv, K, tol):
    kv = np.array([K[0, 0], K[1, 1], K[0, 2], K[1, 2]])
    tab = pnp_ref.mwc_table(len(X), 100)
    thr = np.float32(2.25)
    n_good = n_cmp = 0
    counts_h, counts_o = np.full(100, -1, np.int32), np.full(100, -1, np.int32)
    for h in range(100):
        s = tab[h]
        want = pnp_ref.epnp5(X[s], uv[s], K)
        out = np.zeros(12)
        ok = hm.hm_ref_epnp5(_p(np.ascontiguousarray(X[s].astype(np.float64))), _p(np.ascontiguousarray(uv[s].astype(np.float64))), _p(kv), _p(out))
        assert bool(ok) == (want is not None)
        if not ok:
            continue
        e_o = pnp_ref.reproj_err2(want[0], want[1], K, X, uv)
        e_h = np.zeros(len(X), np.float32)
        pose_o = np.concatenate([want[0].ravel(), want[1]])
        hm.hm_ref_err2(_p(pose_o), _p(kv), _p(np.ascontiguousarray(X)), _p(np.ascontiguousarray(uv)), len(X), _p(e_h))
        assert np.array_equal(e_h, e_o)                                   # scoring arithmetic: bit-identical on the same pose
        counts_o[h] = int((e_o <= thr).sum())
        e_hh = np.zeros(len(X), np.float32)
        hm.hm_ref_err2(_p(out), _p(kv), _p(np.ascontiguousarray(X)), _p(np.ascontiguousarray(uv)), len(X), _p(e_hh))
        counts_h[h] = int((e_hh <= thr).sum())
        if counts_o[h] > 0.3 * len(X):                                    # a usable model: the two eigen-solvers must agree closely
            n_good += 1
            d = max(np.abs(out[:9] - want[0].ravel()).max(), np.abs(out[9:] - want[1]).max())
            assert d < tol, (h, d)
            if tol <= 1e-6:
                straddle = np.abs(e_o - thr) < 1e-3
                assert np.array_equal((e_hh <= thr)[~straddle], (e_o <= thr)[~straddle])
            else:
                assert abs(int(counts_h[h]) - int(counts_o[h])) <= 0.05 * len(X)
            n_cmp += 1
    assert n_good >= 5 and n_cmp == n_good
    for c in (counts_o, counts_h, np.array([-1] * 100, np.int32), np.arange(100, dtype=np.int32) * 9 + 5):
        it_run, bc = ctypes.c_int(), ctypes.c_int()
        b = hm.hm_ref_scan(_p(np.ascontiguousarray(c, dtype=np.int32)), len(X), 100, 0.99, ctypes.byref(it_run), ctypes.byref(bc))
        assert (b, it_run.value, bc.value) == pnp_ref.ransac_scan(c, len(X), 100, 0.99)


def test_restated_epnp_is_statistically_not_bitwise_the_opencv_minimal_solver():
    """Same control flow, the two minimal solvers: winners differ in detail, inlier counts and refit poses agree to the
    reference's own noise floor (SURVEY 3.4: ~1e-3 m / 4e-5 rad when only the point order changes)."""
    import cv2
    from oracle import pnp_ref
    dt, dr, dn = [], [], []
    for seed in range(6):
        X, uv, K = _scene(100 + seed, 1200, 0.3)
        a = pnp_ref.ransac_replica(X, uv, K, solver="cv")
        b = pnp_ref.ransac_replica(X, uv, K, solver="epnp")
        assert a[0] and b[0]
        dt.append(np.abs(a[2].ravel() - b[2].ravel()).max())
        dr.append(np.abs(a[1].ravel() - b[1].ravel()).max())
        dn.append(abs(len(a[3]) - len(b[3])) / len(a[3]))
    print("refit pose difference, cv2 minimal solver vs restated EPnP: dt", np.round(dt, 5), "drvec", np.round(dr, 6), "d#inl", np.round(dn, 3))
    assert max(dt) < 2e-2 and max(dr) < 2e-3 and max(dn) < 0.25


def test_parallel_order_jacobi_is_an_eigen_decomposition(hm):
    """refpnp::jacobi_eig12_rr (rounds of six rotations on disjoint pairs, the order the GPU's warp-wide form runs) on matrices
    shaped like EPnP's M^T M (symmetric positive semi-definite, rank 10, entries spanning many orders of magnitude): eigenvalues
    equal numpy's and the cyclic-by-row order's to round-off, V is orthonormal, A V = V diag(d), and every pair of indices meets
    exactly once per sweep."""
    rng = np.random.default_rng(5)
    for trial in range(20):
        M = rng.standard_normal((10, 12)) * np.exp(rng.uniform(-6, 6, (1, 12)))
        A = M.T @ M
        V, d = np.zeros((12, 12)), np.zeros(12)
        hm.hm_jacobi12(_p(np.ascontiguousarray(A)), 1, _p(V), _p(d))
        Vc, dc = np.zeros((12, 12)), np.zeros(12)
        hm.hm_jacobi12(_p(np.ascontiguousarray(A)), 0, _p(Vc), _p(dc))
        w = np.linalg.eigvalsh(A)[::-1]
        scale = w[0]
        assert np.all(np.diff(d) <= 0)
        assert np.abs(d - w).max() < 1e-12 * scale and np.abs(d - dc).max() < 1e-12 * scale
        assert np.abs(V.T @ V - np.eye(12)).max() < 1e-13
        assert np.abs(A @ V - V * d).max() < 1e-12 * scale
        # the null space (two zero eigenvalues) is spanned by the same vectors in both orders
        Pn, Pc = V[:, 10:] @ V[:, 10:].T, Vc[:, 10:] @ Vc[:, 10:].T
        assert np.abs(Pn - Pc).max() < 1e-6
    seen = set()
    for r in range(11):                                     # the tournament schedule of jacobi12_pair
        rnd = [(11, r)] + [((r + k) % 11, (r + 11 - k) % 11) for k in range(1, 6)]
        assert len({i for pq in rnd for i in pq}) == 12      # six disjoint pairs
        seen |= {tuple(sorted(pq)) for pq in rnd}
    assert len(seen) == 66
