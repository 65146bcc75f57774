"""The fp64 matcher reference (oracle/match64.py) against the fp32 CPU oracle, and its certifier against hand-made
defects: every defect must be rejected, so a GPU result that certifies cannot carry it."""
import numpy as np
import pytest

from oracle import match64 as m64

PAD = 3       # padding rows / columns behind the valid ones, like a ragged batch slot


def _sift(seed, n, m):
    from vo_b200 import synthetic
    p = synthetic.make_pair(seed, n_kp=max(n, 8), n_cur=max(m, 8), kind="sift")
    return p["ref_desc"][:n].copy(), p["cur_desc"][:m].copy()


def _r2d2(seed, n, m):
    from vo_b200 import synthetic
    p = synthetic.make_pair(seed, n_kp=max(n, 8), n_cur=max(m, 8), kind="r2d2")
    return p["ref_desc"][:n].copy(), p["cur_desc"][:m].copy()


def _rootsift(seed, n, m):
    ref, cur = _sift(seed, n, m)
    f = lambda x: np.sqrt(x / np.maximum(x.sum(1, keepdims=True), 1)).astype(np.float32)  # noqa: E731
    return f(ref), f(cur)


def _fp32_output(orc, ref, cur, metric, mode, param):
    """what vo_match_f32 returns for one pair, computed by the fp32 CPU oracle, with PAD padding rows and columns"""
    ridx, rval, cidx = orc.knn_f32(ref, cur, metric)
    pairs, dist = orc.accept(ridx, rval, cidx, mode, param, metric)
    nt = m64._near_tie(metric, rval[:, 0], rval[:, 1], ridx[:, 1] >= 0).astype(np.uint8)
    return dict(knn_idx=np.concatenate([ridx, np.full((PAD, 2), -1, np.int32)]),
                knn_val=np.concatenate([rval, np.zeros((PAD, 2), np.float32)]),
                col_idx=np.concatenate([cidx, np.full(PAD, -1, np.int32)]),
                pairs=pairs, dist=dist, near_tie=np.concatenate([nt, np.zeros(PAD, np.uint8)]))


@pytest.mark.parametrize("n,m", [(300, 280), (1, 50), (50, 1), (40, 2), (0, 10), (10, 0), (700, 650)])
def test_knn64_equals_fp32_oracle_on_integer_data_with_planted_ties(orc, n, m):
    ref, cur = _sift(n * 7 + m, n, m)
    if m >= 250:
        cur[200], cur[130], cur[247] = cur[17], cur[17], cur[17]   # a column tie: the lowest index comes first
        cur[129] = cur[201]
        ref[5] = cur[17]
    if n >= 250:
        ref[211], ref[140] = ref[9], ref[9]                        # a row tie in every column: the lowest row wins
    r = m64.knn64(ref, cur, m64.METRIC_L2)
    assert r.is_int
    want = orc.knn_f32(ref, cur, orc.METRIC_L2)
    got = m64.knn64_as_f32(r)
    for g, w in zip(got, want):
        assert g.dtype == w.dtype and np.array_equal(g, w)
    if m >= 250:      # the planted duplicates really produce ties the reference resolves to the lowest index
        rows = np.nonzero(r.row_idx[:, 0] == 17)[0]
        assert len(rows) and all(r.row_idx[rows, 1] == 130)


_COMMON_MODES = [(m64.MODE_RATIO, 0.85), (m64.MODE_MUTUAL, 0.0), (m64.MODE_RATIO_MUTUAL, 0.9), (m64.MODE_NN, 0.0)]


@pytest.mark.parametrize("family,metric,mode,param",
                         [("r2d2", m64.METRIC_COSINE, md, p) for md, p in
                          _COMMON_MODES + [(m64.MODE_THRESH_MUTUAL, 0.9), (m64.MODE_THRESH, 0.7)]] +
                         [(f, m64.METRIC_L2, md, p) for f in ("rootsift", "sift") for md, p in _COMMON_MODES])
def test_certify_accepts_the_fp32_oracle(orc, family, metric, mode, param):
    ref, cur = {"r2d2": _r2d2, "rootsift": _rootsift, "sift": _sift}[family](5, 600, 550)
    r = m64.knn64(ref, cur, metric)
    gamma = m64.eps(m64.PREC_TF32X3, r)
    assert (gamma == 0) == (family == "sift")
    rep = m64.certify(_fp32_output(orc, ref, cur, metric, mode, param), r, gamma, mode, param)
    assert rep["rows"] == 600 and rep["max_err_ratio"] < 1


def test_eps_model():
    ref, cur = _r2d2(1, 20, 20)
    r = m64.knn64(ref, cur, m64.METRIC_COSINE)
    assert m64.eps(m64.PREC_F16X3, r) == m64.eps(m64.PREC_FP32_SIMT, r) == 2.0 ** -18
    for prec in (m64.PREC_TF32X1, m64.PREC_F16X1):
        with pytest.raises(ValueError):
            m64.eps(prec, r)
    ref, cur = _sift(1, 20, 20)
    r = m64.knn64(ref, cur, m64.METRIC_L2)
    assert all(m64.eps(p, r) == 0.0 for p in range(5))
    assert not m64.knn64(ref + 0.5, cur, m64.METRIC_L2).is_int
    assert not m64.knn64(ref * 2, cur, m64.METRIC_L2).is_int          # values past 255


# ------------------------------------------------------------------------------------------------ planted defects
@pytest.fixture(scope="module")
def real_case():
    """R2D2-like pair plus one near-duplicate column: row 0's best and second best 1e-7 apart (inside eps)"""
    from oracle import oracle as orc
    orc.build()
    ref, cur = _r2d2(11, 400, 380)
    ref[0] = cur[3] + 0.06 * np.random.default_rng(0).standard_normal(128).astype(np.float32)
    cur[300] = cur[3] + np.float32(2e-7) * np.sign(cur[3]) * (np.arange(128) % 2)
    cur[300] /= np.linalg.norm(cur[300])
    r = m64.knn64(ref, cur, m64.METRIC_COSINE)
    return orc, ref, cur, r


def _certain_row(r, out):
    """a row with a wide fp64 margin between its 1st, 2nd and 3rd best that the oracle accepted"""
    S = r.a @ r.b.T
    srt = -np.sort(-S, axis=1)
    margin = np.minimum(srt[:, 0] - srt[:, 1], srt[:, 1] - srt[:, 2])
    kept = np.zeros(r.N, bool)
    kept[out["pairs"][:, 0]] = True
    cand = np.nonzero((margin > 1e-2) & kept)[0]
    assert len(cand)
    return int(cand[0]), S


def _rejects(out, r, gamma, mode, param, match):
    with pytest.raises(m64.CertifyError, match=match):
        m64.certify(out, r, gamma, mode, param)


def test_certify_passes_the_undamaged_real_case(real_case):
    orc, ref, cur, r = real_case
    out = _fp32_output(orc, ref, cur, m64.METRIC_COSINE, m64.MODE_RATIO_MUTUAL, 0.9)
    m64.certify(out, r, 2.0 ** -18, m64.MODE_RATIO_MUTUAL, 0.9)


def test_certify_rejects_swapped_i1_i2(real_case):
    orc, ref, cur, r = real_case
    out = _fp32_output(orc, ref, cur, m64.METRIC_COSINE, m64.MODE_NN, 0.0)
    row, _ = _certain_row(r, out)
    out["knn_idx"][row] = out["knn_idx"][row, ::-1]
    out["knn_val"][row] = out["knn_val"][row, ::-1]
    _rejects(out, r, 2.0 ** -18, m64.MODE_NN, 0.0, "i1 is not optimal")


def test_certify_rejects_third_best_as_second(real_case):
    orc, ref, cur, r = real_case
    out = _fp32_output(orc, ref, cur, m64.METRIC_COSINE, m64.MODE_NN, 0.0)
    row, S = _certain_row(r, out)
    third = int(np.argsort(-S[row], kind="stable")[2])
    out["knn_idx"][row, 1] = third
    out["knn_val"][row, 1] = np.float32(S[row, third])
    _rejects(out, r, 2.0 ** -18, m64.MODE_NN, 0.0, "i2 is not the best of the rest")


def test_certify_rejects_a_tie_broken_to_the_higher_index(orc):
    ref, cur = _sift(21, 300, 280)
    row = 5
    j = int(orc.knn_f32(ref, cur, orc.METRIC_L2)[0][row, 0])
    dup = 279 if j != 279 else 0
    cur[dup] = cur[j]                                      # exact duplicate of row 5's best
    r = m64.knn64(ref, cur, m64.METRIC_L2)
    out = _fp32_output(orc, ref, cur, m64.METRIC_L2, m64.MODE_RATIO, 0.85)
    assert tuple(out["knn_idx"][row]) == tuple(sorted((j, dup))) and out["knn_val"][row, 0] == out["knn_val"][row, 1]
    m64.certify(out, r, 0.0, m64.MODE_RATIO, 0.85)
    out["knn_idx"][row] = out["knn_idx"][row, ::-1]
    _rejects(out, r, 0.0, m64.MODE_RATIO, 0.85, "i1 is not the exact fp64 neighbour")


def test_certify_rejects_a_value_off_by_4_eps(real_case):
    orc, ref, cur, r = real_case
    out = _fp32_output(orc, ref, cur, m64.METRIC_COSINE, m64.MODE_NN, 0.0)
    row, _ = _certain_row(r, out)
    e = 2.0 ** -18 * r.sigma([row], [out["knn_idx"][row, 0]])[0]
    out["knn_val"][row, 0] = np.float32(r.score([row], [out["knn_idx"][row, 0]])[0] + 4 * e)
    k = int(np.nonzero(out["pairs"][:, 0] == row)[0][0])
    out["dist"][k] = m64._dist(m64.METRIC_COSINE, out["knn_val"][row, 0])
    _rejects(out, r, 2.0 ** -18, m64.MODE_NN, 0.0, "off by more than eps")


def test_certify_rejects_a_flipped_acceptance(real_case):
    orc, ref, cur, r = real_case
    out = _fp32_output(orc, ref, cur, m64.METRIC_COSINE, m64.MODE_RATIO_MUTUAL, 0.9)
    row, _ = _certain_row(r, out)
    keep = out["pairs"][:, 0] != row
    out["pairs"], out["dist"] = out["pairs"][keep], out["dist"][keep]
    _rejects(out, r, 2.0 ** -18, m64.MODE_RATIO_MUTUAL, 0.9, "acceptance")
    # the same flip with the k-NN outputs made consistent with it is still caught against fp64
    out["col_idx"][out["knn_idx"][row, 0]] = (row + 1) % r.N
    _rejects(out, r, 2.0 ** -18, m64.MODE_RATIO_MUTUAL, 0.9, "col_idx|acceptance")


def test_certify_rejects_a_missing_near_tie_flag(real_case):
    orc, ref, cur, r = real_case
    out = _fp32_output(orc, ref, cur, m64.METRIC_COSINE, m64.MODE_RATIO, 0.85)
    assert set(out["knn_idx"][0]) == {3, 300} and r.row_idx[0, 0] in (3, 300)
    m64.certify(out, r, 2.0 ** -18, m64.MODE_RATIO, 0.85)
    if out["knn_idx"][0, 0] == r.row_idx[0, 0]:               # make i1 disagree with fp64 (allowed: inside eps)
        out["knn_idx"][0] = out["knn_idx"][0, ::-1]
        out["knn_val"][0] = out["knn_val"][0, ::-1]
    assert out["near_tie"][0] == 1
    m64.certify(out, r, 2.0 ** -18, m64.MODE_RATIO, 0.85)
    out["near_tie"][0] = 0
    _rejects(out, r, 2.0 ** -18, m64.MODE_RATIO, 0.85, "does not carry near_tie")


def test_certify_rejects_a_wrong_near_tie_on_integer_data(orc):
    ref, cur = _sift(23, 300, 280)
    out = _fp32_output(orc, ref, cur, m64.METRIC_L2, m64.MODE_RATIO, 0.85)
    r = m64.knn64(ref, cur, m64.METRIC_L2)
    row = int(np.nonzero(out["near_tie"][:300] == 0)[0][0])
    out["near_tie"][row] = 1
    _rejects(out, r, 0.0, m64.MODE_RATIO, 0.85, "near_tie differs")


def test_certify_rejects_matches_to_padding(real_case):
    orc, ref, cur, r = real_case
    gamma = 2.0 ** -18
    base = _fp32_output(orc, ref, cur, m64.METRIC_COSINE, m64.MODE_NN, 0.0)
    out = {k: v.copy() for k, v in base.items()}
    out["pairs"] = np.concatenate([out["pairs"], [[r.N, 0]]])            # a padding row accepted
    out["dist"] = np.concatenate([out["dist"], [0.5]]).astype(np.float32)
    _rejects(out, r, gamma, m64.MODE_NN, 0.0, "padding row")
    out = {k: v.copy() for k, v in base.items()}
    out["knn_idx"][7, 1] = r.M                                            # a padding column as second best
    _rejects(out, r, gamma, m64.MODE_NN, 0.0, "i2 validity")
    out = {k: v.copy() for k, v in base.items()}
    out["col_idx"][r.M + 1] = 4                                           # a padding column with a neighbour
    _rejects(out, r, gamma, m64.MODE_NN, 0.0, "padding column")
    out = {k: v.copy() for k, v in base.items()}
    out["near_tie"][r.N] = 1
    _rejects(out, r, gamma, m64.MODE_NN, 0.0, "padding row")


def test_certify_rejects_a_loose_eps(orc):
    """non-vacuity: an eps wide enough to excuse anything leaves most rows uncertain, and that is an error"""
    ref, cur = _r2d2(31, 400, 380)
    r = m64.knn64(ref, cur, m64.METRIC_COSINE)
    out = _fp32_output(orc, ref, cur, m64.METRIC_COSINE, m64.MODE_RATIO_MUTUAL, 0.9)
    _rejects(out, r, 0.5, m64.MODE_RATIO_MUTUAL, 0.9, "too many uncertain rows")
