"""vo_match_f32 certified against the fp64 reference (oracle/match64.py) at every precision, at tile, split and
finalize-chunk edges, on exact ties and on ragged batches.

Every call is checked in full: the row top-2 (indices and values), the column arg-best, near_tie, the accepted pairs
and their distances.  Integer-valued data (|x| <= 255) must match fp64 exactly at every precision; real-valued data
must stay inside eps = 2^-18 * sigma (see match64.eps) and leave at most 0.5 % of the rows uncertain.

Kernel paths the shapes reach (pick_split in api.cu, launch_tc / match_f32_tc in match_f32_tc.cu; B200, 148 SMs):
  * column tiles: 128 (TF32X3, F16X3), 160 (TF32X1), 192 (F16X1), 64 (FP32_SIMT); each tile is read as four column
    quarters (32 / 40 / 48 columns), so m in {127..129, 159..161, 191..193, 383, 385} crosses a tile or a quarter;
  * row blocks of 128 and clusters of two blocks (256 rows): n in {127..129, 255..257, 511, 513, 2049};
  * n_split = ceil(296 / (B * row-block pairs * 2)), at most col_tiles / 4 and 64: (1, 40000) gives 64 splits on the
    128-column passes (313 tiles), (129, 33000) 37;
  * F16X1 runs its persistent form when a work item has <= 64 column tiles and the plain form above that
    (VO_TC_PERSIST forces either); a column arg-min (mutual rules, col_idx) moves F16X1 to the TF32X1 kernel;
  * F16X3 with the column side interleaves the row blocks of up to 8 pairs and filters columns against colkey
    (VO_TC_NO_INTERLEAVE turns that off);
  * finalize uses 2048-row chunks and the pack kernel once B * ceil(n / 2048) >= 148: B = 74 pairs of 2049 rows.
"""
import collections
import importlib
import os

import numpy as np
import pytest

from oracle import match64 as m64

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
TF32X3, TF32X1, SIMT, F16X1, F16X3 = range(5)
PREC_NAME = {TF32X3: "TF32X3", TF32X1: "TF32X1", SIMT: "FP32_SIMT", F16X1: "F16X1", F16X3: "F16X3"}
L2, COS = m64.METRIC_L2, m64.METRIC_COSINE
RATIO, MUTUAL, RATIO_MUTUAL, THRESH_MUTUAL, THRESH, NN = range(6)
ALL_PRECS = (TF32X3, TF32X1, SIMT, F16X1, F16X3)
SPLIT_PRECS = (TF32X3, F16X3, SIMT)

REPORT = collections.defaultdict(lambda: [0.0, 0, 0, 0])     # (family, precision) -> max err/eps, uncertain, rows, calls


def _gpu(a):
    import torch
    return torch.from_numpy(np.ascontiguousarray(a)).cuda()


@pytest.fixture(scope="module", autouse=True)
def _report():
    yield
    print("\ncertify report (family, precision): max |err|/eps, uncertain rows / certified rows, calls")
    for (fam, prec), (ratio, unc, rows, calls) in sorted(REPORT.items()):
        print(f"  {fam:9s} {PREC_NAME[prec]:9s} {ratio:8.4f}   {unc:5d} / {rows:8d}   {calls}")


# ------------------------------------------------------------------------------------------------ data families
def _sift_int(seed, n, m):
    from vo_b200 import synthetic
    rng = np.random.default_rng(seed)
    ref, cur = synthetic._descriptors(rng, "sift", int(0.8 * min(n, m)), n, m)
    return ref, cur


def _r2d2(seed, n, m):
    from vo_b200 import synthetic
    rng = np.random.default_rng(seed)
    return synthetic._descriptors(rng, "r2d2", int(0.8 * min(n, m)), n, m)


def _rootsift(seed, n, m):
    f = lambda x: np.sqrt(x / np.maximum(x.sum(1, keepdims=True), 1)).astype(np.float32)  # noqa: E731
    ref, cur = _sift_int(seed, n, m)
    return f(ref), f(cur)


def _wide(seed, n, m):
    """real values in [-255, 255]: R2D2-like directions at per-row scales, with exact +-255 and 254.99 planted"""
    rng = np.random.default_rng(seed)
    ref, cur = _r2d2(seed, n, m)
    out = []
    for x in (ref, cur):
        x = x / np.abs(x).max(1, keepdims=True) * rng.uniform(60, 255, (len(x), 1))
        x = np.clip(x, -255, 255).astype(np.float32)
        k = np.arange(len(x))
        x[k, k % 128] = np.where(k % 3 == 0, 255.0, np.where(k % 3 == 1, -255.0, 254.99)).astype(np.float32)
        out.append(x)
    return out


FAMILIES = {"sift_int": (_sift_int, L2), "r2d2": (_r2d2, COS), "rootsift": (_rootsift, L2), "wide_l2": (_wide, L2),
            "wide_cos": (_wide, COS)}
_CACHE = {}


def _case(family, n, m, seed=None):
    """(ref, cur, knn64) of one frame pair, cached for the module"""
    key = (family, n, m, seed)
    if key not in _CACHE:
        make, metric = FAMILIES[family]
        ref, cur = make(seed if seed is not None else 1000 + 7 * n + m, n, m)
        _CACHE[key] = (ref, cur, m64.knn64(ref, cur, metric))
    return _CACHE[key]


def _run(ref, cur, metric, mode, param, prec, rows_only=False, n_ref=None, n_cur=None):
    from vo_b200 import ops
    return ops.match_f32(_gpu(ref), _gpu(cur), metric, mode, param, precision=prec, n_ref=n_ref, n_cur=n_cur,
                         want_knn="rows" if rows_only else True, want_near_tie=True)


def _certify(family, res, refs, prec, mode, param):
    gamma = m64.eps(prec, refs[0])
    rep = m64.certify_batch(res, refs, gamma, mode, param)
    r = REPORT[(family, prec)]
    r[0], r[1], r[2], r[3] = max(r[0], rep["max_err_ratio"]), r[1] + rep["uncertain"], r[2] + rep["rows"], r[3] + 1
    return rep


def _check(family, n, m, prec, modes):
    ref, cur, r64 = _case(family, n, m)
    metric = FAMILIES[family][1]
    for mode, param in modes:
        # the F16X1 kernel itself runs only without a column arg-min (the row top-2 is then all the k-NN output)
        rows_only = prec == F16X1 and mode in (RATIO, NN, THRESH)
        res = _run(ref, cur, metric, mode, param, prec, rows_only=rows_only)
        try:
            _certify(family, res, [r64], prec, mode, param)
        except m64.CertifyError as e:
            raise AssertionError(f"{family} n={n} m={m} {PREC_NAME[prec]} mode={mode} param={param}: {e}") from None


# ------------------------------------------------------------------------------------------------ shapes
SIFT_SHAPES = [(1, 1), (2, 2), (1, 300), (300, 1), (127, 129), (128, 128), (129, 127), (255, 159), (256, 160),
               (257, 161), (511, 191), (513, 192), (129, 193), (2049, 383), (257, 385), (511, 8193), (257, 12289),
               (129, 33000), (1, 40000)]
SIFT_MODES = [(RATIO, 0.85), (MUTUAL, 0.0), (NN, 0.0)]


@pytest.mark.parametrize("prec", ALL_PRECS, ids=PREC_NAME.get)
@pytest.mark.parametrize("n,m", SIFT_SHAPES)
def test_sift_int_exact_at_every_precision(prec, n, m):
    _check("sift_int", n, m, prec, SIFT_MODES)


R2D2_SHAPES = [(2, 2), (127, 129), (128, 160), (129, 161), (255, 191), (257, 193), (511, 383), (513, 385), (2049, 2049),
               (255, 8193), (129, 33000), (1, 40000)]
R2D2_MODES = [(RATIO_MUTUAL, 0.9), (MUTUAL, 0.0), (THRESH_MUTUAL, 0.7), (THRESH_MUTUAL, 0.9), (THRESH, 0.9), (NN, 0.0),
              (RATIO, 0.85)]


@pytest.mark.parametrize("prec", SPLIT_PRECS, ids=PREC_NAME.get)
@pytest.mark.parametrize("n,m", R2D2_SHAPES)
def test_r2d2_cosine_within_eps(prec, n, m):
    _check("r2d2", n, m, prec, R2D2_MODES)


@pytest.mark.parametrize("prec", SPLIT_PRECS, ids=PREC_NAME.get)
@pytest.mark.parametrize("n,m", [(127, 129), (257, 193), (513, 385), (2049, 2049), (255, 12289)])
def test_rootsift_l2_within_eps(prec, n, m):
    _check("rootsift", n, m, prec, [(RATIO, 0.85), (MUTUAL, 0.0)])


@pytest.mark.parametrize("prec", [TF32X3, F16X3], ids=PREC_NAME.get)
@pytest.mark.parametrize("family", ["wide_l2", "wide_cos"])
@pytest.mark.parametrize("n,m", [(129, 161), (513, 385), (1000, 2000)])
def test_wide_range_operands_within_eps(prec, family, n, m):
    # (cosine similarities of such rows are far above 1: the distance rules would only see sqrt(2 - 2s) = NaN)
    modes = [(RATIO, 0.85), (MUTUAL, 0.0)] if family == "wide_l2" else [(MUTUAL, 0.0), (NN, 0.0)]
    _check(family, n, m, prec, modes)


def test_rootsift_through_the_sift_plugin_takes_a_precision_whose_contract_holds(monkeypatch):
    """feature_extractors._gpu_match picks F16X1 for integer descriptors and TF32X3 otherwise: its pairs must be those
    of a certified call at that precision."""
    from vo_b200 import ops
    monkeypatch.syspath_prepend(os.path.join(ROOT, "visual-odometry-pipeline_b200"))
    gm = importlib.import_module("feature_extractors._gpu_match")
    for family, prec in (("rootsift", TF32X3), ("sift_int", F16X1)):
        ref, cur, r64 = _case(family, 2049, 2049)
        got = gm.knn_ratio_f32(ref, cur, 0.85)
        res = _run(ref, cur, L2, RATIO, 0.85, prec, rows_only=True)
        _certify(family, res, [r64], prec, RATIO, 0.85)
        assert np.array_equal(got, res.numpy()), family
    assert ops.VO_PREC_F16X1 == F16X1


# ------------------------------------------------------------------------------------------------ exact ties
# column pairs (c - 1, c) around every boundary the kernels use: 32/40/48-column quarters, 64/128/160/192 tiles,
# split boundaries (SIMT: 256-column splits here; TF32X3: 512)
TIE_EDGES = [32, 40, 48, 64, 96, 120, 128, 144, 160, 192, 240, 256, 320, 384, 480, 512, 576, 640, 768, 960]


def _plant_ties(ref, cur, rng, integer):
    """Duplicates in cur across boundaries (row ties) and in ref across 128-row blocks / 256-row clusters (column
    ties), each made the clear favourite of one row / column.  Returns {row: (cols...)} and {col: (rows...)}."""
    noise = (lambda x: np.clip(x + rng.integers(-2, 3, x.shape), 0, 255)) if integer else \
        (lambda x: (lambda y: y / np.linalg.norm(y))(x + 0.06 * rng.standard_normal(x.shape)).astype(np.float32))
    row_ties, col_ties = {}, {}
    groups = [(e - 1, e) for e in TIE_EDGES if e < cur.shape[0]]
    groups += [(700, 130, 290), (416, 415, 170), (800, 799, 105),            # triples across tiles, quarters and splits
               (108, 109, 110)]                                             # and one inside a 4-column filter group
    for k, cols in enumerate(groups):
        if max(cols) >= cur.shape[0]:
            continue
        row = 3 + 5 * k
        for c in cols[1:]:
            cur[c] = cur[cols[0]]
        assert not set(cols) & {c for g in row_ties.values() for c in g}
        ref[row] = noise(cur[cols[0]])
        row_ties[row] = tuple(sorted(cols))
    for k, rows in enumerate([(127, 128), (255, 256), (200, 130, 290), (0, 299)]):
        if max(rows) >= ref.shape[0]:
            continue
        col = 900 + 7 * k
        for r in rows[1:]:
            ref[r] = ref[rows[0]]
        cur[col] = noise(ref[rows[0]])
        col_ties[col] = tuple(sorted(rows))
    return row_ties, col_ties


def _check_ties(res, row_ties, col_ties, metric):
    kidx, kval = res.knn_idx[0].cpu().numpy(), res.knn_val[0].cpu().numpy()
    kept = set(res.numpy()[:, 0].tolist())
    nt = res.near_tie[0].cpu().numpy()
    for row, cols in row_ties.items():
        assert tuple(kidx[row]) == cols[:2], (row, cols, kidx[row])           # lowest index first
        assert kval[row, 0].view(np.int32) == kval[row, 1].view(np.int32), (row, kval[row])
        assert row not in kept and nt[row] == 1, row                           # d1 == d2: RATIO rejects; a tie
    if res.col_idx is not None:
        cidx = res.col_idx[0].cpu().numpy()
        for col, rows in col_ties.items():
            assert cidx[col] == rows[0], (col, rows, cidx[col])


@pytest.mark.parametrize("prec", ALL_PRECS, ids=PREC_NAME.get)
def test_exact_ties_on_integer_data(prec):
    rng = np.random.default_rng(77)
    ref, cur = _sift_int(77, 300, 1000)
    row_ties, col_ties = _plant_ties(ref, cur, rng, integer=True)
    r64 = m64.knn64(ref, cur, L2)
    for rows_only in ((True, False) if prec == F16X1 else (False,)):
        res = _run(ref, cur, L2, RATIO, 0.85, prec, rows_only=rows_only)
        _certify("ties_int", res, [r64], prec, RATIO, 0.85)
        _check_ties(res, row_ties, col_ties, L2)


@pytest.mark.parametrize("prec", SPLIT_PRECS, ids=PREC_NAME.get)
def test_exact_ties_and_a_zero_row_on_real_data(prec):
    """Duplicated descriptors give bit-identical scores at every precision, so the lower index must win.  Few are
    planted (each leaves its row uncertain under eps); the all-zero row scores 0 against every column (eps = 0)."""
    rng = np.random.default_rng(78)
    ref, cur = _r2d2(78, 4097, 1000)
    row_ties, col_ties = _plant_ties(ref, cur, rng, integer=False)
    for k in list(row_ties)[8:]:
        del row_ties[k]                                                        # the rows stay planted, checked by certify
    ref[1500] = 0.0
    r64 = m64.knn64(ref, cur, COS)
    for mode, param in ((RATIO, 0.85), (RATIO_MUTUAL, 0.9)):
        res = _run(ref, cur, COS, mode, param, prec)
        _certify("ties_real", res, [r64], prec, mode, param)
        _check_ties(res, row_ties, col_ties, COS)
        kidx, kval = res.knn_idx[0].cpu().numpy(), res.knn_val[0].cpu().numpy()
        assert tuple(kidx[1500]) == (0, 1) and kval[1500, 0] == 0 and kval[1500, 1] == 0, (kidx[1500], kval[1500])


# ------------------------------------------------------------------------------------------------ ragged batches
N_STRIDE, M_STRIDE = 301, 283          # no multiple of any tile


def _ragged(family, B, seed):
    """B pairs with n_ref / n_cur covering 0, 1, stride - 1 and stride; padding rows and columns hold exact copies of
    valid partners (a padding column equal to a ref row would be that row's perfect match if it were read)."""
    rng = np.random.default_rng(seed)
    make, metric = FAMILIES[family]
    sizes_n = [N_STRIDE, 0, 1, N_STRIDE - 1, 150, N_STRIDE, 77, 1, N_STRIDE - 1, 200, N_STRIDE][:B]
    sizes_m = [M_STRIDE, M_STRIDE, M_STRIDE - 1, 0, 1, 140, M_STRIDE, 1, 2, M_STRIDE - 1, 95][:B]
    ref = np.zeros((B, N_STRIDE, 128), np.float32)
    cur = np.zeros((B, M_STRIDE, 128), np.float32)
    refs = []
    for b in range(B):
        a, c = make(seed * 100 + b, N_STRIDE, M_STRIDE)
        n, m = sizes_n[b], sizes_m[b]
        if m:
            a[n:] = c[rng.integers(0, m, N_STRIDE - n)]           # padding ref rows: copies of valid columns
        if n:
            c[m:] = a[rng.integers(0, n, M_STRIDE - m)]           # padding cur columns: copies of valid rows
        ref[b], cur[b] = a, c
        refs.append(m64.knn64(a[:n], c[:m], metric))
    return ref, cur, np.array(sizes_n, np.int32), np.array(sizes_m, np.int32), refs


@pytest.mark.parametrize("B", [3, 9, 11])
@pytest.mark.parametrize("family,precs,modes", [
    ("sift_int", ALL_PRECS, [(RATIO, 0.85), (MUTUAL, 0.0), (NN, 0.0)]),
    ("r2d2", SPLIT_PRECS, [(RATIO_MUTUAL, 0.9), (RATIO, 0.85), (NN, 0.0), (THRESH_MUTUAL, 0.7)])])
def test_ragged_batches(B, family, precs, modes):
    ref, cur, n_ref, n_cur, refs = _ragged(family, B, B)
    metric = FAMILIES[family][1]
    for prec in precs:
        for mode, param in modes:
            rows_only = prec == F16X1 and mode in (RATIO, NN)
            res = _run(ref, cur, metric, mode, param, prec, rows_only=rows_only, n_ref=_gpu(n_ref), n_cur=_gpu(n_cur))
            try:
                _certify(family, res, refs, prec, mode, param)
            except m64.CertifyError as e:
                raise AssertionError(f"{family} B={B} {PREC_NAME[prec]} mode={mode}: {e}") from None
            count = res.count.cpu().numpy()
            kidx = res.knn_idx.cpu().numpy()
            for b in range(B):
                if n_ref[b] == 0 or n_cur[b] == 0:                  # empty pair
                    assert count[b] == 0 and (kidx[b] == -1).all(), (b, count[b])
                    if res.col_idx is not None:
                        assert (res.col_idx[b].cpu().numpy() == -1).all(), b
                elif n_cur[b] == 1 and mode in (RATIO, RATIO_MUTUAL, NN):   # one candidate: no second best
                    assert count[b] == (n_ref[b] if mode == NN else 0), (b, mode, count[b])


# ------------------------------------------------------------------------------------------------ forced paths
def test_f16x1_persistent_and_plain_forms_agree_and_certify(monkeypatch):
    for n, m in ((513, 12289), (129, 1000), (2049, 383)):
        ref, cur, r64 = _case("sift_int", n, m)
        outs = []
        for form in ("0", "1"):
            monkeypatch.setenv("VO_TC_PERSIST", form)
            res = _run(ref, cur, L2, RATIO, 0.85, F16X1, rows_only=True)
            _certify("sift_int", res, [r64], F16X1, RATIO, 0.85)
            outs.append([t.cpu().numpy() for t in (res.knn_idx, res.knn_val, res.pairs[:, :int(res.count[0])], res.near_tie)])
        for x, y in zip(*outs):
            assert np.array_equal(x, y), (n, m)


@pytest.mark.parametrize("family,metric,mode,param", [("r2d2", COS, RATIO_MUTUAL, 0.9), ("rootsift", L2, MUTUAL, 0.0)])
def test_f16x3_interleaved_and_plain_agree_and_certify(monkeypatch, family, metric, mode, param):
    ref, cur, n_ref, n_cur, refs = _ragged(family, 11, 5)
    outs = []
    for interleave in (True, False):
        if interleave:
            monkeypatch.delenv("VO_TC_NO_INTERLEAVE", raising=False)
        else:
            monkeypatch.setenv("VO_TC_NO_INTERLEAVE", "1")
        res = _run(ref, cur, metric, mode, param, F16X3, n_ref=_gpu(n_ref), n_cur=_gpu(n_cur))
        _certify(family, res, refs, F16X3, mode, param)
        outs.append([t.cpu().numpy() for t in (res.knn_idx, res.knn_val, res.col_idx, res.count, res.near_tie)] +
                    [res.pairs[b, :int(res.count[b])].cpu().numpy() for b in range(11)])
    for x, y in zip(*outs):
        assert np.array_equal(x.view(np.uint8), y.view(np.uint8))


# ------------------------------------------------------------------------------------------------ finalize chunks
@pytest.mark.parametrize("family,prec,mode,param", [("sift_int", TF32X1, RATIO, 0.85), ("r2d2", TF32X3, RATIO_MUTUAL, 0.9)])
def test_finalize_2048_row_chunks_and_pack(family, prec, mode, param):
    B, n, m = 74, 2049, 257
    make, metric = FAMILIES[family]
    ref = np.empty((B, n, 128), np.float32)
    cur = np.empty((B, m, 128), np.float32)
    refs = []
    for b in range(B):
        ref[b], cur[b] = make(5000 + b, n, m)
        refs.append(m64.knn64(ref[b], cur[b], metric))
    res = _run(ref, cur, metric, mode, param, prec)
    _certify(family, res, refs, prec, mode, param)
    assert int(res.count.sum()) > B * 100
