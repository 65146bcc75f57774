"""fp64 reference and certifier of the float-descriptor matcher (vo_match_f32) — TEST INFRASTRUCTURE ONLY.

`knn64` scores every (ref row, cur column) pair in float64 (larger is better: cosine a.b, L2 -|a-b|^2) and keeps the
exact row top-2 and column arg-best, ties to the lower index.  On integer-valued descriptors with |x| <= 255 every
score is an exact integer below 2^24, so the result equals oracle.knn_f32 bit for bit.

`eps` is the error model of a precision: a score computed by the GPU is within eps_ij = gamma * sigma_ij of the fp64
score, with P = sum_k |a_k b_k|, sigma = P (cosine) or |a|^2 + |b|^2 + 2P (L2).  gamma = 0 on integer data (every
product and partial sum is exact: the documented contract of TF32X1 and F16X1), 2^-18 on real-valued data for the
22-operand-bit split passes (TF32X3, F16X3) and the CUDA-core FP32 kernel.

`certify` checks one frame pair of GPU output against the reference under that model and raises on the first
violation; decisions that the model cannot pin down (a top-2, mutual status or acceptance that flips inside the
eps interval) are "uncertain" and are only checked for self-consistency.
"""
import numpy as np

MODE_RATIO, MODE_MUTUAL, MODE_RATIO_MUTUAL, MODE_THRESH_MUTUAL, MODE_THRESH, MODE_NN = range(6)
METRIC_L2, METRIC_COSINE = 0, 1
PREC_TF32X3, PREC_TF32X1, PREC_FP32_SIMT, PREC_F16X1, PREC_F16X3 = range(5)

GAMMA_SPLIT = 2.0 ** -18      # TF32X3 / F16X3 / FP32_SIMT on real-valued data
NEAR_TIE_REL = 1e-5           # finalize's near_tie threshold, relative, in the distance domain
MAX_UNCERTAIN = 0.005         # fraction of rows a case may leave uncertain on real-valued data
_CHUNK_BYTES = 256 << 20


def _is_int_data(x):
    return x.size == 0 or bool(np.all((x == np.rint(x)) & (np.abs(x) <= 255)))


def _topk_rows(x, k):
    """indices / values of the k largest entries of each row of x, ties to the lower index (x is modified)."""
    n = x.shape[0]
    idx = np.full((n, k), -1, np.int64)
    val = np.full((n, k), -np.inf)
    r = np.arange(n)
    for t in range(min(k, x.shape[1])):
        j = np.argmax(x, axis=1)         # first maximum = lowest index
        idx[:, t], val[:, t] = j, x[r, j]
        x[r, j] = -np.inf
    return idx, val


class Ref64:
    """Output of knn64 for one frame pair (N ref rows, M cur columns)."""

    def __init__(self, ref, cur, metric):
        self.a = np.asarray(ref, np.float32).astype(np.float64).reshape(-1, 128 if np.size(ref) == 0 else np.shape(ref)[-1])
        self.b = np.asarray(cur, np.float32).astype(np.float64).reshape(-1, self.a.shape[1])
        self.metric = int(metric)
        self.N, self.M = self.a.shape[0], self.b.shape[0]
        self.is_int = _is_int_data(self.a) and _is_int_data(self.b)
        self.na, self.nb = (self.a * self.a).sum(1), (self.b * self.b).sum(1)
        self.abs_a, self.abs_b = np.abs(self.a), np.abs(self.b)
        self._sum = {}
        s = self.summary(0.0)
        self.row_idx, self.row_score, self.col_idx = s["r_idx"], s["r_s"], s["c_idx"]

    # scores and eps at explicit (row, col) pairs
    def score(self, rows, cols):
        rows, cols = np.asarray(rows, np.int64), np.asarray(cols, np.int64)
        dot = np.einsum("ij,ij->i", self.a[rows], self.b[cols])
        if self.metric == METRIC_COSINE:
            return dot
        d = self.a[rows] - self.b[cols]
        return -np.einsum("ij,ij->i", d, d)

    def sigma(self, rows, cols):
        rows, cols = np.asarray(rows, np.int64), np.asarray(cols, np.int64)
        p = np.einsum("ij,ij->i", self.abs_a[rows], self.abs_b[cols])
        return p if self.metric == METRIC_COSINE else self.na[rows] + self.nb[cols] + 2 * p

    def _block(self, r0, r1):
        dot = self.a[r0:r1] @ self.b.T
        p = self.abs_a[r0:r1] @ self.abs_b.T
        if self.metric == METRIC_COSINE:
            return dot, p
        # the GEMM form in fp64: exact on integer data, and its rounding (~2^-50 sigma) is far below any eps on real data
        d2 = (self.na[r0:r1, None] + self.nb[None, :]) - 2 * dot
        return -d2, self.na[r0:r1, None] + self.nb[None, :] + 2 * p

    def summary(self, gamma):
        """Per-row and per-column extremes of S, S + eps and S - eps (cached per gamma)."""
        if gamma in self._sum:
            return self._sum[gamma]
        N, M = self.N, self.M
        out = dict(r_idx=np.full((N, 2), -1, np.int64), r_s=np.full((N, 2), -np.inf),
                   up_idx=np.full((N, 3), -1, np.int64), up=np.full((N, 3), -np.inf),
                   lo_idx=np.full((N, 2), -1, np.int64), lo=np.full((N, 2), -np.inf),
                   c_idx=np.full(M, -1, np.int64), c_s=np.full(M, -np.inf),
                   c_up_idx=np.full((M, 2), -1, np.int64), c_up=np.full((M, 2), -np.inf), c_lo=np.full(M, -np.inf))
        if N and M:
            per_row = 8 * M * 8
            step = max(1, _CHUNK_BYTES // per_row)
            cols = np.arange(M)
            for r0 in range(0, N, step):
                r1 = min(N, r0 + step)
                S, sig = self._block(r0, r1)
                E = gamma * sig
                U, L = S + E, S - E
                out["r_idx"][r0:r1], out["r_s"][r0:r1] = _topk_rows(S.copy(), 2)
                out["lo_idx"][r0:r1], out["lo"][r0:r1] = _topk_rows(L.copy(), 2)
                # column side, merged over chunks in ascending row order (strictly better replaces: lower row wins ties)
                j = np.argmax(S, axis=0)
                v = S[j, cols]
                better = v > out["c_s"]
                out["c_idx"][better], out["c_s"][better] = j[better] + r0, v[better]
                out["c_lo"] = np.maximum(out["c_lo"], L.max(axis=0))
                ut_idx, ut = _topk_rows(U.T.copy(), 2)
                cand_i = np.concatenate([out["c_up_idx"], ut_idx + r0], 1)
                cand_v = np.concatenate([out["c_up"], ut], 1)
                ci, cv = _topk_rows(cand_v.copy(), 2)
                out["c_up_idx"], out["c_up"] = np.take_along_axis(cand_i, ci, 1), cv
                out["up_idx"][r0:r1], out["up"][r0:r1] = _topk_rows(U, 3)
        if M < 2:
            out["r_idx"][:, 1] = -1
        self._sum[gamma] = out
        return out


def knn64(ref, cur, metric):
    """fp64 k-NN of one frame pair.  .row_idx [N,2] (exact top-2, -1 if absent), .row_score [N,2] fp64 scores
    (larger is better), .col_idx [M] (arg-best ref row); .score / .sigma give fp64 values at any (row, col)."""
    return Ref64(ref, cur, metric)


def knn64_as_f32(r):
    """(row_idx int32, row_val f32, col_idx int32) in oracle.knn_f32's conventions (distance for L2, similarity)."""
    ridx = r.row_idx.astype(np.int32)
    s = np.where(ridx >= 0, r.row_score, 0.0)
    val = _value(r.metric, s)
    val[ridx < 0] = 0
    return ridx, val, r.col_idx.astype(np.int32)


def eps(prec, data):
    """gamma of the error model for `prec` on `data` (a Ref64): eps_ij = gamma * sigma_ij."""
    if data.is_int:
        return 0.0
    if prec in (PREC_TF32X1, PREC_F16X1):
        raise ValueError("one 11-bit pass is exact on integer-valued descriptors only (no error model on real data)")
    return GAMMA_SPLIT


# ------------------------------------------------------------------------------------------ acceptance, fp32 like oracle.accept
def _f32(x):
    return np.asarray(x, np.float32)


def _value(metric, s):
    """the value finalize reports for fp64 score(s) s: L2 sqrtf(float(d^2)) (clamped at 0), cosine float(s)."""
    s = np.asarray(s, np.float64)
    if metric == METRIC_L2:
        return np.sqrt(np.maximum(_f32(-s), np.float32(0)), dtype=np.float32)
    return _f32(s)


def _dist(metric, v):
    if metric == METRIC_COSINE:
        with np.errstate(invalid="ignore"):
            return np.sqrt(np.float32(2) - np.float32(2) * _f32(v), dtype=np.float32)
    return _f32(v)


def _keep(mode, param, metric, v1, v2, has1, has2, mutual):
    d1, d2 = _dist(metric, v1), _dist(metric, v2)
    with np.errstate(invalid="ignore", divide="ignore"):
        if mode == MODE_RATIO:
            return has2 & (d1.astype(np.float64) < float(param) * d2.astype(np.float64))
        if mode == MODE_MUTUAL:
            return mutual.copy()
        if mode == MODE_RATIO_MUTUAL:
            return has2 & mutual & ((d1 / (d2 + np.float32(1e-8))).astype(np.float64) <= float(param))
        if mode in (MODE_THRESH_MUTUAL, MODE_THRESH):
            k = has1 & (_f32(v1).astype(np.float64) >= float(param))
            return k & mutual if mode == MODE_THRESH_MUTUAL else k
    return has1.copy()


def _near_tie(metric, v1, v2, has2):
    d1, d2 = _dist(metric, v1), _dist(metric, v2)
    with np.errstate(invalid="ignore"):
        return has2 & ~((d2 - d1) > np.float32(NEAR_TIE_REL) * d2)


class CertifyError(AssertionError):
    pass


def _fail(msg, **kw):
    raise CertifyError(msg + "  " + ", ".join(f"{k}={v}" for k, v in kw.items()))


def certify(gpu, ref64, gamma, mode, param):
    """Check one frame pair of vo_match_f32 output against the fp64 reference.

    gpu: dict of numpy arrays of this pair: knn_idx [n_stride,2], knn_val [n_stride,2], col_idx [m_stride] or None,
    pairs [count,2], dist [count] or None, near_tie [n_stride] or None; ref64 = knn64 of the valid rows / columns;
    gamma from eps().  Returns dict(max_err_ratio, uncertain, rows, uncertain_rows)."""
    r, metric = ref64, ref64.metric
    N, M = r.N, r.M
    sm = r.summary(gamma)
    exact = gamma == 0.0
    kidx = np.asarray(gpu["knn_idx"]).astype(np.int64)
    kval = np.asarray(gpu["knn_val"], np.float32)
    n_stride = kidx.shape[0]
    rows = np.arange(N)
    i1, i2 = kidx[:N, 0], kidx[:N, 1]

    # ---- validity
    if n_stride > N and (kidx[N:] != -1).any():
        row = N + int(np.nonzero((kidx[N:] != -1).any(1))[0][0])
        _fail("padding row has a neighbour", row=row, idx=kidx[row])
    for name, ii, need in (("i1", i1, 1), ("i2", i2, 2)):
        bad = (ii >= 0) != (M >= need)
        bad |= ii >= M
        if bad.any():
            row = int(np.nonzero(bad)[0][0])
            _fail(f"{name} validity", row=row, idx=int(ii[row]), M=M)
    both = (i1 >= 0) & (i2 >= 0)
    if (both & (i1 == i2)).any():
        row = int(np.nonzero(both & (i1 == i2))[0][0])
        _fail("i1 == i2", row=row, idx=int(i1[row]))

    # ---- values at the GPU's own indices
    has1, has2 = i1 >= 0, i2 >= 0
    max_ratio = 0.0
    s_at = [np.full(N, -np.inf), np.full(N, -np.inf)]
    e_at = [np.zeros(N), np.zeros(N)]
    for k, (ii, hh) in enumerate(((i1, has1), (i2, has2))):
        if not hh.any():
            continue
        rr, cc = rows[hh], ii[hh]
        s = r.score(rr, cc)
        e = gamma * r.sigma(rr, cc)
        s_at[k][hh], e_at[k][hh] = s, e
        v = kval[:N, k][hh].astype(np.float64)
        if exact:
            want = _value(metric, s)
            bad = ~(kval[:N, k][hh] == want)
            if bad.any():
                q = int(np.nonzero(bad)[0][0])
                _fail(f"value v{k + 1} is not exact", row=int(rr[q]), col=int(cc[q]), got=float(v[q]), want=float(want[q]))
        else:
            err = np.abs(v * v - (-s)) if metric == METRIC_L2 else np.abs(v - s)
            ratio = np.divide(err, e, out=np.zeros_like(err), where=e > 0)
            if (err > e).any():
                q = int(np.argmax(ratio))
                _fail(f"value v{k + 1} off by more than eps", row=int(rr[q]), col=int(cc[q]), got=float(v[q]),
                      score64=float(s[q]), err=float(err[q]), eps=float(e[q]))
            max_ratio = max(max_ratio, float(ratio.max()) if ratio.size else 0.0)

    # ---- optimality of the row top-2 and certainty
    r1, r2 = sm["r_idx"][:, 0], sm["r_idx"][:, 1]
    if exact:
        for k, (got, want) in enumerate(((i1, r1), (i2, r2))):
            bad = got != want
            if bad.any():
                row = int(np.nonzero(bad)[0][0])
                _fail(f"i{k + 1} is not the exact fp64 neighbour (ties to the lower index)", row=row, got=int(got[row]),
                      want=int(want[row]), s_got=float(s_at[k][row]), s_want=float(sm["r_s"][row, k]))
        top1_ok = np.ones(N, bool)
        top2_ok = np.ones(N, bool)
    else:
        bound1 = sm["lo"][:, 0]
        bad = has1 & (s_at[0] + e_at[0] < bound1)
        if bad.any():
            row = int(np.nonzero(bad)[0][0])
            _fail("i1 is not optimal within eps", row=row, got=int(i1[row]), s_got=float(s_at[0][row]),
                  best=int(r1[row]), s_best=float(sm["r_s"][row, 0]))
        bound2 = np.where(sm["lo_idx"][:, 0] != i1, sm["lo"][:, 0], sm["lo"][:, 1])
        bad = has2 & (s_at[1] + e_at[1] < bound2)
        if bad.any():
            row = int(np.nonzero(bad)[0][0])
            _fail("i2 is not the best of the rest within eps", row=row, i1=int(i1[row]), got=int(i2[row]),
                  s_got=float(s_at[1][row]), want=int(r2[row]), s_want=float(sm["r_s"][row, 1]))
        up_i, up = sm["up_idx"], sm["up"]
        e_r1 = gamma * r.sigma(rows, np.maximum(r1, 0)) if M else np.zeros(N)
        e_r2 = gamma * r.sigma(rows, np.maximum(r2, 0)) if M else np.zeros(N)
        rest1 = np.where(up_i[:, 0] != r1, up[:, 0], up[:, 1])                       # best upper bound among j != r1
        top1_ok = (M <= 1) | (sm["r_s"][:, 0] - e_r1 > rest1)
        rest2 = np.full(N, -np.inf)
        for t in range(3):                                                            # first upper bound not in {r1, r2}
            pick = (rest2 == -np.inf) & (up_i[:, t] != r1) & (up_i[:, t] != r2)
            rest2[pick] = up[pick, t]
        top2_ok = top1_ok & ((M <= 2) | (sm["r_s"][:, 1] - e_r2 > rest2))
        for name, ok, got, want in (("i1", top1_ok, i1, r1), ("i2", top2_ok, i2, r2)):
            bad = ok & (got != want)
            if bad.any():
                row = int(np.nonzero(bad)[0][0])
                _fail(f"{name} differs from fp64 on a row whose margin exceeds the bound", row=row, got=int(got[row]),
                      want=int(want[row]))

    # ---- column arg-best
    cidx = gpu.get("col_idx")
    col_ok = np.ones(M, bool)
    if cidx is not None:
        cidx = np.asarray(cidx).astype(np.int64)
        if (cidx[M:] != -1).any():
            _fail("padding column has a neighbour", col=M + int(np.nonzero(cidx[M:] != -1)[0][0]))
        c = cidx[:M]
        if ((c >= 0) != (N >= 1)).any() or (c >= N).any():
            col = int(np.nonzero(((c >= 0) != (N >= 1)) | (c >= N))[0][0])
            _fail("col_idx validity", col=col, got=int(c[col]), N=N)
        if exact:
            bad = c != sm["c_idx"]
            if bad.any():
                col = int(np.nonzero(bad)[0][0])
                _fail("col_idx is not the exact fp64 arg-best (ties to the lower row)", col=col, got=int(c[col]),
                      want=int(sm["c_idx"][col]))
        elif N:
            cols = np.arange(M)
            s = r.score(c, cols)
            e = gamma * r.sigma(c, cols)
            bad = s + e < sm["c_lo"]
            if bad.any():
                col = int(np.nonzero(bad)[0][0])
                _fail("col_idx is not optimal within eps", col=col, got=int(c[col]), want=int(sm["c_idx"][col]))
            cb = sm["c_idx"]
            e_cb = gamma * r.sigma(cb, cols)
            rest = np.where(sm["c_up_idx"][:, 0] != cb, sm["c_up"][:, 0], sm["c_up"][:, 1])
            col_ok = (N <= 1) | (sm["c_s"] - e_cb > rest)
            bad = col_ok & (c != cb)
            if bad.any():
                col = int(np.nonzero(bad)[0][0])
                _fail("col_idx differs from fp64 on a column whose margin exceeds the bound", col=col, got=int(c[col]),
                      want=int(cb[col]))

    # ---- acceptance
    pairs = np.asarray(gpu["pairs"]).astype(np.int64).reshape(-1, 2)
    if len(pairs) and ((pairs[:, 0] < 0) | (pairs[:, 0] >= N)).any():
        _fail("accepted pair on a padding row", pair=pairs[(pairs[:, 0] < 0) | (pairs[:, 0] >= N)][0])
    if len(pairs) > 1 and not (np.diff(pairs[:, 0]) > 0).all():
        _fail("pairs are not in ascending row order", at=int(np.nonzero(np.diff(pairs[:, 0]) <= 0)[0][0]))
    got_keep = np.zeros(N, bool)
    got_keep[pairs[:, 0]] = True
    if len(pairs) and (pairs[:, 1] != i1[pairs[:, 0]]).any():
        k = int(np.nonzero(pairs[:, 1] != i1[pairs[:, 0]])[0][0])
        _fail("accepted pair is not (row, knn_idx[row, 0])", pair=pairs[k], i1=int(i1[pairs[k, 0]]))
    needs_cols = mode in (MODE_MUTUAL, MODE_RATIO_MUTUAL, MODE_THRESH_MUTUAL)
    uses_d2 = mode in (MODE_RATIO, MODE_RATIO_MUTUAL)
    # the rule applied to the GPU's own outputs (every row: finalize is exact arithmetic on them)
    if cidx is not None or not needs_cols:
        mut_gpu = np.zeros(N, bool)
        if cidx is not None:
            mut_gpu[has1] = cidx[i1[has1]] == rows[has1]
        self_keep = _keep(mode, param, metric, kval[:N, 0], kval[:N, 1], has1, has2, mut_gpu)
        bad = self_keep != got_keep
        if bad.any():
            row = int(np.nonzero(bad)[0][0])
            _fail("acceptance disagrees with the rule applied to the GPU's own k-NN output", row=row, kept=bool(got_keep[row]),
                  v=kval[row], idx=kidx[row])
    # The rule at both ends of the eps interval.  Whichever columns the GPU ranks first and second, the values it ranks
    # there are order statistics of its scores, so they lie between those of S - eps and S + eps.  The rules grow with
    # s1 and fall with s2, so the two corners bound every outcome; mutual status needs the indices themselves.
    h1, h2 = r1 >= 0, r2 >= 0
    s1_lo, s1_hi = sm["lo"][:, 0], sm["up"][:, 0]
    s2_lo, s2_hi = np.where(h2, sm["lo"][:, 1], 0.0), np.where(h2, sm["up"][:, 1], 0.0)
    mut64 = np.zeros(N, bool)
    mut64[h1] = sm["c_idx"][r1[h1]] == rows[h1]
    mut_ok = top1_ok.copy()
    mut_ok[h1] &= col_ok[r1[h1]]
    if needs_cols and not exact and not mut_ok.all():
        # a row whose own top-1 is uncertain is still certainly not mutual when, in every column it may pick, some
        # other row certainly scores higher
        for row in np.nonzero(~mut_ok & h1)[0]:
            cand = np.nonzero(r.score(np.full(M, row), np.arange(M)) + gamma * r.sigma(np.full(M, row), np.arange(M))
                              >= s1_lo[row])[0]
            s = r.score(np.full(len(cand), row), cand) + gamma * r.sigma(np.full(len(cand), row), cand)
            if (s < sm["c_lo"][cand]).all():
                mut_ok[row], mut64[row] = True, False
    yes = np.ones(N, bool)
    k_hi = _keep(mode, param, metric, _value(metric, s1_hi), _value(metric, s2_lo), h1, h2, yes)
    k_lo = _keep(mode, param, metric, _value(metric, s1_lo), _value(metric, s2_hi), h1, h2, yes)
    if metric == METRIC_COSINE and uses_d2 and not exact:
        nan_risk = (s1_hi >= 1.0) | (h2 & (s2_hi >= 1.0))                          # sqrt(2 - 2s) may be NaN
        k_lo &= ~nan_risk
        k_hi |= nan_risk
    want_keep = k_hi & (mut64 if needs_cols else yes)
    certain = ~k_hi | (k_lo & (mut_ok if needs_cols else yes))                        # surely rejected, or surely decided
    bad = certain & (got_keep != want_keep)
    if bad.any():
        row = int(np.nonzero(bad)[0][0])
        _fail("acceptance of a certain row differs from fp64", row=row, kept=bool(got_keep[row]), want=bool(want_keep[row]),
              s64=sm["r_s"][row], idx64=sm["r_idx"][row])

    # ---- dist: derived from knn_val[row, 0] bit for bit
    dist = gpu.get("dist")
    if dist is not None and len(pairs):
        got = _f32(np.asarray(dist)[:len(pairs)])
        want = _dist(metric, kval[pairs[:, 0], 0])
        same = (got.view(np.uint32) == want.view(np.uint32)) | (np.isnan(got) & np.isnan(want))   # any NaN payload
        if not same.all():
            k = int(np.nonzero(~same)[0][0])
            _fail("dist is not the distance of knn_val[row, 0]", pair=pairs[k], got=float(got[k]), want=float(want[k]))

    # ---- near_tie
    nt = gpu.get("near_tie")
    if nt is not None:
        nt = np.asarray(nt).astype(np.int64)
        if (nt[N:] != 0).any():
            _fail("near_tie set on a padding row", row=N + int(np.nonzero(nt[N:])[0][0]))
        nt = nt[:N]
        if ((nt != 0) & (nt != 1)).any():
            _fail("near_tie is not 0 / 1", row=int(np.nonzero((nt != 0) & (nt != 1))[0][0]))
        bad = has1 & (i1 != r1) & (nt != 1)
        if bad.any():
            row = int(np.nonzero(bad)[0][0])
            _fail("row whose i1 differs from fp64 does not carry near_tie", row=row, got=int(i1[row]), want=int(r1[row]),
                  s=(float(s_at[0][row]), float(sm["r_s"][row, 0])))
        # the flag at both ends of the interval (the predicate grows with d1 and falls with d2)
        t_a = _near_tie(metric, _value(metric, s1_hi), _value(metric, s2_lo), h2)
        t_b = _near_tie(metric, _value(metric, s1_lo), _value(metric, s2_hi), h2)
        sure = t_a == t_b
        if metric == METRIC_COSINE and not exact:
            sure &= ~((s1_hi >= 1.0) | (h2 & (s2_hi >= 1.0)))
        bad = sure & (nt != t_a.astype(np.int64))
        if bad.any():
            row = int(np.nonzero(bad)[0][0])
            _fail("near_tie differs from the fp64 gap", row=row, got=int(nt[row]), want=int(t_a[row]),
                  s64=sm["r_s"][row], v=kval[row])

    uncertain = int(N - certain.sum())
    limit = 0 if exact else int(MAX_UNCERTAIN * N)
    if uncertain > limit:
        _fail("too many uncertain rows (eps too loose for this data)", uncertain=uncertain, rows=N, limit=limit)
    return dict(max_err_ratio=max_ratio, uncertain=uncertain, rows=N, uncertain_rows=np.nonzero(~certain)[0])


def certify_batch(res, refs, gamma, mode, param, n_ref=None, n_cur=None):
    """certify every pair of an ops.MatchResult (torch tensors) against refs[b] = knn64 of pair b; merged report."""
    rep = dict(max_err_ratio=0.0, uncertain=0, rows=0)
    B = len(refs)
    t = lambda x: None if x is None else x.cpu().numpy()  # noqa: E731
    kidx, kval, cidx, nt = t(res.knn_idx), t(res.knn_val), t(res.col_idx), t(res.near_tie)
    pairs, dist, count = t(res.pairs), t(res.dist), t(res.count)
    for b in range(B):
        k = int(count[b])
        g = dict(knn_idx=kidx[b], knn_val=kval[b], col_idx=None if cidx is None else cidx[b], pairs=pairs[b, :k],
                 dist=None if dist is None else dist[b, :k], near_tie=None if nt is None else nt[b])
        try:
            one = certify(g, refs[b], gamma, mode, param)
        except CertifyError as e:
            raise CertifyError(f"pair {b}: {e}") from None
        rep["max_err_ratio"] = max(rep["max_err_ratio"], one["max_err_ratio"])
        rep["uncertain"] += one["uncertain"]
        rep["rows"] += one["rows"]
    return rep


__all__ = ["knn64", "knn64_as_f32", "eps", "certify", "certify_batch", "CertifyError", "Ref64"]
