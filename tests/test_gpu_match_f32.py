"""CUDA float-descriptor matcher vs golden vectors and the oracle.  Integer-valued (SIFT) data: bit-exact.
Real-valued (R2D2) data: identical except recorded near-ties (<1e-5 relative, north-star tolerance)."""
import numpy as np
import pytest

pytestmark = pytest.mark.gpu

REL_TIE = 1e-5


def _gpu(a):
    import torch
    return torch.from_numpy(np.ascontiguousarray(a)).cuda()


@pytest.mark.parametrize("prec", [2, 1, 0])
def test_golden_sift_knn_bit_exact(golden, prec):
    from vo_b200 import ops
    g = golden("match_f32_sift.npz")
    r = ops.match_f32(_gpu(g["ref"]), _gpu(g["cur"]), ops.VO_METRIC_L2, ops.VO_MODE_RATIO, 0.85, precision=prec, want_knn=True)
    assert np.array_equal(r.knn_idx[0].cpu().numpy(), g["knn_idx"])
    assert np.array_equal(r.knn_val[0].cpu().numpy(), g["knn_dist"])
    assert np.array_equal(r.numpy(), g["ref_sift_pairs"])


@pytest.mark.parametrize("prec", [2, 0, 4])
def test_golden_r2d2_matchers(golden, orc, prec):
    from vo_b200 import ops
    g = golden("match_f32_r2d2.npz")
    ref, cur = g["ref"], g["cur"]
    cases = [(ops.VO_MODE_RATIO_MUTUAL, 0.90, "ratio_mutual_pairs"), (ops.VO_MODE_THRESH_MUTUAL, 0.9, "mnn_pairs"),
             (ops.VO_MODE_THRESH, 0.9, "sim_pairs"), (ops.VO_MODE_THRESH_MUTUAL, 0.7, "mnn_pairs_t07"),
             (ops.VO_MODE_THRESH, 0.7, "sim_pairs_t07")]
    for mode, param, key in cases:
        r = ops.match_f32(_gpu(ref), _gpu(cur), ops.VO_METRIC_COSINE, mode, param, precision=prec)
        got, want = r.numpy(), g[key].reshape(-1, 2)
        if np.array_equal(got, want):
            continue
        # differences must be explained by rounding-level ties: duplicates (sim ~ 1 -> sqrt(2-2s) NaN or not)
        # or a top-1/top-2 gap below 1e-5 relative
        gd, wd = {int(a): int(b) for a, b in got}, {int(a): int(b) for a, b in want}
        for row in set(gd) ^ set(wd) | {k for k in set(gd) & set(wd) if gd[k] != wd[k]}:
            cols = [c for c in (gd.get(row), wd.get(row)) if c is not None]
            s = orc.pair_scores_f64(ref, cur, [row] * len(cols), cols, orc.METRIC_COSINE)
            near_dup = (1.0 - s.max()) < 1e-6                                 # the sim>1 quirk, SURVEY 3.3
            near_thr = abs(s.max() - param) < 1e-6 if mode != ops.VO_MODE_RATIO_MUTUAL else False
            near_tie = len(cols) == 2 and abs(s[0] - s[1]) <= REL_TIE * abs(s).max()
            assert near_dup or near_thr or near_tie, (key, row, cols, s)


@pytest.mark.parametrize("prec", [2, 1])
@pytest.mark.parametrize("n,m", [(2000, 2000), (777, 1500), (129, 64), (1, 300), (300, 1)])
def test_sift_vs_oracle_sizes(orc, prec, n, m):
    from vo_b200 import ops, synthetic
    p = synthetic.make_pair(n * 3 + m, n_kp=max(n, 8), n_cur=max(m, 8), kind="sift")
    ref, cur = p["ref_desc"][:n], p["cur_desc"][:m]
    r = ops.match_f32(_gpu(ref), _gpu(cur), ops.VO_METRIC_L2, ops.VO_MODE_RATIO, 0.85, precision=prec, want_knn=True)
    ridx, rval, cidx = orc.knn_f32(ref, cur, orc.METRIC_L2)
    assert np.array_equal(r.knn_idx[0].cpu().numpy(), ridx)
    assert np.array_equal(r.knn_val[0].cpu().numpy(), rval)
    assert np.array_equal(r.col_idx[0].cpu().numpy(), cidx)
    want, _ = orc.accept(ridx, rval, cidx, orc.MODE_RATIO, 0.85, orc.METRIC_L2)
    assert np.array_equal(r.numpy(), want)


@pytest.mark.parametrize("prec", [2, 0, 4])
def test_r2d2_vs_oracle_with_recorded_near_ties(orc, prec):
    from vo_b200 import ops, synthetic
    p = synthetic.make_pair(5, n_kp=3000, n_cur=2800, kind="r2d2")
    ref, cur = p["ref_desc"], p["cur_desc"]
    r = ops.match_f32(_gpu(ref), _gpu(cur), ops.VO_METRIC_COSINE, ops.VO_MODE_RATIO_MUTUAL, 0.90, precision=prec,
                      want_knn=True, want_near_tie=True)
    ridx, rval, cidx = orc.knn_f32(ref, cur, orc.METRIC_COSINE)
    gi = r.knn_idx[0].cpu().numpy()
    bad_rows = np.nonzero(gi[:, 0] != ridx[:, 0])[0]
    for row in bad_rows:                      # arg-max may differ only where fp64 calls it a tie
        s = orc.pair_scores_f64(ref, cur, [row, row], [gi[row, 0], ridx[row, 0]], orc.METRIC_COSINE)
        assert abs(s[0] - s[1]) <= REL_TIE * abs(s).max(), (row, s)
    assert len(bad_rows) <= 3
    assert np.allclose(r.knn_val[0].cpu().numpy()[:, 0], rval[:, 0], atol=2e-6, rtol=0)   # 3xTF32 ~ fp32 accuracy
    gc = r.col_idx[0].cpu().numpy()
    bad_cols = np.nonzero(gc != cidx)[0]
    for col in bad_cols:
        s = orc.pair_scores_f64(ref, cur, [gc[col], cidx[col]], [col, col], orc.METRIC_COSINE)
        assert abs(s[0] - s[1]) <= REL_TIE * abs(s).max(), (col, s)
    want, _ = orc.accept(ridx, rval, cidx, orc.MODE_RATIO_MUTUAL, 0.90, orc.METRIC_COSINE)
    got = r.numpy()
    diff = set(map(tuple, got.tolist())) ^ set(map(tuple, want.tolist()))
    assert len(diff) <= 4 and len(got) > 1500, (len(diff), len(got))


def test_ragged_batch(orc):
    from vo_b200 import ops, synthetic
    B, N, M = 3, 300, 280
    ps = [synthetic.make_pair(70 + b, n_kp=N, n_cur=M, kind="sift") for b in range(B)]
    ref = np.stack([p["ref_desc"] for p in ps])
    cur = np.stack([p["cur_desc"] for p in ps])
    n_ref, n_cur = np.array([300, 77, 0], np.int32), np.array([280, 130, 280], np.int32)
    for prec in (2, 1):
        r = ops.match_f32(_gpu(ref), _gpu(cur), ops.VO_METRIC_L2, ops.VO_MODE_RATIO, 0.85, precision=prec,
                          n_ref=_gpu(n_ref), n_cur=_gpu(n_cur))
        for b in range(B):
            want, _ = orc.match_f32(ref[b, :n_ref[b]], cur[b, :n_cur[b]], orc.METRIC_L2, orc.MODE_RATIO, 0.85)
            assert np.array_equal(r.numpy(b), want.reshape(-1, 2)), (prec, b)


# ------------------------------------------------------------------------------------------------ fp16 single pass
def test_golden_sift_f16_pass_bit_exact(golden):
    """VO_PREC_F16X1 (tcgen05 kind::f16, all-warp epilogue): the row top-2 (index and distance) and the accepted pairs
    of the reference's SIFT get_matches, bit for bit.  want_knn="rows" keeps the column side off, so the fp16 kernel
    itself runs (with a column arg-min requested the library takes the tf32 single pass)."""
    from vo_b200 import ops
    g = golden("match_f32_sift.npz")
    r = ops.match_f32(_gpu(g["ref"]), _gpu(g["cur"]), ops.VO_METRIC_L2, ops.VO_MODE_RATIO, 0.85,
                      precision=ops.VO_PREC_F16X1, want_knn="rows")
    assert r.col_idx is None
    assert np.array_equal(r.knn_idx[0].cpu().numpy(), g["knn_idx"])
    assert np.array_equal(r.knn_val[0].cpu().numpy(), g["knn_dist"])
    assert np.array_equal(r.numpy(), g["ref_sift_pairs"])


@pytest.mark.parametrize("n,m", [(2000, 2000), (777, 1500), (129, 64), (1, 300), (300, 1), (5000, 4099), (193, 385)])
def test_sift_f16_pass_vs_oracle_sizes(orc, n, m):
    from vo_b200 import ops, synthetic
    p = synthetic.make_pair(n * 3 + m, n_kp=max(n, 8), n_cur=max(m, 8), kind="sift")
    ref, cur = p["ref_desc"][:n], p["cur_desc"][:m]
    r = ops.match_f32(_gpu(ref), _gpu(cur), ops.VO_METRIC_L2, ops.VO_MODE_RATIO, 0.85, precision=ops.VO_PREC_F16X1,
                      want_knn="rows")
    ridx, rval, cidx = orc.knn_f32(ref, cur, orc.METRIC_L2)
    assert np.array_equal(r.knn_idx[0].cpu().numpy(), ridx)
    assert np.array_equal(r.knn_val[0].cpu().numpy(), rval)
    want, _ = orc.accept(ridx, rval, cidx, orc.MODE_RATIO, 0.85, orc.METRIC_L2)
    assert np.array_equal(r.numpy(), want)


def test_f16_pass_batched_ragged_and_mutual_fallback(orc):
    """B = 3 pairs with ragged counts through the fp16 pass; a mutual rule under VO_PREC_F16X1 (needs the column
    arg-min) must give exactly what the tf32 pass gives."""
    import torch
    from vo_b200 import ops, synthetic
    B, N = 3, 700
    batch = synthetic.make_batch(40, B, n_kp=N, kind="sift")
    n_ref = torch.tensor([700, 333, 1], dtype=torch.int32).cuda()
    n_cur = torch.tensor([512, 700, 64], dtype=torch.int32).cuda()
    ref, cur = _gpu(batch["ref_desc"]), _gpu(batch["cur_desc"])
    r = ops.match_f32(ref, cur, ops.VO_METRIC_L2, ops.VO_MODE_RATIO, 0.85, precision=ops.VO_PREC_F16X1, n_ref=n_ref,
                      n_cur=n_cur, want_knn="rows")
    for b in range(B):
        nr, nc = int(n_ref[b]), int(n_cur[b])
        ridx, rval, cidx = orc.knn_f32(batch["ref_desc"][b][:nr], batch["cur_desc"][b][:nc], orc.METRIC_L2)
        assert np.array_equal(r.knn_idx[b, :nr].cpu().numpy(), ridx)
        assert np.array_equal(r.knn_val[b, :nr].cpu().numpy(), rval)
        want, _ = orc.accept(ridx, rval, cidx, orc.MODE_RATIO, 0.85, orc.METRIC_L2)
        assert np.array_equal(r.numpy(b), want)
    a = ops.match_f32(ref, cur, ops.VO_METRIC_L2, ops.VO_MODE_MUTUAL, 0.0, precision=ops.VO_PREC_F16X1, want_knn=True)
    t = ops.match_f32(ref, cur, ops.VO_METRIC_L2, ops.VO_MODE_MUTUAL, 0.0, precision=ops.VO_PREC_TF32X1, want_knn=True)
    assert torch.equal(a.pairs[0, :int(a.count[0])], t.pairs[0, :int(t.count[0])]) and torch.equal(a.col_idx, t.col_idx)


@pytest.mark.parametrize("B", [3, 8, 11])
def test_split_fp16_batch_equals_single_pair_calls(B):
    """The split fp16 pass deals the clusters of up to 8 consecutive pairs round-robin over the pairs (so that the row
    blocks of a pair run at different times and the column filter sees earlier results).  The remap is an index bijection:
    a ragged batch (sizes that leave a partial last set) must give, pair by pair, exactly what a single-pair call gives."""
    import torch
    from vo_b200 import ops, synthetic
    N = 900
    batch = synthetic.make_batch(70, B, n_kp=N, kind="r2d2")
    rng = np.random.default_rng(B)
    n_ref = torch.from_numpy(rng.integers(1, N + 1, B).astype(np.int32)).cuda()
    n_cur = torch.from_numpy(rng.integers(1, N + 1, B).astype(np.int32)).cuda()
    ref, cur = _gpu(batch["ref_desc"]), _gpu(batch["cur_desc"])
    r = ops.match_f32(ref, cur, ops.VO_METRIC_COSINE, ops.VO_MODE_RATIO_MUTUAL, 0.90, precision=ops.VO_PREC_F16X3,
                      n_ref=n_ref, n_cur=n_cur, want_knn=True)
    for b in range(B):
        nr, nc = int(n_ref[b]), int(n_cur[b])
        s = ops.match_f32(ref[b, :nr].contiguous(), cur[b, :nc].contiguous(), ops.VO_METRIC_COSINE, ops.VO_MODE_RATIO_MUTUAL,
                          0.90, precision=ops.VO_PREC_F16X3, want_knn=True)
        assert int(r.count[b]) == int(s.count[0]), b
        k = int(s.count[0])
        assert torch.equal(r.pairs[b, :k], s.pairs[0, :k]), b
        assert torch.equal(r.knn_idx[b, :nr], s.knn_idx[0, :nr]) and torch.equal(r.knn_val[b, :nr], s.knn_val[0, :nr]), b
        assert torch.equal(r.col_idx[b, :nc], s.col_idx[0, :nc]), b


def test_fp16_passes_random_shapes_vs_oracle(orc):
    """40 random (n, m) shapes around the tile boundaries (192-column tiles of the fp16 single pass, 128-column tiles of the
    split pass, 128-row blocks, cluster pairs): fp16 single pass bit-exact on SIFT-like data, split fp16 near-tie aware
    on R2D2-like data."""
    from vo_b200 import ops, synthetic
    rng = np.random.default_rng(2024)
    edges = [1, 2, 31, 47, 48, 49, 127, 128, 129, 191, 192, 193, 255, 256, 257, 383, 384, 385, 575, 576, 577, 640]
    sift = synthetic.make_pair(901, n_kp=700, n_cur=700, kind="sift")
    r2d2 = synthetic.make_pair(902, n_kp=700, n_cur=700, kind="r2d2")
    for it in range(40):
        n = int(rng.choice(edges)) if it % 2 == 0 else int(rng.integers(1, 700))
        m = int(rng.choice(edges)) if it % 3 == 0 else int(rng.integers(1, 700))
        ref, cur = sift["ref_desc"][:n], sift["cur_desc"][:m]
        r = ops.match_f32(_gpu(ref), _gpu(cur), ops.VO_METRIC_L2, ops.VO_MODE_RATIO, 0.85, precision=ops.VO_PREC_F16X1,
                          want_knn="rows")
        ridx, rval, cidx = orc.knn_f32(ref, cur, orc.METRIC_L2)
        assert np.array_equal(r.knn_idx[0].cpu().numpy(), ridx), (n, m)
        assert np.array_equal(r.knn_val[0].cpu().numpy(), rval), (n, m)
        want, _ = orc.accept(ridx, rval, cidx, orc.MODE_RATIO, 0.85, orc.METRIC_L2)
        assert np.array_equal(r.numpy(), want), (n, m)
        ref, cur = r2d2["ref_desc"][:n], r2d2["cur_desc"][:m]
        r = ops.match_f32(_gpu(ref), _gpu(cur), ops.VO_METRIC_COSINE, ops.VO_MODE_RATIO_MUTUAL, 0.90,
                          precision=ops.VO_PREC_F16X3, want_knn=True)
        ridx, rval, cidx = orc.knn_f32(ref, cur, orc.METRIC_COSINE)
        gi, gc = r.knn_idx[0].cpu().numpy(), r.col_idx[0].cpu().numpy()
        for row in np.nonzero(gi[:, 0] != ridx[:, 0])[0]:
            s = orc.pair_scores_f64(ref, cur, [row, row], [gi[row, 0], ridx[row, 0]], orc.METRIC_COSINE)
            assert abs(s[0] - s[1]) <= REL_TIE * abs(s).max(), (n, m, row, s)
        for col in np.nonzero(gc != cidx)[0]:
            s = orc.pair_scores_f64(ref, cur, [gc[col], cidx[col]], [col, col], orc.METRIC_COSINE)
            assert abs(s[0] - s[1]) <= REL_TIE * abs(s).max(), (n, m, col, s)
        assert np.allclose(r.knn_val[0].cpu().numpy()[:, 0], rval[:, 0], atol=2e-6, rtol=0), (n, m)


@pytest.mark.parametrize("kind", ["sift_f16", "sift_tf32", "r2d2_tf32x3", "r2d2_f16x3", "bits_tc", "bits_l2", "sift_u8"])
def test_consecutive_pairs_prepared_once_equal_separate_buffers(kind):
    """Pairs of one frame sequence (cur = ref one frame on in memory: sequence.FrameSequence) take the path that prepares every
    frame once (match_f32_tc / match_bits_tc, `chained`); the same descriptors in two separate buffers take the two-sided
    path.  Same matches, distances and counts, bit for bit; ragged counts included."""
    import torch
    from vo_b200 import ops
    rng = np.random.default_rng(11)
    B, N = 5, 700 if kind != "sift_u8" else 512
    n_ref = torch.tensor([N, N - 3, 650, N, 1], dtype=torch.int32, device="cuda")
    n_cur = torch.tensor([N - 3, 650, N, 1, N], dtype=torch.int32, device="cuda")
    perms = [rng.permutation(N) for _ in range(B + 1)]      # every frame: the same N features, shuffled and perturbed
    if kind in ("bits_tc", "bits_l2"):
        base = rng.integers(0, 256, (N, 32), dtype=np.uint8)
        seq = torch.from_numpy(np.stack([base[p] ^ (rng.random((N, 32)) < 0.05).astype(np.uint8) for p in perms])).cuda()
        norm, mode = (ops.VO_NORM_HAMMING_TC, ops.VO_MODE_MUTUAL) if kind == "bits_tc" else (ops.VO_NORM_L2_U8, ops.VO_MODE_RATIO)
        call = lambda r, c: ops.match_u8(r, c, norm, mode, 0.85, n_ref=n_ref, n_cur=n_cur)
    elif kind == "sift_u8":
        base = rng.integers(0, 200, (N, 128))
        seq = torch.from_numpy(np.stack([(base[p] + rng.integers(0, 8, (N, 128))).astype(np.uint8) for p in perms])).cuda()
        call = lambda r, c: ops.match_u8(r, c, ops.VO_NORM_L2_U8, ops.VO_MODE_RATIO, 0.85, n_ref=n_ref, n_cur=n_cur)
    elif kind.startswith("sift"):
        base = rng.integers(0, 200, (N, 128))
        seq = torch.from_numpy(np.stack([(base[p] + rng.integers(0, 8, (N, 128))).astype(np.float32) for p in perms])).cuda()
        prec = ops.VO_PREC_F16X1 if kind == "sift_f16" else ops.VO_PREC_TF32X1
        call = lambda r, c: ops.match_f32(r, c, ops.VO_METRIC_L2, ops.VO_MODE_RATIO, 0.85, prec, n_ref=n_ref, n_cur=n_cur)
    else:
        base = rng.standard_normal((N, 128))
        d = np.stack([base[p] + 0.05 * rng.standard_normal((N, 128)) for p in perms]).astype(np.float32)
        seq = torch.from_numpy(d / np.linalg.norm(d, axis=2, keepdims=True)).cuda()
        prec = ops.VO_PREC_TF32X3 if kind == "r2d2_tf32x3" else ops.VO_PREC_F16X3
        call = lambda r, c: ops.match_f32(r, c, ops.VO_METRIC_COSINE, ops.VO_MODE_RATIO_MUTUAL, 0.9, prec, n_ref=n_ref, n_cur=n_cur)
    ref, cur = seq[:-1], seq[1:]
    assert cur.data_ptr() == ref.data_ptr() + ref[0].numel() * ref.element_size()       # the chained layout
    a = call(ref, cur)
    b = call(ref.clone(), cur.clone())
    torch.cuda.synchronize()
    assert torch.equal(a.count, b.count) and int(a.count.sum()) > N
    for i, c in enumerate(a.count.tolist()):                 # rows past count[b] are unspecified
        assert torch.equal(a.pairs[i, :c], b.pairs[i, :c])
        assert torch.equal(a.dist[i, :c].view(torch.int32), b.dist[i, :c].view(torch.int32))
