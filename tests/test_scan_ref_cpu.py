"""GPU-free checks of tests/scan_ref.py: the fp64 reference and canonical bound agree with torch and with an emulation
of the kernels' lane order, and the certificate rejects planted scan defects that parity.check_topk lets through."""
import numpy as np
import pytest
import torch

import scan_ref as R
from parity import check_topk

U = R.U


# ------------------------------------------------------------------------------------------------ helpers
def canonical_dot(rows, q, f32rows):
    """numpy emulation of warp_dot_row / scan_stream_kernel: 16-byte chunk c on lane c % 32, chunks ascending, elements
    ascending, one fp32 fma each (the product is exact in fp64, so one fp64 add then one rounding to fp32), then the
    xor butterfly 16, 8, 4, 2, 1 in fp32.  rows: [n, dim] fp32 values (bf16 values when not f32rows), q: [dim] fp32."""
    n, dim = rows.shape
    E = 4 if f32rows else 8
    nch = dim // E
    it = -(-nch // 32)
    R_ = np.zeros((n, it * 32 * E), np.float64)
    R_[:, :dim] = rows
    Q_ = np.zeros(it * 32 * E, np.float64)
    Q_[:dim] = q
    R_ = R_.reshape(n, it, 32, E)
    Q_ = Q_.reshape(it, 32, E)
    acc = np.zeros((n, 32), np.float32)
    for i in range(it):
        for e in range(E):
            acc = (acc.astype(np.float64) + R_[:, i, :, e] * Q_[i, :, e]).astype(np.float32)
    lanes = np.arange(32)
    for off in (16, 8, 4, 2, 1):
        acc = (acc + acc[:, lanes ^ off]).astype(np.float32)
    return acc[:, 0]


def emulate_search(scores_sel, raw_of, k, weight_mode, levels, allowed=None):
    """A scan as the kernels run it: top-k by (key desc, id asc) over scores_sel [B, n] (fp64), raw_of(b, ids) -> fp32
    raw scores of the rows kept, then finalise_kernel's weight rules.  Returns (ids, raw, score) [B, k]."""
    B, n = scores_sel.shape
    w32 = np.asarray(R.WEIGHTS, np.float32)[levels]
    ids = np.full((B, k), -1, np.int64)
    raw = np.full((B, k), -np.inf, np.float32)
    score = np.full((B, k), -np.inf, np.float32)
    for b in range(B):
        s = scores_sel[b].copy()
        if weight_mode == R.WEIGHT_PRE:
            s = s * w32
        cand = np.arange(n) if allowed is None else np.nonzero(allowed)[0]
        top = cand[np.lexsort((cand, -s[cand]))][:k]
        r = np.asarray(raw_of(b, top), np.float32)
        if weight_mode == R.WEIGHT_PRE:
            key = (r * w32[top]).astype(np.float32)
            o = np.lexsort((top, -key.astype(np.float64)))
            top, r, sc = top[o], r[o], key[o]
        else:
            o = np.lexsort((top, -r.astype(np.float64)))
            top, r = top[o], r[o]
            sc = r.copy()
            if weight_mode == R.WEIGHT_RERANK:
                w = r.astype(np.float64) * np.asarray(R.WEIGHTS)[levels[top]]
                o = np.argsort(-w, kind="stable")
                top, r, sc = top[o], r[o], w[o].astype(np.float32)
        m = len(top)
        ids[b, :m], raw[b, :m], score[b, :m] = top, r, sc
    return ids, raw, score


def _levels(n, seed):
    return np.random.default_rng(seed).choice(np.array([1, 2, 3], np.uint8), size=n, p=[0.12, 0.3, 0.58])


def _exact_raw(rows, q):
    return lambda b, ids: (rows[ids].astype(np.float64) @ q[b].astype(np.float64)).astype(np.float32)


def _oracle_topk(rows, q, k):
    e = rows.astype(np.float64) @ q.astype(np.float64).T
    ids = np.stack([np.lexsort((np.arange(len(rows)), -e[:, b]))[:k] for b in range(q.shape[0])])
    return np.take_along_axis(e.T, ids, 1), ids


# ------------------------------------------------------------------------------------------------ 1. reference and bound
@pytest.mark.parametrize("f32rows", [False, True])
def test_exact_scores_and_bound_equal_torch_float64(f32rows):
    rng = np.random.default_rng(1)
    rows = R.held_rows(rng.standard_normal((300, 256)).astype(np.float32), f32rows)
    q = rng.standard_normal((7, 256)).astype(np.float32)
    want = torch.from_numpy(q).double() @ torch.from_numpy(rows).double().T
    assert torch.equal(R.exact_scores(rows, q), want)
    L = 4 * 2 if f32rows else 8 * 1
    want_b = (L + 5) * U * (torch.from_numpy(q).double().abs() @ torch.from_numpy(rows).double().abs().T)
    assert torch.allclose(R.canonical_bound(q, rows, f32rows), want_b, rtol=1e-15, atol=0)
    assert R.lanes_fmas(768, False) == 24 and R.lanes_fmas(768, True) == 24
    assert R.lanes_fmas(1024, True) == 32 and R.lanes_fmas(8, False) == 8 and R.lanes_fmas(264, False) == 16


@pytest.mark.parametrize("dim", [8, 16, 64, 248, 256, 264, 512, 520, 768, 776, 1016, 1024])
@pytest.mark.parametrize("f32rows", [False, True])
def test_emulated_canonical_dot_stays_within_the_bound(dim, f32rows):
    rng = np.random.default_rng(dim)
    rows = R._unit(rng.standard_normal((400, dim))).astype(np.float32)
    # large-magnitude, mixed-sign rows make the rounding error visible
    rows[:100] *= 1.0 + 60.0 * rng.random((100, 1)).astype(np.float32)
    rows = R.held_rows(rows, f32rows)
    q = rng.standard_normal((3, dim)).astype(np.float32)
    e, d = R.reference(rows, q, f32rows)
    worst = 0.0
    for b in range(q.shape[0]):
        got = canonical_dot(rows, q[b], f32rows).astype(np.float64)
        err = np.abs(got - e[b].numpy())
        worst = max(worst, float((err / d[b].numpy()).max()))
    assert worst <= 1.0, worst
    assert worst > 0.0     # the emulation does round


# ------------------------------------------------------------------------------------------------ 2. planted defects
N_ROWS, DIM, B = 1000, 768, 130       # 7 full row tiles + a partial one (896..999), 12 K blocks, lanes 0..129


@pytest.fixture(scope="module")
def probes():
    rows, q, plants = R.probe_corpus(N_ROWS, DIM, B, seed=7)
    levels = _levels(N_ROWS, 8)
    return rows, q, plants, levels


def _check_topk_passes(ids, raw, rows, q, k):
    """What parity.check_topk (TIE_TOL, the B k / 50 swap budget) says about the same result."""
    ref_s, ref_i = _oracle_topk(rows, q, k)
    ex = lambda b, i: rows[np.asarray(i)].astype(np.float64) @ q[b].astype(np.float64)
    swaps = check_topk(ids, raw, ref_i, ref_s, ex, score_tol=2e-6)
    return swaps <= max(1, ids.shape[0] * k // 50)


def test_correct_result_is_certified(probes):
    rows, q, plants, levels = probes
    e = R.exact_scores(rows, q).numpy()
    for wm in (R.WEIGHT_NONE, R.WEIGHT_PRE, R.WEIGHT_RERANK):
        ids, raw, score = emulate_search(e, _exact_raw(rows, q), 10, wm, levels)
        cert = R.certify(ids, raw, score, rows, q, 10, wm, levels, f32rows=True)
        assert cert.worst <= 1.0, cert
    for l, r in plants.items():
        assert ids[l, :].tolist().count(r) == 1


def test_swap_at_a_3e_5_gap_is_rejected(probes):
    """A true top-10 row replaced by rank 11, 3e-5 below it: a tie for parity.TIE_TOL, 10x the bound here."""
    rows, q, plants, levels = probes
    rows = rows.copy()
    b, k = 3, 10
    e = R.exact_scores(rows, q).numpy()
    order = np.lexsort((np.arange(N_ROWS), -e[b]))
    r10 = order[k - 1]
    spare = order[k + 50]     # a row far down the list becomes rank 11, 3e-5 below rank 10
    rows[spare] = rows[r10] - 3e-5 * q[b] / float(q[b] @ q[b])
    e = R.exact_scores(rows, q).numpy()
    assert np.lexsort((np.arange(N_ROWS), -e[b]))[k] == spare
    ids, raw, score = emulate_search(e, _exact_raw(rows, q), k, R.WEIGHT_NONE, levels)
    ids[b, k - 1], raw[b, k - 1] = spare, _exact_raw(rows, q)(b, [spare])[0]
    score[b] = raw[b]
    assert _check_topk_passes(ids, raw, rows, q, k)
    cert = R.certify(ids, raw, score, rows, q, k, R.WEIGHT_NONE, levels, f32rows=True, strict=False)
    assert cert.gap_ratio >= 10.0, cert


def _defect_ratio(rows, q, levels, sel_scores, k=10, wm=R.WEIGHT_NONE):
    """Selection on defective scores, exact rescoring of what was kept (finalise_kernel): only the certificate's gap rule
    can see the defect."""
    ids, raw, score = emulate_search(sel_scores, _exact_raw(rows, q), k, wm, levels)
    return R.certify(ids, raw, score, rows, q, k, wm, levels, f32rows=True, strict=False), ids, raw


def test_dropped_last_partial_tile_is_rejected(probes):
    rows, q, plants, levels = probes
    e = R.exact_scores(rows, q).numpy()
    sel = e.copy()
    sel[:, 896:] = -np.inf
    cert, ids, raw = _defect_ratio(rows, q, levels, sel)
    assert N_ROWS - 1 in plants.values()
    assert cert.gap_ratio >= 10.0, cert


@pytest.mark.parametrize("kb", [0, 5, 11])
def test_zeroed_k_block_is_rejected(probes, kb):
    rows, q, plants, levels = probes
    bad = rows.copy()
    bad[:, kb * 64:(kb + 1) * 64] = 0
    cert, _, _ = _defect_ratio(rows, q, levels, R.exact_scores(bad, q).numpy())
    assert cert.gap_ratio >= 10.0, cert


@pytest.mark.parametrize("kb", [0, 7])
def test_permuted_k_block_is_rejected(probes, kb):
    """A 128-byte-swizzle error: the eight 16-byte chunks of one 64-wide K block read in xor-permuted order."""
    rows, q, plants, levels = probes
    perm = (np.arange(64) // 8 ^ 3) * 8 + np.arange(64) % 8
    bad = rows.copy()
    bad[:, kb * 64:(kb + 1) * 64] = rows[:, kb * 64 + perm]
    cert, _, _ = _defect_ratio(rows, q, levels, R.exact_scores(bad, q).numpy())
    assert cert.gap_ratio >= 10.0, cert


@pytest.mark.parametrize("lanes", [(31, 32), (63, 64), (0, 127)])
def test_swapped_query_lanes_are_rejected(probes, lanes):
    rows, q, plants, levels = probes
    qb = q.copy()
    qb[list(lanes)] = q[list(lanes[::-1])]
    cert, _, _ = _defect_ratio(rows, q, levels, R.exact_scores(rows, qb).numpy())
    assert cert.gap_ratio >= 10.0, cert


def test_wrong_id_tie_break_is_rejected(probes):
    """Exact duplicates at the k-th place: the lower id must win (cand_before), and within the list come first."""
    rows, q, plants, levels = probes
    rows = rows.copy()
    b, k = 9, 10
    e = R.exact_scores(rows, q).numpy()
    order = np.lexsort((np.arange(N_ROWS), -e[b]))
    j = int(order[k - 1])
    lower = [r for r in order[k + 20:] if r < j]
    i = int(lower[0])
    rows[i] = rows[j]                    # i < j, identical rows: i is the 10th, j the 11th
    e = R.exact_scores(rows, q).numpy()
    ids, raw, score = emulate_search(e, _exact_raw(rows, q), k, R.WEIGHT_NONE, levels)
    assert ids[b, k - 1] == i
    R.certify(ids, raw, score, rows, q, k, R.WEIGHT_NONE, levels, f32rows=True)
    wrong = ids.copy()
    wrong[b, k - 1] = j
    assert _check_topk_passes(wrong, raw, rows, q, k)
    with pytest.raises(AssertionError, match="tied row with a lower id"):
        R.certify(wrong, raw, score, rows, q, k, R.WEIGHT_NONE, levels, f32rows=True)
    # both in the list (k = 11), in the wrong order
    ids, raw, score = emulate_search(e, _exact_raw(rows, q), k + 1, R.WEIGHT_NONE, levels)
    assert ids[b, k - 1] == i and ids[b, k] == j
    ids[b, [k - 1, k]] = [j, i]
    with pytest.raises(AssertionError, match="order"):
        R.certify(ids, raw, score, rows, q, k + 1, R.WEIGHT_NONE, levels, f32rows=True)


def test_pre_weight_applied_after_selection_is_rejected(probes):
    rows, q, plants, levels = probes
    k = 10
    e = R.exact_scores(rows, q).numpy()
    ids, raw, _ = emulate_search(e, _exact_raw(rows, q), k, R.WEIGHT_NONE, levels)
    # weight after selection: same ids, sorted by raw * w
    w32 = np.asarray(R.WEIGHTS, np.float32)[levels]
    key = (raw * w32[ids]).astype(np.float32)
    o = np.lexsort((ids, -key.astype(np.float64)), axis=-1)
    ids, raw, key = (np.take_along_axis(x, o, 1) for x in (ids, raw, key))
    cert = R.certify(ids, raw, key, rows, q, k, R.WEIGHT_PRE, levels, f32rows=True, strict=False)
    assert cert.gap_ratio >= 10.0, cert


def test_mask_rules():
    rows, q, plants = R.probe_corpus(300, 128, 6, seed=3)
    levels = _levels(300, 4)
    allowed = np.random.default_rng(5).random(300) < 0.5
    e = R.exact_scores(rows, q).numpy()
    ids, raw, score = emulate_search(e, _exact_raw(rows, q), 10, R.WEIGHT_NONE, levels, allowed)
    R.certify(ids, raw, score, rows, q, 10, R.WEIGHT_NONE, levels, mask=allowed, f32rows=True)
    # the unmasked result breaks the mask
    ids2, raw2, score2 = emulate_search(e, _exact_raw(rows, q), 10, R.WEIGHT_NONE, levels)
    with pytest.raises(AssertionError, match="masked-out"):
        R.certify(ids2, raw2, score2, rows, q, 10, R.WEIGHT_NONE, levels, mask=allowed, f32rows=True)
    # fewer allowed rows than k: the count is min(k, allowed) with a (-inf, -1) tail
    few = np.zeros(300, bool)
    few[[4, 90, 299]] = True
    ids, raw, score = emulate_search(e, _exact_raw(rows, q), 10, R.WEIGHT_NONE, levels, few)
    R.certify(ids, raw, score, rows, q, 10, R.WEIGHT_NONE, levels, mask=few, f32rows=True)
    ids[0, 3] = 5
    with pytest.raises(AssertionError, match="counts"):
        R.certify(ids, raw, score, rows, q, 10, R.WEIGHT_NONE, levels, mask=few, f32rows=True)


# ------------------------------------------------------------------------------------------------ 3. model of the old tensor path
def clustered_corpus(seed, dim=768, n_background=2000, clusters=((100, 0.015), (300, 0.01), (40, 0.02))):
    """Near-duplicate clusters (member = unit(center + spread * unit noise)) over a random background."""
    rng = np.random.default_rng(seed)
    parts, centers = [R._unit(rng.standard_normal((n_background, dim)))], []
    for size, spread in clusters:
        c = R._unit(rng.standard_normal(dim))
        centers.append(c)
        parts.append(R._unit(c + spread * R._unit(rng.standard_normal((size, dim)))))
    rows = np.concatenate(parts).astype(np.float32)
    return rows, np.stack(centers).astype(np.float32), rng


def test_model_of_the_uncertified_tensor_path_misses_true_top_k():
    """A CPU MODEL of the tensor path as it selected candidates before its certificate existed -- not a test of the
    kernel.  It documents why the certificate and the exact fallback exist: with fp32 master rows the scan kept the
    top kc = 2k + 16 by bf16(row) . bf16(query) (fp64 here, in place of the MMA) and rescored only those against the
    fp32 rows, and in a cluster of near-duplicates the true fp32 top-10 is not always among them."""
    rows, centers, rng = clustered_corpus(seed=2024)
    k, kc = 10, 36
    q = R._unit(centers[rng.integers(0, len(centers), 200)] + 0.05 * R._unit(rng.standard_normal((200, rows.shape[1]))))
    q = q.astype(np.float32)
    levels = _levels(len(rows), 9)
    scan = R.exact_scores(R.bf16_round(rows), R.bf16_round(q)).numpy()
    e = R.exact_scores(rows, q).numpy()
    raw_of = lambda b, ids: e[b, ids].astype(np.float32)
    ids = np.zeros((200, k), np.int64)
    raw = np.zeros((200, k), np.float32)
    for b in range(200):
        cand = np.lexsort((np.arange(len(rows)), -scan[b]))[:kc]
        top = cand[np.lexsort((cand, -e[b, cand]))][:k]
        r = raw_of(b, top)
        o = np.lexsort((top, -r.astype(np.float64)))       # finalise_kernel's (raw desc, id asc)
        ids[b], raw[b] = top[o], r[o]
    true_i = np.stack([np.lexsort((np.arange(len(rows)), -e[b]))[:k] for b in range(200)])
    missed = [b for b in range(200) if set(ids[b].tolist()) != set(true_i[b].tolist())]
    assert len(missed) >= 5, len(missed)
    print(f"model: {len(missed)} of 200 queries miss a true top-{k} row")
    # parity.check_topk's tie rule calls every miss a swap among near-ties; the certificate rejects them by 10x or more
    ref_s, ref_i = _oracle_topk(rows, q, k)
    check_topk(ids, raw, ref_i, ref_s, lambda b, i: e[b, np.asarray(i)], score_tol=2e-6)
    cert = R.certify(ids[missed], raw[missed], raw[missed], rows, q[missed], k, R.WEIGHT_NONE, levels, f32rows=True,
                     strict=False)
    assert cert.gap_ratio >= 10.0, cert
    # the same queries selected on the fp32 scores themselves are certified
    ok_i = true_i[missed]
    ok_r = np.take_along_axis(e[missed], ok_i, 1).astype(np.float32)
    o = np.lexsort((ok_i, -ok_r.astype(np.float64)), axis=-1)
    ok_i, ok_r = np.take_along_axis(ok_i, o, 1), np.take_along_axis(ok_r, o, 1)
    R.certify(ok_i, ok_r, ok_r, rows, q[missed], k, R.WEIGHT_NONE, levels, f32rows=True)
