"""GPU-free checks of the scan-side references in tests/scan_ref.py: the scan bound holds against an emulation of the
tensor cores' blockwise fp32 accumulation and rejects a score off by one K block, the slot-set model of the pre-pass
agrees with a brute-force enumeration of scan_tc.cu's tile split, and the scan kernel shim compiles against the
library headers."""
import os
import subprocess

import numpy as np
import pytest
import torch

import encoder_ref
import scan_ref as R

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CSRC = os.path.join(ROOT, "rag-project-icd10_b200", "csrc")


def test_shim_compiles_against_the_headers(tmp_path):
    nvcc = encoder_ref.nvcc_path()
    if nvcc is None:
        pytest.skip("no nvcc")
    src = os.path.join(ROOT, "tests", "scan_kernel_shim.cu")
    cmd = [nvcc, "-gencode", "arch=compute_100a,code=sm_100a", "-std=c++17", "-Xcompiler", "-fPIC,-Wall",
           "-I", CSRC, "-I", os.path.join(ROOT, "include"), "-c", src, "-o", str(tmp_path / "shim.o")]
    r = subprocess.run(cmd, capture_output=True, text=True)
    assert r.returncode == 0, r.stderr


# ------------------------------------------------------------------------------------------------ scan bound
def _trunc32(x):
    """fp64 -> fp32 rounding toward zero (the worst an accumulator can do per add: one ulp)."""
    f = x.astype(np.float32)
    over = np.abs(f.astype(np.float64)) > np.abs(x)
    f[over] = np.nextafter(f[over], np.float32(0))
    return f


def tc_emulate(q, rows, group):
    """Tensor-core style dot of bf16(q) and bf16(rows): products exact, summed in groups of `group` consecutive K
    elements exactly, each group added to an fp32 accumulator with truncation.  [B, n] fp32."""
    bq = R.bf16_round(q).astype(np.float64)
    bc = R.bf16_round(rows).astype(np.float64)
    acc = np.zeros((bq.shape[0], bc.shape[0]), np.float32)
    for k0 in range(0, bq.shape[1], group):
        part = bq[:, k0:k0 + group] @ bc[:, k0:k0 + group].T
        acc = _trunc32(acc.astype(np.float64) + part)
    return acc


def _inputs(dim, seed):
    rng = np.random.default_rng(seed)
    rows = R._unit(rng.standard_normal((200, dim)))
    rows[:50] *= 2.0 ** rng.uniform(-20, 4, dim)                 # columns spanning 2^-20 .. 2^4
    rows[50:100] *= 10.0 ** rng.uniform(-3, 3, (50, 1))          # row norms far from 1
    rows[100:120, 0::2] = 8.0
    rows[100:120, 1::2] = -8.0                                   # large cancelling pairs
    q = R._unit(rng.standard_normal((6, dim)))
    q[0, 1::2] = q[0, 0::2]
    return rows.astype(np.float32), q.astype(np.float32)


@pytest.mark.parametrize("dim", [64, 128, 448, 768])
@pytest.mark.parametrize("group", [1, 16])
def test_scan_bound_holds_for_truncating_blockwise_accumulation(dim, group):
    rows, q = _inputs(dim, dim)
    # bf16 inputs: T alone
    bq, bc = R.bf16_round(q), R.bf16_round(rows)
    got = tc_emulate(bq, bc, group).astype(np.float64)
    e = R.exact_scores(bc, bq).numpy()
    d = R.scan_bound(bq, bc).numpy()
    assert ((np.abs(got - e) / d).max()) <= 1.0
    # fp32 queries on fp32 master rows: plus the input-rounding terms
    e32 = R.exact_scores(rows, q).numpy()
    d32 = R.scan_bound(q, rows).numpy()
    worst = (np.abs(got - e32) / d32).max()
    assert 0.0 < worst <= 1.0, worst


@pytest.mark.parametrize("dim", [128, 768])
def test_scan_bound_rejects_a_score_off_by_one_k_block(dim):
    rows, q = _inputs(dim, 3 * dim)
    bq, bc = R.bf16_round(q), R.bf16_round(rows)
    got = tc_emulate(bq, bc, 16).astype(np.float64)
    block = bq[:, 64:128].astype(np.float64) @ bc[:, 64:128].T.astype(np.float64)
    d = R.scan_bound(bq, bc).numpy()
    e = R.exact_scores(bc, bq).numpy()
    assert (np.abs(got - block - e) / d).max() >= 10.0


def test_scan_bound_terms():
    """bf16 queries on bf16 rows: exactly T; otherwise T plus the two exact input-rounding terms."""
    rows, q = _inputs(128, 5)
    bq, bc = R.bf16_round(q).astype(np.float64), R.bf16_round(rows).astype(np.float64)
    T = 2 * 128 * R.U * (np.abs(bq) @ np.abs(bc).T)
    assert np.allclose(R.scan_bound(bq.astype(np.float32), bc.astype(np.float32)).numpy(), T, rtol=1e-14, atol=0)
    want = T + np.abs(q - bq) @ np.abs(rows.astype(np.float64)).T + np.abs(bq) @ np.abs(rows - bc).T
    assert np.allclose(R.scan_bound(q, rows).numpy(), want, rtol=1e-14, atol=0)


def test_colstat_slack_is_the_smaller_of_its_two_forms():
    dim = 64
    rng = np.random.default_rng(1)
    q = rng.standard_normal((3, dim)).astype(np.float32)
    cs = np.concatenate([np.full(dim, 2.0), np.full(dim, 0.01), [1e6, 1e6]]).astype(np.float32)
    A, T, C = R.colstat_slack(q, cs, True)
    bq = R.bf16_round(q).astype(np.float64)
    assert np.allclose(A.numpy(), np.abs(q - bq).sum(1) * 2.0 + np.abs(bq).sum(1) * 0.01, rtol=1e-6)
    assert np.allclose(T.numpy(), 2 * dim * R.U * np.abs(bq).sum(1) * 2.0, rtol=1e-12)
    L = R.lanes_fmas(dim, True)
    assert np.allclose(C.numpy(), (L + 5) * R.U * np.abs(q).sum(1) * 2.01, rtol=1e-6)
    cs[-2:] = 1e-3        # small row norms: the Cauchy-Schwarz form wins
    A, T, C = R.colstat_slack(q, cs, True)
    nb = np.linalg.norm(bq, axis=1) * (1 + 1e-6)
    assert np.allclose(T.numpy(), 2 * dim * R.U * nb * np.float32(1e-3), rtol=1e-9)


# ------------------------------------------------------------------------------------------------ slot-set model
def _brute_groups(n_rows, stride, G):
    """scan_tc.cu as written: total_tiles = ceil(ceil(n / 128) / stride), CTA g scans tiles [T g / G, T (g + 1) / G)
    of the pass, sampled tile t starts at row t * stride * 128, and the epilogue puts column c of it in slot c % 32."""
    total = ((n_rows + 127) // 128 + stride - 1) // stride
    out = {}
    for g in range(G):
        t0, t1 = total * g // G, total * (g + 1) // G
        for t in range(t0, t1):
            row0 = t * stride * 128
            for c in range(128):
                if row0 + c < n_rows:
                    out[row0 + c] = (g, c % 32)
    return out


@pytest.mark.parametrize("n_rows,stride,G", [(1000, 3, 2), (6001, 1, 47), (6001, 7, 5), (20011, 2, 74),
                                             (20011, 3, 37), (129, 1, 2), (1, 1, 1), (600001, 64, 13)])
def test_slot_sets_match_a_brute_force_enumeration(n_rows, stride, G):
    rows, g, slot, cls = R.slot_sets(n_rows, stride, G)
    brute = _brute_groups(n_rows, stride, G)
    assert sorted(brute) == sorted(rows.tolist())
    for r, gg, ss, cc in zip(rows.tolist(), g.tolist(), slot.tolist(), cls.tolist()):
        assert brute[r] == (gg, ss) and cc == gg % 4


def test_expected_slot_max_and_bound_match_brute_force():
    rng = np.random.default_rng(4)
    n, stride, G, B = 3001, 3, 7, 5
    scores = (rng.integers(0, 50, (B, n)) / 4.0).astype(np.float32)
    allowed = rng.random(n) < 0.6
    sm = R.expected_slot_max(scores, n, stride, G, allowed)
    brute = _brute_groups(n, stride, G)
    want = np.full((B, G, 32), -np.inf, np.float32)
    for r, (g, s) in brute.items():
        if allowed[r]:
            want[:, g, s] = np.maximum(want[:, g, s], scores[:, r])
    assert np.array_equal(sm, want)
    # bound: the kc-th largest of the 128 class maxima; a set of rows reaching it has >= kc members
    for kc in (1, 2, 17, 64, 128):
        keys = R.bound_from_slots(sm, kc)
        for b in range(B):
            fold = np.full((4, 32), -np.inf, np.float32)
            for g in range(G):
                fold[g % 4] = np.maximum(fold[g % 4], sm[b, g])
            v = np.sort(fold.ravel())[::-1][kc - 1]
            assert keys[b] == (R.MIN_KEY if np.isneginf(v) else R.float_key(np.float32([v]))[0])
            if not np.isneginf(v):
                assert int((scores[b, allowed] >= v).sum()) >= kc      # a lower bound of the kc-th best allowed score


def test_float_key_orders_like_the_floats():
    x = np.array([-np.inf, -3.0, -1e-30, -0.0, 0.0, 1e-45, 1.0, 2.0, np.inf], np.float32)
    k = R.float_key(x)
    assert (np.diff(k.astype(np.int64)) >= 0).all() and k[3] == -1 and k[4] == 0
    # the empty bound's key sits below every finite score a scan can produce above -3.3e38
    assert R.float_key(np.float32([-np.inf]))[0] < R.MIN_KEY < R.float_key(np.float32([-3.3e38]))[0]


# ------------------------------------------------------------------------------------------------ chunked certificate
import test_scan_ref_cpu as REF   # noqa: E402  (the probe corpus and planted defects of the certificate's own tests)

_CERTIFY = R.certify


def _both_forms(*a, **kw):
    """certify from the whole score matrix and from 97-row chunks: the same verdict and ratios, or the same rejection."""
    kw.pop("chunk_rows", None)
    try:
        full = _CERTIFY(*a, **kw)
    except AssertionError as e:
        with pytest.raises(AssertionError) as ei:
            _CERTIFY(*a, chunk_rows=97, **{x: y for x, y in kw.items() if x != "ref"})
        assert str(ei.value).split("\n")[0] == str(e).split("\n")[0]
        raise
    part = _CERTIFY(*a, chunk_rows=97, **{x: y for x, y in kw.items() if x != "ref"})
    # the chunks' fp64 products may round differently from the whole matrix's in the last bit
    assert (part.worst <= 1.0) == (full.worst <= 1.0), (part, full)
    assert np.allclose([part.score_ratio, part.gap_ratio], [full.score_ratio, full.gap_ratio], rtol=1e-6), (part, full)
    return full


DEFECT_CASES = [("test_correct_result_is_certified", ()), ("test_swap_at_a_3e_5_gap_is_rejected", ()),
                ("test_dropped_last_partial_tile_is_rejected", ()), ("test_zeroed_k_block_is_rejected", (5,)),
                ("test_permuted_k_block_is_rejected", (7,)), ("test_swapped_query_lanes_are_rejected", ((31, 32),)),
                ("test_wrong_id_tie_break_is_rejected", ()), ("test_pre_weight_applied_after_selection_is_rejected", ()),
                ("test_mask_rules", None)]


@pytest.mark.parametrize("name,args", DEFECT_CASES)
def test_chunked_certificate_gives_the_same_verdicts(monkeypatch, name, args):
    """The probe corpus of test_scan_ref_cpu.py with each of its planted defects: certify over row chunks accepts and
    rejects exactly what the whole-matrix form does, with the same ratios."""
    monkeypatch.setattr(R, "certify", _both_forms)
    fn = getattr(REF, name)
    if args is None:
        fn()
        return
    rows, q, plants = R.probe_corpus(REF.N_ROWS, REF.DIM, REF.B, seed=7)
    fn((rows, q, plants, REF._levels(REF.N_ROWS, 8)), *args)


def test_chunked_certificate_on_the_clustered_model():
    monkeypatch = pytest.MonkeyPatch()
    monkeypatch.setattr(R, "certify", _both_forms)
    try:
        REF.test_model_of_the_uncertified_tensor_path_misses_true_top_k()
    finally:
        monkeypatch.undo()
