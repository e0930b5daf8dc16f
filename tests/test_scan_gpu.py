"""GPU parity of the exact top-k scan (both kernels) against the CPU oracle, through the C ABI."""
import numpy as np
import pytest

from oracle import search as osearch
from parity import check_topk

pytestmark = pytest.mark.gpu


def _corpus(n, dim, seed, bf16=True):
    rng = np.random.default_rng(seed)
    x = rng.standard_normal((n, dim)).astype(np.float32)
    x /= np.linalg.norm(x, axis=1, keepdims=True)
    return osearch.bf16_round(x) if bf16 else x


def _levels(n, seed):
    rng = np.random.default_rng(seed)
    return rng.choice(np.array([1, 2, 3], np.uint8), size=n, p=[0.1243, 0.2991, 0.5766]).astype(np.uint8)


def _index(pkg, corpus, levels, keep_f32=False):
    from importlib import import_module
    VectorIndex = import_module("rag-project-icd10_b200.engine.index").VectorIndex
    idx = VectorIndex(corpus.shape[1], device=0, keep_f32=keep_f32)
    idx.append(corpus, levels)
    assert len(idx) == corpus.shape[0]
    return idx


def _exact_of(corpus, q):
    return lambda b, ids: corpus[np.asarray(ids)] @ q[b]


@pytest.mark.parametrize("path", [1, 2])
@pytest.mark.parametrize("n,B,k", [(5000, 1, 10), (5000, 3, 5), (40474, 7, 10), (20000, 130, 10),
                                    (3001, 257, 1), (9999, 33, 100), (64, 2, 10), (1, 1, 10), (7, 5, 10)])
def test_scan_matches_oracle(pkg, native, path, n, B, k):
    dim = 768
    corpus = _corpus(n, dim, seed=n + B)
    levels = _levels(n, seed=n)
    q = _corpus(B, dim, seed=999 + B)
    idx = _index(pkg, corpus, levels)
    score, raw, ids = idx.search(q, k, weight_mode=native.WEIGHT_NONE, path=path)
    ref_s, ref_i = osearch.exact_topk(corpus, q, k)
    kk = min(k, n)
    assert np.all(ids[:, kk:] == -1) and np.all(np.isneginf(raw[:, kk:]))
    swaps = check_topk(ids[:, :kk], raw[:, :kk], ref_i, ref_s, _exact_of(corpus, q), score_tol=2e-6)
    assert np.array_equal(score, raw)
    assert swaps <= max(1, B * kk // 50), f"{swaps} tie swaps out of {B * kk}"
    idx.close()


def test_stream_and_tensor_paths_agree_bitwise(pkg, native):
    """Both scan kernels feed the same canonical fp32 rescoring, so scores agree bit for bit."""
    corpus = _corpus(30000, 768, seed=5)
    levels = _levels(30000, seed=6)
    q = _corpus(64, 768, seed=7)
    idx = _index(pkg, corpus, levels)
    s1, r1, i1 = idx.search(q, 10, weight_mode=native.WEIGHT_RERANK, path=native.PATH_STREAM)
    s2, r2, i2 = idx.search(q, 10, weight_mode=native.WEIGHT_RERANK, path=native.PATH_TENSOR)
    assert np.array_equal(i1, i2)
    assert np.array_equal(r1.view(np.uint32), r2.view(np.uint32))
    assert np.array_equal(s1.view(np.uint32), s2.view(np.uint32))
    idx.close()


@pytest.mark.parametrize("path", [1, 2])
def test_rerank_matches_reference_rule(pkg, native, path):
    """ICD_WEIGHT_RERANK == milvus_service.py:290-314: raw top-k, score*w(level), stable re-sort."""
    n, B, k = 40474, 16, 10
    corpus = _corpus(n, 768, seed=11)
    levels = _levels(n, seed=12)
    q = _corpus(B, 768, seed=13)
    idx = _index(pkg, corpus, levels)
    score, raw, ids = idx.search(q, k, weight_mode=native.WEIGHT_RERANK, path=path)
    ref_s, ref_i = osearch.exact_topk(corpus, q, k)
    for b in range(B):
        assert set(ids[b].tolist()) == set(ref_i[b].tolist())
        # re-rank the kernel's own raw list with the oracle rule: must reproduce the kernel's order
        order0 = np.lexsort((ids[b], -raw[b].astype(np.float64)))
        order, weighted = osearch.rerank(raw[b][order0], levels[ids[b][order0]])
        assert [int(ids[b][order0][j]) for j in order] == ids[b].tolist()
        np.testing.assert_allclose(score[b], np.array([weighted[j] for j in order], np.float32), rtol=0, atol=1e-7)
    idx.close()


@pytest.mark.parametrize("path", [1, 2])
def test_pre_weighting_selects_on_weighted_score(pkg, native, path):
    n, B, k = 20000, 9, 10
    corpus = _corpus(n, 768, seed=21)
    levels = _levels(n, seed=22)
    q = _corpus(B, 768, seed=23)
    idx = _index(pkg, corpus, levels)
    score, raw, ids = idx.search(q, k, weight_mode=native.WEIGHT_PRE, path=path)
    w = np.array([1.0, 1.2, 1.0, 0.8], np.float32)[levels]
    full = (q @ corpus.T) * w[None, :]
    for b in range(B):
        ref = np.lexsort((np.arange(n), -full[b].astype(np.float64)))[:k]
        got_w = full[b][ids[b]]
        assert np.all(np.abs(got_w - full[b][ref]) <= 1e-3)
        np.testing.assert_allclose(score[b], got_w, atol=2e-6)
    idx.close()


def test_fp32_master_search_is_exact_fp32(pkg, native):
    """KEEP_F32 tables are searched like Milvus FLAT: fp32 rows, fp32 query, fp32 accumulate."""
    n, k = 40474, 10
    corpus = _corpus(n, 768, seed=31, bf16=False)
    q = _corpus(4, 768, seed=32, bf16=False)
    idx = _index(pkg, corpus, _levels(n, 33), keep_f32=True)
    for path in (native.PATH_AUTO, native.PATH_TENSOR):
        score, raw, ids = idx.search(q, k, weight_mode=native.WEIGHT_NONE, path=path)
        ref_s, ref_i = osearch.exact_topk(corpus, q, k)
        check_topk(ids, raw, ref_i, ref_s, _exact_of(corpus, q), score_tol=2e-6)
    got = idx.read(100, 5)
    assert np.array_equal(got, corpus[100:105])
    idx.close()


def test_device_tensors_and_adopt(pkg, native):
    import torch
    n, B, k = 50000, 200, 10
    corpus = _corpus(n, 768, seed=41)
    levels = _levels(n, 42)
    q = _corpus(B, 768, seed=43)
    t = torch.from_numpy(corpus).cuda().to(torch.bfloat16)
    lv = torch.from_numpy(levels).cuda()
    from importlib import import_module
    VectorIndex = import_module("rag-project-icd10_b200.engine.index").VectorIndex
    idx = VectorIndex(768, device=0)
    idx.adopt(t, lv)
    qd = torch.from_numpy(q).cuda().to(torch.bfloat16)
    score, raw, ids = idx.search(qd, k, weight_mode=native.WEIGHT_NONE)
    torch.cuda.synchronize()
    assert ids.is_cuda and raw.dtype == torch.float32
    ref_s, ref_i = osearch.exact_topk(corpus, q, k)
    check_topk(ids.cpu().numpy(), raw.cpu().numpy(), ref_i, ref_s, _exact_of(corpus, q), score_tol=2e-6)
    with pytest.raises(native.NativeError):
        idx.append(corpus[:4], levels[:4])
    idx.close()


def test_append_grows_and_clear(pkg, native):
    corpus = _corpus(5000, 768, seed=51)
    levels = _levels(5000, 52)
    from importlib import import_module
    VectorIndex = import_module("rag-project-icd10_b200.engine.index").VectorIndex
    idx = VectorIndex(768, device=0, capacity=16)
    for lo in range(0, 5000, 700):
        idx.append(corpus[lo:lo + 700], levels[lo:lo + 700])
    assert len(idx) == 5000
    q = _corpus(2, 768, seed=53)
    _, raw, ids = idx.search(q, 5, weight_mode=native.WEIGHT_NONE)
    ref_s, ref_i = osearch.exact_topk(corpus, q, 5)
    check_topk(ids, raw, ref_i, ref_s, _exact_of(corpus, q), score_tol=2e-6)
    idx.clear()
    assert len(idx) == 0
    _, raw, ids = idx.search(q, 5)
    assert np.all(ids == -1)
    idx.close()


def test_small_dim_golden_vectors(pkg, native, golden_dir):
    """The 8-d vectors of tests/golden/milvus_service_golden.json (reference-generated)."""
    import json, os
    g = json.load(open(os.path.join(golden_dir, "milvus_service_golden.json"), encoding="utf-8"))
    vecs = np.asarray(g["vectors"], np.float32)
    from importlib import import_module
    VectorIndex = import_module("rag-project-icd10_b200.engine.index").VectorIndex
    idx = VectorIndex(vecs.shape[1], device=0, keep_f32=True)
    idx.append(vecs, np.ones(len(vecs), np.uint8))
    for s in g["searches"]:
        q = np.asarray(s["query"], np.float32)
        _, raw, ids = idx.search(q, s["top_k"], weight_mode=native.WEIGHT_NONE)
        want = sorted(s["hits"], key=lambda h: -h["original_score"])
        got_codes = [g["codes"][int(i)] for i in ids[0]]
        assert sorted(got_codes) == sorted(h["code"] for h in want)
        np.testing.assert_allclose(np.sort(raw[0])[::-1], [h["original_score"] for h in want], atol=1e-6)
    idx.close()


def test_full_size_properties(pkg, native):
    """BASELINE-size property checks (no oracle pass over 10 M rows): planted neighbours are found,
    results are sorted, and the two kernels agree."""
    import torch
    n, B, k, dim = 2_000_000, 256, 10, 768
    g = torch.Generator(device="cuda").manual_seed(1234)
    t = torch.empty((n, dim), dtype=torch.bfloat16, device="cuda")
    for lo in range(0, n, 250_000):
        x = torch.randn((250_000, dim), generator=g, device="cuda")
        t[lo:lo + 250_000] = torch.nn.functional.normalize(x, dim=1).to(torch.bfloat16)
    lv = torch.randint(1, 4, (n,), device="cuda", dtype=torch.uint8, generator=g)
    planted = torch.randint(0, n, (B,), device="cuda", generator=g)
    q = torch.nn.functional.normalize(t[planted].float() + 0.3 / dim ** 0.5 * torch.randn((B, dim), device="cuda", generator=g), dim=1)
    q = q.to(torch.bfloat16)
    from importlib import import_module
    VectorIndex = import_module("rag-project-icd10_b200.engine.index").VectorIndex
    idx = VectorIndex(dim, device=0)
    idx.adopt(t, lv)
    _, raw2, ids2 = idx.search(q, k, weight_mode=native.WEIGHT_NONE, path=native.PATH_TENSOR)
    _, raw1, ids1 = idx.search(q[:8], k, weight_mode=native.WEIGHT_NONE, path=native.PATH_STREAM)
    torch.cuda.synchronize()
    assert torch.equal(ids2[:, 0], planted)
    assert torch.all(raw2[:, :-1] >= raw2[:, 1:])
    assert torch.equal(ids1, ids2[:8]) and torch.equal(raw1, raw2[:8])
    # checksum-style property: the k-th score bounds every other row (sampled)
    sample = torch.randint(0, n, (4096,), device="cuda", generator=g)
    s = q.float() @ t[sample].float().T
    assert torch.all(s <= raw2[:, :1] + 1e-6)
    idx.close()


@pytest.mark.parametrize("knobs", [dict(scan_sample=4), dict(scan_sample=3, scan_drift=1), dict(scan_sample=0, scan_drift=0),
                                   dict(scan_sample=8, scan_tmax=2), dict(scan_sample=2, scan_kbs=2), dict(scan_kbs=6), dict(scan_kbs=4, scan_qsplit=0),
                                   dict(scan_qsplit=0), dict(scan_qsplit=1, scan_sample=4), dict(scan_qsplit=1, scan_tmax=1),
                                   dict(scan_sample=4, scan_pre_slots=0), dict(scan_sample=2, scan_pre_slots=0, scan_tmax=2),
                                   dict(scan_sample=16, scan_pair=0), dict(scan_sample=5, scan_generic=1)])
@pytest.mark.parametrize("weight_mode", [2, 1])
def test_tensor_scan_knobs_keep_results_exact(pkg, native, knobs, weight_mode):
    """The sampling pre-pass (admission bound from every s-th row tile), the drift limiter and the
    launch shaping and the placement of the query tile (all of K in tensor memory, or its last third in shared
    memory so that two accumulator buffers fit) are performance devices: with any setting the tensor scan returns the oracle's
    top-k.  Strides forced here at sizes the oracle finishes in seconds (by default: every 2nd row tile below 128 k
    rows, every 4th below 512 k, then whatever keeps the sample near 200 k rows)."""
    n, B, k, dim = 60000, 300, 10, 768
    corpus = _corpus(n, dim, seed=21)
    # duplicate rows make exact score ties across row tiles: the bound must admit equal scores
    corpus[1000:1064] = corpus[50000:50064]
    levels = _levels(n, seed=22)
    q = _corpus(B, dim, seed=23)
    q[:32] = corpus[50000:50032]
    idx = _index(pkg, corpus, levels)
    try:
        native.tune(**knobs)
        score, raw, ids = idx.search(q, k, weight_mode=weight_mode, path=native.PATH_TENSOR)
    finally:
        native.tune(scan_sample=-1, scan_drift=4, scan_tmax=16, scan_kbs=3, scan_qsplit=-1, scan_pre_slots=1, scan_pair=-1, scan_generic=0)
    if weight_mode == native.WEIGHT_PRE:
        w = np.array([1.0, 1.2, 1.0, 0.8], np.float32)[levels]
        full = (q @ corpus.T) * w[None, :]
        for b in range(B):
            ref = np.lexsort((np.arange(n), -full[b].astype(np.float64)))[:k]
            got_w = full[b][ids[b]]
            assert len(set(ids[b].tolist())) == k
            assert np.all(np.abs(got_w - full[b][ref]) <= 1e-3), (b, ids[b], ref)
            np.testing.assert_allclose(score[b], got_w, atol=3e-6)
    else:
        ref_s, ref_i = osearch.exact_topk(corpus, q, k)
        swaps = check_topk(ids, raw, ref_i, ref_s, _exact_of(corpus, q), score_tol=2e-6)
        assert swaps <= B * k // 50
        # the planted duplicates: both copies of the row come back, lower id first
        for b in range(32):
            assert ids[b, 0] == 1000 + b and ids[b, 1] == 50000 + b, (b, ids[b, :3])
    idx.close()


@pytest.mark.parametrize("keep_f32", [False, True])
@pytest.mark.parametrize("k", [10, 26, 27, 60, 128])
def test_pre_pass_bound_is_valid_for_every_k(pkg, native, k, keep_f32):
    """The pre-pass bound must never exceed the true kc-th best score.  Slot maxima: 32 slots x 4 classes of row groups =
    128 disjoint row sets per query, the kc-th largest of their maxima (kc = k + 6, or 2 k + 16 with the fp32 master
    rows: up to 128); a small table with a large forced stride makes the sets sparse (most stay empty: the bound
    falls back to -inf and nothing is pruned)."""
    n, B, dim = 30000, 130, 768
    corpus = _corpus(n, dim, seed=41)
    levels = _levels(n, seed=42)
    q = _corpus(B, dim, seed=43)
    q[:16] = corpus[777:793]
    idx = _index(pkg, corpus, levels, keep_f32=keep_f32)
    try:
        for stride in (2, 7, 64):
            native.tune(scan_sample=stride)
            score, raw, ids = idx.search(q, k, weight_mode=native.WEIGHT_NONE, path=native.PATH_TENSOR)
            ref_s, ref_i = osearch.exact_topk(corpus, q, k)
            check_topk(ids, raw, ref_i, ref_s, _exact_of(corpus, q), score_tol=2e-6)
    finally:
        native.tune(scan_sample=-1)
    idx.close()


@pytest.mark.parametrize("knobs", [dict(), dict(scan_tmax=2), dict(scan_qtmem=8), dict(scan_qsplit=0), dict(scan_sample=4, scan_drift=1),
                                   dict(scan_kbs_pair=2), dict(scan_kbs_pair=4, scan_qsplit=0), dict(scan_kbs_pair=3)])
def test_cta_pair_scan_equals_single_cta_scan(pkg, native, knobs):
    """CTA pairs (tcgen05 cta_group::2: two query tiles per MMA, each CTA loading half of every row tile) are a
    performance device: launches with an even number of query tiles return bit for bit what single CTAs return,
    and both equal the oracle's exact top-k."""
    n, B, k, dim = 70001, 512, 10, 768
    corpus = _corpus(n, dim, seed=31)
    corpus[2000:2032] = corpus[60000:60032]          # exact ties across row tiles and row groups
    levels = _levels(n, seed=32)
    q = _corpus(B, dim, seed=33)
    q[:32] = corpus[60000:60032]
    idx = _index(pkg, corpus, levels)
    try:
        native.tune(scan_pair=0)
        s0, r0, i0 = idx.search(q, k, weight_mode=native.WEIGHT_NONE, path=native.PATH_TENSOR)
        native.tune(scan_pair=-1, **knobs)
        s1, r1, i1 = idx.search(q, k, weight_mode=native.WEIGHT_NONE, path=native.PATH_TENSOR)
        # ragged batch: 3 query tiles + a partly filled 4th (rows of the last tile beyond B are dead lanes)
        s2, r2, i2 = idx.search(q[:400], k, weight_mode=native.WEIGHT_NONE, path=native.PATH_TENSOR)
        # the reference's post-top-k re-rank on top of the pair scan
        s3, r3, i3 = idx.search(q, k, weight_mode=native.WEIGHT_RERANK, path=native.PATH_TENSOR)
    finally:
        native.tune(scan_sample=-1, scan_drift=4, scan_tmax=16, scan_kbs=3, scan_kbs_pair=6, scan_qsplit=-1, scan_pair=-1, scan_qtmem=0)
    assert np.array_equal(i0, i1) and np.array_equal(r0, r1) and np.array_equal(s0, s1)
    assert np.array_equal(i0[:400], i2) and np.array_equal(r0[:400], r2)
    ref_s, ref_i = osearch.exact_topk(corpus, q, k)
    swaps = check_topk(i1, r1, ref_i, ref_s, _exact_of(corpus, q), score_tol=2e-6)
    assert swaps <= B * k // 50
    for b in range(32):
        assert i1[b, 0] == 2000 + b and i1[b, 1] == 60000 + b, (b, i1[b, :3])
    # re-rank = the same k hits, re-sorted by raw * w(level) (milvus_service.py:290-314)
    w = np.array([1.0, 1.2, 1.0, 0.8], np.float32)[levels]
    for b in range(0, B, 37):
        assert sorted(i3[b].tolist()) == sorted(i1[b].tolist())
        np.testing.assert_allclose(s3[b], r3[b] * w[i3[b]], rtol=1e-6)
        assert np.all(s3[b][:-1] >= s3[b][1:])
    idx.close()


@pytest.mark.parametrize("keep_f32", [False, True])
@pytest.mark.parametrize("n,B,k", [(1024, 5, 10), (1500, 64, 1), (4097, 300, 10), (40474, 130, 100), (40474, 1030, 10),
                                    (131072, 257, 10), (200000, 40, 27)])
def test_small_table_pre_pass_is_a_performance_device(pkg, native, n, B, k, keep_f32):
    """Tables below 512 k rows (the reference's own 40 474) run the slot-maxima pre-pass over every 2nd (from 128 k rows:
    every 4th) row tile so that the main scan's lists do not warm up row group by row group.  Same results bit for bit
    with it and without it (icd_tune scan_small_pre = 0, the round-2 behaviour), and both equal the oracle's top-k."""
    dim = 768
    corpus = _corpus(n, dim, seed=n + k)
    corpus[n // 3:n // 3 + 8] = corpus[n - 8:]                       # exact ties between a sampled and an unsampled tile
    levels = _levels(n, seed=n + 1)
    q = _corpus(B, dim, seed=B + k)
    q[:4] = corpus[n - 4:]
    idx = _index(pkg, corpus, levels, keep_f32=keep_f32)
    try:
        got = {}
        for pre in (1, 0):
            native.tune(scan_small_pre=pre)
            for wm in (native.WEIGHT_NONE, native.WEIGHT_RERANK, native.WEIGHT_PRE):
                got[pre, wm] = idx.search(q, k, weight_mode=wm, path=native.PATH_TENSOR)
    finally:
        native.tune(scan_small_pre=1)
    idx.close()
    for wm in (native.WEIGHT_NONE, native.WEIGHT_RERANK, native.WEIGHT_PRE):
        for a, b in zip(got[1, wm], got[0, wm]):
            assert np.array_equal(a, b), (wm, n, B, k)
    score, raw, ids = got[1, native.WEIGHT_NONE]
    ref_s, ref_i = osearch.exact_topk(corpus, q, k)
    swaps = check_topk(ids, raw, ref_i, ref_s, _exact_of(corpus, q), score_tol=2e-6)
    assert swaps <= max(1, B * k // 50)
    for b in range(4):                                                # the planted duplicates, lower id first
        if k >= 2:
            assert ids[b, 0] == n // 3 + 4 + b and ids[b, 1] == n - 4 + b, (b, ids[b, :3])


@pytest.mark.parametrize("keep_f32", [False, True])
def test_large_host_batches_are_pipelined_and_identical(pkg, native, keep_f32):
    """Batches of >= 4096 queries handed over in host memory run in chunks of 2048 on two streams (copy-in of the next
    chunk under the scan of the current one, two sets of staging buffers, copy-back one chunk behind): same results,
    bit for bit, as the same queries in small calls and as one call with device-resident buffers; repeated calls and a
    ragged last chunk included."""
    import torch
    n, dim, k = 40474, 768, 10
    corpus = _corpus(n, dim, seed=301)
    levels = _levels(n, seed=302)
    idx = _index(pkg, corpus, levels, keep_f32=keep_f32)
    for B in (4096, 4096 + 777, 10_000):
        q = _corpus(B, dim, seed=303 + B)
        small = [idx.search(q[lo:lo + 1000], k, weight_mode=native.WEIGHT_RERANK) for lo in range(0, B, 1000)]
        want = [np.concatenate([p[i] for p in small]) for i in range(3)]
        for _ in range(2):
            got = idx.search(q, k, weight_mode=native.WEIGHT_RERANK)
            for a, b in zip(got, want):
                assert np.array_equal(a, b), B
        dev = idx.search(torch.from_numpy(q).cuda(), k, weight_mode=native.WEIGHT_RERANK)
        for a, b in zip(dev, want):
            assert np.array_equal(a.cpu().numpy(), b), B
    ref_s, ref_i = osearch.exact_topk(corpus, q[:256], k)
    s, r, i = idx.search(q, k, weight_mode=native.WEIGHT_NONE)
    check_topk(i[:256], r[:256], ref_i, ref_s, _exact_of(corpus, q), score_tol=2e-6)
    idx.close()


def test_config1_10k_queries_against_the_icd_sized_corpus(pkg, native):
    """BASELINE.json configs[1]: batched exact top-10 of 10 000 synthetic diagnosis queries against a 40 474-row
    corpus (the size of data/ICD_10v601.csv) with the hierarchical level weights, one GPU.  Queries go through in
    batches of 1024 + remainder (SURVEY 8d); every one of the 10 000 result rows is checked against the oracle:
    the raw top-10 (ids identical up to 1e-3 ties) and the reference's post-top-k re-rank (milvus_service.py:290-314)."""
    import time
    n, nq, k, dim = 40474, 10_000, 10, 768
    corpus = _corpus(n, dim, seed=101)
    levels = _levels(n, seed=102)
    rng = np.random.default_rng(103)
    # half i.i.d. queries (worst case for ties), half planted near a corpus row (unambiguous neighbour)
    q = _corpus(nq, dim, seed=104)
    planted = rng.integers(0, n, size=nq // 2)
    q[nq // 2:] = osearch.bf16_round(corpus[planted] + 0.3 / np.sqrt(dim) * rng.standard_normal((nq // 2, dim)).astype(np.float32))
    idx = _index(pkg, corpus, levels)
    idx.search(q[:1024], k, weight_mode=native.WEIGHT_RERANK)          # warm-up (workspace allocation)
    t0 = time.perf_counter()
    parts = [idx.search(q[lo:lo + 1024], k, weight_mode=native.WEIGHT_RERANK) for lo in range(0, nq, 1024)]
    wall = time.perf_counter() - t0
    score = np.concatenate([p[0] for p in parts]); raw = np.concatenate([p[1] for p in parts]); ids = np.concatenate([p[2] for p in parts])
    idx.close()
    assert ids.shape == (nq, k)
    ref_s, ref_i = osearch.exact_topk(corpus, q, k)
    w = np.array([1.0, 1.2, 1.0, 0.8], np.float64)[levels]
    # (1) the k hits are the exact top-k (as a set, up to 1e-3 ties at the boundary), raw scores exact to 2e-6
    swaps = 0
    for b in range(nq):
        o = np.lexsort((ids[b], -raw[b].astype(np.float64)))
        swaps += check_topk(ids[b][o][None, :], raw[b][o][None, :], ref_i[b][None, :], ref_s[b][None, :],
                            lambda _b, ii: corpus[np.asarray(ii)] @ q[b], score_tol=2e-6)
        # (2) weighted score = raw * w(level), list sorted by it, descending (the reference's re-rank)
        np.testing.assert_allclose(score[b], raw[b].astype(np.float64) * w[ids[b]], rtol=2e-7, atol=1e-7)
        assert np.all(score[b][:-1] >= score[b][1:])
    assert swaps <= nq * k // 100, swaps
    assert np.array_equal(ids[nq // 2:][np.arange(nq // 2), np.argmax(raw[nq // 2:], axis=1)], planted)
    print(f"configs[1]: {nq} queries x {n} rows in {wall * 1e3:.1f} ms through the C ABI with host buffers "
          f"({nq / wall:.0f} queries/s; corpus 62 MB, L2-resident)")


# ---------------------------------------------------------------------------------------------- BASELINE configs[3]
@pytest.fixture(scope="module")
def corpus_10m():
    """10 M x 768 bf16 rows on the GPU (configs[3]), built like bench.py's corpus, + 1024 queries of which every 4th is a
    perturbed corpus row."""
    import torch
    import bench
    dev = torch.device("cuda", 0)
    table, levels = bench.make_corpus(torch, 10_000_000, dev, seed=4321)
    q, pos, gid = bench.make_planted_queries(torch, None, table, 0, 10_000_000, 10_000_000, 1024, dev, 0, 1)
    yield table, levels, q, pos, gid
    del table, levels
    torch.cuda.empty_cache()


@pytest.mark.parametrize("B", [128, 256, 1024])
def test_config3_10m_rows_against_an_independent_exact_search(pkg, native, corpus_10m, B):
    """configs[3] with the DEFAULT launch configuration (sampling pre-pass, cross-CTA pruning, drift limiter, CTA pairs,
    unrolled issue loop), checked with the exactness certificate of scan_ref.certify over row chunks in fp64 (no row
    left out beats a returned one by more than the two rows' combined rounding bounds); planted rows first."""
    import torch
    from importlib import import_module
    import scan_ref as R
    table, levels, q_all, pos, gid = corpus_10m
    q = q_all[:B].contiguous()
    VectorIndex = import_module("rag-project-icd10_b200.engine.index").VectorIndex
    idx = VectorIndex(768, device=0)
    idx.adopt(table, levels)
    score, raw, ids = idx.search(q, 10, weight_mode=native.WEIGHT_NONE)
    torch.cuda.synchronize()
    assert idx.take_fallbacks() == 0        # bf16 queries on bf16 rows: the scan scores are the canonical products
    cert = R.certify(ids, raw, score, table, q.float(), 10, native.WEIGHT_NONE, levels, chunk_rows=(1 << 27) // B)
    print(f"configs[3] B={B}: worst error / bound {cert.worst:.3f}")
    planted = [j for j in range(len(pos)) if pos[j] < B]
    assert ids[[pos[j] for j in planted], 0].cpu().tolist() == [gid[j] for j in planted]
    # the level re-rank on top of the same raw list
    s2, r2, i2 = idx.search(q, 10, weight_mode=native.WEIGHT_RERANK)
    assert torch.equal(i2.sort(dim=1).values, ids.sort(dim=1).values) and bool((s2[:, 1:] <= s2[:, :-1]).all())
    idx.close()
