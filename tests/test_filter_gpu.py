"""Filtered exact search on the GPU: a row bitmap applied inside both scan kernels (and the sampling pre-pass), against the
oracle's exact top-k over the allowed rows; the C ABI edge cases; the `filter` argument of the store and the services."""
import ctypes as C
import importlib
import os
import subprocess
import sys

import numpy as np
import pytest

from oracle import search as osearch
from oracle import text as otext
from parity import check_topk

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
F = importlib.import_module("rag-project-icd10_b200.engine.filter_expr")
W = np.array([1.0, 1.2, 1.0, 0.8], np.float32)          # level weights by level byte (1, 2, 3; else 1.0)
DEFAULT_KNOBS = dict(scan_sample=-1, scan_drift=4, scan_tmax=16, scan_kbs=3, scan_kbs_pair=6, scan_qsplit=-1,
                     scan_pre_slots=1, scan_pair=-1, scan_generic=0, scan_small_pre=1)


def _corpus(n, dim, seed, bf16=True):
    rng = np.random.default_rng(seed)
    x = rng.standard_normal((n, dim)).astype(np.float32)
    x /= np.linalg.norm(x, axis=1, keepdims=True)
    return osearch.bf16_round(x) if bf16 else x


def _levels(n, seed):
    rng = np.random.default_rng(seed)
    return rng.choice(np.array([1, 2, 3], np.uint8), size=n, p=[0.1243, 0.2991, 0.5766]).astype(np.uint8)


def _index(corpus, levels, keep_f32=False):
    VectorIndex = importlib.import_module("rag-project-icd10_b200.engine.index").VectorIndex
    idx = VectorIndex(corpus.shape[1], device=0, keep_f32=keep_f32)
    idx.append(corpus, levels)
    return idx


def _masks(n, seed):
    rng = np.random.default_rng(seed)
    lo = int(rng.integers(0, n - n // 100))
    contiguous = np.zeros(n, bool)
    contiguous[lo:lo + max(1, n // 100)] = True
    return {"all": np.ones(n, bool), "half": rng.random(n) < 0.5, "range1pct": contiguous,
            "rand1pct": rng.random(n) < 0.01}


def _oracle(corpus, allowed, q, k, weights=None):
    """(scores [B, k], ids [B, k]) of the exact top-k over the allowed rows, (-inf, -1) past their count; `weights`:
    select on score * weight (ICD_WEIGHT_PRE)."""
    sub = np.nonzero(allowed)[0]
    B = q.shape[0]
    s = np.full((B, k), -np.inf, np.float32)
    i = np.full((B, k), -1, np.int64)
    if sub.size:
        if weights is None:
            rs, ri = osearch.exact_topk(corpus[sub], q, k)
        else:   # weighted scores of the k best (ties at the boundary do not matter: compared within 1e-3)
            full = (q @ corpus[sub].T) * weights[sub][None, :]
            kk = min(k, sub.size)
            ri = np.argpartition(-full, kk - 1, axis=1)[:, :kk] if sub.size > kk else np.tile(np.arange(kk), (B, 1))
            rs = np.take_along_axis(full, ri, axis=1)
            o = np.argsort(-rs, axis=1, kind="stable")
            ri, rs = np.take_along_axis(ri, o, 1), np.take_along_axis(rs, o, 1).astype(np.float32)
        kk = ri.shape[1]
        s[:, :kk], i[:, :kk] = rs, sub[ri]
    return s, i


def _check(corpus, levels, q, allowed, k, wm, got, what, ref=None):
    """ref: a dict that keeps the oracle's answers for further calls with the same corpus, queries and mask."""
    ref = {} if ref is None else ref
    score, raw, ids = got
    exact = lambda b, ii: corpus[np.asarray(ii)] @ q[b]                        # noqa: E731
    kk = min(k, int(allowed.sum()))
    assert np.all(ids[:, kk:] == -1) and np.all(np.isneginf(raw[:, kk:])), what
    assert np.all(allowed[ids[:, :kk]]), what
    if wm == 1:
        if "w" not in ref:
            ref["w"] = _oracle(corpus, allowed, q, k, W[levels])
        ref_s = ref["w"][0]
        for b in range(q.shape[0]):
            w_b = (corpus[ids[b, :kk]] @ q[b]) * W[levels][ids[b, :kk]]
            assert len(set(ids[b, :kk].tolist())) == kk, (what, b)
            assert np.all(np.abs(w_b - ref_s[b, :kk]) <= 1e-3), (what, b)
            np.testing.assert_allclose(score[b, :kk], w_b, atol=3e-6, err_msg=what)
        return
    if "raw" not in ref:
        ref["raw"] = _oracle(corpus, allowed, q, k)
    ref_s, ref_i = ref["raw"]
    if wm == 0:   # the re-rank re-sorts the raw top-k: compare the raw list in (raw desc, id asc) order
        order = np.lexsort((ids, -raw.astype(np.float64)), axis=1)
        ids, raw = np.take_along_axis(ids, order, 1), np.take_along_axis(raw, order, 1)
    swaps = check_topk(ids[:, :kk], raw[:, :kk], ref_i[:, :kk], ref_s[:, :kk], exact, score_tol=2e-6)
    assert swaps <= max(1, q.shape[0] * kk // 50), (what, swaps)


# ---------------------------------------------------------------------------------------------- 1. parity
@pytest.mark.parametrize("keep_f32", [False, True])
@pytest.mark.parametrize("n,B,k", [(5000, 1, 10), (5000, 7, 5), (40474, 130, 10), (12345, 1030, 7), (40474, 3, 100)])
def test_filtered_search_matches_oracle_on_allowed_rows(pkg, native, n, B, k, keep_f32):
    """Both paths x the three weight modes x four selectivities (every row, 50 % random, a contiguous 1 %, 1 % random)."""
    dim = 768
    corpus = _corpus(n, dim, seed=n + B, bf16=not keep_f32)
    levels = _levels(n, seed=n)
    q = _corpus(B, dim, seed=B + 7, bf16=not keep_f32)
    idx = _index(corpus, levels, keep_f32)
    try:
        for name, allowed in _masks(n, seed=n + k).items():
            words = F.pack_bits(allowed)
            ref = {}
            for path in (native.PATH_STREAM, native.PATH_TENSOR):
                for wm in (native.WEIGHT_RERANK, native.WEIGHT_PRE, native.WEIGHT_NONE):
                    got = idx.search(q, k, weight_mode=wm, path=path, mask=words)
                    _check(corpus, levels, q, allowed, k, wm, got, (name, path, wm), ref)
    finally:
        idx.close()


# ---------------------------------------------------------------------------------------------- 2. all-ones mask
@pytest.mark.parametrize("keep_f32", [False, True])
def test_all_ones_mask_is_bitwise_the_unfiltered_search(pkg, native, keep_f32):
    n, B, k = 70001, 300, 10
    corpus = _corpus(n, 768, seed=3, bf16=not keep_f32)
    levels = _levels(n, seed=4)
    q = _corpus(B, 768, seed=5, bf16=not keep_f32)
    idx = _index(corpus, levels, keep_f32)
    ones = F.pack_bits(np.ones(n, bool))
    for path in (native.PATH_STREAM, native.PATH_TENSOR):
        qq = q[:5] if path == native.PATH_STREAM else q
        for wm in (native.WEIGHT_RERANK, native.WEIGHT_PRE, native.WEIGHT_NONE):
            a = idx.search(qq, k, weight_mode=wm, path=path)
            b = idx.search(qq, k, weight_mode=wm, path=path, mask=ones)
            for x, y in zip(a, b):
                assert np.array_equal(x.view(np.uint8), y.view(np.uint8)), (path, wm)
    idx.close()


# ---------------------------------------------------------------------------------------------- 3. adversarial pre-pass
KNOBS = [dict(), dict(scan_sample=4, scan_pre_slots=0),
         dict(scan_sample=4), dict(scan_sample=3, scan_drift=1), dict(scan_sample=0, scan_drift=0),
         dict(scan_sample=8, scan_tmax=2), dict(scan_sample=2, scan_kbs=2), dict(scan_kbs=6), dict(scan_kbs=4, scan_qsplit=0),
         dict(scan_qsplit=0), dict(scan_qsplit=1, scan_sample=4), dict(scan_qsplit=1, scan_tmax=1),
         dict(scan_sample=2, scan_pre_slots=0, scan_tmax=2), dict(scan_sample=16, scan_pair=0),
         dict(scan_sample=5, scan_generic=1), dict(scan_small_pre=0), dict(scan_pair=0, scan_sample=2)]


@pytest.fixture(scope="module")
def adversarial():
    """Half of the rows are near copies of one of the queries (score ~0.99 against it, spread over every row tile, slot
    and row group) and exactly those rows are masked out: a pre-pass or a list that admitted a masked-out row would
    prove a bound no allowed row reaches and prune every correct answer."""
    n, dim, B = 60000, 768, 32
    rng = np.random.default_rng(2024)
    q = _corpus(B, dim, seed=2025)
    corpus = rng.standard_normal((n, dim)).astype(np.float32)
    corpus /= np.linalg.norm(corpus, axis=1, keepdims=True)
    planted = rng.random(n) < 0.5
    owner = rng.integers(0, B, size=n)
    near = q[owner[planted]] + 0.15 / np.sqrt(dim) * rng.standard_normal((int(planted.sum()), dim)).astype(np.float32)
    corpus[planted] = near / np.linalg.norm(near, axis=1, keepdims=True)
    corpus = osearch.bf16_round(corpus)
    return corpus, _levels(n, seed=9), q, ~planted


@pytest.mark.parametrize("keep_f32", [False, True])
@pytest.mark.parametrize("k", [10, 60])
def test_pre_pass_bound_comes_from_allowed_rows_only(pkg, native, adversarial, k, keep_f32):
    """kc = 16 / 66 (bf16 queries) and 36 / 128 (fp32 master rows), with the slot-maxima pre-pass and the list-based one
    (forced on a small table: scan_sample=4, scan_pre_slots=0)."""
    corpus, levels, q, allowed = adversarial
    idx = _index(corpus, levels, keep_f32)
    qq = osearch.to_bf16_bits(q) if not keep_f32 else q
    words = F.pack_bits(allowed)
    try:
        for knobs in KNOBS[:2]:
            native.tune(**knobs)
            got = idx.search(qq, k, weight_mode=native.WEIGHT_NONE, path=native.PATH_TENSOR, mask=words)
            native.tune(**DEFAULT_KNOBS)
            _check(corpus, levels, q, allowed, k, native.WEIGHT_NONE, got, knobs)
            # without the mask the planted rows win: the test data does exercise the bound
            _, _, ids = idx.search(qq, k, weight_mode=native.WEIGHT_NONE, path=native.PATH_TENSOR)
            assert not allowed[ids].any()
    finally:
        native.tune(**DEFAULT_KNOBS)
        idx.close()


@pytest.mark.parametrize("knobs", KNOBS[2:], ids=[",".join(f"{a}={b}" for a, b in kn.items()) for kn in KNOBS[2:]])
@pytest.mark.parametrize("weight_mode", [2, 1])
def test_filtered_tensor_scan_under_the_knob_matrix(pkg, native, adversarial, knobs, weight_mode):
    corpus, levels, q, allowed = adversarial
    idx = _index(corpus, levels)
    try:
        native.tune(**knobs)
        got = idx.search(q, 10, weight_mode=weight_mode, path=native.PATH_TENSOR, mask=F.pack_bits(allowed))
    finally:
        native.tune(**DEFAULT_KNOBS)
        idx.close()
    _check(corpus, levels, q, allowed, 10, weight_mode, got, knobs)


# ---------------------------------------------------------------------------------------------- 4. edge cases
@pytest.mark.parametrize("path", [1, 2])
def test_mask_edge_cases(pkg, native, path):
    n, B, k = 5000, 9, 10                                   # 5000 = 156 words + 8 rows: a partial last word
    corpus = _corpus(n, 768, seed=61)
    levels = _levels(n, seed=62)
    q = _corpus(B, 768, seed=63)
    idx = _index(corpus, levels)
    # fewer allowed rows than k: (-inf, -1) tail
    few = np.zeros(n, bool)
    few[[4, 2500, 4999]] = True
    s, r, i = idx.search(q, k, weight_mode=native.WEIGHT_RERANK, path=path, mask=F.pack_bits(few))
    assert np.all(np.sort(i[:, :3], axis=1) == [4, 2500, 4999]) and np.all(i[:, 3:] == -1)
    assert np.all(np.isneginf(r[:, 3:])) and np.all(np.isneginf(s[:, 3:])) and np.all(np.isfinite(r[:, :3]))
    _check(corpus, levels, q, few, k, native.WEIGHT_RERANK, (s, r, i), "few")
    # an empty mask
    s, r, i = idx.search(q, k, weight_mode=native.WEIGHT_NONE, path=path, mask=F.pack_bits(np.zeros(n, bool)))
    assert np.all(i == -1) and np.all(np.isneginf(r)) and np.all(np.isneginf(s))
    # set bits past n (and extra words) are ignored
    half = np.random.default_rng(64).random(n) < 0.5
    clean = F.pack_bits(half)
    dirty = np.concatenate([clean, np.full(3, 0xFFFFFFFF, np.uint32)])
    dirty[len(clean) - 1] |= np.uint32(0xFFFFFFFF << (n % 32) & 0xFFFFFFFF)
    want = idx.search(q, k, weight_mode=native.WEIGHT_NONE, path=path, mask=clean)
    got = idx.search(q, k, weight_mode=native.WEIGHT_NONE, path=path, mask=dirty)
    for a, b in zip(want, got):
        assert np.array_equal(a, b)
    _check(corpus, levels, q, half, k, native.WEIGHT_NONE, want, "half")
    # a device mask gives what the host mask gives
    import torch
    dev = idx.search(q, k, weight_mode=native.WEIGHT_NONE, path=path, mask=torch.from_numpy(clean.view(np.int32)).cuda())
    for a, b in zip(want, dev):
        assert np.array_equal(a, b)
    # mask_rows must equal the table size
    out = [np.empty((B, k), np.float32), np.empty((B, k), np.float32), np.empty((B, k), np.int64)]
    L = native.lib()
    for rows in (n + 1, n - 1, 0):
        st = L.icd_index_search_filtered(idx._h, native.buf_ptr(q), native.F32, B, k, 0, path, native.buf_ptr(clean), rows,
                                         *[native.buf_ptr(o) for o in out], C.c_void_p(0), 1)
        assert st == -1 and b"row mask" in L.icd_last_error()
    # NULL mask = every row, whatever mask_rows says
    st = L.icd_index_search_filtered(idx._h, native.buf_ptr(q), native.F32, B, k, 0, path, None, 12345,
                                     *[native.buf_ptr(o) for o in out], C.c_void_p(0), 1)
    assert st == 0 and np.array_equal(out[2], idx.search(q, k, weight_mode=0, path=path)[2])
    idx.close()


@pytest.mark.parametrize("keep_f32", [False, True])
def test_pipelined_host_batch_uses_the_mask_for_every_chunk(pkg, native, keep_f32):
    import torch
    n, B, k = 40474, 8192, 10
    corpus = _corpus(n, 768, seed=71, bf16=not keep_f32)
    levels = _levels(n, seed=72)
    q = _corpus(B, 768, seed=73, bf16=not keep_f32)
    allowed = np.random.default_rng(74).random(n) < 0.3
    words = F.pack_bits(allowed)
    idx = _index(corpus, levels, keep_f32)
    host = idx.search(q, k, weight_mode=native.WEIGHT_RERANK, mask=words)                 # chunks of 2048, two streams
    dev = idx.search(torch.from_numpy(q).cuda(), k, weight_mode=native.WEIGHT_RERANK,
                     mask=torch.from_numpy(words.view(np.int32)).cuda())
    for a, b in zip(host, dev):
        assert np.array_equal(a, b.cpu().numpy())
    sample = np.arange(0, B, 257)
    _check(corpus, levels, q[sample], allowed, k, native.WEIGHT_RERANK, tuple(x[sample] for x in host), "pipelined")
    idx.close()


# ---------------------------------------------------------------------------------------------- 5. 10 M rows
@pytest.fixture(scope="module")
def corpus_10m():
    import torch
    import bench
    dev = torch.device("cuda", 0)
    table, levels = bench.make_corpus(torch, 10_000_000, dev, seed=4321)
    q, pos, gid = bench.make_planted_queries(torch, None, table, 0, 10_000_000, 10_000_000, 1024, dev, 0, 1)
    yield table, levels, q
    del table, levels
    torch.cuda.empty_cache()


@pytest.mark.parametrize("sel", ["half", "range1pct"])
@pytest.mark.parametrize("B", [128, 1024])
def test_10m_rows_filtered_against_an_independent_exact_search(pkg, native, corpus_10m, B, sel):
    """Default launch configuration (pre-pass, pruning, drift limiter, CTA pairs) with a mask, against chunked fp32
    torch.matmul + topk over the allowed rows on the same GPU, merged by (score desc, id asc)."""
    import torch
    table, levels, q_all = corpus_10m
    n = table.shape[0]
    q = q_all[:B].contiguous()
    if sel == "half":
        allowed = np.random.default_rng(5).random(n) < 0.5
    else:
        allowed = np.zeros(n, bool)
        allowed[3_333_333:3_333_333 + n // 100] = True
    VectorIndex = importlib.import_module("rag-project-icd10_b200.engine.index").VectorIndex
    idx = VectorIndex(768, device=0)
    idx.adopt(table, levels)
    _, raw, ids = idx.search(q, 10, weight_mode=native.WEIGHT_NONE, mask=F.pack_bits(allowed))
    torch.cuda.synchronize()
    allowed_d = torch.from_numpy(allowed).cuda()
    qf = q.float()
    best_s = torch.full((B, 0), -float("inf"), device=q.device)
    best_i = torch.zeros((B, 0), dtype=torch.int64, device=q.device)
    prev = torch.backends.cuda.matmul.allow_tf32
    torch.backends.cuda.matmul.allow_tf32 = False
    try:
        for lo in range(0, n, 1 << 20):
            s = qf @ table[lo:lo + (1 << 20)].float().T
            s[:, ~allowed_d[lo:lo + (1 << 20)]] = -float("inf")
            ts, ti = s.topk(16, dim=1)
            best_s = torch.cat([best_s, ts], 1)
            best_i = torch.cat([best_i, ti + lo], 1)
    finally:
        torch.backends.cuda.matmul.allow_tf32 = prev
    order = best_i.argsort(dim=1, stable=True)
    best_s, best_i = best_s.gather(1, order), best_i.gather(1, order)
    order = (-best_s).argsort(dim=1, stable=True)[:, :10]
    ref_s, ref_i = best_s.gather(1, order).cpu().numpy(), best_i.gather(1, order).cpu().numpy()
    ids_h = ids.cpu().numpy()
    assert allowed[ids_h].all()
    swaps = check_topk(ids_h, raw.cpu().numpy(), ref_i, ref_s,
                       lambda b, i: (table[torch.as_tensor(np.asarray(i), device=q.device)].float() @ qf[b]).cpu().numpy(),
                       tie_tol=1e-6, score_tol=2e-6)
    assert swaps <= B // 16, swaps
    idx.close()


# ---------------------------------------------------------------------------------------------- 6. services
class _Emb768:
    def encode_query(self, q):
        return np.ones(768, np.float32) / np.sqrt(768.0)


def _py_filter(recs, fn):
    return np.array([bool(fn(r)) for r in recs])


def test_service_filter_on_the_icd_table(tmp_path, monkeypatch):
    monkeypatch.setenv("MILVUS_DB_PATH", str(tmp_path / "db" / "f.db"))
    monkeypatch.setenv("MILVUS_COLLECTION_NAME", "icd10")
    M = importlib.import_module("rag-project-icd10_b200.services.milvus_service")
    Bm = importlib.import_module("rag-project-icd10_b200.services.batched_retrieval")
    ms = M.MilvusService(embedding_service=_Emb768())
    recs = otext.load_records(os.path.join(ROOT, "data", "ICD_10v601.csv"))
    rng = np.random.default_rng(11)
    corpus = rng.standard_normal((len(recs), 768)).astype(np.float32)
    corpus /= np.linalg.norm(corpus, axis=1, keepdims=True)
    assert ms.insert_records_array(recs, corpus) is True
    q = corpus[rng.integers(0, len(recs), size=6)] + 0.3 * rng.standard_normal((6, 768)).astype(np.float32)
    q /= np.linalg.norm(q, axis=1, keepdims=True)
    cases = [('code like "J%"', lambda r: r["code"].startswith("J")),
             ("level == 3 and has_complication == false", lambda r: r["level"] == 3 and not r["has_complication"]),
             ('parent_code == "A00.0"', lambda r: r["parent_code"] == "A00.0")]
    for expr, fn in cases:
        allowed = _py_filter(recs, fn)
        sub = np.nonzero(allowed)[0]
        recs_sub = [recs[j] for j in sub]
        batch = ms.search_batch(q, 5, filter=expr)
        for b in range(q.shape[0]):
            want = osearch.search_hits(corpus[sub], recs_sub, q[b], 5)
            got = ms.search(q[b], 5, filter=expr)
            assert [h["code"] for h in got] == [h["code"] for h in want], (expr, b)
            assert np.allclose([h["original_score"] for h in got], [h["original_score"] for h in want], atol=2e-6)
            assert all(fn(recs[int(j)]) for j in batch[b].row_ids)
            assert list(batch[b]) == got, (expr, b)
    # the unfiltered calls are what they were
    assert ms.search(q[0], 5) == ms.search(q[0], 5, filter="") == ms.search(q[0], 5, filter="   ")
    # an invalid expression: logged, []
    for bad in ('level == "3"', "nope == 1", 'code like "A_0"', "level == 3 level"):
        assert ms.search(q[0], 5, filter=bad) == []
        assert ms.search_batch(q, 5, filter=bad) == []
    # BatchedRetrieval passes the filter through
    class _EmbQ:
        def encode_queries(self, texts):
            return q[:len(texts)]
    br = Bm.BatchedRetrieval(_EmbQ(), ms)
    got = br.retrieve(["a", "b"], top_k=3, filter='code like "J%"')
    assert [list(x) for x in got] == [ms.search(q[b], 6, filter='code like "J%"') for b in range(2)]
    assert [list(x) for x in br.retrieve(["a"], top_k=3)] == [ms.search(q[0], 6)]
    # query / get
    cl = ms.client
    rows = cl.query("icd10", filter='parent_code == "A00"', output_fields=["code", "level"])
    want = [{"id": int(j), "code": recs[j]["code"], "level": recs[j]["level"]} for j in range(len(recs))
            if recs[j]["parent_code"] == "A00"]
    assert rows == want and len(rows) >= 2
    assert cl.query("icd10", filter="level == 1", limit=3) == [{"id": int(j)} for j in np.nonzero(_py_filter(recs, lambda r: r["level"] == 1))[0][:3]]
    assert cl.query("icd10", filter="level == 1", ids=[0, 1, 2, 40000]) == [{"id": j} for j in (0, 1, 2, 40000) if recs[j]["level"] == 1]
    got = cl.get("icd10", [7, 3, 99999], output_fields=["code", "preferred_zh"])
    assert got == [{"id": 7, "code": recs[7]["code"], "preferred_zh": recs[7]["preferred_zh"]},
                   {"id": 3, "code": recs[3]["code"], "preferred_zh": recs[3]["preferred_zh"]}]
    assert cl.get("icd10", 5, output_fields=["*"])[0]["semantic_text"] == recs[5]["semantic_text"]
    with pytest.raises(ValueError):
        cl.query("icd10", filter="nope == 1")
    # an append rebuilds the cached mask
    expr = 'code like "ZZ%"'
    assert ms.search(q[0], 5, filter=expr) == []
    extra = [dict(recs[0], code="ZZ1", preferred_zh="新增"), dict(recs[1], code="ZZ2", preferred_zh="新增二")]
    assert ms.insert_records_array(extra, q[:2]) is True
    got = ms.search(q[0], 5, filter=expr)
    assert [h["code"] for h in got] == ["ZZ1", "ZZ2"]
    assert cl.query("icd10", filter=expr) == [{"id": len(recs)}, {"id": len(recs) + 1}]
    ms.disconnect()


def test_example_query_returns_only_the_chapter(tmp_path, monkeypatch):
    """One chapter (code like "A0%") over the first 3 000 ICD rows: hits in the reference's dict layout, all of them in the
    chapter, equal to the oracle's search over the chapter's rows."""
    monkeypatch.setenv("MILVUS_DB_PATH", str(tmp_path / "db" / "e.db"))
    monkeypatch.setenv("MILVUS_COLLECTION_NAME", "icd10")
    M = importlib.import_module("rag-project-icd10_b200.services.milvus_service")
    ms = M.MilvusService(embedding_service=_Emb768())
    recs = otext.load_records(os.path.join(ROOT, "data", "ICD_10v601.csv"))[:3000]
    vecs = _corpus(len(recs), 768, seed=12)
    assert ms.insert_records_array(recs, vecs) is True
    v = vecs[2500] + vecs[10]
    hits = ms.search(v, 5, filter='code like "A0%"')
    assert len(hits) == 5 and all(h["code"].startswith("A0") for h in hits)
    assert set(hits[0]) == {"code", "title", "score", "original_score", "metadata"}
    sub = [j for j, r in enumerate(recs) if r["code"].startswith("A0")]
    want = osearch.search_hits(vecs[sub], [recs[j] for j in sub], v, 5)
    assert [h["code"] for h in hits] == [h["code"] for h in want]
    assert hits[0]["code"] == recs[10]["code"]
    ms.disconnect()


# ---------------------------------------------------------------------------------------------- 7. two GPUs
def test_filtered_shard_group_equals_the_single_table():
    import torch
    if torch.cuda.device_count() < 2:
        pytest.skip("needs >= 2 GPUs")
    world = 2
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", f"--nproc-per-node={world}",
           "--master-addr", "127.0.0.1", "--master-port", "29547", os.path.join(ROOT, "tests", "filter_shard_worker.py")]
    out = subprocess.run(cmd, capture_output=True, text=True, timeout=600)
    assert out.returncode == 0 and "FILTER_SHARD_OK" in out.stdout, out.stdout[-3000:] + out.stderr[-3000:]
