"""icd_index_search_page on the GPU: offset + limit up to 16 384, offset paging and range search (include/icdrag.h).

- Below the old cap the new call returns exactly what icd_index_search_filtered(k = offset + limit, PATH_STREAM)[:,
  offset:] returns, bit for bit, at every dim class, for bf16 and fp32 master rows, fp32 and bf16 queries, every weight
  mode, with and without a mask.
- Above it, scan_ref.certify checks K = 129, 1 000 and 16 384 on probe corpora, the clustered near-duplicate corpus, a
  40 474-row table and a 2 000 003-row table.
- Paging, ranges, ties at the K-th rank, query chunking, guard regions and sync=0 are checked bit for bit against the
  call itself or against tests/page_ref.py applied to the call's own canonical scores.
"""
import ctypes as C
import importlib
import os

import numpy as np
import pytest
import torch

import page_ref as P
import scan_ref as R
from test_scan_exact_gpu import _cluster_queries, _levels, clustered_corpus

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
DEV = torch.device("cuda", 0)
WMS = (R.WEIGHT_RERANK, R.WEIGHT_PRE, R.WEIGHT_NONE)


def _mods():
    N = importlib.import_module("rag-project-icd10_b200._native")
    VI = importlib.import_module("rag-project-icd10_b200.engine.index").VectorIndex
    F = importlib.import_module("rag-project-icd10_b200.engine.filter_expr")
    return N, VI, F


def _p(t):
    return C.c_void_p(0 if t is None else t.data_ptr())


def page_call(idx, q, offset, limit, wm, allowed=None, radius=None, range_filter=None, sync=1, stream=None, out=None):
    """icd_index_search_page with device buffers -> (score, raw, ids) [B, limit] torch tensors on the GPU."""
    N, _, F = _mods()
    B = q.shape[0]
    if out is None:
        out = (torch.empty(B, limit, dtype=torch.float32, device=DEV), torch.empty(B, limit, dtype=torch.float32, device=DEV),
               torch.empty(B, limit, dtype=torch.int64, device=DEV))
    mask = None if allowed is None else torch.from_numpy(F.pack_bits(allowed).view(np.int32)).to(DEV)
    page = N.SearchPage(offset=offset, limit=limit,
                        range_flags=(N.RANGE_RADIUS if radius is not None else 0) | (N.RANGE_FILTER if range_filter is not None else 0),
                        radius=0.0 if radius is None else radius, range_filter=0.0 if range_filter is None else range_filter)
    n = len(idx)
    st = N.lib().icd_index_search_page(idx._h, _p(q), N.vec_dtype(q), B, C.byref(page), wm, _p(mask), n, _p(out[0]),
                                       _p(out[1]), _p(out[2]), C.c_void_p(0 if stream is None else stream.cuda_stream), sync)
    N.check(st, "icd_index_search_page")
    return out


def _same(a, b, what=""):
    for x, y, name in zip(a, b, ("score", "raw", "ids")):
        x = x.cpu().numpy() if isinstance(x, torch.Tensor) else np.asarray(x)
        y = y.cpu().numpy() if isinstance(y, torch.Tensor) else np.asarray(y)
        assert x.shape == y.shape, (what, name, x.shape, y.shape)
        bad = np.nonzero((x.view(np.uint8).reshape(x.shape[0], -1) != y.view(np.uint8).reshape(y.shape[0], -1)).any(1))[0]
        assert bad.size == 0, f"{what} {name}: query {bad[0]} differs: {x[bad[0]][:8]} vs {y[bad[0]][:8]}"


def _table(rows, levels, keep_f32):
    _, VI, _ = _mods()
    idx = VI(rows.shape[1], device=0, keep_f32=keep_f32)
    idx.append(rows, levels)
    return idx


def _q(q, qdtype):
    t = torch.from_numpy(np.ascontiguousarray(q)).to(DEV)
    return t.to(torch.bfloat16) if qdtype == "bf16" else t


# ------------------------------------------------------------------------------------------------ below the cap
@pytest.mark.parametrize("dim", [8, 64, 264, 768, 776, 1024])
@pytest.mark.parametrize("keep_f32", [False, True])
@pytest.mark.parametrize("qdtype", ["f32", "bf16"])
def test_equivalent_to_the_stream_path_below_the_cap(native, dim, keep_f32, qdtype):
    N = native
    rng = np.random.default_rng(dim)
    n = 3001
    rows = R._unit(rng.standard_normal((n, dim))).astype(np.float32)
    rows[n - 40:] = rows[:40]                                       # exact duplicates: ties by id
    levels = _levels(n, dim + 1)
    q = _q(R._unit(rng.standard_normal((6, dim))).astype(np.float32), qdtype)
    allowed = rng.random(n) < 0.5
    idx = _table(rows, levels, keep_f32)
    try:
        for wm in WMS:
            for mask in (None, allowed):
                for offset, limit in ((0, 10), (3, 20), (0, 128), (100, 28)):
                    for qb in (q, q[:1]):                 # 8 queries per score CTA, and the one-query variant
                        K = offset + limit
                        want = idx.search(qb, K, weight_mode=wm, path=N.PATH_STREAM,
                                          mask=None if mask is None else torch.from_numpy(
                                              _mods()[2].pack_bits(mask).view(np.int32)).to(DEV))
                        torch.cuda.synchronize()
                        got = page_call(idx, qb, offset, limit, wm, mask)
                        _same(got, tuple(t[:, offset:] for t in want), f"dim {dim} wm {wm} mask {mask is not None} "
                                                                        f"B {qb.shape[0]} page [{offset}, {K})")
    finally:
        idx.close()


# ------------------------------------------------------------------------------------------------ above the cap
def _certify(res, held, q_used, K, wm, levels, allowed=None, keep_f32=False, chunk_rows=None):
    score, raw, ids = res
    return R.certify(ids, raw, score, held, q_used, K, wm, levels, mask=allowed, f32rows=keep_f32, chunk_rows=chunk_rows)


@pytest.mark.parametrize("keep_f32", [False, True])
def test_probe_corpora_are_certified_above_the_cap(native, keep_f32):
    for dim, n in ((768, 20011), (1024, 17003), (264, 30001)):
        rows, q, _ = R.probe_corpus(n, dim, 9, seed=dim)
        levels = _levels(n, 3)
        idx = _table(rows, levels, keep_f32)
        held = torch.from_numpy(R.held_rows(rows, keep_f32)).to(DEV)
        qt = _q(q, "f32")
        allowed = np.random.default_rng(dim).random(n) < 0.5
        try:
            for K, wm, mask in ((129, R.WEIGHT_NONE, None), (1000, R.WEIGHT_RERANK, allowed), (1000, R.WEIGHT_PRE, None),
                                (16384, R.WEIGHT_NONE, None), (16384, R.WEIGHT_RERANK, allowed)):
                qq = qt[:2] if K == 16384 else qt
                res = page_call(idx, qq, 0, K, wm, mask)
                _certify(res, held, qq, K, wm, levels, mask, keep_f32)
        finally:
            idx.close()


@pytest.fixture(scope="module")
def clustered40k():
    n, dim = 40474, 768
    rows, centers, rng = clustered_corpus(n, dim, seed=404)
    q = _cluster_queries(centers, rng, 64, dim)
    return rows, _levels(n, 405), q


@pytest.mark.parametrize("keep_f32", [False, True])
@pytest.mark.parametrize("qdtype", ["f32", "bf16"])
def test_clustered_40474_rows_are_certified(native, clustered40k, keep_f32, qdtype):
    rows, levels, q = clustered40k
    idx = _table(rows, levels, keep_f32)
    held = torch.from_numpy(R.held_rows(rows, keep_f32)).to(DEV)
    qt = _q(q, qdtype)
    allowed = np.random.default_rng(6).random(len(rows)) < 0.5
    try:
        for K, wm, mask, B in ((129, R.WEIGHT_RERANK, None, 64), (1000, R.WEIGHT_NONE, allowed, 64),
                               (1000, R.WEIGHT_PRE, None, 64), (16384, R.WEIGHT_RERANK, None, 2),
                               (16384, R.WEIGHT_PRE, allowed, 2)):
            res = page_call(idx, qt[:B], 0, K, wm, mask)
            _certify(res, held, qt[:B].float(), K, wm, levels, mask, keep_f32)
    finally:
        idx.close()


@pytest.fixture(scope="module")
def big():
    """2 000 003 clustered rows built on the GPU (test_scan_large_gpu.py's corpus, smaller query set)."""
    n, dim = 2_000_003, 768
    g = torch.Generator(device=DEV).manual_seed(2000003)
    centers = torch.randn(4000, dim, generator=g, device=DEV)
    centers /= centers.norm(dim=1, keepdim=True)
    rows = torch.empty(n, dim, dtype=torch.float32, device=DEV)
    spreads = torch.tensor([0.01, 0.02, 0.05, 0.1], device=DEV)
    for r0 in range(0, n, 1 << 18):
        m = min(n, r0 + (1 << 18)) - r0
        noise = torch.randn(m, dim, generator=g, device=DEV)
        noise /= noise.norm(dim=1, keepdim=True)
        c = centers[torch.randint(0, 4000, (m,), generator=g, device=DEV)]
        s = spreads[torch.randint(0, 4, (m, 1), generator=g, device=DEV)]
        x = torch.where(torch.rand(m, 1, generator=g, device=DEV) < 0.75, c + s * noise, noise)
        rows[r0:r0 + m] = x / x.norm(dim=1, keepdim=True)
    qn = torch.randn(80, dim, generator=g, device=DEV)
    q = centers[torch.randint(0, 4000, (80,), generator=g, device=DEV)] + 0.05 * qn / qn.norm(dim=1, keepdim=True)
    q = (q / q.norm(dim=1, keepdim=True)).contiguous()
    levels = _levels(n, 77)
    _, VI, _ = _mods()
    idx = VI(dim, device=0)
    idx.append(rows, torch.from_numpy(levels).to(DEV))
    held = rows.to(torch.bfloat16).float()
    del rows
    yield idx, held, q, levels
    idx.close()
    del held
    torch.cuda.empty_cache()


def test_two_million_rows_are_certified(native, big):
    idx, held, q, levels = big
    allowed = np.random.default_rng(78).random(len(levels)) < 0.5
    for K, wm, mask, B in ((129, R.WEIGHT_NONE, None, 8), (1000, R.WEIGHT_RERANK, allowed, 8),
                           (16384, R.WEIGHT_PRE, None, 2)):
        res = page_call(idx, q[:B], 0, K, wm, mask)
        _certify(res, held, q[:B], K, wm, levels, mask, chunk_rows=1 << 19)


def test_query_chunks_match_per_query_calls(native, big):
    """At 2 000 003 rows one workspace pass holds about 66 queries: 80 queries run as two passes."""
    idx, _, q, _ = big
    allowed = np.random.default_rng(79).random(idx.__len__()) < 0.5
    for K, wm, mask in ((200, R.WEIGHT_RERANK, None), (1000, R.WEIGHT_NONE, allowed)):
        whole = page_call(idx, q, 10, K - 10, wm, mask)
        for b in range(q.shape[0]):
            one = page_call(idx, q[b:b + 1], 10, K - 10, wm, mask)
            _same(tuple(t[b:b + 1] for t in whole), one, f"query {b} K {K}")


# ------------------------------------------------------------------------------------------------ paging, ranges, ties
@pytest.fixture(scope="module")
def small():
    """12 000 rows: a page of 12 000 holds every row, so one NONE call gives each query's canonical score of every row."""
    n, dim = 12000, 768
    rows, centers, rng = clustered_corpus(n, dim, seed=12)
    q = _cluster_queries(centers, rng, 5, dim)
    levels = _levels(n, 13)
    idx = _table(rows, levels, True)
    qt = _q(q, "f32")
    _, raw, ids = page_call(idx, qt, 0, n, R.WEIGHT_NONE)
    full = np.empty((q.shape[0], n), np.float32)
    np.put_along_axis(full, ids.cpu().numpy(), raw.cpu().numpy(), 1)
    yield idx, qt, full, levels
    idx.close()


def test_pages_concatenate_to_one_call(native, small):
    idx, qt, _, _ = small
    allowed = np.random.default_rng(14).random(len(idx)) < 0.5
    for wm in (R.WEIGHT_PRE, R.WEIGHT_NONE):
        for mask in (None, allowed):
            whole = page_call(idx, qt, 0, 3000, wm, mask)
            pages = [page_call(idx, qt, o, 500, wm, mask) for o in range(0, 3000, 500)]
            _same(whole, tuple(torch.cat([p[i] for p in pages], 1) for i in range(3)), f"wm {wm}")
    s, r, ids = page_call(idx, qt, int(allowed.sum()), 100, R.WEIGHT_NONE, allowed)     # past the allowed rows
    assert bool((ids == -1).all()) and bool(torch.isneginf(r).all()) and bool(torch.isneginf(s).all())


@pytest.mark.parametrize("wm", WMS)
def test_every_rule_against_the_model_on_the_calls_own_scores(native, small, wm):
    """Ranges (both bounds, radius only, empty), masks and offsets: page_ref over the canonical scores, bit for bit."""
    idx, qt, full, levels = small
    rng = np.random.default_rng(15)
    allowed = rng.random(len(idx)) < 0.5
    med = float(np.median(full))
    for offset, limit, mask, radius, rf in ((0, 129, None, None, None), (0, 2000, None, med, None),
                                            (37, 900, allowed, med - 0.05, med + 0.2), (0, 50, None, 0.99, 0.995),
                                            (5, 300, allowed, None, med), (0, 16384, None, None, None),
                                            (2, 400, None, 2.0, None), (16000, 384, None, None, None)):
        got = page_call(idx, qt, offset, limit, wm, mask, radius, rf)
        want = P.page_ref(full, levels, wm, offset, limit, mask, radius, rf)
        _same(got, want, f"page [{offset}, {offset + limit}) range ({radius}, {rf}] mask {mask is not None}")


def test_ranged_list_is_the_unranged_list_filtered(native, small):
    idx, qt, full, _ = small
    med = float(np.median(full))
    for wm in (R.WEIGHT_PRE, R.WEIGHT_NONE):
        s, r, i = (t.cpu().numpy() for t in page_call(idx, qt, 0, len(idx), wm))
        for radius, rf in ((med, med + 0.3), (med, None), (0.9, 0.9001)):
            got = page_call(idx, qt, 0, 3000, wm, None, radius, rf)
            keep = (r > np.float32(radius)) & ((r <= np.float32(rf)) if rf is not None else True)
            want = P._out(qt.shape[0], 3000)
            for b in range(qt.shape[0]):
                sel = np.nonzero(keep[b])[0][:3000]
                want[0][b, :len(sel)], want[1][b, :len(sel)], want[2][b, :len(sel)] = s[b, sel], r[b, sel], i[b, sel]
            _same(got, want, f"wm {wm} range ({radius}, {rf}]")


def test_ties_across_row_blocks_and_zero_queries(native):
    """Identical rows at ids i and n - 1 - i (8 192-row select blocks apart) straddle the K-th rank: lowest id first.
    An all-zero query scores every row 0: ids come back ascending."""
    n, dim = 20000, 64
    rng = np.random.default_rng(16)
    rows = R._unit(rng.standard_normal((n, dim))).astype(np.float32)
    q = R._unit(rng.standard_normal((1, dim))).astype(np.float32)
    s = rows @ q[0]
    top = np.argsort(-s)[:1200]
    rows[n - 1 - top] = rows[top]
    levels = np.full(n, 2, np.uint8)
    idx = _table(rows, levels, False)
    try:
        qt = _q(np.concatenate([q, np.zeros((1, dim), np.float32)]), "f32")
        for K in (999, 1000, 1001, 1500):
            _, raw, ids = (t.cpu().numpy() for t in page_call(idx, qt, 0, K, R.WEIGHT_NONE))
            for j in range(K - 1):
                assert raw[0, j] > raw[0, j + 1] or (raw[0, j] == raw[0, j + 1] and ids[0, j] < ids[0, j + 1]), (K, j)
            assert ids[1].tolist() == list(range(K))
            _certify(page_call(idx, qt[:1], 0, K, R.WEIGHT_NONE), torch.from_numpy(R.held_rows(rows, False)).to(DEV),
                     qt[:1], K, R.WEIGHT_NONE, levels)
    finally:
        idx.close()


# ------------------------------------------------------------------------------------------------ buffers, async, API
def test_guard_regions_and_async(native, small):
    idx, qt, _, _ = small
    B, limit, G = qt.shape[0], 700, 4096
    want = page_call(idx, qt, 50, limit, R.WEIGHT_RERANK, None, 0.0, None)
    bufs = [torch.full((B * limit + G,), v, dtype=dt, device=DEV)
            for v, dt in ((1234.5, torch.float32), (-77.0, torch.float32), (0x5A5A5A5A, torch.int64))]
    out = tuple(b[:B * limit].view(B, limit) for b in bufs)
    st = torch.cuda.Stream()
    page_call(idx, qt, 50, limit, R.WEIGHT_RERANK, None, 0.0, None, sync=0, stream=st, out=out)
    st.synchronize()
    _same(out, want, "sync=0")
    assert bool((bufs[0][B * limit:] == 1234.5).all()) and bool((bufs[1][B * limit:] == -77.0).all())
    assert bool((bufs[2][B * limit:] == 0x5A5A5A5A).all())
    # host buffers through VectorIndex.search (paged because of the offset)
    s, r, i = idx.search(qt.cpu().numpy(), limit, weight_mode=R.WEIGHT_RERANK, offset=50, radius=0.0)
    _same((s, r, i), want, "host buffers")


def test_argument_errors_and_unchanged_calls(native, small):
    N = native
    idx, qt, _, _ = small
    for offset, limit, rad, rf in ((0, 0, None, None), (-1, 10, None, None), (16000, 385, None, None),
                                   (0, 10, 0.5, 0.5), (0, 10, 0.6, 0.5)):
        with pytest.raises(N.NativeError):
            page_call(idx, qt, offset, limit, R.WEIGHT_NONE, None, rad, rf)
    F = _mods()[2]
    bad_mask = torch.from_numpy(F.pack_bits(np.ones(len(idx) + 64, bool)).view(np.int32)).to(DEV)
    page = N.SearchPage(offset=0, limit=10, range_flags=0, radius=0.0, range_filter=0.0)
    out = torch.empty(qt.shape[0], 10, device=DEV)
    assert N.lib().icd_index_search_page(idx._h, _p(qt), N.F32, qt.shape[0], C.byref(page), 0, _p(bad_mask),
                                         len(idx) + 64, _p(out), None, None, None, 1) == -1
    # the k <= 128 calls keep their contract
    ids = torch.empty(qt.shape[0], 129, dtype=torch.int64, device=DEV)
    assert N.lib().icd_index_search(idx._h, _p(qt), N.F32, qt.shape[0], 129, 0, 0, None, None, _p(ids), None, 1) == -1
    with pytest.raises(ValueError, match="PATH_AUTO"):
        idx.search(qt, 200, path=N.PATH_STREAM)


# ------------------------------------------------------------------------------------------------ service and client
def test_service_and_client_beyond_128(native, tmp_path, monkeypatch):
    monkeypatch.setenv("MILVUS_DB_PATH", str(tmp_path / "db" / "big.db"))
    monkeypatch.setenv("MILVUS_COLLECTION_NAME", "icd10")
    M = importlib.import_module("rag-project-icd10_b200.services.milvus_service")
    otext = importlib.import_module("oracle.text")

    class Emb:
        def encode_query(self, q):
            return np.ones(768, np.float32) / np.sqrt(768.0)

    ms = M.MilvusService(embedding_service=Emb())
    recs = otext.load_records(os.path.join(ROOT, "data", "ICD_10v601.csv"))
    rng = np.random.default_rng(21)
    corpus = R._unit(rng.standard_normal((len(recs), 768))).astype(np.float32)
    assert ms.insert_records_array(recs, corpus) is True
    q = R._unit(corpus[rng.integers(0, len(recs), 6)] + 0.05 * rng.standard_normal((6, 768))).astype(np.float32)
    held = torch.from_numpy(corpus).to(DEV)            # the store keeps fp32 master rows
    batch = ms.search_batch(q, top_k=1000)
    ids, raw = batch.row_ids, batch.raw_scores
    lv = np.array([ms.client.field(ms.collection_name, "level", int(i)) for i in range(len(recs))], np.int64)
    w = np.array([1.0, 1.2, 1.0, 0.8])[np.where((lv >= 1) & (lv <= 3), lv, 0)]
    score = np.where(ids >= 0, (raw.astype(np.float64) * w[np.maximum(ids, 0)]).astype(np.float32), -np.inf)
    R.certify(ids, raw, score, held, torch.from_numpy(q).to(DEV), 1000, R.WEIGHT_RERANK, lv.astype(np.uint8),
              f32rows=True)
    for b in range(len(q)):
        one = ms.search(q[b], top_k=500)
        assert len(one) == 500 and len(batch[b]) == 1000
        exact = corpus.astype(np.float64) @ q[b].astype(np.float64)
        assert {recs[i]["code"] for i in np.argsort(-exact)[:480]} <= {c["code"] for c in one}   # clear of near-ties
        assert one == list(ms.search_batch(q[b:b + 1], top_k=500)[0])
    # the client: filter + offset + search_params on the ICD schema
    c = ms.client
    whole = c.search(ms.collection_name, [q[0]], limit=2000, filter="level == 3", output_fields=["code", "level"])[0]
    page = c.search(ms.collection_name, [q[0]], limit=300, filter="level == 3", offset=200,
                    search_params={"metric_type": "IP", "params": {"radius": -1.0, "range_filter": 1.0}},
                    output_fields=["code", "level"])[0]
    assert [h["id"] for h in page] == [h["id"] for h in whole if -1.0 < h["distance"] <= 1.0][200:500]
    assert all(h["entity"]["level"] == 3 for h in page)
