"""Paged and range search without a GPU: the reference model of icd_index_search_page (tests/page_ref.py) against a
brute-force statement of the rules, the kernels' algorithm (radix select, block-ordered gather, level-run merge)
emulated in numpy against the model, and the store's pymilvus argument handling against a recording fake index."""
import functools
import importlib

import numpy as np
import pytest

import page_ref as P

WMS = (P.WEIGHT_RERANK, P.WEIGHT_PRE, P.WEIGHT_NONE)


def _brute(raw, levels, wm, offset, limit, mask=None, radius=None, range_filter=None):
    """The contract in plain Python: allowed rows, cmp-sorted by (key desc, id asc), cut to K, stable re-rank."""
    B, n = raw.shape
    K = offset + limit
    score = np.full((B, limit), -np.inf, np.float32)
    rw = np.full((B, limit), -np.inf, np.float32)
    ids = np.full((B, limit), -1, np.int64)
    w = {1: 1.2, 3: 0.8}
    for b in range(B):
        rows = [i for i in range(n) if (mask is None or mask[i])
                and (radius is None or raw[b, i] > np.float32(radius))
                and (range_filter is None or raw[b, i] <= np.float32(range_filter))]

        def key(i):
            r = raw[b, i]
            return float(r * np.float32(w.get(int(levels[i]), 1.0))) if wm == P.WEIGHT_PRE else float(r)

        def cmp(i, j):
            ki, kj = key(i), key(j)
            if ki != kj:                      # -0.0 == +0.0 here: the id decides
                return -1 if ki > kj else 1
            return -1 if i < j else 1

        lst = sorted(rows, key=functools.cmp_to_key(cmp))[:K]
        if wm == P.WEIGHT_RERANK:
            lst = sorted(lst, key=lambda i: -(float(raw[b, i]) * w.get(int(levels[i]), 1.0)))   # Python sort is stable
        for s, i in enumerate(lst[offset:K]):
            ids[b, s], rw[b, s] = i, raw[b, i]
            if wm == P.WEIGHT_RERANK:
                score[b, s] = np.float32(float(raw[b, i]) * w.get(int(levels[i]), 1.0))
            elif wm == P.WEIGHT_PRE:
                score[b, s] = raw[b, i] * np.float32(w.get(int(levels[i]), 1.0))
            else:
                score[b, s] = raw[b, i]
    return score, rw, ids


def _same(a, b):
    for x, y in zip(a, b):
        assert x.shape == y.shape
        assert np.array_equal(np.asarray(x).view(np.uint8), np.asarray(y).view(np.uint8)), (x, y)


def _tied_scores(B, n, seed):
    """Scores drawn from a few values, +0.0 and -0.0 among them, so that ties (and the zero pair) straddle the K-th."""
    rng = np.random.default_rng(seed)
    vals = np.array([0.5, 0.25, 0.0, -0.0, -0.25, 0.125, 1.0, -1.0], np.float32)
    return vals[rng.integers(0, len(vals), (B, n))]


@pytest.mark.parametrize("wm", WMS)
def test_model_matches_brute_force(wm):
    rng = np.random.default_rng(1)
    n = 300
    levels = rng.integers(0, 5, n).astype(np.uint8)
    for raw in (_tied_scores(3, n, 2), rng.standard_normal((3, n)).astype(np.float32)):
        for offset, limit in ((0, 7), (5, 40), (0, 300), (250, 100), (400, 3)):
            for mask, radius, rf in ((None, None, None), (rng.random(n) < 0.5, None, None), (None, 0.0, None),
                                     (None, None, 0.25), (rng.random(n) < 0.7, -0.25, 0.5), (None, 2.0, None)):
                _same(P.page_ref(raw, levels, wm, offset, limit, mask, radius, rf),
                      _brute(raw, levels, wm, offset, limit, mask, radius, rf))


def test_plus_and_minus_zero_are_one_key_broken_by_id():
    raw = np.array([[-0.0, 0.0, -0.0, 0.0, 0.5]], np.float32)
    levels = np.ones(5, np.uint8)
    for wm in WMS:
        for f in (P.page_ref, P.page_emulate):
            _, r, ids = f(raw, levels, wm, 0, 5)
            assert ids[0].tolist() == [4, 0, 1, 2, 3], (f.__name__, wm, ids)
            assert np.signbit(r[0, 1:]).tolist() == [True, False, True, False]    # the raw bits come back as stored


@pytest.mark.parametrize("wm", WMS)
def test_kernel_algorithm_matches_model(wm):
    rng = np.random.default_rng(3)
    n = 5000
    levels = rng.integers(0, 5, n).astype(np.uint8)
    for raw in (_tied_scores(2, n, 4), rng.standard_normal((2, n)).astype(np.float32),
                (rng.standard_normal((2, n)) * 1e-3).astype(np.float32)):
        for offset, limit in ((0, 129), (100, 900), (0, 4999), (0, 5000), (4000, 2000), (16384 - 10, 10)):
            for mask, radius, rf in ((None, None, None), (rng.random(n) < 0.5, None, None), (None, 0.0, 0.5),
                                     (rng.random(n) < 0.02, None, None)):
                _same(P.page_emulate(raw, levels, wm, offset, limit, mask, radius, rf, block_rows=512),
                      P.page_ref(raw, levels, wm, offset, limit, mask, radius, rf))


def test_ties_straddling_the_kth_rank_come_back_lowest_id_first():
    """Identical rows at ids i and n - 1 - i, in different row blocks, tie at the K-th rank."""
    n, K = 4096, 1000
    raw = np.linspace(1.0, 0.0, n, dtype=np.float32)[None, :].copy()
    raw[0, n - 1 - np.arange(600)] = raw[0, :600]
    levels = np.full(n, 2, np.uint8)
    _, _, ids = P.page_emulate(raw, levels, P.WEIGHT_NONE, 0, K, block_rows=256)
    _same(P.page_emulate(raw, levels, P.WEIGHT_NONE, 0, K, block_rows=256), P.page_ref(raw, levels, P.WEIGHT_NONE, 0, K))
    got = ids[0].tolist()
    for i in range(500):                               # pairs well inside the top K: lower id first
        assert got[2 * i] == i and got[2 * i + 1] == n - 1 - i


def test_pages_concatenate_to_one_call():
    rng = np.random.default_rng(5)
    n = 3000
    raw = _tied_scores(2, n, 6)
    levels = rng.integers(1, 4, n).astype(np.uint8)
    for wm in (P.WEIGHT_PRE, P.WEIGHT_NONE):
        whole = P.page_ref(raw, levels, wm, 0, 1200)
        pages = [P.page_ref(raw, levels, wm, o, 300) for o in range(0, 1200, 300)]
        _same(whole, tuple(np.concatenate([p[i] for p in pages], 1) for i in range(3)))
    # past the allowed rows: an all-tail page
    s, r, ids = P.page_ref(raw, levels, P.WEIGHT_NONE, n, 10)
    assert (ids == -1).all() and np.isneginf(r).all() and np.isneginf(s).all()


# ------------------------------------------------------------------------------------------------ store arguments
class SearchFake:
    """engine.index.VectorIndex stand-in: keeps the rows and answers searches with the reference model."""
    calls = []

    def __init__(self, dim, device=0, capacity=0, keep_f32=False):
        self.vecs = np.zeros((0, dim), np.float32)
        self.levels = np.zeros((0,), np.uint8)

    def append(self, vecs, levels=None):
        self.vecs = np.concatenate([self.vecs, np.asarray(vecs, np.float32)])
        self.levels = np.concatenate([self.levels, np.asarray(levels, np.uint8)])

    def __len__(self):
        return len(self.vecs)

    def close(self):
        pass

    def search(self, q, k, weight_mode=0, path=0, mask=None, offset=0, radius=None, range_filter=None):
        SearchFake.calls.append(dict(k=k, weight_mode=weight_mode, offset=offset, radius=radius,
                                     range_filter=range_filter, masked=mask is not None))
        allowed = None
        if mask is not None:
            allowed = ((np.asarray(mask).view(np.uint32)[np.arange(len(self)) >> 5] >> (np.arange(len(self)) & 31)) & 1) > 0
        raw = (np.asarray(q, np.float32) @ self.vecs.T).astype(np.float32)
        return P.page_ref(raw, self.levels, weight_mode, offset, k, allowed, radius, range_filter)


@pytest.fixture()
def client(monkeypatch, tmp_path):
    S = importlib.import_module("rag-project-icd10_b200.engine.store")
    N = importlib.import_module("rag-project-icd10_b200._native")
    F = importlib.import_module("rag-project-icd10_b200.engine.filter_expr")
    monkeypatch.setattr(N, "require_gpu", lambda: None)
    monkeypatch.setattr(S, "VectorIndex", SearchFake)

    def host_mask(self, col, expr):   # the device bitmap, kept on the host
        pred = F.compile(expr)
        return None if pred.is_all else F.pack_bits(pred.mask(col.rows, col.row_lo, col.row_hi))

    monkeypatch.setattr(S.IcdStoreClient, "_row_mask", host_mask)
    SearchFake.calls = []
    c = S.IcdStoreClient(uri=str(tmp_path / "m.db"))
    sch = c.create_schema(enable_dynamic_field=True)
    sch.add_field(field_name="id", datatype=S.DataType.INT64, is_primary=True, auto_id=True)
    sch.add_field(field_name="vector", datatype=S.DataType.FLOAT_VECTOR, dim=8)
    c.create_collection("icd10", schema=sch, index_params=c.prepare_index_params())
    c.load_collection("icd10")
    n = 400
    rng = np.random.default_rng(7)
    rows = [{"code": f"A{i:03d}", "preferred_zh": f"疾病{i}", "has_complication": False, "main_code": f"A{i}",
             "secondary_code": "", "level": 1 + i % 3, "parent_code": "A", "category_path": "A",
             "semantic_text": f"t{i}"} for i in range(n)]
    vecs = rng.standard_normal((n, 8)).astype(np.float32)
    c.insert_arrays("icd10", rows, vecs)
    yield c, S, N, vecs
    c.close()


def _ids(hits):
    return [h["id"] for h in hits[0]]


def test_store_offset_in_both_spellings_and_limit_beyond_128(client):
    c, S, N, vecs = client
    q = vecs[3] + 0.1
    whole = _ids(c.search("icd10", [q], limit=300))
    assert len(whole) == 300 and SearchFake.calls[-1]["k"] == 300          # no clamp to 128
    assert _ids(c.search("icd10", [q], limit=50, offset=120)) == whole[120:170]
    assert _ids(c.search("icd10", [q], limit=50, search_params={"offset": 120})) == whole[120:170]
    assert _ids(c.search("icd10", [q], limit=50, offset=120, search_params={"offset": 120})) == whole[120:170]
    with pytest.raises(ValueError, match="conflicting offsets"):
        c.search("icd10", [q], limit=50, offset=10, search_params={"offset": 20})
    assert c.search("icd10", [q], limit=10, offset=395)[0].__len__() == 5
    assert c.search("icd10", [q], limit=10, offset=1000) == [[]]
    _, _, ids = c.search_ranked("icd10", q[None, :], 300)
    assert ids.shape == (1, 300) and SearchFake.calls[-1]["k"] == 300


def test_store_rejects_out_of_range_pages_like_pymilvus(client):
    c, S, N, vecs = client
    q = [vecs[0]]
    assert len(c.search("icd10", q, limit=16384)[0]) == 400
    assert len(c.search("icd10", q, limit=16000, offset=384)[0]) == 16
    for kw in (dict(limit=16385), dict(limit=0), dict(limit=-3), dict(limit=10, offset=-1),
               dict(limit=16000, offset=385), dict(limit=1, search_params={"offset": 16384})):
        with pytest.raises(ValueError):
            c.search("icd10", q, **kw)
    for lim in (0, 16385):
        with pytest.raises(ValueError):
            c.search_ranked("icd10", np.asarray(q), lim)


def test_store_range_search_params(client):
    c, S, N, vecs = client
    q = vecs[5]
    raw = (q[None, :] @ vecs.T).astype(np.float32)[0]
    hits = c.search("icd10", [q], limit=400, search_params={"params": {"radius": 0.5, "range_filter": 2.0}})[0]
    want = [int(i) for i in np.lexsort((np.arange(400), -raw.astype(np.float64))) if 0.5 < raw[i] <= 2.0]
    assert [h["id"] for h in hits] == want and all(0.5 < h["distance"] <= 2.0 for h in hits)
    assert SearchFake.calls[-1]["radius"] == 0.5 and SearchFake.calls[-1]["range_filter"] == 2.0
    hits = c.search("icd10", [q], limit=400, search_params={"metric_type": "IP", "params": {"radius": 1.0}})[0]
    order = np.lexsort((np.arange(400), -raw.astype(np.float64)))
    assert [h["id"] for h in hits] == [int(i) for i in order if raw[i] > 1.0]
    assert SearchFake.calls[-1]["radius"] == 1.0 and SearchFake.calls[-1]["range_filter"] is None
    for params in ({"radius": 1.0, "range_filter": 1.0}, {"radius": 2.0, "range_filter": 0.5}):
        with pytest.raises(ValueError, match="radius < range_filter"):
            c.search("icd10", [q], limit=10, search_params={"params": params})
    with pytest.raises(ValueError):
        c.search("icd10", [q], limit=10, search_params=[("offset", 1)])


def test_store_filter_offset_and_range_together(client):
    c, S, N, vecs = client
    q = vecs[9]
    raw = (q[None, :] @ vecs.T).astype(np.float32)[0]
    level = np.array([1 + i % 3 for i in range(400)])
    order = [int(i) for i in np.lexsort((np.arange(400), -raw.astype(np.float64)))]
    want = [i for i in order if level[i] == 2 and -1.0 < raw[i] <= 1.5]
    got = c.search("icd10", [q], limit=20, filter="level == 2", offset=5,
                   search_params={"params": {"radius": -1.0, "range_filter": 1.5}}, output_fields=["level"])[0]
    assert [h["id"] for h in got] == want[5:25] and all(h["entity"]["level"] == 2 for h in got)
    assert SearchFake.calls[-1]["masked"]


def test_sharded_collection_refuses_what_it_cannot_serve(client):
    c, S, N, vecs = client

    class Group:
        def search(self, q, k, weight_mode=0, mask=None):
            return (np.zeros((len(q), k), np.float32), np.zeros((len(q), k), np.float32),
                    np.tile(np.arange(k), (len(q), 1)))

    c.attach_group("icd10", Group())
    q = [vecs[0]]
    assert len(c.search("icd10", q, limit=128)[0]) == 128
    for kw in (dict(limit=129), dict(limit=10, offset=1), dict(limit=10, search_params={"params": {"radius": 0.1}}),
               dict(limit=10, search_params={"params": {"range_filter": 0.1}})):
        with pytest.raises(NotImplementedError, match="sharded"):
            c.search("icd10", q, **kw)
    with pytest.raises(NotImplementedError, match="sharded"):
        c.search_ranked("icd10", np.asarray(q), 500)
