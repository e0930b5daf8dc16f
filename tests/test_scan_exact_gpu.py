"""Both scan kernels against the exactness certificate of tests/scan_ref.py, at the shapes where they go wrong.

Every result is checked with scan_ref.certify: the returned ids are the canonical fp32 top-k of what the index holds
(bf16 image or fp32 master, fp32 query), up to differences the derived fp32 rounding bound cannot resolve, with the
kernels' order, tie and weight rules.  Planted probes (scan_ref.probe_corpus) turn a dropped or misplaced K block, row
tile or query lane into a miss by a wide margin, and a clustered corpus of near-duplicates, like the ICD table's, puts
rows within 1e-4 of each other.  A session-end summary prints the worst error / bound per (kernel, dim).
"""
import importlib
import os

import numpy as np
import pytest
import torch

import scan_ref as R

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
WORST = {}        # (kernel, dim) -> worst error / bound
FALLBACKS = {}    # what -> (queries re-searched by the exact stream scan, queries)
TC_DIMS = list(range(64, 769, 64))
QF32, QBF16 = "f32", "bf16"


@pytest.fixture(scope="module", autouse=True)
def _report(request):
    yield
    tr = request.config.pluginmanager.get_plugin("terminalreporter")
    capman = request.config.pluginmanager.get_plugin("capturemanager")
    if tr is None or capman is None or not WORST:
        return
    with capman.global_and_fixture_disabled():
        tr.write_line("")
        tr.write_line("worst error / bound per (kernel, dim) (<= 1 passes):")
        for key in sorted(WORST):
            tr.write_line(f"  {key[0]:<8s} dim {key[1]:<5d} {WORST[key]:.3f}")
        if FALLBACKS:
            tr.write_line("queries re-searched by the exact fallback:")
            for what in sorted(FALLBACKS):
                f, b = FALLBACKS[what]
                tr.write_line(f"  {what:<56s} {f} of {b}")


def _record(kernel, dim, cert):
    WORST[(kernel, dim)] = max(WORST.get((kernel, dim), 0.0), cert.worst)


def _count_fallbacks(what, idx, B):
    f = idx.take_fallbacks()
    old = FALLBACKS.get(what, (0, 0))
    FALLBACKS[what] = (old[0] + f, old[1] + B)
    return f


def _levels(n, seed):
    rng = np.random.default_rng(seed)
    return rng.choice(np.array([1, 2, 3], np.uint8), size=n, p=[0.1243, 0.2991, 0.5766]).astype(np.uint8)


class Table:
    """One index and, on the GPU, the rows it holds (fp32 master or bf16 image) for the fp64 reference."""

    def __init__(self, rows, levels, keep_f32):
        VectorIndex = importlib.import_module("rag-project-icd10_b200.engine.index").VectorIndex
        self.idx = VectorIndex(rows.shape[1], device=0, keep_f32=keep_f32)
        self.idx.append(rows, levels)
        self.keep_f32 = keep_f32
        self.held = torch.from_numpy(R.held_rows(rows, keep_f32)).cuda()
        self.levels = levels
        self.dim = rows.shape[1]

    def search(self, native, q, k, wm, path, qdtype=QF32, allowed=None):
        """-> (score, raw, ids) on the GPU and the fp32 queries the index used."""
        F = importlib.import_module("rag-project-icd10_b200.engine.filter_expr")
        qt = torch.from_numpy(np.ascontiguousarray(q)).cuda()
        if qdtype == QBF16:
            qt = qt.to(torch.bfloat16)
        mask = None if allowed is None else F.pack_bits(allowed)
        score, raw, ids = self.idx.search(qt, k, weight_mode=wm, path=path, mask=mask)
        torch.cuda.synchronize()
        return (score, raw, ids), qt.float()

    def certify(self, res, q_used, k, wm, allowed=None, ref=None):
        score, raw, ids = res
        return R.certify(ids, raw, score, self.held, q_used, k, wm, self.levels, mask=allowed, f32rows=self.keep_f32,
                         ref=ref)

    def close(self):
        self.idx.close()


def _queries(q, plants, B):
    """The first B probe queries, with the batch's last lane taken by the probe planted for the full batch's last."""
    last = q.shape[0] - 1
    qb = q[:B].copy()
    pl = {l: r for l, r in plants.items() if l < B - 1}
    if B - 1 < last and last in plants:
        qb[B - 1] = q[last]
        pl[B - 1] = plants[last]
    elif B - 1 in plants:
        pl[B - 1] = plants[B - 1]
    return qb, pl


def _check_plants(ids, plants, allowed):
    ids = ids.cpu().numpy()
    for l, r in plants.items():
        if allowed is None or allowed[r]:
            assert ids[l, 0] == r, f"probe lane {l}: planted row {r}, got {ids[l, :4]}"


def _reset(native):
    native.tune(scan_pair=-1, scan_qsplit=-1, scan_generic=0, scan_small_pre=1)


# ------------------------------------------------------------------------------------------------ tensor path
@pytest.mark.parametrize("dim", TC_DIMS)
def test_tensor_scan_is_certified_at_every_dim(native, dim):
    """PATH_TENSOR at every dim it accepts: generic and specialised issue loops, odd and prime K-block counts, shared-
    memory query tails, nkb = 1, CTA pairs (B = 256) and single CTAs (B = 384: an odd tile count), several launches
    (B = 2049), kc at and past its cap of 128 (k = 56/57 with fp32 queries, 122/123 with bf16), all weight modes and a
    50 % row mask, on the bf16 image and on fp32 master rows."""
    rng = np.random.default_rng(dim)
    # tiny tables: one row; one full row tile plus one row
    for n in (1, 129):
        rows, q, plants = R.probe_corpus(n, dim, 130, seed=dim + n)
        levels = _levels(n, dim + n)
        for keep_f32 in (False, True):
            tab = Table(rows, levels, keep_f32)
            for B, k, wm in ((5, 1, R.WEIGHT_NONE), (130, 10, R.WEIGHT_PRE), (130, 128, R.WEIGHT_RERANK)):
                qb, pl = _queries(q, plants, B)
                res, qu = tab.search(native, qb, k, wm, native.PATH_TENSOR)
                _record("tensor", dim, tab.certify(res, qu, k, wm))
                _check_plants(res[2], pl, None)
            tab.close()
    n = 20011
    rows, q, plants = R.probe_corpus(n, dim, 2049, seed=dim)
    levels = _levels(n, dim + 1)
    allowed = rng.random(n) < 0.5
    cases = [(5, 1, R.WEIGHT_NONE, False, QF32, {}),
             (130, 10, R.WEIGHT_RERANK, False, QF32, {}),
             (256, 56, R.WEIGHT_NONE, False, QBF16, {}),
             (256, 57, R.WEIGHT_PRE, False, QF32, {"scan_pair": 0}),
             (256, 10, R.WEIGHT_NONE, True, QF32, {}),
             (384, 122, R.WEIGHT_NONE, True, QF32, {}),
             (384, 123, R.WEIGHT_RERANK, False, QBF16, {"scan_small_pre": 0}),
             (384, 57, R.WEIGHT_NONE, False, QF32, {"scan_small_pre": 0}),
             (2049, 128, R.WEIGHT_PRE, True, QF32, {}),
             (2049, 10, R.WEIGHT_NONE, False, QBF16, {})]
    if dim >= 576:
        cases += [(256, 10, R.WEIGHT_NONE, False, QF32, {"scan_qsplit": 0}),
                  (130, 10, R.WEIGHT_PRE, False, QBF16, {"scan_qsplit": 0, "scan_pair": 0})]
    if dim == 768:
        cases += [(384, 10, R.WEIGHT_PRE, False, QF32, {"scan_generic": 1}),
                  (256, 56, R.WEIGHT_NONE, True, QBF16, {"scan_generic": 1})]
    for keep_f32 in (False, True):
        tab = Table(rows, levels, keep_f32)
        refs = {}
        try:
            for B, k, wm, masked, qdtype, knobs in cases:
                qb, pl = _queries(q, plants, B)
                al = allowed if masked else None
                native.tune(**knobs)
                try:
                    res, qu = tab.search(native, qb, k, wm, native.PATH_TENSOR, qdtype, al)
                finally:
                    _reset(native)
                _count_fallbacks(f"tensor probes keep_f32={keep_f32} q={qdtype}", tab.idx, B)
                key = (B, qdtype)
                if key not in refs:
                    refs[key] = R.reference(tab.held, qu, keep_f32)
                cert = tab.certify(res, qu, k, wm, al, refs[key])
                _record("tensor", dim, cert)
                _check_plants(res[2], pl, al)
        finally:
            tab.close()


# ------------------------------------------------------------------------------------------------ stream path
STREAM_CASES = [(d, False) for d in (8, 16, 248, 256, 264, 512, 520, 760, 768, 776, 1016, 1024)] + \
               [(d, True) for d in (8, 128, 264, 512, 520, 640, 768, 776, 1024)]


@pytest.mark.parametrize("dim,keep_f32", STREAM_CASES)
def test_stream_scan_is_certified_at_every_width(native, dim, keep_f32):
    """PATH_STREAM at the widths where its chunks-per-lane variant changes (bf16: 256/264, 512/520, 768/776; fp32
    master rows: CPL up to 8), with 1, 2, 3 and 5 queries (ragged passes of 4, and of 2 above dim 768), tables of 1, 31
    and 33 rows (a warp step cut short) and 20 011, k = 1, 10 and 128, with and without a row mask."""
    kernel = "stream32" if keep_f32 else "stream"
    for n in (1, 31, 33, 20011):
        rows, q, plants = R.probe_corpus(n, dim, 5, seed=dim * 7 + n)
        levels = _levels(n, dim + n)
        allowed = np.random.default_rng(n).random(n) < 0.5
        allowed[0] = True
        tab = Table(rows, levels, keep_f32)
        i = 0
        for B in (1, 2, 3, 5):
            qb, pl = _queries(q, plants, B)
            for k in (1, 10, 128):
                wm = (R.WEIGHT_NONE, R.WEIGHT_PRE, R.WEIGHT_RERANK)[i % 3]
                al = allowed if i % 2 else None
                i += 1
                res, qu = tab.search(native, qb, k, wm, native.PATH_STREAM, QF32 if i % 4 else QBF16, al)
                _record(kernel, dim, tab.certify(res, qu, k, wm, al))
                if dim >= R.BK:   # below 64 dimensions random rows come close enough to outweigh a plant's level
                    _check_plants(res[2], pl, al)
        tab.close()


# ------------------------------------------------------------------------------------------------ clustered corpora
def clustered_corpus(n, dim, seed):
    """Near-duplicate clusters of 20 - 300 rows (member = unit(center + spread * unit noise), spreads 0.01 - 0.1), exact
    duplicates (the ICD table has 5 500 rows that share their text with another row) and random rows, shuffled."""
    rng = np.random.default_rng(seed)
    parts, centers = [], []
    total = 0
    while total < n * 3 // 4:
        size = int(rng.integers(20, 301))
        spread = float(rng.choice([0.01, 0.02, 0.05, 0.1]))
        c = R._unit(rng.standard_normal(dim))
        centers.append(c)
        parts.append(R._unit(c + spread * R._unit(rng.standard_normal((size, dim)))))
        total += size
    parts.append(R._unit(rng.standard_normal((n - total, dim))) if n > total else np.zeros((0, dim)))
    rows = np.concatenate(parts)[:n]
    rows = rows[rng.permutation(n)].astype(np.float32)
    dup = rng.choice(n, 2 * (n // 16), replace=False)
    rows[dup[: n // 16]] = rows[dup[n // 16:]]
    return rows, np.stack(centers).astype(np.float32), rng


def _cluster_queries(centers, rng, B, dim):
    q = R._unit(centers[rng.integers(0, len(centers), B)] + 0.05 * R._unit(rng.standard_normal((B, dim))))
    return q.astype(np.float32)


@pytest.fixture(scope="module")
def clustered():
    n, dim = 40474, 768
    rows, centers, rng = clustered_corpus(n, dim, seed=404)
    q = _cluster_queries(centers, rng, 1024, dim)
    return rows, _levels(n, 405), q


@pytest.mark.parametrize("k", [10, 100])
def test_clustered_keep_f32_corpus_is_exact(native, clustered, k):
    """The store's configuration (fp32 master rows, fp32 queries) on near-duplicate clusters: the default path
    (tensor at B = 1024) returns the certified exact top-k in every weight mode."""
    rows, levels, q = clustered
    tab = Table(rows, levels, keep_f32=True)
    ref = None
    for wm in (R.WEIGHT_NONE, R.WEIGHT_PRE, R.WEIGHT_RERANK):
        res, qu = tab.search(native, q, k, wm, native.PATH_AUTO)
        _count_fallbacks(f"clustered keep_f32 k={k}", tab.idx, q.shape[0])
        ref = ref or R.reference(tab.held, qu, True)
        _record("auto32", 768, tab.certify(res, qu, k, wm, None, ref))
        st, _ = tab.search(native, q, k, wm, native.PATH_STREAM)
        for a, b in zip(res, st):
            assert torch.equal(a, b), "tensor path result differs from the stream path's"
    tab.close()


@pytest.mark.parametrize("keep_f32", [False, True])
@pytest.mark.parametrize("qdtype", [QF32, QBF16])
def test_a_query_result_does_not_depend_on_its_batch(native, clustered, keep_f32, qdtype):
    """A query alone (B = 1: the stream path), in a batch of 3 (the tensor path with master rows) and in a batch of
    1 024 (the tensor path) returns the same bits.  The one allowed difference: bf16 queries on bf16 rows, where both
    paths score the canonical products and may differ by a swap the certificate accepts as an fp32 accumulation tie."""
    rows, levels, q = clustered
    tab = Table(rows, levels, keep_f32)
    k, wm = 10, R.WEIGHT_RERANK
    full, qu = tab.search(native, q, k, wm, native.PATH_AUTO, qdtype)
    ref = R.reference(tab.held, qu, keep_f32)
    _record("auto32" if keep_f32 else "auto", 768, tab.certify(full, qu, k, wm, None, ref))
    exact_tie_only = not keep_f32 and qdtype == QBF16
    for j in range(0, 1024, 31):
        for sub in (q[j:j + 1], q[j:j + 3]):
            got, qs = tab.search(native, sub, k, wm, native.PATH_AUTO, qdtype)
            same = all(torch.equal(a[0], b[j]) for a, b in zip(got, full))
            if not same:
                assert exact_tie_only, f"query {j}: batch of {sub.shape[0]} differs from the batch of 1024"
                tab.certify(got, qs, k, wm, None, tuple(x[j:j + sub.shape[0]] for x in ref))
    tab.close()


def test_service_search_equals_search_batch(tmp_path, monkeypatch, clustered):
    """MilvusService.search(q) (one query: the stream scan over the fp32 rows) equals search_batch(...)[i] (the tensor
    path) on the ICD table's 40 474 records with clustered embeddings."""
    monkeypatch.setenv("MILVUS_DB_PATH", str(tmp_path / "db" / "c.db"))
    monkeypatch.setenv("MILVUS_COLLECTION_NAME", "icd10")
    otext = importlib.import_module("oracle.text")
    M = importlib.import_module("rag-project-icd10_b200.services.milvus_service")

    class _Emb:
        def encode_query(self, q):
            return np.ones(768, np.float32) / np.sqrt(768.0)

    rows, _, q = clustered
    recs = otext.load_records(os.path.join(ROOT, "data", "ICD_10v601.csv"))
    assert len(recs) == rows.shape[0]
    ms = M.MilvusService(embedding_service=_Emb())
    assert ms.insert_records_array(recs, rows) is True
    qs = q[:96]
    batch = ms.search_batch(qs, 10)
    for b in range(qs.shape[0]):
        assert list(batch[b]) == ms.search(qs[b], 10), b
    ms.disconnect()


# ------------------------------------------------------------------------------------------------ path agreement
@pytest.mark.parametrize("dim", TC_DIMS)
def test_paths_agree_bit_for_bit(native, dim):
    """Where both paths hold the same candidates, raw and score agree bit for bit (one canonical rescoring).  With fp32
    queries or master rows every query holds them (the certificate sends the others to the stream scan); bf16 queries
    on bf16 rows may differ by an accumulation tie the certificate accepts."""
    n = 20011
    rows, centers, rng = clustered_corpus(n, dim, seed=dim + 3)
    levels = _levels(n, dim)
    q = _cluster_queries(centers, rng, 300, dim)
    for keep_f32 in (False, True):
        tab = Table(rows, levels, keep_f32)
        for qdtype in (QF32, QBF16):
            st, qu = tab.search(native, q, 10, R.WEIGHT_RERANK, native.PATH_STREAM, qdtype)
            tc, _ = tab.search(native, q, 10, R.WEIGHT_RERANK, native.PATH_TENSOR, qdtype)
            _count_fallbacks(f"path agreement keep_f32={keep_f32} q={qdtype}", tab.idx, q.shape[0])
            ref = R.reference(tab.held, qu, keep_f32)
            _record("stream32" if keep_f32 else "stream", dim, tab.certify(st, qu, 10, R.WEIGHT_RERANK, None, ref))
            _record("tensor", dim, tab.certify(tc, qu, 10, R.WEIGHT_RERANK, None, ref))
            same = (st[2] == tc[2]).all(1)
            for a, b in zip(st, tc):
                assert torch.equal(a[same].view(torch.int32) if a.dtype == torch.float32 else a[same],
                                   b[same].view(torch.int32) if b.dtype == torch.float32 else b[same])
            if keep_f32 or qdtype == QF32:
                assert bool(same.all()), f"{int((~same).sum())} queries differ between the paths"
        tab.close()


@pytest.mark.parametrize("dim", [1024, 72, 32, 8])
def test_tensor_path_refuses_unsupported_dims_and_auto_falls_back(native, dim):
    rows, q, _ = R.probe_corpus(2000, dim, 64, seed=dim)
    tab = Table(rows, _levels(2000, dim), keep_f32=False)
    with pytest.raises(native.NativeError, match=rf"status -5: tensor scan needs dim % 64 == 0, dim <= 768 \(dim={dim}\)"):
        tab.search(native, q, 10, R.WEIGHT_NONE, native.PATH_TENSOR)
    auto, qu = tab.search(native, q, 10, R.WEIGHT_NONE, native.PATH_AUTO)
    st, _ = tab.search(native, q, 10, R.WEIGHT_NONE, native.PATH_STREAM)
    for a, b in zip(auto, st):
        assert torch.equal(a, b)
    tab.certify(auto, qu, 10, R.WEIGHT_NONE)
    tab.close()
