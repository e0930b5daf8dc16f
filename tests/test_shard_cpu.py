"""Host-side logic of the row-sharded search, on CPU: shard bounds, the merge rule the GPU
exchange implements (oracle level), and the torch.distributed bootstrap under gloo, world 2."""
import importlib
import os
import socket
import sys

import numpy as np
import pytest

from oracle import search as osearch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_shard_bounds_partition():
    shard = importlib.import_module("rag-project-icd10_b200.engine.shard")
    for total in (0, 1, 7, 40474, 100_000_000):
        for world in (1, 2, 3, 4, 8):
            spans = [shard.shard_bounds(total, r, world) for r in range(world)]
            assert spans[0][0] == 0 and spans[-1][1] == total
            assert all(a[1] == b[0] for a, b in zip(spans, spans[1:]))
            sizes = [hi - lo for lo, hi in spans]
            assert max(sizes) - min(sizes) <= 1


def test_merge_of_shard_topk_equals_global_topk():
    rng = np.random.default_rng(9)
    c = rng.standard_normal((9000, 64)).astype(np.float32)
    c[7000] = c[12]
    q = np.concatenate([c[12:13], rng.standard_normal((5, 64)).astype(np.float32)])
    ref_s, ref_i = osearch.exact_topk(c, q, 10)
    shard = importlib.import_module("rag-project-icd10_b200.engine.shard")
    for world in (2, 4, 8):
        ss, ii = [], []
        for r in range(world):
            lo, hi = shard.shard_bounds(len(c), r, world)
            s, i = osearch.exact_topk(c[lo:hi], q, 10)
            ss.append(s); ii.append(i + lo)
        m_s, m_i = osearch.merge_shards(ss, ii, 10)
        assert np.array_equal(m_i, ref_i) and np.allclose(m_s, ref_s, atol=1e-6)


def _free_port():
    s = socket.socket(); s.bind(("127.0.0.1", 0)); p = s.getsockname()[1]; s.close(); return p


def _gloo_worker(rank, world, port, q):
    import torch.distributed as dist
    sys.path.insert(0, ROOT)
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    dist.init_process_group("gloo", rank=rank, world_size=world)
    shard = importlib.import_module("rag-project-icd10_b200.engine.shard")
    ident, table = shard.bootstrap_exchange(dist, rank, world, (bytes([rank + 1]) * 128) if rank == 0 else None,
                                            bytes([10 + rank]) * 64, share_ident=True)
    # each rank searches its rows with the oracle; merged result must equal the global one
    rng = np.random.default_rng(4)
    c = rng.standard_normal((2001, 32)).astype(np.float32)
    qs = rng.standard_normal((4, 32)).astype(np.float32)
    lo, hi = shard.shard_bounds(len(c), rank, world)
    s, i = osearch.exact_topk(c[lo:hi], qs, 5)
    gathered = [None] * world
    dist.all_gather_object(gathered, (s, i + lo))
    m_s, m_i = osearch.merge_shards([g[0] for g in gathered], [g[1] for g in gathered], 5)
    ref_s, ref_i = osearch.exact_topk(c, qs, 5)
    q.put((rank, ident == bytes([1]) * 128, table == bytes([10]) * 64 + bytes([11]) * 64, bool(np.array_equal(m_i, ref_i))))
    dist.destroy_process_group()


def test_bootstrap_exchange_gloo_world2():
    import torch.multiprocessing as mp
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    port = _free_port()
    procs = [ctx.Process(target=_gloo_worker, args=(r, 2, port, q)) for r in range(2)]
    for p in procs:
        p.start()
    res = [q.get(timeout=120) for _ in procs]
    for p in procs:
        p.join(timeout=60)
    assert sorted(r[0] for r in res) == [0, 1]
    assert all(r[1] and r[2] and r[3] for r in res), res


def test_partition_by_tokens_balances_and_covers():
    shard = importlib.import_module("rag-project-icd10_b200.engine.shard")
    rng = np.random.default_rng(3)
    counts = rng.integers(3, 129, size=1001).tolist()
    for world in (1, 2, 3, 8):
        parts = shard.partition_by_tokens(counts, world)
        assert sorted(j for p in parts for j in p) == list(range(len(counts)))
        loads = [sum(counts[j] for j in p) for p in parts]
        assert max(loads) - min(loads) <= 128          # within one longest sentence
    assert shard.partition_by_tokens([], 4) == [[], [], [], []]
    assert shard.partition_by_tokens([5], 2) == [[0], []]


def _dp_worker(rank, world, port, q):
    import torch.distributed as dist
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    dist.init_process_group("gloo", rank=rank, world_size=world)
    shard = importlib.import_module("rag-project-icd10_b200.engine.shard")
    texts = ["t%03d" % i + "x" * (i % 17) for i in range(53)]
    counts = [len(t) + 2 for t in texts]

    def fake_encode(batch):           # a deterministic stand-in for an encoder replica
        return np.stack([np.full(8, float(int(t[1:4])), np.float32) for t in batch]) if batch else np.zeros((0, 8), np.float32)
    full = shard.encode_data_parallel(fake_encode, texts, counts, rank, world, dist=dist, dim=8)
    local = shard.encode_data_parallel(fake_encode, texts, counts, rank, world, dist=None, dim=8)
    mine = shard.partition_by_tokens(counts, world)[rank]
    ok_full = bool(np.array_equal(full[:, 0], np.arange(53, dtype=np.float32)))
    ok_local = bool(np.array_equal(local[mine, 0], np.asarray(mine, np.float32))) and float(np.abs(local).sum()) == float(sum(mine)) * 8
    q.put((rank, ok_full, ok_local))
    dist.destroy_process_group()


def test_encode_data_parallel_gloo_world2():
    import torch.multiprocessing as mp
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    port = _free_port()
    procs = [ctx.Process(target=_dp_worker, args=(r, 2, port, q)) for r in range(2)]
    for p in procs:
        p.start()
    res = [q.get(timeout=120) for _ in procs]
    for p in procs:
        p.join(timeout=60)
    assert sorted(r[0] for r in res) == [0, 1]
    assert all(r[1] and r[2] for r in res), res


# ---------------------------------------------------------------------------------------------- sharded build, host side
class _FakeIndex:
    def __init__(self, dim, device=0, capacity=0, keep_f32=False):
        self.dim = dim
        self.vecs = np.zeros((0, dim), np.float32)

    def append(self, vecs, levels=None):
        self.vecs = np.concatenate([self.vecs, np.asarray(vecs, np.float32)])

    def __len__(self):
        return len(self.vecs)

    def close(self):
        pass


class _FakeGroup:
    def __init__(self, index, row_offset, rank, world):
        self.index, self.row_offset = index, row_offset


class _FakeEmb:
    """Deterministic stand-in for an encoder replica: the vector of a text depends on the text only."""
    def _vec(self, text):
        import zlib
        rng = np.random.default_rng(zlib.crc32(text.encode("utf-8")))
        v = rng.standard_normal(8).astype(np.float32)
        return v / np.linalg.norm(v)

    def encode_query(self, q):
        return self._vec("query: " + q)

    def encode_queries(self, qs):
        return np.stack([self._vec("query: " + q) for q in qs])

    encode_queries_device = encode_queries

    def test_embedding(self, t):
        return {"success": True}

    def get_model_info(self):
        return {"loaded": True}


def _patched_builder(rank, world, dist, db_path):
    os.environ.update(MILVUS_DB_PATH=db_path, MILVUS_COLLECTION_NAME="icd10", MILVUS_MODE="local", PYTHONHASHSEED="0")
    N = importlib.import_module("rag-project-icd10_b200._native")
    S = importlib.import_module("rag-project-icd10_b200.engine.store")
    sh = importlib.import_module("rag-project-icd10_b200.engine.shard")
    B = importlib.import_module("rag-project-icd10_b200.tools.build_database")
    M = importlib.import_module("rag-project-icd10_b200.services.milvus_service")
    N.require_gpu = lambda: None
    S.VectorIndex = _FakeIndex
    sh.ShardGroup = _FakeGroup
    B.EmbeddingService = _FakeEmb
    M.MilvusService.client_kwargs = {}
    return B, B.DatabaseBuilder(rank=rank, world=world, dist=dist)


def _build_worker(rank, world, port, work, q):
    import torch.distributed as dist
    sys.path.insert(0, ROOT)
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    dist.init_process_group("gloo", rank=rank, world_size=world)
    B, builder = _patched_builder(rank, world, dist, os.path.join(work, "sharded.db"))
    ok = builder.build_full_database(os.path.join(work, "subset.csv"), rebuild=True)
    col = builder.milvus_service.client.cols["icd10"]
    q.put((rank, bool(ok), len(col.rows), col.row_lo, col.row_hi, len(col.index), isinstance(getattr(col, "group", None), _FakeGroup)))
    dist.barrier()
    dist.destroy_process_group()


def test_sharded_build_writes_the_same_files_as_a_single_process_build(tmp_path, monkeypatch):
    """tools/build_database.py with the records split over 2 ranks (gloo, fake encoder / device table): rank 0 writes the
    scalar columns and commits, every rank fills its slice of the vector files; the result is byte-identical to the
    single-process build and every rank ends up serving rows shard_bounds(n, r, 2)."""
    import torch.multiprocessing as mp
    monkeypatch.chdir(tmp_path)     # the builder appends to ./logs/database_build.log; the workers inherit the directory
    os.environ["PYTHONHASHSEED"] = "0"
    src = open(os.path.join(ROOT, "data", "ICD_10v601.csv"), encoding="utf-8-sig").read().splitlines()
    (tmp_path / "subset.csv").write_text("﻿" + "\n".join(src[:702]) + "\n", encoding="utf-8")
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    port = _free_port()
    procs = [ctx.Process(target=_build_worker, args=(r, 2, port, str(tmp_path), q)) for r in range(2)]
    for p in procs:
        p.start()
    res = sorted(q.get(timeout=180) for _ in procs)
    for p in procs:
        p.join(timeout=60)
    n = res[0][2]
    assert n == 701 and all(r[1] and r[2] == n and r[6] for r in res), res
    assert [(r[3], r[4]) for r in res] == [(0, n // 2), (n // 2, n)] and [r[5] for r in res] == [n // 2, n - n // 2]
    # single-process build of the same CSV in this process
    saved = {k: os.environ.get(k) for k in ("MILVUS_DB_PATH", "MILVUS_COLLECTION_NAME", "MILVUS_MODE")}
    mods = [importlib.import_module("rag-project-icd10_b200." + m) for m in ("_native", "engine.store", "engine.shard", "tools.build_database")]
    keep = (mods[0].require_gpu, mods[1].VectorIndex, mods[2].ShardGroup, mods[3].EmbeddingService)
    try:
        B, single = _patched_builder(0, 1, None, str(tmp_path / "single.db"))
        assert single.build_full_database(str(tmp_path / "subset.csv"), rebuild=True)
        single.milvus_service.disconnect()
    finally:
        mods[0].require_gpu, mods[1].VectorIndex, mods[2].ShardGroup, mods[3].EmbeddingService = keep
        for k, v in saved.items():
            if v is None:
                os.environ.pop(k, None)
            else:
                os.environ[k] = v
    d1, d2 = tmp_path / "sharded.db.icdb" / "icd10", tmp_path / "single.db.icdb" / "icd10"
    names = sorted(os.listdir(d2))
    assert names == sorted(os.listdir(d1)) and "vectors.f32" in names and "code.off" in names
    for fn in names:
        assert (d1 / fn).read_bytes() == (d2 / fn).read_bytes(), fn
