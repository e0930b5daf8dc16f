"""Exact search on tables larger than L2, through the public API, checked with the exactness certificate.

The certified tests of test_scan_exact_gpu.py use tables of at most 40 474 rows (<= 64 MB: no drift limiter, pre-pass
stride 2).  Here a clustered near-duplicate corpus of 2 000 003 rows (3 GB of bf16: pre-pass stride 8, drift limiter on,
a partial last tile) is searched with bf16 and fp32 master rows, fp32 and bf16 queries, B = 1 024 (one launch),
4 096 (two launches with their own drift-limiter regions) and 8 193 (two passes of at most 8 192 queries), k = 10 and
100, every weight mode and a 50 % mask.  certify runs over row chunks (scan_ref.summarise), so no [B, n] score matrix is
ever held.  The host pipeline is checked on the 40 474-row clustered master table, with fallbacks counted per chunk.
The worst error / bound and the fallback counts are printed at the end of the module."""
import importlib

import numpy as np
import pytest
import torch

import scan_ref as R
from test_scan_exact_gpu import clustered_corpus, _cluster_queries, _levels

pytestmark = pytest.mark.gpu

DEV = "cuda"
QF32, QBF16 = "f32", "bf16"
WORST = {}        # case -> worst error / bound
FALLBACKS = {}    # case -> (queries re-searched by the exact stream scan, queries)


@pytest.fixture(scope="module", autouse=True)
def _report(request):
    yield
    tr = request.config.pluginmanager.get_plugin("terminalreporter")
    capman = request.config.pluginmanager.get_plugin("capturemanager")
    if tr is None or capman is None or not WORST:
        return
    with capman.global_and_fixture_disabled():
        tr.write_line("")
        tr.write_line("worst error / bound per case (<= 1 passes) and queries re-searched by the exact fallback:")
        for key in sorted(WORST):
            f, b = FALLBACKS.get(key, (0, 0))
            tr.write_line(f"  {key:<58s} {WORST[key]:.3f}   fallback {f} of {b}")


def _vector_index():
    return importlib.import_module("rag-project-icd10_b200.engine.index").VectorIndex


def _pack(allowed):
    return importlib.import_module("rag-project-icd10_b200.engine.filter_expr").pack_bits(allowed)


def _chunk_rows(B):
    return max(4096, (1 << 27) // B)      # about 1 GB per fp64 [B, chunk] matrix


# ------------------------------------------------------------------------------------------------ 2 000 003 rows
N_BIG, DIM = 2_000_003, 768


@pytest.fixture(scope="module")
def big():
    """Near-duplicate clusters (unit(center + spread * unit noise), spreads 0.01 - 0.1) over 4 000 centers for three
    quarters of the rows, random unit rows for the rest, n / 16 exact duplicates; built on the GPU in fp32."""
    g = torch.Generator(device=DEV).manual_seed(2000003)
    centers = torch.randn(4000, DIM, generator=g, device=DEV)
    centers /= centers.norm(dim=1, keepdim=True)
    rows = torch.empty(N_BIG, DIM, dtype=torch.float32, device=DEV)
    spreads = torch.tensor([0.01, 0.02, 0.05, 0.1], device=DEV)
    for r0 in range(0, N_BIG, 1 << 18):
        m = min(N_BIG, r0 + (1 << 18)) - r0
        noise = torch.randn(m, DIM, generator=g, device=DEV)
        noise /= noise.norm(dim=1, keepdim=True)
        c = centers[torch.randint(0, 4000, (m,), generator=g, device=DEV)]
        s = spreads[torch.randint(0, 4, (m, 1), generator=g, device=DEV)]
        x = torch.where(torch.rand(m, 1, generator=g, device=DEV) < 0.75, c + s * noise, noise)
        rows[r0:r0 + m] = x / x.norm(dim=1, keepdim=True)
    dup = torch.randperm(N_BIG, generator=g, device=DEV)[:2 * (N_BIG // 16)]
    rows[dup[:N_BIG // 16]] = rows[dup[N_BIG // 16:]]
    qn = torch.randn(8193, DIM, generator=g, device=DEV)
    q = centers[torch.randint(0, 4000, (8193,), generator=g, device=DEV)] + 0.05 * qn / qn.norm(dim=1, keepdim=True)
    q = (q / q.norm(dim=1, keepdim=True)).contiguous()
    levels = _levels(N_BIG, 77)
    allowed = np.random.default_rng(78).random(N_BIG) < 0.5
    yield rows, q, levels, allowed
    del rows
    torch.cuda.empty_cache()


# (keep_f32, query dtype, B, k, weight mode, masked)
BIG_CASES = [(False, QF32, 1024, 10, R.WEIGHT_NONE, False),
             (False, QBF16, 1024, 100, R.WEIGHT_RERANK, True),
             (False, QBF16, 4096, 10, R.WEIGHT_PRE, False),
             (False, QF32, 4096, 100, R.WEIGHT_NONE, True),
             (False, QF32, 8193, 10, R.WEIGHT_RERANK, False),
             (False, QBF16, 8193, 10, R.WEIGHT_NONE, False),
             (True, QF32, 1024, 10, R.WEIGHT_PRE, True),
             (True, QF32, 1024, 100, R.WEIGHT_NONE, False),
             (True, QBF16, 1024, 10, R.WEIGHT_RERANK, False),
             (True, QF32, 4096, 10, R.WEIGHT_RERANK, True),
             (True, QBF16, 8193, 10, R.WEIGHT_PRE, False)]


@pytest.mark.parametrize("keep_f32", [False, True])
def test_two_million_rows_are_certified(native, big, keep_f32):
    rows, q_all, levels, allowed = big
    idx = _vector_index()(DIM, device=0, keep_f32=keep_f32)
    try:
        idx.append(rows, torch.from_numpy(levels).to(DEV))
        held = rows if keep_f32 else rows.to(torch.bfloat16).float()
        mask = _pack(allowed)
        for kf, qdtype, B, k, wm, masked in BIG_CASES:
            if kf != keep_f32:
                continue
            q = q_all[:B]
            if qdtype == QBF16:
                q = q.to(torch.bfloat16)
            score, raw, ids = idx.search(q, k, weight_mode=wm, path=native.PATH_AUTO,
                                         mask=mask if masked else None)
            torch.cuda.synchronize()
            case = f"2M keep_f32={keep_f32} q={qdtype} B={B} k={k} wm={wm} mask={masked}"
            old = FALLBACKS.get(case, (0, 0))
            FALLBACKS[case] = (old[0] + idx.take_fallbacks(), old[1] + B)
            cert = R.certify(ids, raw, score, held, q.float(), k, wm, levels, mask=allowed if masked else None,
                             f32rows=keep_f32, chunk_rows=_chunk_rows(B))
            WORST[case] = max(WORST.get(case, 0.0), cert.worst)
    finally:
        idx.close()


# ------------------------------------------------------------------------------------------------ host pipeline
@pytest.fixture(scope="module")
def clustered_master():
    n = 40474
    rows, centers, rng = clustered_corpus(n, DIM, seed=404)
    q = _cluster_queries(centers, rng, 6144, DIM)
    return rows, _levels(n, 405), q


def test_host_pipeline_is_certified_with_fallbacks_inside_its_chunks(native, clustered_master):
    """6 144 host fp32 queries on the clustered 40 474-row master table run as three pipelined chunks of 2 048.  The
    result is certified, and equals the three chunks searched one call at a time, whose fallbacks add up to the
    pipelined call's: uncertified queries are re-searched inside the pipelined chunks."""
    rows, levels, q = clustered_master
    idx = _vector_index()(DIM, device=0, keep_f32=True)
    try:
        idx.append(rows, levels)
        k, wm = 10, R.WEIGHT_RERANK
        score, raw, ids = idx.search(q, k, weight_mode=wm)
        total = idx.take_fallbacks()
        held = torch.from_numpy(rows).to(DEV)
        cert = R.certify(ids, raw, score, held, torch.from_numpy(q).to(DEV), k, wm, levels, f32rows=True,
                         chunk_rows=8192)
        per_chunk = []
        for b0 in range(0, q.shape[0], 2048):
            s, r, i = idx.search(q[b0:b0 + 2048], k, weight_mode=wm)
            per_chunk.append(idx.take_fallbacks())
            assert np.array_equal(i, ids[b0:b0 + 2048]) and np.array_equal(s.view(np.int32),
                                                                         score[b0:b0 + 2048].view(np.int32))
        assert sum(per_chunk) == total, (per_chunk, total)
        assert sum(1 for f in per_chunk if f > 0) >= 2, per_chunk
        case = f"host pipeline 40474 keep_f32 B=6144 per chunk {per_chunk}"
        WORST[case] = cert.worst
        FALLBACKS[case] = (total, q.shape[0])
    finally:
        idx.close()
