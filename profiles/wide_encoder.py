"""The 1024-wide encoder (XLM-RoBERTa-large shape: 24 layers, hidden 1024, 16 heads, FFN 4096) on one GPU.

Prints one JSON line per measurement (and writes them to --out):
  * card: name and power limit (nvidia-smi), read in the same run;
  * throughput: sentences/s of forward_ids at S = 64, B = 4096 over >= 2 s windows, and the achieved TFLOP/s of the
    algorithmic work, 24 x [2 (4 H^2 + 2 H I) + 4 S H] per token = 610.3 MFLOP (39.06 GFLOP per 64-token sentence),
    against the repository's measured sustained bf16 peak (MEASURED_PEAKS.json, DESIGN.md §4: 1 373 TFLOP/s);
  * encode_query-shaped latency: p50 / p90 of a batch-1 forward at 12 / 32 / 64 tokens (host ids in, host vector out);
  * text in: sentences/s of EmbeddingService.encode_batch over the ICD table's query texts through the HF Unigram
    tokenizer of a synthetic multilingual-e5-large directory, and the feeder's (tokeniser's) share of the wall time;
  * the exact search at dim 1024, which takes the stream path (the tensor scan needs dim <= 768): a 10 000-query
    search over the 40 474-row ICD-sized table, fp32 master rows kept as the service keeps them.
Synthetic seeded weights (the throughput does not depend on the values); vocabulary 8 000 rows.
usage: python profiles/wide_encoder.py [--out FILE.jsonl]   (profiles/wide_encoder.jsonl holds a recorded run)
"""
import argparse
import importlib
import json
import os
import subprocess
import sys
import tempfile
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
import wide_model as WM  # noqa: E402

SUSTAINED_BF16_TFLOPS = 1373.0
LAYERS, H, I = 24, 1024, 4096


def flops_per_token(S):
    return LAYERS * (2 * (4 * H * H + 2 * H * I) + 4 * S * H)


def emit(fh, rec):
    line = json.dumps(rec)
    print(line, flush=True)
    fh.write(line + "\n")
    fh.flush()


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True).stdout.strip().splitlines()
    return q[0] if q else "unknown"


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None, help="also write the JSON lines to this file")
    ap.add_argument("--window", type=float, default=2.0)
    args = ap.parse_args()
    fh = open(args.out, "w") if args.out else open(os.devnull, "w")
    emit(fh, {"what": "card", "nvidia_smi": card()})
    N = importlib.import_module("rag-project-icd10_b200._native")
    E = importlib.import_module("rag-project-icd10_b200.engine.encoder")
    W = importlib.import_module("rag-project-icd10_b200.engine.weights")
    cfg = WM.xlmr_config(layers=LAYERS, vocab_size=8000)
    state = WM.state_dict(cfg, seed=7)
    ncfg = W.config_from_dict(dict(cfg.to_dict(), model_type="xlm-roberta"))
    eng = E.EncoderEngine(cfg=ncfg, blob=W.pack_state_dict(state, ncfg), tokenizer=object(), device=0,
                          max_tokens=4096 * 64, position_offset=2, unk_id=3, max_seq_length=512)

    # ---- throughput at S = 64, B = 4096 (device-resident ids, lengths and output)
    B, S = 4096, 64
    rng = np.random.default_rng(0)
    ids = torch.from_numpy(rng.integers(4, 8000, size=(B, S)).astype(np.int32)).cuda()
    lens = torch.full((B,), S, dtype=torch.int32).cuda()
    out = torch.empty((B, H), dtype=torch.float32, device="cuda")
    for _ in range(3):
        eng.forward_ids(ids, lens, out=out)
    torch.cuda.synchronize()
    for w in range(3):
        n, t0 = 0, time.perf_counter()
        while time.perf_counter() - t0 < args.window:
            eng.forward_ids(ids, lens, out=out, sync=False)
            n += 1
            if n % 4 == 0:
                torch.cuda.synchronize()
        torch.cuda.synchronize()
        dt = time.perf_counter() - t0
        sps = n * B / dt
        tflops = sps * S * flops_per_token(S) / 1e12
        emit(fh, {"what": "throughput", "window": w, "B": B, "S": S, "batches": n, "seconds": dt, "sentences_per_s": sps,
                  "gflop_per_sentence": S * flops_per_token(S) / 1e9, "tflops": tflops,
                  "of_sustained_bf16": tflops / SUSTAINED_BF16_TFLOPS})

    # ---- batch-1 latency (encode_query shape: host ids in, host vector out)
    for S1 in (12, 32, 64):
        ids1 = rng.integers(4, 8000, size=(1, S1)).astype(np.int32)
        lens1 = np.array([S1], np.int32)
        for _ in range(20):
            eng.forward_ids(ids1, lens1)
        ts = []
        for _ in range(300):
            t0 = time.perf_counter()
            eng.forward_ids(ids1, lens1)
            ts.append(time.perf_counter() - t0)
        ts.sort()
        emit(fh, {"what": "batch1_latency", "tokens": S1, "p50_ms": ts[len(ts) // 2] * 1e3, "p90_ms": ts[int(len(ts) * 0.9)] * 1e3})
    eng.close()

    # ---- text in through EmbeddingService (HF Unigram tokenizer of a synthetic e5-large directory)
    from oracle import text as otext
    recs = otext.load_records(os.path.join(ROOT, "data", "ICD_10v601.csv"))
    texts = [r["semantic_text"] for r in recs]
    tok = WM.unigram_tokenizer([otext.query_text(t) for t in texts])
    d = tempfile.mkdtemp()
    WM.save_e5_dir(d, cfg, state, tok)
    os.environ["EMBEDDING_MODEL_NAME"] = d
    S_mod = importlib.import_module("rag-project-icd10_b200.services.embedding_service")
    es = S_mod.EmbeddingService()
    es.encode_batch(texts[:5000], show_progress=False)
    for w in range(2):
        t0 = time.perf_counter()
        v = es.encode_batch(texts, show_progress=False)
        dt = time.perf_counter() - t0
        st = dict(es.model.last_stats)
        emit(fh, {"what": "text_in", "window": w, "sentences": len(texts), "tokens": st.get("tokens"), "seconds": dt,
                  "sentences_per_s": len(texts) / dt, "tokenize_wait_s": st.get("tokenize_wait_s"),
                  "feeder_share": (st.get("tokenize_wait_s") or 0.0) / dt, "tokenizer": st.get("tokenizer"),
                  "dim": len(v[0])})
    prepared = [es._prepare_text_for_embedding(t) for t in texts]
    t0 = time.perf_counter()
    es.model.tokenizer(prepared, truncation=True, max_length=512)
    emit(fh, {"what": "hf_tokenizer_alone", "sentences": len(texts), "seconds": time.perf_counter() - t0})
    es.model.close()

    # ---- exact search at dim 1024: the stream path
    VectorIndex = importlib.import_module("rag-project-icd10_b200.engine.index").VectorIndex
    n_rows, nq = len(recs), 10000
    corpus = rng.standard_normal((n_rows, H)).astype(np.float32)
    corpus /= np.linalg.norm(corpus, axis=1, keepdims=True)
    q = rng.standard_normal((nq, H)).astype(np.float32)
    q /= np.linalg.norm(q, axis=1, keepdims=True)
    levels = np.full(n_rows, 3, np.uint8)
    for keep in (True, False):
        idx = VectorIndex(H, device=0, keep_f32=keep)
        idx.append(corpus, levels)
        idx.search(q[:64], 10)
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        idx.search(q, 10)
        torch.cuda.synchronize()
        emit(fh, {"what": "search_1024d", "rows": n_rows, "queries": nq, "k": 10, "keep_f32": keep,
                  "ms": (time.perf_counter() - t0) * 1e3})
        idx.close()
    emit(fh, {"what": "card_after", "nvidia_smi": card()})


if __name__ == "__main__":
    main()
