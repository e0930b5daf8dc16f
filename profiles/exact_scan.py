"""Cost of the tensor path's exactness certificate and exact fallback at BASELINE configs[1]: 40 474 rows, fp32 master
rows (keep_f32, the store's default), B = 1 024 fp32 queries in host memory, k = 10, through VectorIndex.search.

Two corpora: random unit rows (every query certified) and near-duplicate clusters like the ICD table's (some queries
go to the stream scan).  Prints one JSON line per (corpus, weight mode) with the GPU's name and power limit; run it on the
parent commit and on this one for the before / after (profiles/exact_scan.jsonl).

  python profiles/exact_scan.py [--reps 50] [--out FILE]
"""
import argparse
import importlib
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))


def _gpu():
    try:
        return subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"],
                              capture_output=True, text=True).stdout.strip().splitlines()[0]
    except Exception:
        return "unknown"


def _clustered(n, dim, seed):
    from test_scan_exact_gpu import clustered_corpus, _cluster_queries
    rows, centers, rng = clustered_corpus(n, dim, seed)
    return rows, _cluster_queries(centers, rng, 1024, dim)


def _random(n, dim, seed):
    rng = np.random.default_rng(seed)
    u = lambda x: (x / np.linalg.norm(x, axis=1, keepdims=True)).astype(np.float32)
    return u(rng.standard_normal((n, dim))), u(rng.standard_normal((1024, dim)))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=50)
    ap.add_argument("--out", default="")
    args = ap.parse_args()
    VectorIndex = importlib.import_module("rag-project-icd10_b200.engine.index").VectorIndex
    N = importlib.import_module("rag-project-icd10_b200._native")
    n, dim, k = 40474, 768, 10
    levels = np.random.default_rng(1).choice(np.array([1, 2, 3], np.uint8), size=n, p=[0.1243, 0.2991, 0.5766])
    gpu = _gpu()
    lines = []
    for corpus, make in (("random", _random), ("clustered", _clustered)):
        rows, q = make(n, dim, 404)
        idx = VectorIndex(dim, device=0, keep_f32=True)
        idx.append(rows, levels)
        for wm in (N.WEIGHT_NONE, N.WEIGHT_RERANK):
            for _ in range(5):
                idx.search(q, k, weight_mode=wm)
            fb = idx.take_fallbacks() // 5 if hasattr(idx, "take_fallbacks") else None
            times = []
            for _ in range(args.reps):
                t0 = time.perf_counter()
                idx.search(q, k, weight_mode=wm)     # host in, host out: returns after a device synchronise
                times.append(time.perf_counter() - t0)
            if hasattr(idx, "take_fallbacks"):
                idx.take_fallbacks()
            t = np.array(times) * 1e3
            line = dict(corpus=corpus, rows=n, dim=dim, B=1024, k=k, weight_mode=int(wm), keep_f32=True,
                        ms_p50=round(float(np.median(t)), 4), ms_p10=round(float(np.percentile(t, 10)), 4),
                        ms_p90=round(float(np.percentile(t, 90)), 4), fallback_queries=fb, gpu=gpu,
                        tree=os.environ.get("EXACT_SCAN_TREE", "this"))
            print(json.dumps(line), flush=True)
            lines.append(line)
        idx.close()
    if args.out:
        with open(args.out, "a") as f:
            for line in lines:
                f.write(json.dumps(line) + "\n")


if __name__ == "__main__":
    main()
