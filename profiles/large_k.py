"""Device time of the paged search (icd_index_search_page) beyond k = 128, next to the k = 128 scan on the same shape.

Grid: the 40 474-row table at dims 768 and 1024, bf16 rows and fp32 master rows, B = 1, 64 and 1 024, K = 129, 1 000
and 16 384; and 10 000 000 x 768 bf16 rows at B = 1 and 16, K = 1 000.  Queries and results stay on the device; each
time is CUDA events around `--reps` back-to-back calls (after warm-up), divided by the count.  The 40 474-row tables fit
in L2 after the first pass; the 10 M-row table (15 GB) does not.  Writes one JSON line per shape, with the card's name
and power limit read in the same run.

  python profiles/large_k.py [--reps 10] [--out profiles/large_k.jsonl] [--quick]
"""
import argparse
import importlib
import json
import os
import subprocess
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def _gpu():
    out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"],
                         capture_output=True, text=True).stdout.strip().splitlines()
    return out[0] if out else "unknown"


def _time(fn, reps):
    for _ in range(2):
        fn()
    torch.cuda.synchronize()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(reps):
        fn()
    b.record()
    b.synchronize()
    return a.elapsed_time(b) / reps


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=10)
    ap.add_argument("--out", default="")
    ap.add_argument("--quick", action="store_true", help="one small shape only (a rehearsal of the script)")
    args = ap.parse_args()
    VectorIndex = importlib.import_module("rag-project-icd10_b200.engine.index").VectorIndex
    N = importlib.import_module("rag-project-icd10_b200._native")
    gpu = _gpu()
    dev = torch.device("cuda", 0)
    g = torch.Generator(device=dev).manual_seed(5)
    grid = []
    for dim in (768, 1024):
        for keep_f32 in (False, True):
            for B in (1, 64, 1024):
                grid.append((40474, dim, keep_f32, B, (129, 1000, 16384)))
    grid.append((10_000_000, 768, False, 1, (1000,)))
    grid.append((10_000_000, 768, False, 16, (1000,)))
    if args.quick:
        grid = [(40474, 768, False, 4, (129,))]
    lines = []
    tables = {}
    for n, dim, keep_f32, B, Ks in grid:
        key = (n, dim, keep_f32)
        if key not in tables:
            tables.clear()
            torch.cuda.empty_cache()
            idx = VectorIndex(dim, device=0, keep_f32=keep_f32, capacity=n)
            for r0 in range(0, n, 1 << 20):
                m = min(n, r0 + (1 << 20)) - r0
                x = torch.randn(m, dim, generator=g, device=dev)
                idx.append((x / x.norm(dim=1, keepdim=True)).contiguous(),
                           torch.randint(1, 4, (m,), generator=g, device=dev, dtype=torch.uint8))
            tables[key] = idx
        idx = tables[key]
        q = torch.randn(B, dim, generator=g, device=dev)
        q = (q / q.norm(dim=1, keepdim=True)).contiguous()
        base = _time(lambda: idx.search(q, 128, weight_mode=N.WEIGHT_RERANK, sync=False), args.reps)
        for K in Ks:
            reps = max(2, args.reps // (4 if K == 16384 and B == 1024 else 1))
            ms = _time(lambda: idx.search(q, K, weight_mode=N.WEIGHT_RERANK, sync=False), reps)
            line = dict(rows=n, dim=dim, rows_dtype="f32 master" if keep_f32 else "bf16", B=B, K=K,
                        ms_per_call=round(ms, 4), ms_k128=round(base, 4), ratio_to_k128=round(ms / base, 2),
                        table_reads=-(-B // 8), weight_mode="rerank", gpu=gpu)
            print(json.dumps(line), flush=True)
            lines.append(line)
    if args.out:
        with open(args.out, "w") as f:
            for line in lines:
                f.write(json.dumps(line) + "\n")


if __name__ == "__main__":
    main()
