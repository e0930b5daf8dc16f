"""Worker for the two-GPU filter test: run under torch.distributed.run, one rank per GPU.  Each rank passes the mask of its
LOCAL rows; the filtered ShardGroup search (both exchanges, both paths, every weight mode) must equal the filtered search
of one table holding every row, bit for bit."""
import importlib
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def main():
    import torch
    import torch.distributed as dist
    from oracle import search as osearch
    rank, world = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"])
    local = int(os.environ.get("LOCAL_RANK", rank))
    torch.cuda.set_device(local)
    dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    N = importlib.import_module("rag-project-icd10_b200._native")
    VectorIndex = importlib.import_module("rag-project-icd10_b200.engine.index").VectorIndex
    shard = importlib.import_module("rag-project-icd10_b200.engine.shard")
    F = importlib.import_module("rag-project-icd10_b200.engine.filter_expr")

    n, dim, B, k = 60_001, 768, 150, 10
    rng = np.random.default_rng(78)          # same data on every rank
    corpus = rng.standard_normal((n, dim)).astype(np.float32)
    corpus /= np.linalg.norm(corpus, axis=1, keepdims=True)
    corpus = osearch.bf16_round(corpus)
    levels = rng.integers(1, 4, size=n).astype(np.uint8)
    q = osearch.bf16_round(corpus[rng.integers(0, n, size=B)] + 0.02 * rng.standard_normal((B, dim)).astype(np.float32))
    masks = {"half": rng.random(n) < 0.5, "range": (np.arange(n) >= 29_000) & (np.arange(n) < 31_000),
             "one_shard": np.arange(n) < 1000, "none": np.zeros(n, bool)}
    lo, hi = shard.shard_bounds(n, rank, world)
    idx = VectorIndex(dim, device=local)
    idx.append(corpus[lo:hi], levels[lo:hi])
    grp = shard.ShardGroup(idx, row_offset=lo, rank=rank, world=world)
    whole = VectorIndex(dim, device=local)
    whole.append(corpus, levels)
    ok = True
    for name, allowed in masks.items():
        gm, lm = F.pack_bits(allowed), F.pack_bits(allowed[lo:hi])
        for mode in (N.WEIGHT_RERANK, N.WEIGHT_NONE, N.WEIGHT_PRE):
            for path in (N.PATH_STREAM, N.PATH_TENSOR):
                qq = q[:6] if path == N.PATH_STREAM else q
                ws, wr, wi = whole.search(qq, k, weight_mode=mode, path=path, mask=gm)
                for exchange in (0, 1):
                    s, r, i = grp.search(qq, k, weight_mode=mode, path=path, exchange=exchange, mask=lm)
                    good = np.array_equal(i, wi) and np.array_equal(r, wr) and np.array_equal(s, ws)
                    good = good and bool(np.all(allowed[i[i >= 0]]))
                    if not good:
                        bad = np.nonzero((i != wi).any(1))[0][:3]
                        print(f"rank {rank} MISMATCH mask={name} mode={mode} exchange={exchange} path={path} "
                              f"queries={bad} {i[bad[:1]]} vs {wi[bad[:1]]}", flush=True)
                    ok = ok and good
    flag = torch.tensor([1 if ok else 0], device="cuda")
    dist.all_reduce(flag, op=dist.ReduceOp.MIN)
    grp.close(); idx.close(); whole.close()
    dist.barrier()
    dist.destroy_process_group()
    if rank == 0:
        print("FILTER_SHARD_OK" if int(flag) == 1 else "FILTER_SHARD_FAIL", flush=True)
    sys.exit(0 if int(flag) == 1 else 1)


if __name__ == "__main__":
    main()
