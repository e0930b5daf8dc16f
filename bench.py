#!/usr/bin/env python3
"""bench.py -- headline benchmark of the retrieval hot path (BASELINE.json metric).

  python bench.py --gpus N --steps K --warmup W            our arm (libicdrag.so on B200)
  python bench.py --impl reference --gpus N --steps K ...  the reference's CPU path (oracle port)
  python bench.py ... --dump-outputs DIR                    also write the last timed step's results as DIR/*.npy, so
                                                            two builds can be compared output for output (same inputs)

Workload (config.workload): exact top-10 inner-product search of a batch of 1024 synthetic
768-d bf16 queries over a synthetic 100 M x 768 bf16 corpus -- BASELINE.json configs[4].  The
corpus is row-sharded over the N GPUs (strong scaling: total rows fixed, 100 M / N per GPU; at
N = 1 the whole 153.6 GB table sits in one B200's 180 GB).  One "step" = one batch through the
scan.  `value` is queries/s with queries and corpus resident in HBM; `e2e` is the same metric
through the C ABI with HOST query/result buffers (H2D + D2H inside the timed region).

A quarter of the queries are PLANTED: perturbed copies of corpus rows spread evenly over all shards, so every
driver-run line carries its own correctness evidence (`checks`): the planted row must come back first, scores
must be sorted, host and device paths must agree, and at N > 1 the sharded search must equal a single-table
search (on a 1 M-row check corpus gathered onto every rank) and an independent torch merge of the local lists.

Besides the headline (batch 1024: tensor-bound by arithmetic, SURVEY 8d) the same resident table is measured at
batch 128 (`hbm_point`, HBM-bound) and batch 256 (`ridge_point`), each over >= 1 s of load with its own clocks.
`config1_point` (N = 1) is BASELINE configs[1]: 10 000 queries against a table of the reference's own 40 474 rows.
The `encoder` object is BASELINE configs[2] (S = 64, B = 4096) plus `e2e_text`: EmbeddingService text in ->
embeddings out over >= 200 k real ICD strings (native tokeniser, pinned staging, GPU encoder).

The corpus (15x-1200x the 126 MB L2) is far larger than L2, so every step streams it from HBM:
no L2 flush is needed between iterations (config.l2 says so).
"""
import argparse
import importlib
import json
import math
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

DIM = 768
K_TOP = 10
PKG = "rag-project-icd10_b200"
DUMP_MAX_BYTES = 64 << 20


def _peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        with open(p) as fh:
            d = json.load(fh)
        return {"hbm_gbs": d["hbm_gbs"], "bf16_tflops": d["bf16_tflops"],
                "bf16_tflops_sustained": d.get("bf16_tflops_sustained", d["bf16_tflops"]), "source": "measured"}
    return {"hbm_gbs": 6650.0, "bf16_tflops": 1590.0, "bf16_tflops_sustained": 1400.0, "source": "fallback"}


def _ncu_traffic(key):
    """DRAM bytes per launch of the dominant kernel from the committed `ncu --set full` capture of this
    exact workload (profiles/ncu_traffic.json), or (None, None) when no capture matches."""
    try:
        with open(os.path.join(ROOT, "profiles", "ncu_traffic.json")) as fh:
            ent = json.load(fh).get(key)
        return (ent["bytes"], ent["capture"]) if ent else (None, None)
    except Exception:
        return None, None


def dump_outputs(out_dir, score, raw, ids):
    """--dump-outputs: what search() hands its caller for the headline batch -- level-weighted scores, raw inner
    products and global row ids, [B, k] each -- as out_dir/<name>.npy in float32 / float64 (ids are exact in float64).
    Above DUMP_MAX_BYTES in all, a fixed seeded sample of query rows is written, its row numbers in query_rows.npy."""
    import numpy as np
    import torch
    arrays = {"scores": score.float(), "raw_scores": raw.float(), "ids": ids.double()}
    n = score.shape[0]
    row_bytes = sum(a.element_size() * a.shape[1] for a in arrays.values())
    if n * row_bytes > DUMP_MAX_BYTES:
        rows = np.sort(np.random.default_rng(0).choice(n, DUMP_MAX_BYTES // (row_bytes + 8), replace=False))
        sel = torch.from_numpy(rows).to(score.device)
        arrays = {name: a[sel] for name, a in arrays.items()}
        arrays["query_rows"] = torch.from_numpy(rows.astype(np.float64))
    os.makedirs(out_dir, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(out_dir, name + ".npy"), a.cpu().numpy())


def _icd_env():
    """ICD_* environment variables seen by this run (knobs that could change the measured path)."""
    return {k: v for k, v in sorted(os.environ.items()) if k.startswith("ICD")}


class ClockSampler:
    """nvidia-smi clocks + throttle reasons during the timed region (B200_PROFILING.md recipe)."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,"
         "clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        self.gpu = gpu_index
        self.proc = None
        self.lines = []       # (arrival time, csv line)
        self.t0 = self.t1 = None

    def begin(self):
        """Start of the load window (the process was started earlier: nvidia-smi takes ~0.2 s to come up)."""
        self.t0 = time.time()

    def end(self):
        self.t1 = time.time()

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.gpu), f"--query-gpu={self.Q}",
                                          "--format=csv,noheader,nounits", "-lms", "100"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._pump, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _pump(self):
        for line in self.proc.stdout:
            self.lines.append((time.time(), line.strip()))

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:
            self.proc.kill()
        sm, mx, pw, reasons = [], [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        t0 = self.t0 if self.t0 is not None else 0.0
        t1 = self.t1 if self.t1 is not None else time.time()
        for ts, ln in self.lines:
            if ts < t0 + 0.05 or ts > t1 + 0.02:   # a sample describes the period before it arrives
                continue
            f = [x.strip() for x in ln.split(",")]
            if len(f) < 9:
                continue
            try:
                sm.append(float(f[1])); mx.append(float(f[2]))
            except ValueError:
                continue
            try:
                pw.append(float(f[3]))
            except ValueError:
                pass
            for name, val in zip(names, f[5:9]):
                if val.lower().startswith("active"):
                    reasons.add(name)
        sm.sort()
        pw.sort()
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "power_w": pw[len(pw) // 2] if pw else None, "samples": len(sm), "reasons": sorted(reasons)}


def make_corpus(torch, rows, device, seed):
    """SURVEY 8d: i.i.d. N(0,1) -> fp32 L2-normalise -> bf16 (the bf16 values ARE the corpus);
    level bytes ~ Categorical(0.1243, 0.2991, 0.5766).  Built in 1 M-row chunks."""
    g = torch.Generator(device=device).manual_seed(seed)
    table = torch.empty((rows, DIM), dtype=torch.bfloat16, device=device)
    chunk = 1 << 20
    for lo in range(0, rows, chunk):
        n = min(chunk, rows - lo)
        x = torch.randn((n, DIM), generator=g, device=device, dtype=torch.float32)
        x = torch.nn.functional.normalize(x, dim=1)
        table[lo:lo + n] = x.to(torch.bfloat16)
        del x
    u = torch.rand((rows,), generator=g, device=device)
    levels = torch.full((rows,), 3, dtype=torch.uint8, device=device)
    levels[u < 0.1243 + 0.2991] = 2
    levels[u < 0.1243] = 1
    return table, levels


def make_queries(torch, batch, device, seed=999):
    g = torch.Generator(device=device).manual_seed(seed)
    q = torch.randn((batch, DIM), generator=g, device=device, dtype=torch.float32)
    return torch.nn.functional.normalize(q, dim=1).to(torch.bfloat16)


def planted_ids(batch, rows_total):
    """Query positions 0, 4, 8, ... are planted; planted query j looks for global row (j + 1/2) rows / P, so the
    planted rows are spread evenly over the whole table (every shard at every N <= P)."""
    pos = list(range(0, batch, 4))
    n = len(pos)
    return pos, [min(rows_total - 1, int((j + 0.5) * rows_total / n)) for j in range(n)]


def make_planted_queries(torch, dist, table, lo, hi, rows_total, batch, dev, rank, world):
    """[batch, 768] bf16 queries, identical on every rank: i.i.d. directions, every 4th one replaced by a corpus row
    plus N(0, 0.01^2) noise per component (cosine ~0.96 with its row; the best i.i.d. row scores ~0.2)."""
    q = make_queries(torch, batch, dev).float()
    pos, gids = planted_ids(batch, rows_total)
    rows = torch.zeros((len(pos), DIM), dtype=torch.float32, device=dev)
    for j, g in enumerate(gids):
        if lo <= g < hi:
            rows[j] = table[g - lo].float()
    if world > 1:
        dist.all_reduce(rows)      # exactly one rank holds each planted row: the sum is that row
    gen = torch.Generator(device=dev).manual_seed(4242)
    noise = torch.randn(rows.shape, generator=gen, device=dev, dtype=torch.float32) * 0.01
    q[pos] = torch.nn.functional.normalize(rows + noise, dim=1)
    q = q.to(torch.bfloat16).contiguous()
    if world > 1:
        dist.broadcast(q, 0)       # bit-identical queries everywhere (no reliance on equal RNG streams)
    return q, pos, gids


def _use_all_host_threads():
    """torchrun exports OMP_NUM_THREADS=1; the CPU arm is meant to use every host core, so undo
    that before numpy / BLAS load (and through threadpoolctl if they already have)."""
    cores = os.cpu_count() or 1
    for var in ("OMP_NUM_THREADS", "OPENBLAS_NUM_THREADS", "MKL_NUM_THREADS"):
        os.environ[var] = str(cores)
    try:
        from threadpoolctl import threadpool_limits
        threadpool_limits(limits=cores)
    except Exception:
        pass
    return cores


class CpuScanSample:
    """The reference's CPU search path (Milvus FLAT/IP restated: oracle/search.py::fast_topk, fp32 numpy GEMM over
    all host threads + argpartition) on a bounded sample of the workload: the REAL batch against a row slice.
    The synthetic corpus slice is generated ONCE; step() only runs the search."""

    def __init__(self, rows, batch):
        _use_all_host_threads()
        import numpy as np
        from oracle import search as osearch
        self.np, self.osearch = np, osearch
        rng = np.random.default_rng(1234)
        corpus = rng.standard_normal((rows, DIM), dtype=np.float32)
        corpus /= np.linalg.norm(corpus, axis=1, keepdims=True)
        u = corpus.view(np.uint32)                 # round to bf16 in place (nearest even), values stay fp32
        u += np.uint32(0x7FFF) + ((u >> np.uint32(16)) & np.uint32(1))
        u &= np.uint32(0xFFFF0000)
        self.corpus = corpus
        q = rng.standard_normal((batch, DIM), dtype=np.float32)
        self.q = q / np.linalg.norm(q, axis=1, keepdims=True)
        self.rows, self.batch = rows, batch

    def calibrate(self, calls, budget_s):
        """Warm the BLAS threads on 1/8 of the slice and shrink the slice so that `calls` searches fit the budget."""
        n8 = max(1024, self.rows // 8)
        self.osearch.fast_topk(self.corpus[:n8], self.q[: max(1, self.batch // 8)], K_TOP)
        t0 = time.perf_counter()
        self.osearch.fast_topk(self.corpus[:n8], self.q, K_TOP)
        est = (time.perf_counter() - t0) * self.rows / n8
        if calls * est > budget_s:
            self.rows = max(n8, int(self.rows * budget_s / (calls * est)) // 1024 * 1024)
            self.corpus = self.corpus[: self.rows]
        return est

    def step(self):
        t0 = time.perf_counter()
        self.osearch.fast_topk(self.corpus, self.q, K_TOP)
        return time.perf_counter() - t0

    def describe(self, total_rows, batch):
        s = (f"{self.batch} queries x {self.rows} rows per step (numpy fp32 GEMM + argpartition top-k, "
             f"oracle/search.py::fast_topk; corpus slice generated once), extrapolated linearly in rows to {total_rows}")
        if self.batch != batch:
            s += f" and in batch to {batch}"
        return s


def cpu_encoder_sample(n_sent=256, seq=64, batch=32):
    """The reference's CPU encoder path (SentenceTransformer.encode restated: HF BertModel fp32 + masked mean +
    L2 normalise, oracle/encoder.py) on a bounded sample: n_sent synthetic sentences of `seq` tokens in batches of
    32 (encode_batch's batch_size, embedding_service.py:97-102), all host threads."""
    cores = _use_all_host_threads()
    import torch
    torch.set_num_threads(cores)
    from transformers import BertModel
    from oracle import encoder as oenc
    torch.manual_seed(0)
    model = BertModel(oenc.bert_config(12, 21128, 512), add_pooling_layer=False).eval()
    g = torch.Generator().manual_seed(7)
    ids = torch.randint(1000, 21128, (n_sent, seq), generator=g)
    ids[:, 0], ids[:, -1] = 101, 102
    mask = torch.ones_like(ids)

    def run():
        with torch.no_grad():
            for lo in range(0, n_sent, batch):
                h = model(input_ids=ids[lo:lo + batch], attention_mask=mask[lo:lo + batch]).last_hidden_state
                m = mask[lo:lo + batch].unsqueeze(-1).float()
                torch.nn.functional.normalize((h * m).sum(1) / m.sum(1).clamp(min=1e-9), p=2, dim=1)
    run()   # warm-up (thread pools, allocator)
    t0 = time.perf_counter()
    run()
    dt = time.perf_counter() - t0
    # batch 1, what encode_query does once per ICD row in the reference's build loop (build_database.py:221)
    n1 = 32
    with torch.no_grad():
        model(input_ids=ids[:1], attention_mask=mask[:1])
        t1 = time.perf_counter()
        for i in range(n1):
            h = model(input_ids=ids[i:i + 1], attention_mask=mask[i:i + 1]).last_hidden_state
            torch.nn.functional.normalize(h.mean(1), p=2, dim=1)
        dt1 = time.perf_counter() - t1
    return {"value": n_sent / dt, "unit": "sentences/s", "cores": cores, "kind": "port",
            "batch1_sentences_per_s": n1 / dt1,
            "sample": f"{n_sent} synthetic sentences x {seq} tokens, batch {batch} (and {n1} at batch 1), 12-layer HF "
                      f"BertModel fp32 (oracle/encoder.py arithmetic), torch {torch.get_num_threads()} threads"}


def workload_config(args, world, rows_total=None, note=None):
    """The `config` object: shared by both arms so the driver compares like with like."""
    rows_total = rows_total or args.rows
    rows_local = rows_total * 1 // world if world > 1 else rows_total
    w = f"exact top-{K_TOP} IP, {rows_total} x {DIM} bf16 corpus row-sharded over {world} GPU(s), batch {args.batch}"
    if note:
        w += f" ({note})"
    return {"workload": w, "rows": rows_total, "rows_per_gpu": rows_local, "dim": DIM, "batch": args.batch,
            "k": K_TOP, "weight_mode": "rerank", "l2": "corpus >> L2 (no flush needed)", "tune": args.tune or None,
            "exchange": ("peer-store" if args.exchange else "nccl-allgather") if world > 1 else None,
            "planted_queries": len(range(0, args.batch, 4))}


def run_reference(args, rank, world):
    """--impl reference: the reference's own CPU implementation of the path (restated: numpy
    fp32 exact IP + top-k; pymilvus/milvus-lite are not installable offline), host cores only.
    Same config as our arm: the real batch (1024) against a row slice generated once; every step is one search of
    the slice; `ms_per_step` is the MEASURED step, `value` its extrapolation in rows (exact scan cost is linear in
    rows) to the full table.  The slice shrinks if warmup + steps would not fit --cpu-budget-s."""
    if rank != 0:
        return
    cores = _use_all_host_threads()
    import torch
    torch.set_num_threads(cores)
    total_rows = args.rows
    t_setup = time.perf_counter()
    sample = CpuScanSample(args.cpu_rows, args.cpu_batch or args.batch)
    sample.calibrate(args.warmup + args.steps, args.cpu_budget_s)
    setup_s = time.perf_counter() - t_setup
    times = []
    for i in range(args.warmup + args.steps):
        dt = sample.step()
        if i >= args.warmup:
            times.append(dt)
    dt = sum(times) / len(times)
    # one step of the real workload = batch x total_rows; the sample is the same arithmetic on a row slice
    full_step_s = dt * (total_rows / sample.rows) * (args.batch / sample.batch)
    qps = args.batch / full_step_s
    line = {
        "impl": "reference", "metric": "top-10 cosine QPS (100M x 768)", "value": qps, "unit": "queries/s",
        "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": dt * 1e3,
        "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": workload_config(args, max(1, args.gpus)),
        "cpu_baseline": {"value": qps, "unit": "queries/s", "cores": cores, "kind": "port",
                         "torch_threads": torch.get_num_threads(),
                         "sample": sample.describe(total_rows, args.batch),
                         "sample_rows": sample.rows, "sample_batch": sample.batch,
                         "measured_ms_per_sample_step": dt * 1e3, "extrapolated_ms_per_full_step": full_step_s * 1e3,
                         "setup_s": setup_s},
        "e2e": {"value": qps, "unit": "queries/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "env": _icd_env(),
    }
    if not args.no_encoder:
        try:
            cb = cpu_encoder_sample()
            line["encoder"] = {"metric": "text2vec sentences/sec", "value": cb["value"], "unit": "sentences/s",
                               "batch": 32, "seq_len": 64, "layers": 12, "dtype": "f32", "cpu_baseline": cb}
        except Exception as e:
            line["encoder"] = {"error": repr(e)[:200]}
    emit(line)


_REAL_STDOUT = None


def quiet_stdout():
    """Libraries (NCCL prints its version banner) write to fd 1; the contract is ONE JSON line on
    stdout, so fd 1 is pointed at stderr for the run and the line goes to the saved descriptor."""
    global _REAL_STDOUT
    if _REAL_STDOUT is None:
        sys.stdout.flush()
        _REAL_STDOUT = os.dup(1)
        os.dup2(2, 1)


def emit(line):
    data = (json.dumps(line) + "\n").encode()
    if _REAL_STDOUT is None:
        sys.stdout.write(data.decode())
        sys.stdout.flush()
    else:
        os.write(_REAL_STDOUT, data)


# ---------------------------------------------------------------------------------------------- encoder
def synthetic_engine(num_layers=12, seed=0, device=0, vocab_size=21128, max_tokens=4096 * 64, tokenizer=None,
                     vocab_path=None):
    """Random-init encoder of the text2vec-base-chinese architecture (no checkpoint exists offline): HF-style
    N(0, 0.02) init from a numpy generator, LayerNorm gains near 1."""
    import numpy as np
    N = importlib.import_module(PKG + "._native")
    E = importlib.import_module(PKG + ".engine.encoder")
    cfg = N.BertCfg(vocab_size=vocab_size, hidden=768, layers=num_layers, heads=12, intermediate=3072,
                    max_position=512, type_vocab=2, ln_eps=1e-12)
    n = int(N.lib().icd_encoder_weight_count(cfg))
    rng = np.random.default_rng(seed)
    blob = (rng.standard_normal(n, dtype=np.float32) * 0.02)
    H, I = 768, 3072
    off = vocab_size * H + 512 * H + 2 * H
    blob[off:off + H] = 1.0 + 0.1 * rng.standard_normal(H, dtype=np.float32); off += 2 * H
    for _ in range(num_layers):
        off += 3 * H * H + 3 * H + H * H + H
        blob[off:off + H] = 1.0 + 0.1 * rng.standard_normal(H, dtype=np.float32); off += 2 * H
        off += I * H + I + H * I + H
        blob[off:off + H] = 1.0 + 0.1 * rng.standard_normal(H, dtype=np.float32); off += 2 * H
    assert off == n

    class _NoTok:
        def __call__(self, *a, **k):
            raise RuntimeError("synthetic engine has no tokenizer; use forward_ids")
    return E.EncoderEngine(cfg=cfg, blob=blob, tokenizer=tokenizer or _NoTok(), device=device, max_tokens=max_tokens,
                           vocab_path=vocab_path)


def icd_texts():
    """The 40 474 real texts of the reference's build: "query: " + semantic_text of every CSV record
    (tools/build_database.py:221 through encode_query, embedding_service.py:117-120)."""
    B = importlib.import_module(PKG + ".tools.build_database")
    recs = B.DatabaseBuilder.load_csv_data(B.DatabaseBuilder.__new__(B.DatabaseBuilder),
                                           os.path.join(ROOT, "data", "ICD_10v601.csv"))
    return [r["semantic_text"] for r in recs]


def write_synthetic_vocab(texts, path, size=21128):
    """vocab.txt in the bert-base-chinese layout (specials at 0 / 100-103) holding every character of `texts`,
    printable ASCII, a few word pieces, padded with [unusedN] -- there is no real vocab.txt offline."""
    vocab = ["[unused%d]" % i for i in range(size)]
    for tok, idx in {"[PAD]": 0, "[UNK]": 100, "[CLS]": 101, "[SEP]": 102, "[MASK]": 103}.items():
        vocab[idx] = tok
    chars = set()
    for t in texts:
        chars.update(t.lower())
    chars.update(chr(c) for c in range(33, 127))
    pieces = sorted(c for c in chars if not c.isspace())
    pieces += ["##" + c for c in "abcdefghijklmnopqrstuvwxyz0123456789"] + ["icd", "query", "passage", "##cd"]
    seen, slot = set(vocab), 104
    for p in pieces:
        if p in seen:
            continue
        vocab[slot] = p
        seen.add(p)
        slot += 1
    with open(path, "w", encoding="utf-8") as fh:
        fh.write("\n".join(vocab) + "\n")
    return path


def bench_encoder(dev, peaks, batch=4096, seq=64, warmup=3, min_window_s=2.0, barrier=None, sampler_gpu=None):
    """BASELINE configs[2]: encoder throughput at S=64, B=4096 on synthetic ids, random-init weights of the
    text2vec-base-chinese architecture.  `value` with ids and outputs resident in HBM over >= 50 steps / >= 2 s with
    its own clock sample; `e2e` through icd_encoder_forward with pinned HOST ids / lens / output (copies inside the
    timed region)."""
    import torch
    N = importlib.import_module(PKG + "._native")
    eng = synthetic_engine(device=dev.index or 0, max_tokens=batch * seq)
    g = torch.Generator(device=dev).manual_seed(7)
    ids = torch.randint(1000, 21128, (batch, seq), generator=g, device=dev, dtype=torch.int32)
    ids[:, 0] = 101
    ids[:, -1] = 102
    lens = torch.full((batch,), seq, dtype=torch.int32, device=dev)
    out = torch.empty((batch, 768), dtype=torch.float32, device=dev)
    stream = torch.cuda.current_stream(dev)
    launches0 = N.lib().icd_launch_count()
    eng.forward_ids(ids, lens, out=out, stream=stream.cuda_stream, sync=False)
    launches = int(N.lib().icd_launch_count() - launches0)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record(stream)
    for _ in range(warmup):
        eng.forward_ids(ids, lens, out=out, stream=stream.cuda_stream, sync=False)
    e1.record(stream)
    torch.cuda.synchronize(dev)
    est_ms = max(e0.elapsed_time(e1) / warmup, 1e-3)
    steps = max(50, int(math.ceil(min_window_s * 1e3 / est_ms)))
    sampler = ClockSampler(sampler_gpu) if sampler_gpu is not None else None
    if sampler:
        sampler.start()
        time.sleep(0.25)
    if barrier is not None:
        barrier()
    if sampler:
        sampler.begin()
    e0.record(stream)
    for _ in range(steps):
        eng.forward_ids(ids, lens, out=out, stream=stream.cuda_stream, sync=False)
    e1.record(stream)
    torch.cuda.synchronize(dev)
    if sampler:
        sampler.end()
    if barrier is not None:
        barrier()
    clocks = sampler.stop() if sampler else None
    ms = e0.elapsed_time(e1) / steps
    # end to end: host token ids in, host embeddings out, every step
    h_ids, h_lens = ids.cpu().pin_memory(), lens.cpu().pin_memory()
    h_out = torch.empty((batch, 768), dtype=torch.float32).pin_memory()
    eng.forward_ids(h_ids, h_lens, out=h_out, stream=stream.cuda_stream, sync=True)
    e2e_steps = 10
    e0.record(stream)
    for _ in range(e2e_steps):
        eng.forward_ids(h_ids, h_lens, out=h_out, stream=stream.cuda_stream, sync=True)
    e1.record(stream)
    torch.cuda.synchronize(dev)
    ms_e2e = e0.elapsed_time(e1) / e2e_steps
    same = bool(torch.allclose(h_out, out.cpu(), atol=1e-6))
    flops = batch * seq * 12 * (2 * (4 * 768 * 768 + 2 * 768 * 3072) + 4 * seq * 768)
    tf = flops / (ms * 1e-3) / 1e12
    norm = float(out.norm(dim=1).mean())
    eng.close()
    traffic, traffic_src = _ncu_traffic(f"encoder:{batch}:{seq}")
    return {"metric": "text2vec sentences/sec", "value": batch / (ms * 1e-3), "unit": "sentences/s",
            "ms_per_batch": ms, "steps": steps, "warmup": warmup, "flops_per_batch": flops, "batch": batch,
            "seq_len": seq, "layers": 12, "dtype": "bf16",
            "tflops": tf, "frac_of_bf16_sustained": tf / peaks["bf16_tflops_sustained"], "mean_norm": norm,
            "roofline": {"bound": "tensor", "achieved": tf, "peak": peaks["bf16_tflops_sustained"], "unit": "TFLOP/s",
                         "frac": tf / peaks["bf16_tflops_sustained"], "traffic": traffic, "traffic_source": traffic_src,
                         "traffic_is": "sum over the launches of one batch",
                         "kernel": "gemm_tc_kernel (4 of the 5 launches per layer)", "peak_source": peaks["source"] + " (sustained)"},
            "clocks": clocks,
            "e2e": {"value": batch / (ms_e2e * 1e-3), "unit": "sentences/s", "h2d_bytes_per_step": batch * seq * 4 + batch * 4,
                    "d2h_bytes_per_step": batch * 768 * 4, "host_equals_device": same, "input": "token ids"},
            "gpu_launches_per_batch": launches,
            "data": "synthetic ids, random-init weights"}


def bench_encoder_text(dev, rank, world, min_texts=200_000):
    """Text in -> embeddings out through the public service API (EmbeddingService.encode_queries, the call
    tools/build_database.py makes; and encode_batch, whose .tolist() return the reference's signature imposes) over
    >= 200 k real ICD strings: host tokenisation + staging + H2D + encoder + D2H, all inside the timed region.
    At N > 1 every rank encodes its 1/N share (data-parallel replicas); rank 0 reports total / max time."""
    import tempfile
    import numpy as np
    N = importlib.import_module(PKG + "._native")
    E = importlib.import_module(PKG + ".engine.encoder")
    S = importlib.import_module(PKG + ".services.embedding_service")
    base = icd_texts()
    reps = (min_texts + len(base) - 1) // len(base)
    texts = base * reps
    mine = texts[rank::world]
    tmp = tempfile.mkdtemp(prefix="icd_bench_vocab_")
    vocab_path = write_synthetic_vocab(["query: " + t for t in base], os.path.join(tmp, "vocab.txt"))
    tok = E.bert_tokenizer_from_vocab(vocab_path)
    eng = synthetic_engine(device=dev.index or 0, tokenizer=tok, vocab_path=vocab_path)
    prev = S.EmbeddingService.engine_factory
    S.EmbeddingService.engine_factory = staticmethod(lambda name, device=None: eng)
    try:
        os.environ.setdefault("EMBEDDING_MODEL_NAME", "synthetic-text2vec-base-chinese")
        svc = S.EmbeddingService()
        svc.encode_queries(mine[:20000])                     # warm-up: allocations, thread pools
        runs = []
        for _ in range(3):                                   # three full passes; the median one is reported
            launches0 = N.lib().icd_launch_count()
            t0 = time.perf_counter()
            vecs = svc.encode_queries(mine)
            dt = time.perf_counter() - t0
            runs.append((dt, int(N.lib().icd_launch_count() - launches0), dict(getattr(eng, "last_stats", {}) or {})))
        dt, launches, stats = sorted(runs, key=lambda r: r[0])[1]
        ok = bool(vecs.shape == (len(mine), 768) and np.all(np.abs(np.linalg.norm(vecs, axis=1) - 1.0) < 1e-3))
        # the reference-typed call: encode_batch returns vectors.tolist() (embedding_service.py:104)
        n_b = min(len(mine), 40_000)
        t0 = time.perf_counter()
        lst = svc.encode_batch(mine[:n_b], show_progress=False)
        dt_b = time.perf_counter() - t0
        ok = ok and isinstance(lst, list) and len(lst) == n_b and isinstance(lst[0], list)
        tokens = int(stats.get("tokens", 0))
        return {"value": len(mine) / dt, "unit": "sentences/s", "seconds": dt, "sentences": len(mine),
                "api": "EmbeddingService.encode_queries(list[str]) -> ndarray [n, 768] float32",
                "texts": f"{len(base)} real 'query: ' + semantic_text strings of data/ICD_10v601.csv x {reps}",
                "mean_tokens": tokens / max(1, len(mine)), "host_threads": os.cpu_count(), "gpu_launches": launches,
                "h2d_bytes": int(stats.get("h2d_bytes", 0)), "d2h_bytes": len(mine) * 768 * 4,
                "stages_s": {k: v for k, v in stats.items() if k.endswith("_s")},
                "all_runs_s": [r[0] for r in runs],
                "tokenizer": stats.get("tokenizer"),
                "encode_batch_tolist": {"value": n_b / dt_b, "unit": "sentences/s", "sentences": n_b,
                                        "note": "returns list[list[float]] like the reference; .tolist() of n x 768 "
                                                "Python floats is host-bound"},
                "ok": ok}
    finally:
        S.EmbeddingService.engine_factory = prev
        eng.close()


# ---------------------------------------------------------------------------------------------- scan
def bench_config1(torch, dev, native, VectorIndex, peaks, k=10, rows=40474, nq=10_000, steps=20):
    """BASELINE configs[1]: exact top-10 of 10 000 queries against a table of the reference's own size (40 474 rows,
    62 MB of bf16: L2-sized) with the level re-rank, one GPU.  `value` = queries/s with queries and results resident
    (CUDA events over `steps` calls), `e2e` = the same call with numpy fp32 queries and numpy results (pageable host
    memory, what MilvusService.search_batch hands over).  256 of the result rows are compared with an exact fp32
    torch search."""
    table, levels = make_corpus(torch, rows, dev, 4242)
    q = make_queries(torch, nq, dev, seed=4243).float()   # fp32 in, as the service hands them over
    idx = VectorIndex(DIM, device=dev.index)
    idx.adopt(table, levels)
    stream = torch.cuda.current_stream(dev)
    o = (torch.empty((nq, k), dtype=torch.float32, device=dev), torch.empty((nq, k), dtype=torch.float32, device=dev),
         torch.empty((nq, k), dtype=torch.int64, device=dev))
    run = lambda: idx.search(q, k, weight_mode=native.WEIGHT_RERANK, out=o, stream=stream.cuda_stream, sync=False)  # noqa: E731
    for _ in range(3):
        run()
    torch.cuda.synchronize(dev)
    l0 = native.lib().icd_launch_count()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record(stream)
    for _ in range(steps):
        run()
    e1.record(stream)
    torch.cuda.synchronize(dev)
    ms = e0.elapsed_time(e1) / steps
    launches = (native.lib().icd_launch_count() - l0) // steps
    q_np = q.float().cpu().numpy()
    for _ in range(2):
        idx.search(q_np, k, weight_mode=native.WEIGHT_RERANK)
    t0 = time.perf_counter()
    for _ in range(steps):
        hs, hr, hi = idx.search(q_np, k, weight_mode=native.WEIGHT_RERANK)
    ms_e2e = (time.perf_counter() - t0) / steps * 1e3
    # exact fp32 check of a sample (raw top-k as sets up to ties within 1e-6, re-rank order by weighted score)
    sample = torch.arange(0, nq, nq // 256, device=dev)[:256]
    exact = q[sample].float() @ table.float().T
    ref_s, ref_i = exact.topk(k, dim=1)
    got_i, got_r, got_s = o[2][sample], o[1][sample], o[0][sample]
    kth = ref_s[:, -1:]
    ok = bool(((got_r >= kth - 1e-6).all()) and (got_s[:, 1:] <= got_s[:, :-1]).all() and
              torch.allclose(got_r, exact.gather(1, got_i), atol=2e-6) and
              torch.equal(torch.from_numpy(hi).to(dev)[sample], got_i))
    same = float((got_i.sort(dim=1).values == ref_i.sort(dim=1).values).all(dim=1).float().mean())
    idx.close()
    flops = 2.0 * nq * rows * DIM
    return {"workload": f"exact top-{k} + level re-rank, {nq} queries x {rows} rows x {DIM} bf16 (BASELINE configs[1]), one call",
            "value": nq / (ms * 1e-3), "unit": "queries/s", "ms_per_call": ms, "steps": steps, "gpu_launches_per_call": int(launches),
            "tflops": flops / (ms * 1e-3) / 1e12, "frac_of_bf16_sustained": flops / (ms * 1e-3) / 1e12 / peaks["bf16_tflops_sustained"],
            "e2e": {"value": nq / (ms_e2e * 1e-3), "unit": "queries/s", "ms_per_call": ms_e2e, "h2d_bytes_per_step": nq * DIM * 4,
                    "d2h_bytes_per_step": nq * k * 16, "buffers": "numpy fp32 queries, numpy results (pageable)"},
            "checks": {"sample_matches_exact_fp32": ok, "sample_rows_with_identical_id_sets": same, "sample": 256}}


def scan_roofline(peaks, rows_local, B, k, scan_us, calls, kernel):
    flops = 2.0 * B * rows_local * DIM                     # per scan launch (per GPU)
    bytes_alg = rows_local * DIM * 2 + B * DIM * 2 + B * k * 16
    tensor_bound = flops / (peaks["bf16_tflops_sustained"] * 1e12) > bytes_alg / (peaks["hbm_gbs"] * 1e9)
    scan_s = scan_us * 1e-6
    if tensor_bound:
        roof = {"bound": "tensor", "achieved": flops / scan_s / 1e12, "peak": peaks["bf16_tflops_sustained"],
                "unit": "TFLOP/s"}
    else:
        roof = {"bound": "hbm", "achieved": bytes_alg / scan_s / 1e9, "peak": peaks["hbm_gbs"], "unit": "GB/s"}
    roof["frac"] = roof["achieved"] / roof["peak"]
    roof["kernel"] = kernel
    roof["traffic"], roof["traffic_source"] = _ncu_traffic(f"{kernel}:{rows_local}:{B}")
    roof["algorithmic_bytes"] = bytes_alg
    roof["algorithmic_flops"] = flops
    roof["kernel_us"] = scan_us
    roof["kernel_us_over"] = "mean of %d timed launches (max over ranks)" % calls
    roof["peak_source"] = peaks["source"] + (" (sustained)" if tensor_bound else "")
    roof["hbm_gbs_of_scan"] = bytes_alg / scan_s / 1e9
    roof["tflops_of_scan"] = flops / scan_s / 1e12
    return roof


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--rows", type=int, default=100_000_000, help="total corpus rows over all GPUs")
    ap.add_argument("--batch", type=int, default=1024)
    ap.add_argument("--path", type=int, default=0, help="0 auto, 1 stream, 2 tensor")
    ap.add_argument("--exchange", type=int, default=1, help="multi-GPU candidate exchange: 0 NCCL all-gather, 1 peer stores")
    ap.add_argument("--cpu-rows", type=int, default=500_000, help="rows of the CPU arm's corpus slice")
    ap.add_argument("--cpu-batch", type=int, default=0, help="CPU arm batch (0 = --batch, the real one)")
    ap.add_argument("--cpu-budget-s", type=float, default=60.0, help="wall budget of the CPU arm's warmup + steps")
    ap.add_argument("--tune", default="", help="comma list of icd_tune knobs, e.g. scan_sample=0,scan_drift=0")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-encoder", action="store_true")
    ap.add_argument("--no-points", action="store_true", help="skip the hbm_point / ridge_point measurements")
    ap.add_argument("--no-text", action="store_true", help="skip the encoder's text-in e2e")
    ap.add_argument("--dump-outputs", metavar="DIR", default="",
                    help="write the headline search results of the last timed step as DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be >= 1")
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs writes the GPU arm's results (--impl ours)")

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    quiet_stdout()
    if args.impl == "reference":
        run_reference(args, rank, world)
        return

    import torch
    import torch.distributed as dist
    native = importlib.import_module(PKG + "._native")
    VectorIndex = importlib.import_module(PKG + ".engine.index").VectorIndex
    native.require_gpu()
    for kv in filter(None, args.tune.split(",")):
        key, _, val = kv.partition("=")
        native.tune(**{key.strip(): int(val)})
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    assert world == args.gpus, f"--gpus {args.gpus} but WORLD_SIZE={world}: launch with torch.distributed.run"

    peaks = _peaks()
    rows_total = args.rows
    lo = rows_total * rank // world
    hi = rows_total * (rank + 1) // world
    rows_local = hi - lo
    note = None
    try:
        table, levels = make_corpus(torch, rows_local, dev, 1234 + rank)
    except torch.OutOfMemoryError:
        if world > 1:
            raise
        rows_total = rows_local = 10_000_000
        lo, hi = 0, rows_total
        note = "configs[3]: 100 M rows did not fit this GPU"
        torch.cuda.empty_cache()
        table, levels = make_corpus(torch, rows_local, dev, 1234)
    config = workload_config(args, world, rows_total, note)
    config["rows_per_gpu"] = rows_local
    q_all, p_pos, p_gid = make_planted_queries(torch, dist, table, lo, hi, rows_total, args.batch, dev, rank, world)
    stream = torch.cuda.current_stream(dev)
    k = K_TOP
    checks = {}

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize(dev)

    def all_true(flag):
        t = torch.tensor([1 if flag else 0], device=dev)
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MIN)
        return bool(int(t) == 1)

    ShardGroup = importlib.import_module(PKG + ".engine.shard").ShardGroup if world > 1 else None

    # ------------------------------------------------ start-up check (N > 1): sharded search == single table
    if world > 1:
        # check corpus: the first 1 M / N rows of every shard; gathered onto every rank as one table
        m_r = min(rows_local, 1_000_000 // world)
        piece_t, piece_l = table[:m_r].contiguous(), levels[:m_r].contiguous()
        whole_t = torch.empty((m_r * world, DIM), dtype=torch.bfloat16, device=dev)
        whole_l = torch.empty((m_r * world,), dtype=torch.uint8, device=dev)
        dist.all_gather_into_tensor(whole_t, piece_t)
        dist.all_gather_into_tensor(whole_l, piece_l)
        small = VectorIndex(DIM, device=local_rank)
        small.adopt(piece_t, piece_l)
        whole = VectorIndex(DIM, device=local_rank)
        whole.adopt(whole_t, whole_l)
        grp = ShardGroup(small, row_offset=m_r * rank, rank=rank, world=world)
        ws, wr, wi = whole.search(q_all, k, weight_mode=native.WEIGHT_RERANK)
        same = True
        for exchange in (0, 1):
            s, r, i = grp.search(q_all, k, weight_mode=native.WEIGHT_RERANK, exchange=exchange)
            same = same and bool(torch.equal(i, wi) and torch.equal(r, wr) and torch.equal(s, ws))
        checks["shard_equals_single"] = all_true(same)
        checks["shard_check"] = f"{m_r * world}-row check corpus ({m_r} rows of every shard), both exchanges, ids + scores bit-equal on every rank"
        grp.close(); small.close(); whole.close()
        del whole_t, whole_l, piece_t, piece_l
        torch.cuda.empty_cache()

    idx = VectorIndex(DIM, device=local_rank)
    idx.adopt(table, levels)
    idx.set_timing(True)
    group = ShardGroup(idx, row_offset=lo, rank=rank, world=world) if world > 1 else None

    def measure(B, steps, warmup, min_window_s, with_e2e, sample_clocks=True):
        """One operating point on the resident table: `steps` timed searches of the first B queries (CUDA events on
        the launch stream, max over ranks), continued untimed until min_window_s of identical load for the clocks."""
        q_dev = q_all[:B].contiguous()
        o = (torch.empty((B, k), dtype=torch.float32, device=dev), torch.empty((B, k), dtype=torch.float32, device=dev),
             torch.empty((B, k), dtype=torch.int64, device=dev))

        def step_device():
            if group is not None:
                group.search(q_dev, k, out=o, path=args.path, exchange=args.exchange, stream=stream.cuda_stream, sync=False)
            else:
                idx.search(q_dev, k, weight_mode=native.WEIGHT_RERANK, path=args.path, out=o,
                           stream=stream.cuda_stream, sync=False)

        sampler = ClockSampler(local_rank)
        if rank == 0 and sample_clocks:
            sampler.start()
        for _ in range(warmup):
            step_device()
        barrier()
        launches0 = native.lib().icd_launch_count()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        barrier()
        idx.set_timing(True)   # restart the library's per-search event ring: the timed steps are what gets averaged
        sampler.begin()
        e0.record(stream)
        for _ in range(steps):
            step_device()
        e1.record(stream)
        barrier()
        last = tuple(t.clone() for t in o)     # results of the last timed step (the untimed steps below rewrite o)
        ms_total = e0.elapsed_time(e1)
        launches = native.lib().icd_launch_count() - launches0
        tm = idx.mean_timing()
        tm["launches"] = idx.last_timing()["launches"]
        t = torch.tensor([ms_total, tm["scan_us"]], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms_total, scan_us_max = float(t[0]), float(t[1])
        # nvidia-smi samples every 100 ms: a timed region shorter than the window is followed by the SAME steps,
        # untimed, until the window is full, so the clocks line always describes this workload under load (every
        # rank runs the same number of extra steps: the count comes from the max-over-ranks time)
        extra = 0
        if ms_total < min_window_s * 1e3:
            extra = min(int((min_window_s * 1e3 - ms_total) / max(ms_total / steps, 1e-3)) + 1, 100000)
            for _ in range(extra):
                step_device()
            barrier()
        sampler.end()
        clocks = sampler.stop() if (rank == 0 and sample_clocks) else None
        if clocks is not None:
            clocks["window"] = ("timed region" if extra == 0 else
                                "timed region + %d identical untimed steps (%.0f s of load)" % (extra, min_window_s))
        ms_step = ms_total / steps
        res = {"B": B, "ms_per_step": ms_step, "qps": B / (ms_step * 1e-3), "scan_us": scan_us_max, "calls": tm["calls"],
               "launches": int(launches), "launches_per_step": tm["launches"], "clocks": clocks, "steps": steps, "out": o,
               "last": last,
               "kernel": "scan_tc_kernel" if B > 4 else "scan_stream_kernel"}
        if with_e2e:
            q_host = q_dev.cpu().pin_memory()
            h = (torch.empty((B, k), dtype=torch.float32).pin_memory(), torch.empty((B, k), dtype=torch.float32).pin_memory(),
                 torch.empty((B, k), dtype=torch.int64).pin_memory())

            def step_host():
                if group is not None:
                    group.search(q_host, k, out=h, path=args.path, exchange=args.exchange, stream=stream.cuda_stream, sync=True)
                else:
                    idx.search(q_host, k, weight_mode=native.WEIGHT_RERANK, path=args.path, out=h,
                               stream=stream.cuda_stream, sync=True)
            for _ in range(2):
                step_host()
            barrier()
            t0 = time.perf_counter()
            for _ in range(steps):
                step_host()
            barrier()
            t = torch.tensor([time.perf_counter() - t0], dtype=torch.float64, device=dev)
            if world > 1:
                dist.all_reduce(t, op=dist.ReduceOp.MAX)
            res["e2e_qps"] = B / (float(t[0]) / steps)
            step_device()
            torch.cuda.synchronize(dev)
            res["host_equals_device"] = bool(torch.equal(o[2].cpu(), h[2]) and torch.equal(o[0].cpu(), h[0]))
        return res

    # ------------------------------------------------ headline: device-resident timing (value) + e2e
    B = args.batch
    head = measure(B, args.steps, args.warmup, 1.0, with_e2e=True)
    o_score, o_raw, o_id = head["out"]

    # ------------------------------------------------ correctness of the timed configuration
    gid = torch.tensor(p_gid, dtype=torch.int64, device=dev)
    checks["planted_top1_ok"] = all_true(bool(torch.equal(o_id[p_pos, 0], gid)))
    checks["planted"] = f"{len(p_pos)} of {B} queries are corpus rows + noise, spread over all shards"
    checks["scores_sorted"] = all_true(bool((o_score[:, 1:] <= o_score[:, :-1]).all()))
    checks["ids_unique"] = all_true(bool((o_id.sort(dim=1).values.diff(dim=1) != 0).all()))
    if world > 1:
        # independent merge: every rank's local top-k (raw scores, global ids) gathered and merged by torch sorts
        gs, gr, gi = group.search(q_all, k, weight_mode=native.WEIGHT_NONE, path=args.path, exchange=args.exchange)
        ls, lr, li = idx.search(q_all, k, weight_mode=native.WEIGHT_NONE, path=args.path)
        li = li + lo
        all_r = torch.empty((world, B, k), dtype=torch.float32, device=dev)
        all_i = torch.empty((world, B, k), dtype=torch.int64, device=dev)
        dist.all_gather_into_tensor(all_r, lr.contiguous())
        dist.all_gather_into_tensor(all_i, li.contiguous())
        cat_r = all_r.permute(1, 0, 2).reshape(B, world * k)
        cat_i = all_i.permute(1, 0, 2).reshape(B, world * k)
        by_id = cat_i.argsort(dim=1, stable=True)
        cat_r, cat_i = cat_r.gather(1, by_id), cat_i.gather(1, by_id)
        by_score = (-cat_r).argsort(dim=1, stable=True)[:, :k]
        checks["merge_equals_torch"] = all_true(bool(torch.equal(cat_i.gather(1, by_score), gi) and
                                                     torch.equal(cat_r.gather(1, by_score), gr)))

    # ------------------------------------------------ HBM-bound and ridge operating points (same resident table)
    points = {}
    if not args.no_points:
        for name, pb in (("hbm_point", 128), ("ridge_point", 256)):
            if pb > B:
                continue
            probe = measure(pb, 3, 2, 0.0, with_e2e=False, sample_clocks=False)      # sizes the step count
            n_steps = max(5, int(math.ceil(1000.0 / max(probe["ms_per_step"], 1e-3))))
            points[name] = measure(pb, n_steps, 2, 1.0, with_e2e=False)

    # ------------------------------------------------ BASELINE configs[1]: the reference's own table size (rank 0, N = 1)
    config1 = None
    if not args.no_points and world == 1:
        try:
            config1 = bench_config1(torch, dev, native, VectorIndex, peaks)
        except Exception as e:  # auxiliary: the headline must still print
            config1 = {"error": repr(e)[:300]}

    # ------------------------------------------------ encoder (BASELINE configs[2]), data-parallel replicas
    enc = None
    if not args.no_encoder:
        torch.cuda.empty_cache()
        try:
            enc = bench_encoder(dev, peaks, barrier=barrier, sampler_gpu=local_rank if rank == 0 else None)
            ok = 1.0
        except Exception as e:  # encoder line is auxiliary; the headline must still print
            enc = {"error": repr(e)[:200]}
            ok = 0.0
        t = torch.tensor([enc.get("ms_per_batch", 0.0), -ok], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        if float(t[1]) == -1.0 and "error" not in enc:
            ms = float(t[0])  # max over ranks; every rank encodes its own batch (weak scaling, no exchange)
            enc.update({"ms_per_batch": ms, "value": world * enc["batch"] / (ms * 1e-3), "n_gpus": world,
                        "tflops": world * enc["flops_per_batch"] / (ms * 1e-3) / 1e12,
                        "frac_of_bf16_sustained": enc["flops_per_batch"] / (ms * 1e-3) / 1e12 / peaks["bf16_tflops_sustained"],
                        "scaling": "weak (one batch per GPU, replicas, no collective)"})
            if "roofline" in enc:   # per-GPU figure from the max-over-ranks time, like frac_of_bf16_sustained
                enc["roofline"]["achieved"] = enc["flops_per_batch"] / (ms * 1e-3) / 1e12
                enc["roofline"]["frac"] = enc["roofline"]["achieved"] / enc["roofline"]["peak"]
        if not args.no_text and "error" not in enc:
            try:
                txt = bench_encoder_text(dev, rank, world)
                t = torch.tensor([txt["seconds"], float(txt["sentences"])], dtype=torch.float64, device=dev)
                tmax = t.clone()
                if world > 1:
                    dist.all_reduce(tmax, op=dist.ReduceOp.MAX)
                    dist.all_reduce(t, op=dist.ReduceOp.SUM)
                    txt["value"] = float(t[1]) / float(tmax[0])
                    txt["seconds"], txt["sentences"] = float(tmax[0]), int(t[1])
                    txt["scaling"] = "strong (the texts are split over the ranks; host threads are shared)"
                enc["e2e_text"] = txt
            except Exception as e:
                enc["e2e_text"] = {"error": repr(e)[:300]}
                if world > 1:   # keep the collectives matched
                    z = torch.zeros(2, dtype=torch.float64, device=dev)
                    dist.all_reduce(z, op=dist.ReduceOp.MAX)
                    dist.all_reduce(z, op=dist.ReduceOp.SUM)

    if rank == 0:
        roof = scan_roofline(peaks, rows_local, B, k, head["scan_us"], head["calls"], head["kernel"])
        checks["ids_match_host_device"] = head["host_equals_device"]
        line = {
            "metric": "top-10 cosine QPS (100M x 768)", "value": head["qps"], "unit": "queries/s", "n_gpus": world,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": head["ms_per_step"], "higher_is_better": True,
            "scaling": "strong", "vs_baseline": None, "dtype": "bf16", "data": "synthetic",
            "config": config,
            "e2e": {"value": head["e2e_qps"], "unit": "queries/s", "h2d_bytes_per_step": B * DIM * 2,
                    "d2h_bytes_per_step": B * k * 16},
            "gpu_launches": head["launches"], "launches_per_step": head["launches_per_step"],
            "roofline": roof, "clocks": head["clocks"], "ids_match_host_device": head["host_equals_device"],
            "checks": checks, "planted_top1_ok": checks["planted_top1_ok"],
            "shard_equals_single": checks.get("shard_equals_single"), "env": _icd_env(),
        }
        for name, pt in points.items():
            line[name] = {"batch": pt["B"], "value": pt["qps"], "unit": "queries/s", "ms_per_step": pt["ms_per_step"],
                          "steps": pt["steps"], "n_gpus": world,
                          "roofline": scan_roofline(peaks, rows_local, pt["B"], k, pt["scan_us"], pt["calls"], pt["kernel"]),
                          "clocks": pt["clocks"], "gpu_launches": pt["launches"]}
        if config1 is not None:
            line["config1_point"] = config1
        if not args.no_cpu_baseline and world == 1:
            sample = CpuScanSample(args.cpu_rows, args.cpu_batch or B)
            sample.calibrate(5, 25.0)
            sample.step()
            dts = [sample.step() for _ in range(4)]
            dt = sum(dts) / len(dts)
            qps_cpu = B / (dt * (rows_total / sample.rows) * (B / sample.batch))
            line["cpu_baseline"] = {"value": qps_cpu, "unit": "queries/s", "cores": os.cpu_count(), "kind": "port",
                                    "sample": sample.describe(rows_total, B), "measured_ms_per_sample_step": dt * 1e3}
        if enc is not None:
            if not args.no_cpu_baseline and world == 1 and "error" not in enc:
                try:
                    enc["cpu_baseline"] = cpu_encoder_sample()
                except Exception as e:
                    enc["cpu_baseline"] = {"error": repr(e)[:200]}
            line["encoder"] = enc
        if args.dump_outputs:
            dump_outputs(args.dump_outputs, *head["last"])
        emit(line)
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


if __name__ == "__main__":
    sys.dont_write_bytecode = True     # the checkout may be read-only: the bench writes nothing into it
    try:
        main()
    except BaseException as exc:      # a rank that dies must take the job down (torchrun then stops the others): never hang
        if isinstance(exc, SystemExit) and not exc.code:
            raise
        import traceback
        traceback.print_exc()
        sys.stderr.flush()
        os._exit(1)
