"""bench.py's own arm on a small table: the JSON line the driver parses carries every contract key, the correctness flags
are true, the HBM / ridge points and the roofline objects are there; with >= 2 GPUs the same under torchrun (start-up
shard check, merged result against an independent torch merge)."""
import json
import os
import subprocess
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
pytestmark = pytest.mark.gpu


def _check_line(d, n_gpus):
    for key in ("metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling",
                "vs_baseline", "dtype", "data", "config", "e2e", "gpu_launches", "roofline", "clocks", "checks", "env"):
        assert key in d, key
    assert d["n_gpus"] == n_gpus and d["steps"] == 3 and d["warmup"] == 3 and d["higher_is_better"] is True
    assert d["unit"] == "queries/s" and d["value"] > 0 and d["vs_baseline"] is None and d["dtype"] == "bf16"
    assert "workload" in d["config"] and d["config"]["rows"] == 4_000_000 and d["config"]["batch"] == 1024
    e = d["e2e"]
    assert e["value"] > 0 and e["h2d_bytes_per_step"] == 1024 * 768 * 2 and e["d2h_bytes_per_step"] == 1024 * 10 * 16
    r = d["roofline"]
    assert r["bound"] in ("hbm", "tensor") and r["unit"] in ("GB/s", "TFLOP/s") and 0 < r["frac"] < 1.5
    assert abs(r["frac"] - r["achieved"] / r["peak"]) < 1e-9 and "traffic" in r and r["kernel_us"] > 0
    assert d["gpu_launches"] >= 3 * 3
    c = d["checks"]
    assert c["planted_top1_ok"] is True and c["scores_sorted"] is True and c["ids_unique"] is True
    assert c["ids_match_host_device"] is True and d["planted_top1_ok"] is True
    if n_gpus > 1:
        assert c["shard_equals_single"] is True and c["merge_equals_torch"] is True and d["shard_equals_single"] is True
    for name, batch, bound in (("hbm_point", 128, "hbm"), ("ridge_point", 256, "tensor")):
        p = d[name]
        assert p["batch"] == batch and p["value"] > 0 and p["roofline"]["bound"] == bound and p["steps"] >= 5
        assert p["clocks"] is None or "sm_mhz" in p["clocks"]
    assert isinstance(d["env"], dict)


def test_bench_line_contract_and_checks_one_gpu(tmp_path):
    import numpy as np
    sys.path.insert(0, ROOT)
    import bench
    cmd = [sys.executable, os.path.join(ROOT, "bench.py"), "--rows", "4000000", "--steps", "3", "--warmup", "3",
           "--no-encoder", "--no-cpu-baseline", "--dump-outputs", str(tmp_path)]
    out = subprocess.run(cmd, capture_output=True, text=True, timeout=900, cwd=ROOT)
    assert out.returncode == 0, out.stderr[-3000:]
    lines = [l for l in out.stdout.splitlines() if l.strip()]
    assert len(lines) == 1, out.stdout[-2000:]
    _check_line(json.loads(lines[0]), 1)
    # the dumped results are the checked ones: planted rows first, scores sorted
    d = {n: np.load(tmp_path / f"{n}.npy") for n in ("scores", "raw_scores", "ids")}
    assert all(a.shape == (1024, 10) for a in d.values()) and d["ids"].dtype == np.float64
    pos, gids = bench.planted_ids(1024, 4_000_000)
    assert np.array_equal(d["ids"][pos, 0], np.asarray(gids, np.float64))
    assert np.all(np.diff(d["scores"], axis=1) <= 0)


def test_bench_line_contract_and_checks_multi_gpu():
    import torch
    n = torch.cuda.device_count()
    if n < 2:
        pytest.skip("needs >= 2 GPUs (run with gpurun --gpus 2)")
    world = 8 if n >= 8 else (4 if n >= 4 else 2)
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", f"--nproc-per-node={world}", "--master-addr",
           "127.0.0.1", "--master-port", "29547", os.path.join(ROOT, "bench.py"), "--gpus", str(world), "--rows", "4000000",
           "--steps", "3", "--warmup", "3", "--no-encoder", "--no-cpu-baseline"]
    out = subprocess.run(cmd, capture_output=True, text=True, timeout=900, cwd=ROOT)
    assert out.returncode == 0, out.stderr[-3000:]
    lines = [l for l in out.stdout.splitlines() if l.strip().startswith("{")]
    assert len(lines) == 1, out.stdout[-2000:]
    _check_line(json.loads(lines[0]), world)
