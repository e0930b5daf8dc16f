"""bench.py's reference arm runs on the host cores only, so its output contract can be checked without a GPU:
one JSON line with the keys the driver reads, `impl: reference`, a cpu_baseline describing the run and an e2e
object that repeats the line's own value (tier rules, section 4)."""
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _run(*extra):
    cmd = [sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "1", "--warmup", "0",
           "--cpu-rows", "20000", "--cpu-batch", "8", *extra]
    out = subprocess.run(cmd, capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert out.returncode == 0, out.stderr[-2000:]
    lines = [l for l in out.stdout.splitlines() if l.strip()]
    assert len(lines) == 1, out.stdout
    return json.loads(lines[0])


def test_reference_arm_prints_one_contract_line():
    d = _run("--no-encoder")
    for key in ("metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling",
                "vs_baseline", "dtype", "data", "config", "cpu_baseline", "e2e", "impl"):
        assert key in d, key
    assert d["impl"] == "reference" and d["vs_baseline"] is None and d["higher_is_better"] is True
    assert d["unit"] == "queries/s" and d["value"] > 0
    assert d["cpu_baseline"]["kind"] == "port" and d["cpu_baseline"]["cores"] >= 1 and "sample" in d["cpu_baseline"]
    assert d["cpu_baseline"]["value"] == d["value"]
    assert d["e2e"] == {"value": d["value"], "unit": d["unit"], "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    assert d["config"]["rows"] == 100_000_000 and d["config"]["batch"] == 1024 and "workload" in d["config"]


def test_clock_sampler_parses_nvidia_smi_lines():
    sys.path.insert(0, ROOT)
    import bench
    s = bench.ClockSampler(0)
    s.proc = type("P", (), {"terminate": lambda self: None, "wait": lambda self, timeout=None: 0, "kill": lambda self: None})()
    s.t0, s.t1 = 100.0, 101.0
    s.lines = [(99.0, "0, 1965, 1965, 200.0, 0x0, Not Active, Not Active, Not Active, Not Active"),     # before the window
               (100.2, "0, 1500, 1965, 990.1, 0x4, Not Active, Not Active, Not Active, Active"),
               (100.5, "0, 1470, 1965, 995.0, 0x4, Not Active, Not Active, Not Active, Active"),
               (100.9, "0, 1440, 1965, 996.0, 0x4, Not Active, Not Active, Not Active, Active"),
               (102.0, "0, 1965, 1965, 150.0, 0x0, Not Active, Not Active, Not Active, Not Active")]    # after it
    c = s.stop()
    assert c["samples"] == 3 and c["sm_mhz"] == 1470.0 and c["sm_max_mhz"] == 1965.0 and c["reasons"] == ["sw_power_cap"]


def test_dump_outputs_writes_float_arrays_and_samples_large_outputs(tmp_path, monkeypatch):
    import numpy as np
    import torch
    sys.path.insert(0, ROOT)
    import bench
    g = torch.Generator().manual_seed(0)
    raw = torch.rand((1024, 10), generator=g).sort(dim=1, descending=True).values
    ids = torch.randint(0, 100_000_000, (1024, 10), generator=g)
    bench.dump_outputs(str(tmp_path / "all"), raw * 1.5, raw, ids)
    got = {f.stem: np.load(f) for f in (tmp_path / "all").iterdir()}
    assert sorted(got) == ["ids", "raw_scores", "scores"]
    assert got["ids"].dtype == np.float64 and np.array_equal(got["ids"], ids.numpy())
    assert got["scores"].dtype == got["raw_scores"].dtype == np.float32 and np.array_equal(got["raw_scores"], raw.numpy())
    monkeypatch.setattr(bench, "DUMP_MAX_BYTES", 16 << 10)
    for name in ("s1", "s2"):
        bench.dump_outputs(str(tmp_path / name), raw * 1.5, raw, ids)
    s1 = {f.stem: np.load(f) for f in (tmp_path / "s1").iterdir()}
    s2 = {f.stem: np.load(f) for f in (tmp_path / "s2").iterdir()}
    rows = s1["query_rows"].astype(np.int64)
    assert sum(a.nbytes for a in s1.values()) <= 16 << 10 and len(rows) > 0 and np.all(np.diff(rows) > 0)
    assert np.array_equal(s1["ids"], ids.numpy()[rows]) and np.array_equal(s1["scores"], (raw * 1.5).numpy()[rows])
    assert all(np.array_equal(s1[k], s2[k]) for k in s1)      # the sample is fixed
