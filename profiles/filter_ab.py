#!/usr/bin/env python3
"""A/B of the row mask of filtered search (DESIGN.md, "Filtered search"): scan time with and without a mask, and of the
unfiltered scan against another build of libicdrag.so (the parent commit's), alternating in one process on one GPU.

  python profiles/filter_ab.py --parent-lib PATH/libicdrag.so --out profiles/filter_ab.jsonl

Variants per point: `parent` (the other library, no mask; skipped without --parent-lib), `nomask`, `ones` (an
all-ones mask), `range1` (a contiguous 1 % of the rows), `rand1` (1 % of the rows at random).  Points: 10 M x 768 bf16
rows at B = 128 and B = 1024 (tensor path), the 40 474-row table at B = 1024, and 10 M rows at B = 1 on the stream
path.  Each measurement is a window of >= 1 s of back-to-back searches on device buffers; the figure is the library's
own CUDA-event stage time (icd_index_mean_timing: scan + merge + finalise, mean over the window's last 64 searches)
next to the wall time per search of the window.  Variants rotate inside every repetition; the median over the
repetitions is reported.  Each library is loaded with RTLD_DEEPBIND so that neither resolves the other's symbols.
"""
import argparse
import ctypes as C
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


class Lib:
    def __init__(self, path):
        self.L = C.CDLL(path, mode=os.RTLD_LOCAL | os.RTLD_DEEPBIND)
        vp, i32, i64, f32p = C.c_void_p, C.c_int, C.c_int64, C.POINTER(C.c_float)
        L = self.L
        L.icd_last_error.restype = C.c_char_p
        L.icd_index_create.argtypes = [i32, i32, i64, i32, C.POINTER(vp)]
        L.icd_index_destroy.argtypes = [vp]
        L.icd_index_adopt.argtypes = [vp, vp, vp, i64]
        L.icd_index_search.argtypes = [vp, vp, i32, i32, i32, i32, i32, vp, vp, vp, vp, i32]
        L.icd_index_set_timing.argtypes = [vp, i32]
        L.icd_index_mean_timing.argtypes = [vp, f32p, C.POINTER(i32)]
        self.filtered = hasattr(L, "icd_index_search_filtered")
        if self.filtered:
            L.icd_index_search_filtered.argtypes = [vp, vp, i32, i32, i32, i32, i32, vp, i64, vp, vp, vp, vp, i32]

    def check(self, st, what):
        if st != 0:
            raise RuntimeError(f"{what}: {st} {self.L.icd_last_error().decode()}")

    def index(self, table, levels):
        h = C.c_void_p()
        self.check(self.L.icd_index_create(table.shape[1], 0, 0, 0, C.byref(h)), "create")
        self.check(self.L.icd_index_adopt(h, table.data_ptr(), levels.data_ptr(), table.shape[0]), "adopt")
        return h


def window(lib, h, n, q, out, k, path, mask, min_s):
    """Back-to-back searches for >= min_s seconds; returns (library stage time us, wall us per search)."""
    import torch
    B = q.shape[0]
    args = (h, q.data_ptr(), 1, B, k, 2, path)
    outs = tuple(o.data_ptr() for o in out) + (None, 0)
    call = (lambda: lib.L.icd_index_search_filtered(*args, mask, n, *outs)) if mask is not None else \
        (lambda: lib.L.icd_index_search(*args, *outs))
    for _ in range(3):
        lib.check(call(), "search")
    torch.cuda.synchronize()
    lib.check(lib.L.icd_index_set_timing(h, 1), "timing")
    calls, t0 = 0, time.perf_counter()
    while True:
        for _ in range(16):
            lib.check(call(), "search")
        calls += 16
        torch.cuda.synchronize()
        dt = time.perf_counter() - t0
        if dt >= min_s:
            break
    us = (C.c_float * 3)()
    cnt = C.c_int()
    lib.check(lib.L.icd_index_mean_timing(h, us, C.byref(cnt)), "mean_timing")
    lib.check(lib.L.icd_index_set_timing(h, 0), "timing")
    return float(us[0] + us[1] + us[2]), dt / calls * 1e6, float(us[0])


def device_info():
    import torch
    info = {"device": torch.cuda.get_device_name(0)}
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                             capture_output=True, text=True, timeout=30).stdout.strip()
        info["power_limit"], info["max_sm_clock"] = [x.strip() for x in out.split(",")]
    except Exception as e:   # the figure is still labelled with the device name
        info["power_limit"] = f"unknown ({e})"
    return info


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--lib", default=os.path.join(ROOT, "rag-project-icd10_b200", "csrc", "libicdrag.so"))
    ap.add_argument("--parent-lib", default="")
    ap.add_argument("--rows", type=int, default=10_000_000)
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--min-s", type=float, default=1.0)
    ap.add_argument("--out", default="")
    a = ap.parse_args()
    import torch
    import bench
    from importlib import import_module
    F = import_module("rag-project-icd10_b200.engine.filter_expr")
    if not torch.cuda.is_available():
        raise SystemExit("filter_ab.py measures on the GPU: no CUDA device")
    dev = torch.device("cuda", 0)
    libs = {"new": Lib(a.lib)}
    if a.parent_lib:
        libs["parent"] = Lib(a.parent_lib)
    info = device_info()
    big_t, big_l = bench.make_corpus(torch, a.rows, dev, seed=4321)
    small_t, small_l = bench.make_corpus(torch, 40474, dev, seed=99)
    q_all, _, _ = bench.make_planted_queries(torch, None, big_t, 0, a.rows, a.rows, 1024, dev, 0, 1)
    tables = {"big": (big_t, big_l), "small": (small_t, small_l)}
    handles = {(ln, tn): lib.index(*tables[tn]) for ln, lib in libs.items() for tn in tables}

    def masks(n):
        rng = np.random.default_rng(n)
        rng1 = np.zeros(n, bool)
        rng1[n // 3:n // 3 + n // 100] = True
        out = {"ones": np.ones(n, bool), "range1": rng1, "rand1": rng.random(n) < 0.01}
        return {k: torch.from_numpy(F.pack_bits(v).view(np.int32)).to(dev) for k, v in out.items()}
    mask_of = {"big": masks(a.rows), "small": masks(40474)}
    points = [("big", 128, 2), ("big", 1024, 2), ("small", 1024, 2), ("big", 1, 1)]
    rows_out = []
    for tn, B, path in points:
        n = tables[tn][0].shape[0]
        q = q_all[:B].contiguous()
        k = 10
        out = (torch.empty((B, k), dtype=torch.float32, device=dev), torch.empty((B, k), dtype=torch.float32, device=dev),
               torch.empty((B, k), dtype=torch.int64, device=dev))
        variants = ([("parent", None)] if "parent" in libs else []) + [("nomask", None)] + \
            [(m, mask_of[tn][m]) for m in ("ones", "range1", "rand1")]
        res = {v: [] for v, _ in variants}
        for rep in range(a.reps):
            order = variants[rep % len(variants):] + variants[:rep % len(variants)]
            for v, m in order:
                ln = "parent" if v == "parent" else "new"
                res[v].append(window(libs[ln], handles[ln, tn], n, q, out, k, path, None if m is None else m.data_ptr(),
                                     a.min_s))
        for v, _ in variants:
            r = np.array(res[v])
            rec = dict(info, rows=n, B=B, path="tensor" if path == 2 else "stream", variant=v,
                       stage_us_median=float(np.median(r[:, 0])), scan_us_median=float(np.median(r[:, 2])),
                       wall_us_median=float(np.median(r[:, 1])), stage_us=r[:, 0].round(2).tolist(),
                       wall_us=r[:, 1].round(2).tolist())
            rows_out.append(rec)
            print(json.dumps(rec), flush=True)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as fh:
            for r in rows_out:
                fh.write(json.dumps(r) + "\n")


if __name__ == "__main__":
    main()
