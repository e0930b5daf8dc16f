"""VectorIndex -- Python handle over the icd_index_* C ABI (include/icdrag.h).

Stands where the Milvus FLAT/IP collection stands in the reference
(/root/reference/services/milvus_service.py:163-206 schema, :259 insert, :280-285 search).
All arithmetic happens in libicdrag.so on the GPU; this class only moves pointers.
"""
from __future__ import annotations

import ctypes as C
import threading
from typing import Optional, Tuple

import numpy as np

from .. import _native as N


class VectorIndex:
    def __init__(self, dim: int, device: int = 0, capacity: int = 0, keep_f32: bool = False):
        N.require_gpu()
        self._h = C.c_void_p()
        self.dim, self.device, self.keep_f32 = int(dim), int(device), bool(keep_f32)
        N.check(N.lib().icd_index_create(self.dim, self.device, int(capacity),
                                         N.INDEX_KEEP_F32 if keep_f32 else 0, C.byref(self._h)),
                "icd_index_create")
        self._adopted = None  # keeps adopted tensors alive
        self._lock = threading.RLock()   # one in-flight call per handle (the workspace is per handle); ctypes drops the GIL

    # ---------------------------------------------------------------- lifetime
    def close(self) -> None:
        if getattr(self, "_h", None) is not None and self._h.value:
            N.lib().icd_index_destroy(self._h)
            self._h = C.c_void_p()
            self._adopted = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def __len__(self) -> int:
        return int(N.lib().icd_index_size(self._h))

    # ---------------------------------------------------------------- writes
    def append(self, vecs, levels=None) -> None:
        """vecs: [n, dim] float32 / bfloat16 (numpy or torch, host or device); levels: [n] uint8."""
        n = int(vecs.shape[0])
        if n == 0:
            return
        if int(vecs.shape[1]) != self.dim:
            raise ValueError(f"expected dim {self.dim}, got {vecs.shape[1]}")
        if levels is not None:
            if int(levels.shape[0]) != n:
                raise ValueError("levels length mismatch")
            if N._is_torch(levels) != N._is_torch(vecs) or (N._is_torch(vecs) and levels.device != vecs.device):
                raise ValueError("vecs and levels must live in the same memory space")
        with self._lock:
            N.check(N.lib().icd_index_append(self._h, N.buf_ptr(vecs), N.vec_dtype(vecs), N.buf_ptr(levels), n),
                    "icd_index_append")

    def adopt(self, table_bf16, levels_u8) -> None:
        """Zero-copy: scan caller-owned device tensors ([n, dim] bfloat16, [n] uint8)."""
        n = int(table_bf16.shape[0])
        N.check(N.lib().icd_index_adopt(self._h, N.buf_ptr(table_bf16), N.buf_ptr(levels_u8), n),
                "icd_index_adopt")
        self._adopted = (table_bf16, levels_u8)

    def clear(self) -> None:
        N.check(N.lib().icd_index_clear(self._h), "icd_index_clear")

    def read(self, row0: int, n: int) -> np.ndarray:
        out = np.empty((n, self.dim), np.float32)
        with self._lock:
            N.check(N.lib().icd_index_read(self._h, int(row0), int(n), N.buf_ptr(out)), "icd_index_read")
        return out

    # ---------------------------------------------------------------- search
    def search(self, q, k: int, weight_mode: int = N.WEIGHT_RERANK, path: int = N.PATH_AUTO,
               out: Optional[Tuple] = None, stream: int = 0, sync: bool = True, mask=None, offset: int = 0,
               radius: Optional[float] = None, range_filter: Optional[float] = None):
        """q: [B, dim] float32/bfloat16, numpy (host) or torch (host/device).

        Returns (score [B,k] f32, raw [B,k] f32, ids [B,k] i64) in the memory space of q
        (numpy for numpy, torch tensors on q's device for torch), or fills `out`.
        mask: packed uint32 row bitmap (engine/filter_expr.py::pack_bits; numpy or a CUDA tensor): the exact top-k over
        the rows whose bit is set; fewer than k such rows leave a (-inf, -1) tail.  None = every row.
        offset / radius / range_filter (pymilvus's paging and FLAT/IP range search): the hits [offset, offset + k) of
        the exact list over the rows whose raw inner product lies in (radius, range_filter]; offset + k <= MAX_LIMIT.
        k <= MAX_K with no offset and no range is today's icd_index_search_filtered call; anything else is
        icd_index_search_page, which has one exact path (path must be PATH_AUTO)."""
        if q.ndim == 1:
            q = q[None, :]
        B = int(q.shape[0])
        if int(q.shape[1]) != self.dim:
            raise ValueError(f"expected dim {self.dim}, got {q.shape[1]}")
        if out is None:
            if N._is_torch(q):
                import torch
                score = torch.empty((B, k), dtype=torch.float32, device=q.device)
                raw = torch.empty((B, k), dtype=torch.float32, device=q.device)
                ids = torch.empty((B, k), dtype=torch.int64, device=q.device)
            else:
                score = np.empty((B, k), np.float32)
                raw = np.empty((B, k), np.float32)
                ids = np.empty((B, k), np.int64)
        else:
            score, raw, ids = out
        paged = k > N.MAX_K or offset != 0 or radius is not None or range_filter is not None
        if paged and path != N.PATH_AUTO:
            raise ValueError("searches beyond k = 128, with an offset or with a range have one exact path: "
                             "path must be PATH_AUTO")
        if paged:
            page = N.SearchPage(offset=int(offset), limit=int(k),
                                range_flags=(N.RANGE_RADIUS if radius is not None else 0)
                                | (N.RANGE_FILTER if range_filter is not None else 0),
                                radius=float(radius) if radius is not None else 0.0,
                                range_filter=float(range_filter) if range_filter is not None else 0.0)
            with self._lock:
                n = len(self)
                N.check(N.lib().icd_index_search_page(self._h, N.buf_ptr(q), N.vec_dtype(q), B, C.byref(page),
                                                      int(weight_mode), N.mask_ptr(mask, n), n, N.buf_ptr(score),
                                                      N.buf_ptr(raw), N.buf_ptr(ids), C.c_void_p(stream),
                                                      1 if sync else 0), "icd_index_search_page")
            return score, raw, ids
        with self._lock:
            n = len(self)
            N.check(N.lib().icd_index_search_filtered(self._h, N.buf_ptr(q), N.vec_dtype(q), B, int(k), int(weight_mode),
                                                      int(path), N.mask_ptr(mask, n), n, N.buf_ptr(score),
                                                      N.buf_ptr(raw), N.buf_ptr(ids), C.c_void_p(stream),
                                                      1 if sync else 0), "icd_index_search")
        return score, raw, ids

    def take_fallbacks(self) -> int:
        """Queries the tensor path re-searched with the exact stream scan since the previous call (DESIGN.md, "Exact
        search"); waits for the device."""
        n = C.c_int64()
        with self._lock:
            N.check(N.lib().icd_index_take_fallbacks(self._h, C.byref(n)), "icd_index_take_fallbacks")
        return int(n.value)

    def set_timing(self, on: bool) -> None:
        N.check(N.lib().icd_index_set_timing(self._h, 1 if on else 0), "icd_index_set_timing")

    def last_timing(self):
        us = (C.c_float * 3)()
        launches = C.c_int()
        N.check(N.lib().icd_index_last_timing(self._h, us, C.byref(launches)), "icd_index_last_timing")
        return {"scan_us": us[0], "merge_us": us[1], "finalise_us": us[2], "launches": launches.value}

    def mean_timing(self):
        """Stage times averaged over the searches since set_timing(True) (most recent 64)."""
        us = (C.c_float * 3)()
        calls = C.c_int()
        N.check(N.lib().icd_index_mean_timing(self._h, us, C.byref(calls)), "icd_index_mean_timing")
        return {"scan_us": us[0], "merge_us": us[1], "finalise_us": us[2], "calls": calls.value}
