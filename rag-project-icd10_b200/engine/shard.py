"""ShardGroup -- row-sharded exact search over the GPUs of one box (one process per GPU).

New work relative to the reference (single process, SURVEY.md section 5): rank r holds rows
[row_offset, row_offset + n_r); every rank calls ``search`` with the same queries and gets the
merged top-k.  torch.distributed is plumbing only: it carries the NCCL id and the cudaIpc slab
handles at start-up; the data path is libicdrag's own kernels (+ ncclAllGather for exchange 0).
"""
from __future__ import annotations

import ctypes as C

import numpy as np

from .. import _native as N


class ShardGroup:
    def __init__(self, index, row_offset: int, rank: int, world: int, peer_slabs: bool = True):
        import torch
        import torch.distributed as dist
        self.index, self.rank, self.world = index, rank, world
        self._h = C.c_void_p()
        idbuf = np.zeros(N_ID_BYTES, np.uint8)
        if world > 1:
            if rank == 0:
                N.check(N.lib().icd_nccl_unique_id(N.buf_ptr(idbuf)), "icd_nccl_unique_id")
            ident, _ = bootstrap_exchange(dist, rank, world, idbuf.tobytes() if rank == 0 else None, None, share_ident=True)
            idbuf = np.frombuffer(ident, np.uint8).copy()
        N.check(N.lib().icd_shard_group_create(N.buf_ptr(idbuf) if world > 1 else None, rank, world, int(row_offset),
                                               index._h, C.byref(self._h)), "icd_shard_group_create")
        self.peer_ready = False
        if world > 1 and peer_slabs:
            mine = np.zeros(64, np.uint8)
            N.check(N.lib().icd_shard_group_export_slab(self._h, N.buf_ptr(mine)), "icd_shard_group_export_slab")
            _, table_b = bootstrap_exchange(dist, rank, world, None, mine.tobytes())
            table = np.frombuffer(table_b, np.uint8).copy()
            N.check(N.lib().icd_shard_group_import_slabs(self._h, N.buf_ptr(table)), "icd_shard_group_import_slabs")
            self.peer_ready = True
            dist.barrier()

    def search(self, q, k: int, weight_mode: int = N.WEIGHT_RERANK, path: int = N.PATH_AUTO, exchange: int = 1,
               out=None, stream: int = 0, sync: bool = True, mask=None):
        """mask: packed uint32 bitmap of THIS rank's local rows (VectorIndex.search), None = every row."""
        if q.ndim == 1:
            q = q[None, :]
        B = int(q.shape[0])
        if exchange == 1 and not self.peer_ready and self.world > 1:
            exchange = 0
        if out is None:
            if N._is_torch(q):
                import torch
                out = (torch.empty((B, k), dtype=torch.float32, device=q.device),
                       torch.empty((B, k), dtype=torch.float32, device=q.device),
                       torch.empty((B, k), dtype=torch.int64, device=q.device))
            else:
                out = (np.empty((B, k), np.float32), np.empty((B, k), np.float32), np.empty((B, k), np.int64))
        score, raw, ids = out
        with self.index._lock:       # the group searches through the local index's workspace
            n = len(self.index)
            N.check(N.lib().icd_shard_group_search_filtered(self._h, N.buf_ptr(q), N.vec_dtype(q), B, int(k),
                                                            int(weight_mode), int(path), int(exchange),
                                                            N.mask_ptr(mask, n), n, N.buf_ptr(score), N.buf_ptr(raw),
                                                            N.buf_ptr(ids), C.c_void_p(stream), 1 if sync else 0),
                    "icd_shard_group_search")
        return score, raw, ids

    def close(self) -> None:
        if getattr(self, "_h", None) is not None and self._h.value:
            N.lib().icd_shard_group_destroy(self._h)
            self._h = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


N_ID_BYTES = 128


def bootstrap_exchange(dist, rank: int, world: int, ident, handle, share_ident: bool = False):
    """Start-up plumbing over torch.distributed (any backend): rank 0's NCCL id to everyone
    (share_ident=True; ident is only read on rank 0) and/or an all-gather of one opaque 64-byte handle per rank.
    Returns (ident_bytes | None, concatenated_handles | None)."""
    out_ident, out_table = None, None
    if share_ident:
        obj = [ident if rank == 0 else None]
        dist.broadcast_object_list(obj, src=0)
        out_ident = obj[0]
    if handle is not None:
        allh = [None] * world
        dist.all_gather_object(allh, handle)
        out_table = b"".join(allh)
    return out_ident, out_table


def shard_bounds(total_rows: int, rank: int, world: int):
    """Rows [lo, hi) of rank r: contiguous, sizes differ by at most one."""
    return total_rows * rank // world, total_rows * (rank + 1) // world


# ------------------------------------------------------------------ data-parallel encoder (SURVEY 8e, encoder row)
def partition_by_tokens(token_counts, world: int):
    """Splits sentence indices over `world` ranks with (nearly) equal TOKEN totals: longest-first onto the
    least-loaded rank.  Replicas share no state, so balance is the only thing that matters; each rank then
    length-buckets its own share (EncoderEngine._encode_ids).  Returns a list of index lists, each ascending."""
    order = sorted(range(len(token_counts)), key=lambda j: (-int(token_counts[j]), j))
    loads = [0] * world
    parts = [[] for _ in range(world)]
    for j in order:
        r = min(range(world), key=lambda x: (loads[x], x))
        parts[r].append(j)
        loads[r] += int(token_counts[j])
    return [sorted(p) for p in parts]


def encode_data_parallel(encode_fn, texts, token_counts, rank: int, world: int, dist=None, dim: int = 768):
    """Every rank encodes its share of `texts` with its own encoder replica (`encode_fn(list[str]) -> [m, dim]
    float32 array`); no collective on the data path.  With `dist` (torch.distributed, any backend) the shares are
    all-gathered so every rank returns the full [n, dim] matrix in input order; without it only this rank's rows
    are filled (the build tool's case: shard r encodes exactly the rows it will hold)."""
    parts = partition_by_tokens(token_counts, world)
    mine = parts[rank]
    out = np.zeros((len(texts), dim), np.float32)
    local = np.asarray(encode_fn([texts[j] for j in mine]), np.float32).reshape(len(mine), dim) if mine else \
        np.zeros((0, dim), np.float32)
    out[mine] = local
    if dist is not None and world > 1:
        gathered = [None] * world
        dist.all_gather_object(gathered, local)
        for r in range(world):
            if parts[r]:
                out[parts[r]] = gathered[r]
    return out
