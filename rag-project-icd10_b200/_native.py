"""ctypes binding of libicdrag.so (include/icdrag.h).

This is the only place Python touches the C ABI.  There is no CPU fallback: when the shared
library is missing or no sm_100 GPU is present, every entry point raises ``NativeError``.
"""
from __future__ import annotations

import ctypes as C
import os
import subprocess
import threading
from typing import Optional, Tuple

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
LIB_PATH = os.path.join(CSRC, "libicdrag.so")

F32, BF16 = 0, 1
WEIGHT_RERANK, WEIGHT_PRE, WEIGHT_NONE = 0, 1, 2
PATH_AUTO, PATH_STREAM, PATH_TENSOR = 0, 1, 2
INDEX_KEEP_F32 = 1
MAX_K = 128
MAX_LIMIT = 16384          # offset + limit of icd_index_search_page, as pymilvus
RANGE_RADIUS, RANGE_FILTER = 1, 2

# every symbol include/icdrag.h declares (tests check the library exports each one)
SYMBOLS = [
    "icd_version", "icd_last_error", "icd_launch_count", "icd_device_count", "icd_tune",
    "icd_index_create", "icd_index_destroy", "icd_index_append", "icd_index_adopt", "icd_index_clear",
    "icd_index_size", "icd_index_dim", "icd_index_read", "icd_index_search", "icd_index_last_timing",
    "icd_index_set_timing", "icd_index_mean_timing", "icd_index_search_filtered", "icd_index_take_fallbacks",
    "icd_index_search_page",
    "icd_nccl_unique_id", "icd_shard_group_create", "icd_shard_group_destroy",
    "icd_shard_group_export_slab", "icd_shard_group_import_slabs", "icd_shard_group_search",
    "icd_shard_group_search_filtered",
    "icd_encoder_weight_count", "icd_encoder_create", "icd_encoder_destroy", "icd_encoder_reserve",
    "icd_encoder_forward", "icd_encoder_read_hidden", "icd_encoder_set_token_head", "icd_encoder_token_logits",
    "icd_encoder_set_embedding_ids",
    "icd_tokenizer_create", "icd_tokenizer_destroy", "icd_tokenizer_encode", "icd_pack_batch",
]
MAX_LABELS = 64


class NativeError(RuntimeError):
    pass


class BertCfg(C.Structure):
    _fields_ = [("vocab_size", C.c_int32), ("hidden", C.c_int32), ("layers", C.c_int32),
                ("heads", C.c_int32), ("intermediate", C.c_int32), ("max_position", C.c_int32),
                ("type_vocab", C.c_int32), ("ln_eps", C.c_float)]


class SearchPage(C.Structure):
    """icd_search_page: the page [offset, offset + limit) of the exact list, after the range (radius, range_filter]
    on the raw inner product (range_flags = RANGE_RADIUS | RANGE_FILTER)."""
    _fields_ = [("offset", C.c_int32), ("limit", C.c_int32), ("range_flags", C.c_int32),
                ("radius", C.c_float), ("range_filter", C.c_float)]


_lib = None
_lock = threading.Lock()


def build(verbose: bool = False) -> str:
    """Compile csrc/ into csrc/libicdrag.so with nvcc for sm_100a (in-tree)."""
    out = subprocess.run(["make", "-C", CSRC, "-j", str(os.cpu_count() or 4)], capture_output=True, text=True)
    if verbose or out.returncode != 0:
        print(out.stdout[-4000:])
        print(out.stderr[-4000:])
    if out.returncode != 0:
        raise NativeError("building libicdrag.so failed")
    return LIB_PATH


def _preload_nccl() -> None:
    """libicdrag resolves NCCL lazily with dlopen; make torch's bundled copy findable."""
    try:
        import nvidia.nccl  # type: ignore
        root = list(nvidia.nccl.__path__)[0]
        cand = os.path.join(root, "lib", "libnccl.so.2")
        if os.path.exists(cand):
            os.environ.setdefault("ICDRAG_NCCL_LIB", cand)
    except Exception:
        pass


def lib() -> C.CDLL:
    global _lib
    if _lib is not None:
        return _lib
    with _lock:
        if _lib is not None:
            return _lib
        if not os.path.exists(LIB_PATH):
            raise NativeError(f"{LIB_PATH} is missing: run `python -c 'import __graft_entry__ as g; g.build()'` "
                              "(there is no CPU fallback)")
        _preload_nccl()
        L = C.CDLL(LIB_PATH, mode=C.RTLD_GLOBAL)
        _declare(L)
        _lib = L
        return L


def _declare(L: C.CDLL) -> None:
    vp, i32, i64, f32p = C.c_void_p, C.c_int, C.c_int64, C.POINTER(C.c_float)
    L.icd_version.restype = i32
    L.icd_last_error.restype = C.c_char_p
    L.icd_launch_count.restype = i64
    L.icd_device_count.restype = i32
    L.icd_tune.argtypes = [C.c_char_p, i32]
    L.icd_index_create.argtypes = [i32, i32, i64, i32, C.POINTER(vp)]
    L.icd_index_destroy.argtypes = [vp]
    L.icd_index_append.argtypes = [vp, vp, i32, vp, i64]
    L.icd_index_adopt.argtypes = [vp, vp, vp, i64]
    L.icd_index_clear.argtypes = [vp]
    L.icd_index_size.argtypes = [vp]
    L.icd_index_size.restype = i64
    L.icd_index_dim.argtypes = [vp]
    L.icd_index_read.argtypes = [vp, i64, i64, vp]
    L.icd_index_search.argtypes = [vp, vp, i32, i32, i32, i32, i32, vp, vp, vp, vp, i32]
    L.icd_index_search_filtered.argtypes = [vp, vp, i32, i32, i32, i32, i32, vp, i64, vp, vp, vp, vp, i32]
    L.icd_index_last_timing.argtypes = [vp, f32p, C.POINTER(i32)]
    L.icd_index_set_timing.argtypes = [vp, i32]
    L.icd_index_mean_timing.argtypes = [vp, f32p, C.POINTER(i32)]
    L.icd_index_take_fallbacks.argtypes = [vp, C.POINTER(i64)]
    L.icd_index_search_page.argtypes = [vp, vp, i32, i32, C.POINTER(SearchPage), i32, vp, i64, vp, vp, vp, vp, i32]
    if hasattr(L, "icd_nccl_unique_id"):
        L.icd_nccl_unique_id.argtypes = [vp]
        L.icd_shard_group_create.argtypes = [vp, i32, i32, i64, vp, C.POINTER(vp)]
        L.icd_shard_group_destroy.argtypes = [vp]
        L.icd_shard_group_export_slab.argtypes = [vp, vp]
        L.icd_shard_group_import_slabs.argtypes = [vp, vp]
        L.icd_shard_group_search.argtypes = [vp, vp, i32, i32, i32, i32, i32, i32, vp, vp, vp, vp, i32]
        L.icd_shard_group_search_filtered.argtypes = [vp, vp, i32, i32, i32, i32, i32, i32, vp, i64, vp, vp, vp, vp, i32]
    if hasattr(L, "icd_encoder_create"):
        L.icd_encoder_weight_count.argtypes = [C.POINTER(BertCfg)]
        L.icd_encoder_weight_count.restype = i64
        L.icd_encoder_create.argtypes = [vp, i64, C.POINTER(BertCfg), i32, C.POINTER(vp)]
        L.icd_encoder_destroy.argtypes = [vp]
        L.icd_encoder_reserve.argtypes = [vp, i32]
        L.icd_encoder_forward.argtypes = [vp, vp, vp, i32, i32, vp, i32, vp, i32]
        L.icd_encoder_read_hidden.argtypes = [vp, i32, vp, i64]
        L.icd_encoder_set_token_head.argtypes = [vp, vp, vp, i32]
        L.icd_encoder_token_logits.argtypes = [vp, vp, vp, i32, i32, vp, vp, i32]
        L.icd_encoder_set_embedding_ids.argtypes = [vp, i32, i32]
    if hasattr(L, "icd_tokenizer_create"):
        L.icd_tokenizer_create.argtypes = [C.c_char_p, i64, vp, i64, vp, vp, vp, i64, C.POINTER(vp)]
        L.icd_tokenizer_destroy.argtypes = [vp]
        L.icd_tokenizer_encode.argtypes = [vp, C.c_char_p, i64, i64, i32, vp, i32, vp, vp, i32]
        L.icd_pack_batch.argtypes = [vp, i32, vp, vp, i32, i32, vp, vp]


def check(status: int, what: str = "") -> None:
    if status != 0:
        msg = lib().icd_last_error().decode("utf-8", "replace")
        raise NativeError(f"{what} failed with status {status}: {msg}")


def tune(**knobs: int) -> None:
    """icd_tune: process-wide knobs of the tensor-core scan, e.g. tune(scan_sample=4)."""
    for key, value in knobs.items():
        check(lib().icd_tune(key.encode(), int(value)), f"icd_tune({key})")


def require_gpu() -> None:
    if lib().icd_device_count() <= 0:
        raise NativeError("no CUDA device visible: libicdrag has no CPU fallback")


# ------------------------------------------------------------------ buffer helpers
def _is_torch(x) -> bool:
    return type(x).__module__.startswith("torch")


def buf_ptr(x) -> int:
    """Address of a contiguous numpy array or torch tensor (host or device)."""
    if x is None:
        return 0
    if _is_torch(x):
        if not x.is_contiguous():
            raise ValueError("tensor must be contiguous")
        return int(x.data_ptr())
    if isinstance(x, np.ndarray):
        if not x.flags["C_CONTIGUOUS"]:
            raise ValueError("array must be C-contiguous")
        return int(x.ctypes.data)
    raise TypeError(f"unsupported buffer type {type(x)}")


def vec_dtype(x) -> int:
    """ICD_F32 / ICD_BF16 of a buffer; numpy uint16 is read as raw bf16 bits."""
    if _is_torch(x):
        import torch
        if x.dtype == torch.float32:
            return F32
        if x.dtype == torch.bfloat16:
            return BF16
        raise TypeError(f"unsupported tensor dtype {x.dtype}")
    if x.dtype == np.float32:
        return F32
    if x.dtype == np.uint16:
        return BF16
    raise TypeError(f"unsupported array dtype {x.dtype}")


def mask_ptr(mask, n_rows: int) -> int:
    """Address of a packed row mask (engine/filter_expr.py::pack_bits): uint32 words, numpy or a CUDA tensor, at least
    ceil(n_rows / 32) of them.  0 for None (every row)."""
    if mask is None:
        return 0
    words = (int(n_rows) + 31) // 32
    if _is_torch(mask):
        import torch
        if mask.dtype not in (torch.uint32, torch.int32):
            raise TypeError(f"row mask must be uint32 words, got {mask.dtype}")
    elif not isinstance(mask, np.ndarray) or mask.dtype not in (np.uint32, np.int32):
        raise TypeError("row mask must be a uint32 numpy array or tensor (engine/filter_expr.py::pack_bits)")
    if mask.ndim != 1 or int(mask.shape[0]) < words:
        raise ValueError(f"row mask of {n_rows} rows needs {words} uint32 words, got shape {tuple(mask.shape)}")
    return buf_ptr(mask)


def current_stream_ptr(device_index: Optional[int] = None) -> int:
    import torch
    return int(torch.cuda.current_stream(device_index).cuda_stream)
