"""IcdStoreClient -- the object MilvusService holds where the reference holds a
``pymilvus.MilvusClient`` (/root/reference/services/milvus_service.py:81,100-110).

It offers the slice of the MilvusClient surface the reference touches (has_collection,
create_schema / add_field, prepare_index_params / add_index, create_collection,
get_load_state, load_collection, release_collection, drop_collection, get_collection_stats,
insert, search (with a boolean ``filter`` over the scalar fields: engine/filter_expr.py), query, get, close) over:
  * a device-resident vector table searched by libicdrag.so (engine/index.py): bf16 scan copy
    plus an fp32 master, so single-query search is exact fp32 inner product like Milvus FLAT/IP;
  * a COLUMNAR on-disk form next to MILVUS_DB_PATH (format 2), one directory per collection:
        <db_path>.icdb/<collection>/header.json     dim, metric, fields, committed_rows  (the commit point)
                                    vectors.f32     [n, dim] little-endian float32 (the fp32 master image)
                                    vectors.bf16    [n, dim] bfloat16 bits (the scan table image)
                                    levels.u8       [n] level bytes (1, 2, 3)
                                    <field>.str/.off  UTF-8 bytes + uint64 end offsets of every VARCHAR field
                                    <field>.u8 / .i32 BOOL / INT32 fields
                                    extra.str/.off  JSON of any dynamic fields of a row (enable_dynamic_field)
    Every file is a flat array: ``load_collection`` is an mmap plus ONE host-to-device copy per array (no parsing),
    a shard loads only its row range, and scalar fields are decoded lazily, per hit, from the mapped columns.
    Appends write the column tails first and replace header.json (write + fsync + rename) last; opening a collection
    truncates every column back to the committed row count, so a torn append can never pair a row with another
    row's vector.  The reference's append / drop semantics are kept (auto-id primary key; re-running the build
    appends duplicates; drop removes everything).
There is no CPU search path: loading a collection needs a GPU.
"""
from __future__ import annotations

import json
import mmap
import os
import shutil
from collections import OrderedDict
from typing import Any, Dict, Iterable, List, Optional, Sequence, Tuple

import numpy as np

from .. import _native as N
from . import filter_expr
from .index import VectorIndex

SCALAR_FIELDS = ["code", "preferred_zh", "has_complication", "main_code", "secondary_code", "level",
                 "parent_code", "category_path", "semantic_text"]
_STR_FIELDS = ["code", "preferred_zh", "main_code", "secondary_code", "parent_code", "category_path", "semantic_text"]
_BOOL_FIELDS = ["has_complication"]
_INT_FIELDS = ["level"]
_FORMAT = 2
# fsync column tails and header on every append (power-loss durability).  Off by default: the commit protocol (tails
# first, header replaced last, tails truncated to the committed count on open) already survives a crashed or failed
# append, and the reference's build makes hundreds of small inserts.
DURABLE = os.environ.get("ICD_STORE_DURABLE", "0") == "1"


class Hit(dict):
    """pymilvus Hit look-alike: ``hit.get(field)`` falls through to the entity fields
    (the reference relies on it at milvus_service.py:293,298-309)."""

    def get(self, key, default=None):
        if key in self:
            return dict.get(self, key)
        return dict.get(self, "entity", {}).get(key, default)


class _Schema:
    def __init__(self, **kw):
        self.options = kw
        self.fields: List[Dict[str, Any]] = []

    def add_field(self, field_name: str, datatype=None, **kw):
        self.fields.append({"field_name": field_name, "datatype": datatype, **kw})
        return self

    @property
    def dim(self) -> Optional[int]:
        for f in self.fields:
            if "dim" in f:
                return int(f["dim"])
        return None


class _IndexParams:
    def __init__(self):
        self.indexes: List[Dict[str, Any]] = []

    def add_index(self, field_name: str, index_type: str = "FLAT", metric_type: str = "IP", **kw):
        self.indexes.append({"field_name": field_name, "index_type": index_type, "metric_type": metric_type, **kw})


class DataType:
    """Names the reference imports from pymilvus (milvus_service.py:6,174-186)."""
    INT64, FLOAT_VECTOR, VARCHAR, BOOL, INT32 = "INT64", "FLOAT_VECTOR", "VARCHAR", "BOOL", "INT32"


# ---------------------------------------------------------------------------------------------- columns
class _Column:
    """One append-only flat array on disk (or in memory for a non-persistent store), mapped read-only."""

    def __init__(self, path: Optional[str], dtype, width: int = 1):
        self.path, self.dtype, self.width = path, np.dtype(dtype), int(width)
        self.count = 0                      # committed elements (rows * width)
        self._pending = 0                   # elements written so far (committed + the uncommitted tail)
        self._mem: List[np.ndarray] = []    # non-persistent stores keep the pieces here
        self._map: Optional[np.ndarray] = None
        self._mm = None
        self._fh = None

    @property
    def item_bytes(self) -> int:
        return self.dtype.itemsize

    def open(self, committed: int) -> None:
        """Bring the file to exactly `committed` elements (a longer file is the tail of a torn append)."""
        self.count = self._pending = int(committed)
        if self.path is None:
            return
        want = self.count * self.item_bytes
        if not os.path.exists(self.path):
            if want:
                raise N.NativeError(f"{self.path} is missing")
            open(self.path, "wb").close()
        size = os.path.getsize(self.path)
        if size < want:
            raise N.NativeError(f"{self.path} holds {size} bytes, the committed header needs {want}")
        if size > want:
            with open(self.path, "r+b") as fh:
                fh.truncate(want)
        self._remap()

    def _remap(self) -> None:
        self._map = None
        if self._mm is not None:
            try:
                self._mm.close()
            except BufferError:     # a caller still holds a view of the old map: it stays valid, the map goes with it
                pass
            self._mm = None
        if self._fh is not None:
            self._fh.close()
            self._fh = None
        if self.path is None or self.count == 0:
            return
        self._fh = open(self.path, "rb")
        self._mm = mmap.mmap(self._fh.fileno(), self.count * self.item_bytes, access=mmap.ACCESS_READ)
        self._map = np.frombuffer(self._mm, dtype=self.dtype, count=self.count)

    def append(self, arr: np.ndarray) -> None:
        """Write the tail (not yet committed: `commit` makes it visible)."""
        arr = np.ascontiguousarray(arr, self.dtype).reshape(-1)
        if self.path is None:
            self._mem.append(arr.copy())
        else:
            with open(self.path, "r+b" if os.path.exists(self.path) else "wb") as fh:
                fh.seek(self.count * self.item_bytes)
                fh.write(arr.tobytes())
                fh.truncate()
                if DURABLE:
                    fh.flush()
                    os.fsync(fh.fileno())
        self._pending = self.count + arr.size

    def presize(self, count: int) -> None:
        """Extend the (uncommitted) tail to `count` elements so that several writers can fill disjoint slices."""
        if self.path is None:
            raise N.NativeError("sharded appends need a persistent store")
        with open(self.path, "r+b") as fh:
            fh.truncate(int(count) * self.item_bytes)
        self._pending = int(count)

    def write_at(self, elem_offset: int, arr: np.ndarray) -> None:
        """Write into the pre-sized tail (any process; rows at or above the committed count only)."""
        arr = np.ascontiguousarray(arr, self.dtype).reshape(-1)
        if elem_offset < self.count:
            raise N.NativeError("write_at below the committed row count")
        with open(self.path, "r+b") as fh:
            fh.seek(int(elem_offset) * self.item_bytes)
            fh.write(arr.tobytes())
            if DURABLE:
                fh.flush()
                os.fsync(fh.fileno())

    def commit(self) -> None:
        self.count = self._pending
        if self.path is None:
            if len(self._mem) > 1:
                self._mem = [np.concatenate(self._mem)]
            self._map = self._mem[0] if self._mem else None
        else:
            self._remap()

    def rollback(self) -> None:
        self._pending = self.count
        if self.path is None:
            have = sum(a.size for a in self._mem)
            while self._mem and have > self.count:
                have -= self._mem.pop().size
        elif os.path.exists(self.path):
            with open(self.path, "r+b") as fh:
                fh.truncate(self.count * self.item_bytes)

    def view(self) -> np.ndarray:
        """The committed elements (a read-only map of the file)."""
        if self._map is None:
            return np.zeros((0,), self.dtype)
        return self._map

    def close(self) -> None:
        self.count_closed = self.count
        self._map = None
        if self._mm is not None:
            try:
                self._mm.close()
            except BufferError:     # a caller still holds a view: the map goes away with it
                pass
            self._mm = None
        if self._fh is not None:
            self._fh.close()
            self._fh = None


class _StrColumn:
    """VARCHAR column: UTF-8 bytes + uint64 END offset of every row."""

    def __init__(self, base: Optional[str]):
        self.data = _Column(base + ".str" if base else None, np.uint8)
        self.off = _Column(base + ".off" if base else None, np.uint64)

    def open(self, rows: int) -> None:
        self.off.open(rows)
        nbytes = int(self.off.view()[rows - 1]) if rows else 0
        self.data.open(nbytes)

    def append(self, values: Sequence[str]) -> None:
        enc = [("" if v is None else str(v)).encode("utf-8") for v in values]
        start = int(self.off.view()[self.off.count - 1]) if self.off.count else 0
        ends = start + np.cumsum([len(b) for b in enc], dtype=np.uint64) if enc else np.zeros((0,), np.uint64)
        self.data.append(np.frombuffer(b"".join(enc), np.uint8))
        self.off.append(ends.astype(np.uint64))

    def commit(self) -> None:
        self.data.commit()
        self.off.commit()

    def rollback(self) -> None:
        self.data.rollback()
        self.off.rollback()

    def get(self, i: int) -> str:
        off = self.off.view()
        lo = int(off[i - 1]) if i else 0
        return bytes(self.data.view()[lo:int(off[i])]).decode("utf-8")

    def close(self) -> None:
        self.data.close()
        self.off.close()


class ColumnTable:
    """The scalar fields of a collection, row id == insertion order.  ``table[i]`` decodes one row to the dict the
    reference stores (lazily: nothing is parsed when the collection is opened)."""

    def __init__(self, directory: Optional[str], dim: int):
        self.dir, self.dim = directory, int(dim)
        p = (lambda name: os.path.join(directory, name)) if directory else (lambda name: None)
        self.f32 = _Column(p("vectors.f32"), "<f4", dim)
        self.bf16 = _Column(p("vectors.bf16"), "<u2", dim)
        self.levels = _Column(p("levels.u8"), np.uint8)
        self.strs = {f: _StrColumn(p(f)) for f in _STR_FIELDS}
        self.bools = {f: _Column(p(f + ".u8"), np.uint8) for f in _BOOL_FIELDS}
        self.ints = {f: _Column(p(f + ".i32"), "<i4") for f in _INT_FIELDS}
        self.extra = _StrColumn(p("extra"))
        self.n = 0

    def _all(self):
        return [self.f32, self.bf16, self.levels, *self.strs.values(), *self.bools.values(), *self.ints.values(), self.extra]

    def open(self, rows: int) -> None:
        self.n = int(rows)
        self.__dict__.pop("_row_cache", None)
        self.f32.open(rows * self.dim)
        self.bf16.open(rows * self.dim)
        self.levels.open(rows)
        for c in [*self.strs.values(), self.extra]:
            c.open(rows)
        for c in [*self.bools.values(), *self.ints.values()]:
            c.open(rows)

    def __len__(self) -> int:
        return self.n

    def __getitem__(self, i: int) -> Dict[str, Any]:
        i = int(i)
        if not 0 <= i < self.n:
            raise IndexError(i)
        row: Dict[str, Any] = {}
        extra = self.extra.get(i)
        if extra:
            row.update(json.loads(extra))
        for f, c in self.strs.items():
            row[f] = c.get(i)
        for f, c in self.bools.items():
            row[f] = bool(c.view()[i])
        for f, c in self.ints.items():
            row[f] = int(c.view()[i])
        return row

    _ROW_CACHE_MAX = 131072

    def cached_row(self, i: int) -> Dict[str, Any]:
        """Decoded row i, memoised: rows are immutable once committed and a serving process returns the same few thousand
        ICD rows over and over (9 field decodes per hit otherwise).  Callers must not mutate the dict."""
        cache = self.__dict__.setdefault("_row_cache", {})
        row = cache.get(i)
        if row is None:
            if len(cache) >= self._ROW_CACHE_MAX:
                cache.clear()
            row = cache[i] = self[i]
        return row

    def field(self, name: str, i: int):
        if name in self.strs:
            return self.strs[name].get(i)
        if name in self.bools:
            return bool(self.bools[name].view()[i])
        if name in self.ints:
            return int(self.ints[name].view()[i])
        extra = self.extra.get(i)
        return json.loads(extra).get(name) if extra else None

    def stage(self, rows: List[Dict[str, Any]], vecs_f32: Optional[np.ndarray], bf16_bits: Optional[np.ndarray],
              levels: Optional[np.ndarray]) -> None:
        """Validate and serialise everything FIRST (a value that cannot be stored raises before any file is touched),
        then write the column tails.  Nothing is visible until commit().  With vecs_f32 = None only the scalar columns
        are written and the three fixed-width vector files are pre-sized: the slices are filled by write_vectors()
        (the sharded build: every rank writes the rows it encoded)."""
        known = set(_STR_FIELDS) | set(_BOOL_FIELDS) | set(_INT_FIELDS)
        strs = {f: ["" if r.get(f) is None else str(r.get(f)) for r in rows] for f in _STR_FIELDS}
        bools = {f: np.asarray([1 if r.get(f, False) else 0 for r in rows], np.uint8) for f in _BOOL_FIELDS}
        ints = {f: np.asarray([int(r.get(f, 1)) for r in rows], "<i4") for f in _INT_FIELDS}
        extra = []
        for r in rows:
            rest = {k: v for k, v in r.items() if k not in known}
            extra.append(json.dumps(rest, ensure_ascii=False) if rest else "")
        try:
            if vecs_f32 is None:
                total = self.n + len(rows)
                self.f32.presize(total * self.dim)
                self.bf16.presize(total * self.dim)
                self.levels.presize(total)
            else:
                self.f32.append(vecs_f32)
                self.bf16.append(bf16_bits)
                self.levels.append(levels)
            for f in _STR_FIELDS:
                self.strs[f].append(strs[f])
            for f in _BOOL_FIELDS:
                self.bools[f].append(bools[f])
            for f in _INT_FIELDS:
                self.ints[f].append(ints[f])
            self.extra.append(extra)
        except Exception:
            self.rollback()
            raise
        self._staged = self.n + len(rows)

    def write_vectors(self, row0: int, vecs_f32: np.ndarray, bf16_bits: np.ndarray, levels: np.ndarray) -> None:
        """Fill rows [row0, row0 + m) of the pre-sized vector files (disjoint slices, any process)."""
        self.f32.write_at(row0 * self.dim, vecs_f32)
        self.bf16.write_at(row0 * self.dim, bf16_bits)
        self.levels.write_at(row0, levels)

    def commit(self) -> None:
        for c in self._all():
            c.commit()
        self.n = getattr(self, "_staged", self.n)

    def rollback(self) -> None:
        for c in self._all():
            c.rollback()
        self._staged = self.n

    def close(self) -> None:
        for c in self._all():
            c.close()


def f32_to_bf16_bits(x: np.ndarray) -> np.ndarray:
    """Round-to-nearest-even fp32 -> bf16 bit patterns (what f32_to_bf16_kernel does on the device)."""
    u = np.ascontiguousarray(x, np.float32).view(np.uint32)
    return ((u + np.uint32(0x7FFF) + ((u >> np.uint32(16)) & np.uint32(1))) >> np.uint32(16)).astype(np.uint16)


def shard_rows(total_rows: int, rank: int, world: int) -> Tuple[int, int]:
    """Rows [lo, hi) of shard `rank` (engine/shard.py::shard_bounds)."""
    return total_rows * rank // world, total_rows * (rank + 1) // world


class _Collection:
    def __init__(self, name: str, dim: int, directory: Optional[str], metric: str = "IP", index_type: str = "FLAT"):
        self.name, self.dim, self.metric, self.index_type = name, dim, metric, index_type
        self.dir = directory
        self.rows = ColumnTable(directory, dim)    # scalar fields + vector images, insertion order == row id
        self.index: Optional[VectorIndex] = None   # device table when loaded
        self.loaded = False
        self.row_lo, self.row_hi = 0, 0            # rows resident on this device (a shard when the client is sharded)

    @property
    def levels(self) -> np.ndarray:
        return self.rows.levels.view()


class IcdStoreClient:
    def __init__(self, uri: str = "./db/milvus_icd10.db", device: int = 0, shard: Optional[Tuple[int, int]] = None,
                 keep_f32: bool = True, **_remote_kwargs):
        """shard=(rank, world): this client serves rows shard_rows(n, rank, world) of every collection (8-GPU serving:
        one client per rank over the same files; search results carry GLOBAL row ids)."""
        N.require_gpu()
        self.uri, self.device = uri, device
        self.shard = shard
        # keep_f32=False: load only the bf16 image (half the HBM; scores are then those of the bf16-rounded rows) --
        # for corpora far larger than the ICD table.  The default keeps Milvus FLAT's exact fp32 inner products.
        self.keep_f32 = bool(keep_f32)
        self.root = uri + ".icdb" if not uri.endswith(".icdb") else uri
        self.persist = not uri.startswith(("http://", "https://"))
        self.cols: Dict[str, _Collection] = {}
        # device row masks of recent filter expressions: (collection, expression) -> (committed rows, mask words)
        self._masks: "OrderedDict[Tuple[str, str], Tuple[int, Any]]" = OrderedDict()
        if self.persist:
            os.makedirs(self.root, exist_ok=True)
            for fn in sorted(os.listdir(self.root)):
                if os.path.exists(os.path.join(self.root, fn, "header.json")):
                    self._open(fn)

    # ---------------------------------------------------------------- persistence
    def _dir(self, name: str) -> Optional[str]:
        return os.path.join(self.root, name) if self.persist else None

    def _write_header(self, col: _Collection, rows: int, fields: Optional[List[str]] = None) -> None:
        if not self.persist:
            return
        head = os.path.join(col.dir, "header.json")
        if fields is None and os.path.exists(head):
            with open(head, encoding="utf-8") as fh:
                fields = json.load(fh).get("fields", [])
        tmp = head + ".tmp"
        with open(tmp, "w", encoding="utf-8") as fh:
            json.dump({"format": _FORMAT, "dim": col.dim, "metric": col.metric, "index_type": col.index_type,
                       "fields": fields or [], "committed_rows": int(rows)}, fh)
            if DURABLE:
                fh.flush()
                os.fsync(fh.fileno())
        os.replace(tmp, head)      # the commit point

    def _open(self, name: str) -> None:
        d = self._dir(name)
        with open(os.path.join(d, "header.json"), encoding="utf-8") as fh:
            h = json.load(fh)
        if h.get("format") != _FORMAT:
            raise N.NativeError(f"collection {name}: store format {h.get('format')} is not format {_FORMAT}")
        col = _Collection(name, int(h["dim"]), d, h.get("metric", "IP"), h.get("index_type", "FLAT"))
        col.rows.open(int(h.get("committed_rows", 0)))
        self.cols[name] = col

    # ---------------------------------------------------------------- MilvusClient surface
    def has_collection(self, collection_name: str) -> bool:
        return collection_name in self.cols

    def create_schema(self, **kw) -> _Schema:
        return _Schema(**kw)

    def prepare_index_params(self) -> _IndexParams:
        return _IndexParams()

    def create_collection(self, collection_name: str, schema: _Schema = None, index_params: _IndexParams = None,
                          dimension: Optional[int] = None, **_kw) -> None:
        dim = dimension or (schema.dim if schema is not None else None)
        if not dim:
            raise ValueError("create_collection needs a FLOAT_VECTOR field with dim")
        metric, itype = "IP", "FLAT"
        if index_params is not None and index_params.indexes:
            metric = index_params.indexes[0].get("metric_type", "IP")
            itype = index_params.indexes[0].get("index_type", "FLAT")
        if metric != "IP":
            raise N.NativeError(f"only the IP metric is implemented (got {metric})")
        d = self._dir(collection_name)
        if d is not None:
            if os.path.isdir(d):
                shutil.rmtree(d)
            os.makedirs(d)
        col = _Collection(collection_name, int(dim), d, metric, itype)
        col.rows.open(0)
        self.cols[collection_name] = col
        self._write_header(col, 0, [f["field_name"] for f in (schema.fields if schema else [])])

    def drop_collection(self, collection_name: str) -> None:
        self._forget_masks(collection_name)
        col = self.cols.pop(collection_name, None)
        if col is not None:
            if col.index is not None:
                col.index.close()
            col.rows.close()
        d = self._dir(collection_name)
        if d is not None and os.path.isdir(d):
            shutil.rmtree(d)

    def get_load_state(self, collection_name: str) -> str:
        # The reference compares this value with the string "Loaded" (milvus_service.py:143,154).
        return "Loaded" if self.cols[collection_name].loaded else "NotLoad"

    def _resident_range(self, col: _Collection) -> Tuple[int, int]:
        n = len(col.rows)
        return shard_rows(n, *self.shard) if self.shard else (0, n)

    def load_collection(self, collection_name: str) -> None:
        """mmap -> device: one host-to-device copy of the bf16 image (the scan table), one of the fp32 image (the
        master) and one of the level bytes, for the rows this client serves."""
        col = self.cols[collection_name]
        if col.loaded and col.index is not None:
            return
        if col.index is None:
            lo, hi = self._resident_range(col)
            col.index = VectorIndex(col.dim, device=self.device, capacity=max(hi - lo, 1024), keep_f32=self.keep_f32)
            if hi > lo:
                image = col.rows.f32 if self.keep_f32 else col.rows.bf16
                col.index.append(image.view().reshape(-1, col.dim)[lo:hi], np.ascontiguousarray(col.levels[lo:hi]))
            col.row_lo, col.row_hi = lo, hi
        col.loaded = True

    def release_collection(self, collection_name: str) -> None:
        self._forget_masks(collection_name)
        col = self.cols[collection_name]
        if col.index is not None and self.persist:
            col.index.close()          # frees the HBM table; load_collection maps it back from the column files
            col.index = None
        col.loaded = False

    def get_collection_stats(self, collection_name: str) -> Dict[str, Any]:
        return {"row_count": len(self.cols[collection_name].rows)}

    def _append_rows(self, col: _Collection, rows: List[Dict[str, Any]], vecs: Optional[np.ndarray], vecs_dev=None):
        """The one append path: validate -> column tails -> device table -> header (commit).  Any failure before the
        header is replaced rolls the column tails back, so files, host state and device table stay in step."""
        if self.shard is not None:
            raise N.NativeError("a sharded client is read-only for plain inserts: use the sharded_append_* protocol "
                                "(tools/build_database.py under torchrun) or an unsharded client")
        first = len(col.rows)
        if vecs is None:
            vecs = vecs_dev.detach().to("cpu").numpy()
        vecs = np.ascontiguousarray(vecs, np.float32)
        if vecs.ndim != 2 or vecs.shape[1] != col.dim or vecs.shape[0] != len(rows):
            raise ValueError(f"vector dimension mismatch: expected [{len(rows)}, {col.dim}], got {vecs.shape}")
        if not np.all(np.isfinite(vecs)):
            raise ValueError("vectors must be finite")
        levels = np.asarray([_level_byte(r.get("level", 1)) for r in rows], np.uint8)
        if col.index is None and (col.loaded or not self.persist):
            col.index = VectorIndex(col.dim, device=self.device, keep_f32=self.keep_f32)
            if first:   # rows persisted earlier must be on the device before new ones are appended behind them
                col.index.append(col.rows.f32.view().reshape(-1, col.dim)[:first], np.ascontiguousarray(col.levels[:first]))
        col.rows.stage(rows, vecs, f32_to_bf16_bits(vecs), levels)
        try:
            if col.index is not None:
                if vecs_dev is not None:
                    import torch
                    col.index.append(vecs_dev.contiguous(), torch.from_numpy(levels).to(vecs_dev.device))
                else:
                    col.index.append(vecs, levels)
            self._write_header(col, first + len(rows))
        except Exception:
            col.rows.rollback()
            if col.index is not None:   # the device table may hold the new rows: rebuild it from the committed files
                col.index.close()
                col.index = None
                was_loaded, col.loaded = col.loaded, False
                if was_loaded:
                    self.load_collection(col.name)
            raise
        col.rows.commit()
        col.row_hi = len(col.rows)
        self._forget_masks(col.name)
        return first

    def insert(self, collection_name: str, data: Iterable[Dict[str, Any]]) -> Dict[str, Any]:
        col = self.cols[collection_name]
        data = list(data)
        if not data:
            return {"insert_count": 0}
        vecs = np.asarray([d["vector"] for d in data], dtype=np.float32)
        if vecs.ndim != 2 or vecs.shape[1] != col.dim:
            raise ValueError(f"vector dimension mismatch: expected {col.dim}, got {vecs.shape}")
        rows = [{k: v for k, v in d.items() if k != "vector"} for d in data]
        first = self._append_rows(col, rows, vecs)
        return {"insert_count": len(rows), "ids": list(range(first, first + len(rows)))}

    def insert_arrays(self, collection_name: str, rows: List[Dict[str, Any]], vectors) -> Dict[str, Any]:
        """Build path (SURVEY 8e): the embeddings of many records as ONE [n, dim] float32 array -- numpy, or a torch
        tensor that is still on the GPU (appended to the device table without a host round trip; the host copy made
        for the column files is the only transfer) -- instead of n Python lists."""
        col = self.cols[collection_name]
        if not rows:
            return {"insert_count": 0}
        if N._is_torch(vectors) and vectors.is_cuda:
            first = self._append_rows(col, list(rows), None, vecs_dev=vectors)
        elif N._is_torch(vectors):
            first = self._append_rows(col, list(rows), vectors.numpy())
        else:
            first = self._append_rows(col, list(rows), np.asarray(vectors, np.float32))
        return {"insert_count": len(rows), "ids": list(range(first, first + len(rows)))}

    # ---------------------------------------------------------------- sharded build (SURVEY 8e, encoder row)
    # Every rank encodes exactly the rows it will hold; the embeddings go from the encoder's output buffer into that
    # rank's device table and never visit another GPU.  On disk the collection is still ONE set of flat column files:
    # rank 0 writes the scalar columns of all rows and pre-sizes the vector files, every rank then fills its own slice
    # (fixed-width rows: plain offset writes), rank 0 replaces the header.  The caller provides the barriers between
    # the phases (tools/build_database.py over torch.distributed).
    def sharded_append_prepare(self, collection_name: str, rows_all: List[Dict[str, Any]]) -> None:
        """Phase 1, rank 0 only: scalar columns of ALL new rows + pre-sized vector files.  The collection must be empty
        (a sharded build is a rebuild: shard r serves rows shard_rows(n, r, world))."""
        col = self.cols[collection_name]
        if len(col.rows):
            raise N.NativeError("a sharded build needs an empty collection (use --rebuild)")
        col.rows.stage(list(rows_all), None, None, None)

    def sharded_append_slice(self, collection_name: str, row_lo: int, rows_local: List[Dict[str, Any]], vectors) -> None:
        """Phase 2, every rank: this rank's rows [row_lo, row_lo + m): vectors (numpy or a CUDA tensor) into the device
        table of this client and into its slice of the vector files."""
        col = self.cols[collection_name]
        dev = vectors if (N._is_torch(vectors) and vectors.is_cuda) else None
        host = vectors.detach().to("cpu").numpy() if N._is_torch(vectors) else np.asarray(vectors, np.float32)
        host = np.ascontiguousarray(host, np.float32)
        if host.ndim != 2 or host.shape != (len(rows_local), col.dim) or not np.all(np.isfinite(host)):
            raise ValueError(f"expected finite vectors of shape [{len(rows_local)}, {col.dim}], got {host.shape}")
        levels = np.asarray([_level_byte(r.get("level", 1)) for r in rows_local], np.uint8)
        if col.index is not None:
            col.index.close()
        col.index = VectorIndex(col.dim, device=self.device, capacity=max(len(rows_local), 1024), keep_f32=self.keep_f32)
        if len(rows_local):
            if dev is not None:
                import torch
                col.index.append(dev.contiguous(), torch.from_numpy(levels).to(dev.device))
            else:
                col.index.append(host, levels)
            col.rows.write_vectors(int(row_lo), host, f32_to_bf16_bits(host), levels)
        col.row_lo, col.row_hi = int(row_lo), int(row_lo) + len(rows_local)

    def sharded_append_commit(self, collection_name: str, total_rows: int, is_writer: bool) -> None:
        """Phase 3: rank 0 (is_writer) replaces the header; every rank calls this AFTER the writer has (barrier in
        between) to map the committed columns."""
        self._forget_masks(collection_name)
        col = self.cols[collection_name]
        if is_writer:
            self._write_header(col, int(total_rows))
            col.rows.commit()
        else:
            col.rows.open(int(total_rows))
        col.loaded = True

    def attach_group(self, collection_name: str, group) -> None:
        """Serve this collection through a ShardGroup (engine/shard.py): search() then returns the merged top-k of all
        shards with GLOBAL row ids; every rank must issue the same searches."""
        self.cols[collection_name].group = group

    # ---------------------------------------------------------------- filters
    _MASK_CACHE = 8   # masks kept on the device (12.5 MB each at 100 M rows)

    def _forget_masks(self, collection_name: str) -> None:
        for key in [k for k in self._masks if k[0] == collection_name]:
            del self._masks[key]

    def _row_mask(self, col: _Collection, expr: str):
        """Device bitmap of the rows this client serves ([row_lo, row_hi): a shard's LOCAL rows) that satisfy `expr`, or
        None for an empty expression.  Cached per (collection, expression) while the committed row count holds."""
        pred = filter_expr.compile(expr)        # ValueError on a bad expression, before any cache lookup
        if pred.is_all:
            return None
        key = (col.name, str(expr).strip())
        stamp = (len(col.rows), col.row_lo, col.row_hi)
        hit = self._masks.get(key)
        if hit is not None and hit[0] == stamp:
            self._masks.move_to_end(key)
            return hit[1]
        import torch
        words = filter_expr.pack_bits(pred.mask(col.rows, col.row_lo, col.row_hi))
        dev = torch.from_numpy(words.view(np.int32)).to(torch.device("cuda", self.device))
        self._masks[key] = (stamp, dev)
        self._masks.move_to_end(key)
        while len(self._masks) > self._MASK_CACHE:
            self._masks.popitem(last=False)
        return dev

    @staticmethod
    def _page(limit, search_params=None, offset=None):
        """pymilvus's paging and range arguments -> (limit, offset, radius, range_filter), checked by pymilvus's rules:
        1 <= limit, 0 <= offset, offset + limit <= 16 384; offset given as `offset=` or search_params["offset"] (both
        only when equal); radius / range_filter from search_params["params"] (FLAT/IP range search: the hits whose
        inner product lies in (radius, range_filter]), radius < range_filter when both are given."""
        sp = search_params or {}
        if not isinstance(sp, dict):
            raise ValueError(f"search_params must be a dict, got {type(sp).__name__}")
        sp_offset = sp.get("offset")
        if offset is not None and sp_offset is not None and int(offset) != int(sp_offset):
            raise ValueError(f"conflicting offsets: offset={offset} and search_params['offset']={sp_offset}")
        offset = int(offset if offset is not None else (sp_offset or 0))
        limit = int(limit)
        if limit < 1:
            raise ValueError(f"limit must be >= 1, got {limit}")
        if offset < 0:
            raise ValueError(f"offset must be >= 0, got {offset}")
        if offset + limit > N.MAX_LIMIT:
            raise ValueError(f"offset + limit must be in [1, {N.MAX_LIMIT}], got {offset} + {limit}")
        params = sp.get("params") or {}
        radius, range_filter = params.get("radius"), params.get("range_filter")
        radius = None if radius is None else float(radius)
        range_filter = None if range_filter is None else float(range_filter)
        if radius is not None and range_filter is not None and not radius < range_filter:
            raise ValueError(f"range search on IP needs radius < range_filter, got {radius} and {range_filter}")
        return limit, offset, radius, range_filter

    @staticmethod
    def _group_refuses(limit, offset, radius, range_filter) -> None:
        if limit > N.MAX_K or offset or radius is not None or range_filter is not None:
            raise NotImplementedError(f"a sharded collection serves limit <= {N.MAX_K} without offset or range "
                                      "(paged and range search run on a single-table collection)")

    def search(self, collection_name: str, data, limit: int = 10, output_fields: Optional[List[str]] = None,
               filter: str = "", search_params: Optional[Dict[str, Any]] = None, offset: Optional[int] = None,
               **_kw) -> List[List[Hit]]:
        """MilvusClient.search; `filter` = a boolean expression over the scalar fields (engine/filter_expr.py): the exact
        top-`limit` over the rows it allows (fewer hits when fewer rows match).  ValueError on a bad expression.
        `offset` (or search_params["offset"]) skips the first hits, search_params["params"] may hold `radius` /
        `range_filter` (range search on the raw inner product); offset + limit <= 16 384 (_page)."""
        col = self.cols[collection_name]
        if not col.loaded or col.index is None:
            raise N.NativeError(f"collection {collection_name} is not loaded")
        k, offset, radius, range_filter = self._page(limit, search_params, offset)
        q = np.ascontiguousarray(np.asarray(data, dtype=np.float32))
        if q.ndim == 1:
            q = q[None, :]
        mask = self._row_mask(col, filter)
        group = getattr(col, "group", None)
        if group is not None:
            self._group_refuses(k, offset, radius, range_filter)
            _, raw, ids = group.search(q, k, weight_mode=N.WEIGHT_NONE, mask=mask)
            base = 0
        else:
            _, raw, ids = col.index.search(q, k, weight_mode=N.WEIGHT_NONE, mask=mask, offset=offset, radius=radius,
                                           range_filter=range_filter)
            base = col.row_lo
        fields = output_fields or []
        out = []
        for b in range(q.shape[0]):
            hits = []
            for s, j in zip(raw[b], ids[b]):
                if j < 0:
                    break
                g = int(j) + base
                row = col.rows.cached_row(g)
                hits.append(Hit(id=g, distance=float(s), entity={f: row.get(f) for f in fields}))
            out.append(hits)
        return out

    def search_ranked(self, collection_name: str, queries, limit: int, filter: str = ""):
        """Batched search with the level re-rank done on the GPU (ICD_WEIGHT_RERANK: raw top-k, score x w(level),
        stable re-sort -- milvus_service.py:290-314): returns (score [B,k] f32, raw [B,k] f32, ids [B,k] i64 GLOBAL
        row ids, -1 = no hit) as numpy arrays; scalar fields are fetched lazily through row() / field().  `filter` as
        in search(); limit <= 16 384."""
        col = self.cols[collection_name]
        if not col.loaded or col.index is None:
            raise N.NativeError(f"collection {collection_name} is not loaded")
        k, _, _, _ = self._page(limit)
        q = np.ascontiguousarray(np.asarray(queries, dtype=np.float32))
        if q.ndim == 1:
            q = q[None, :]
        mask = self._row_mask(col, filter)
        group = getattr(col, "group", None)
        if group is not None:
            self._group_refuses(k, 0, None, None)
            return group.search(q, k, weight_mode=N.WEIGHT_RERANK, mask=mask)
        score, raw, ids = col.index.search(q, k, weight_mode=N.WEIGHT_RERANK, mask=mask)
        if col.row_lo:
            ids = np.where(ids >= 0, ids + col.row_lo, ids)
        return score, raw, ids

    def _entities(self, col: _Collection, rows, output_fields: Optional[List[str]]) -> List[Dict[str, Any]]:
        fields = list(output_fields or [])
        if "*" in fields:
            fields = [f for f in fields if f != "*"] + [f for f in SCALAR_FIELDS if f not in fields]
        out = []
        for g in rows:
            row = col.rows.cached_row(int(g))
            ent = {"id": int(g)}
            for f in fields:
                if f != "id":
                    ent[f] = row.get(f)
            out.append(ent)
        return out

    def query(self, collection_name: str, filter: str = "", output_fields: Optional[List[str]] = None,
              ids=None, limit: Optional[int] = None, **_kw) -> List[Dict[str, Any]]:
        """MilvusClient.query: the rows (ascending id) that satisfy `filter` (and are among `ids` when given), as dicts
        {"id": row, <field>: value, ...} of output_fields ("*" = every scalar field).  Reads the column files, so a
        sharded client answers for every row of the collection."""
        col = self.cols[collection_name]
        n = len(col.rows)
        allowed = filter_expr.compile(filter).mask(col.rows, 0, n)
        if ids is not None:
            sel = np.zeros(n, bool)
            want = np.asarray([ids] if np.isscalar(ids) else list(ids), np.int64)
            sel[want[(want >= 0) & (want < n)]] = True
            allowed &= sel
        rows = np.nonzero(allowed)[0]
        if limit is not None:
            rows = rows[:max(0, int(limit))]
        return self._entities(col, rows, output_fields)

    def get(self, collection_name: str, ids, output_fields: Optional[List[str]] = None, **_kw) -> List[Dict[str, Any]]:
        """MilvusClient.get: the rows with these primary keys (row ids), in the order given; unknown ids are skipped."""
        col = self.cols[collection_name]
        n = len(col.rows)
        want = [ids] if np.isscalar(ids) else list(ids)
        return self._entities(col, [int(i) for i in want if 0 <= int(i) < n], output_fields)

    def row(self, collection_name: str, row_id: int) -> Dict[str, Any]:
        return self.cols[collection_name].rows[row_id]

    def field(self, collection_name: str, name: str, row_id: int):
        return self.cols[collection_name].rows.cached_row(int(row_id)).get(name)

    def close(self) -> None:
        self._masks.clear()
        for col in self.cols.values():
            if col.index is not None:
                col.index.close()
                col.index = None
            col.loaded = False
            col.rows.close()


def _level_byte(level) -> int:
    try:
        v = int(level)
    except Exception:
        return 0
    return v if 0 <= v <= 255 else 0
