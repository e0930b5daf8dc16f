"""MilvusService -- drop-in mirror of /root/reference/services/milvus_service.py.

Same class name, methods, arguments, return shapes and error behaviour (search never raises
and degrades to [], insert_records raises ValueError on a length mismatch and otherwise
returns bool, ...).  ``self.client`` is engine.store.IcdStoreClient -- a device-resident exact
inner-product table searched by libicdrag.so -- where the reference holds a
pymilvus.MilvusClient over Milvus Lite FLAT/IP.
"""
from __future__ import annotations

import datetime
import os
from typing import Any, Dict, List

import numpy as np

try:
    from loguru import logger
except Exception:  # pragma: no cover
    import logging
    logger = logging.getLogger("icd10_b200")

from ..engine.store import DataType, IcdStoreClient

MilvusClient = IcdStoreClient  # the name the reference constructs (milvus_service.py:81,110)


class LazyCandidates:
    """What MilvusService.search returns for one query -- a list of candidate dicts in the reference's order -- with
    the dicts built on access.  Compares equal to the list; ``list(x)`` materialises it."""

    def __init__(self, service, raw, ids, trimmed: bool = False):
        if not trimmed:
            keep = ids >= 0
            raw, ids = raw[keep], ids[keep]
        self._svc, self._raw, self._ids = service, raw, ids
        self._cache: Dict[int, Dict[str, Any]] = {}

    def __len__(self) -> int:
        return int(self._ids.shape[0])

    def _one(self, i: int) -> Dict[str, Any]:
        if i not in self._cache:
            self._cache[i] = self._svc._candidate_of_row(int(self._ids[i]), float(self._raw[i]))
        return self._cache[i]

    def __getitem__(self, i):
        if isinstance(i, slice):
            return [self._one(j) for j in range(*i.indices(len(self)))]
        n = len(self)
        if i < 0:
            i += n
        if not 0 <= i < n:
            raise IndexError(i)
        return self._one(i)

    def __iter__(self):
        return (self._one(i) for i in range(len(self)))

    def __eq__(self, other):
        return list(self) == list(other)

    def __repr__(self) -> str:
        return repr(list(self))

    @property
    def row_ids(self):
        return self._ids

    @property
    def raw_scores(self):
        return self._raw


class LazyBatch:
    """What MilvusService.search_batch returns: a read-only sequence whose element b is the LazyCandidates of query b,
    created on access from the [B, k] result arrays (10 000 queries used to cost 20 ms of per-query numpy slicing
    before anything was read; missing hits are -1 at the tail of a row, counted once for the whole batch)."""

    def __init__(self, service, raw, ids):
        self._svc, self._raw, self._ids = service, raw, ids
        self._n = (ids >= 0).sum(axis=1)
        self._rows: Dict[int, LazyCandidates] = {}

    def __len__(self) -> int:
        return int(self._ids.shape[0])

    def _one(self, b: int) -> LazyCandidates:
        row = self._rows.get(b)
        if row is None:
            n = int(self._n[b])
            row = self._rows[b] = LazyCandidates(self._svc, self._raw[b, :n], self._ids[b, :n], trimmed=True)
        return row

    def __getitem__(self, b):
        if isinstance(b, slice):
            return [self._one(j) for j in range(*b.indices(len(self)))]
        n = len(self)
        if b < 0:
            b += n
        if not 0 <= b < n:
            raise IndexError(b)
        return self._one(b)

    def __iter__(self):
        return (self._one(b) for b in range(len(self)))

    def __eq__(self, other):
        return len(self) == len(other) and all(a == b for a, b in zip(self, other))

    def __repr__(self) -> str:
        return f"LazyBatch({len(self)} queries)"

    @property
    def row_ids(self):
        """[B, k] int64 global row ids in the reference's order (-1 = no hit)."""
        return self._ids

    @property
    def raw_scores(self):
        return self._raw


_OUTPUT_FIELDS = ["code", "preferred_zh", "has_complication", "main_code", "secondary_code", "level",
                  "parent_code", "category_path", "semantic_text"]
_LEVEL_WEIGHTS = {1: 1.2, 2: 1.0, 3: 0.8}  # reference :550-558


class MilvusService:
    # extra keyword arguments for the store client: device=<gpu index>, shard=(rank, world) when one process per GPU
    # serves a row shard each (set by tools/build_database.py under torchrun); empty for the reference's single process
    client_kwargs: Dict[str, Any] = {}

    def __init__(self, embedding_service=None):
        self.config = self._load_config()
        self.collection_name = self.config.get("milvus", {}).get("collection_name", "icd10")
        self.embedding_service = embedding_service
        self.dimension = self._get_vector_dimension()
        self.client = None
        self._connect()
        self._setup_collection()

    # reference :21-37
    def _load_config(self) -> Dict[str, Any]:
        env = os.getenv
        return {"milvus": {
            "mode": env("MILVUS_MODE", "local"),
            "host": env("MILVUS_HOST", "localhost"),
            "port": int(env("MILVUS_PORT", "19530")),
            "username": env("MILVUS_USERNAME", ""),
            "password": env("MILVUS_PASSWORD", ""),
            "db_name": env("MILVUS_DB_NAME", "default"),
            "db_path": env("MILVUS_DB_PATH", "./db/milvus_icd10.db"),
            "collection_name": env("MILVUS_COLLECTION_NAME", "icd10"),
            "index_type": "FLAT",
            "metric_type": "IP",
            "secure": env("MILVUS_SECURE", "false").lower() == "true",
        }}

    # reference :39-55
    def _get_vector_dimension(self) -> int:
        if self.embedding_service:
            try:
                dim = len(self.embedding_service.encode_query("测试文本"))
                logger.info(f"从嵌入模型获取向量维度: {dim}")
                return dim
            except Exception as e:
                logger.warning(f"无法从嵌入服务获取维度: {e}")
        logger.warning("使用默认向量维度: 1024")
        return 1024

    # reference :57-118
    def _connect(self):
        cfg = self.config.get("milvus", {})
        mode = cfg.get("mode", "local")
        try:
            if getattr(self, "client", None):
                try:
                    self.client.close()
                except Exception:
                    pass
            if mode == "local":
                db_path = cfg.get("db_path", "./db/milvus_icd10.db")
                db_dir = os.path.dirname(db_path)
                if db_dir and not os.path.exists(db_dir):
                    os.makedirs(db_dir, exist_ok=True)
                    logger.info(f"创建数据库目录: {db_dir}")
                self.client = MilvusClient(uri=db_path, **type(self).client_kwargs)
                logger.info(f"成功连接到本地向量库: {db_path}")
            elif mode == "remote":
                # a remote Milvus server is outside this engine: the table lives in this process's HBM
                raise ValueError("MILVUS_MODE=remote is not served by the B200 engine; use 'local'")
            else:
                raise ValueError(f"不支持的Milvus模式: {mode}，请使用 'local' 或 'remote'")
        except Exception as e:
            logger.error(f"Milvus连接失败 (模式: {mode}): {e}")
            raise

    # reference :120-161
    def _setup_collection(self):
        try:
            if self.client.has_collection(collection_name=self.collection_name):
                logger.info(f"集合 {self.collection_name} 已存在")
            else:
                logger.info(f"集合 {self.collection_name} 不存在，创建新集合")
                self._create_collection()
            self._load_collection_to_memory()
        except Exception as e:
            logger.error(f"设置集合失败: {e}")
            raise

    def _load_collection_to_memory(self):
        try:
            if self.client.get_load_state(collection_name=self.collection_name) == "Loaded":
                logger.info(f"✅ 集合 {self.collection_name} 已经在内存中")
                return
            logger.info(f"📤 正在加载集合 {self.collection_name} 到内存...")
            self.client.load_collection(collection_name=self.collection_name)
            state = self.client.get_load_state(collection_name=self.collection_name)
            if state == "Loaded":
                logger.info(f"✅ 集合 {self.collection_name} 已成功加载到内存")
            else:
                logger.warning(f"⚠️  集合 {self.collection_name} 加载状态: {state}")
        except Exception as e:
            logger.error(f"❌ 加载集合到内存失败: {e}")
            raise

    # reference :163-206 -- same schema, FLAT / IP
    def _create_collection(self):
        logger.info(f"创建新集合: {self.collection_name}")
        try:
            schema = self.client.create_schema(enable_dynamic_field=True)
            schema.add_field(field_name="id", datatype=DataType.INT64, is_primary=True, auto_id=True)
            schema.add_field(field_name="vector", datatype=DataType.FLOAT_VECTOR, dim=self.dimension)
            for name, length in (("code", 50), ("preferred_zh", 500)):
                schema.add_field(field_name=name, datatype=DataType.VARCHAR, max_length=length)
            schema.add_field(field_name="has_complication", datatype=DataType.BOOL)
            for name in ("main_code", "secondary_code"):
                schema.add_field(field_name=name, datatype=DataType.VARCHAR, max_length=50)
            schema.add_field(field_name="level", datatype=DataType.INT32)
            for name, length in (("parent_code", 50), ("category_path", 200), ("semantic_text", 1000)):
                schema.add_field(field_name=name, datatype=DataType.VARCHAR, max_length=length)
            index_params = self.client.prepare_index_params()
            index_params.add_index(field_name="vector",
                                   index_type=self.config.get("milvus", {}).get("index_type", "FLAT"),
                                   metric_type=self.config.get("milvus", {}).get("metric_type", "IP"))
            self.client.create_collection(collection_name=self.collection_name, schema=schema,
                                          index_params=index_params)
            logger.info("集合创建完成")
        except Exception as e:
            logger.error(f"创建集合失败: {e}")
            raise

    # reference :208-269
    def insert_records(self, records: List[Dict[str, Any]], embeddings: List[np.ndarray]) -> bool:
        if len(records) != len(embeddings):
            raise ValueError("记录数量与向量数量不匹配")
        logger.info(f"准备插入 {len(records)} 条记录到集合 {self.collection_name}")
        try:
            data = []
            for rec, vec in zip(records, embeddings):
                main_code = rec.get("main_code")
                secondary = rec.get("secondary_code")
                data.append({
                    "vector": vec.tolist(),     # a plain list raises here, as in the reference (:231)
                    "code": rec["code"],
                    "preferred_zh": rec.get("preferred_zh", ""),
                    "has_complication": rec.get("has_complication", False),
                    "main_code": "" if main_code is None else main_code,
                    "secondary_code": "" if secondary is None else secondary,
                    "level": rec.get("level", 1),
                    "parent_code": rec.get("parent_code", ""),
                    "category_path": rec.get("category_path", ""),
                    "semantic_text": rec.get("semantic_text", ""),
                })
            filled: Dict[str, int] = {}
            for row in data:
                for name, value in row.items():
                    filled.setdefault(name, 0)
                    if value is not None and value != "":
                        filled[name] += 1
            logger.info(f"字段数据统计: {filled}")
            self.client.insert(collection_name=self.collection_name, data=data)
            logger.info(f"成功插入 {len(records)} 条记录")
            return True
        except Exception as e:
            logger.error(f"插入记录失败: {e}")
            return False

    # reference :271-320
    # extension: `filter` -- a Milvus boolean expression over the scalar fields (e.g. 'code like "J%"', 'level == 3'),
    # applied inside the scan (exact top_k over the matching rows); an invalid expression is logged and gives []
    def search(self, query_vector: np.ndarray, top_k: int = 10, filter: str = "") -> List[Dict[str, Any]]:
        try:
            if not self.client.has_collection(collection_name=self.collection_name):
                logger.error(f"集合 {self.collection_name} 不存在")
                return []
            results = self.client.search(collection_name=self.collection_name, data=[query_vector.tolist()],
                                         limit=top_k, output_fields=_OUTPUT_FIELDS, filter=filter)
            candidates = []
            if results and len(results) > 0:
                candidates = [self._candidate(hit) for hit in results[0]]
                candidates.sort(key=lambda c: c["score"], reverse=True)
            return candidates
        except Exception as e:
            logger.error(f"搜索失败: {e}")
            return []

    def _candidate(self, hit) -> Dict[str, Any]:
        """One hit -> the reference's candidate dict (milvus_service.py:290-311)."""
        base = float(hit.get("distance", 0))
        level = hit.get("level", 1)
        adjusted = float(base * self._calculate_level_weight(level))
        return {
            "code": hit.get("code"),
            "title": hit.get("preferred_zh"),
            "score": float(adjusted),
            "original_score": float(base),
            "metadata": {
                "has_complication": hit.get("has_complication", False),
                "main_code": hit.get("main_code", ""),
                "secondary_code": hit.get("secondary_code", ""),
                "level": level,
                "parent_code": hit.get("parent_code", ""),
                "category_path": hit.get("category_path", ""),
                "semantic_text": hit.get("semantic_text", ""),
            },
        }

    # extension (SURVEY 8f-1): all diagnoses of a request in ONE scan launch, level re-rank on the GPU
    # (ICD_WEIGHT_RERANK == the sort at :314).  Element b is what search(query_vectors[b], top_k) returns; the hit
    # dicts are built lazily, on access, from the mapped columns -- 10 000 queries do not cost 100 000 dicts up front.
    def search_batch(self, query_vectors, top_k: int = 10, filter: str = "") -> "LazyBatch":
        try:
            if not self.client.has_collection(collection_name=self.collection_name):
                logger.error(f"集合 {self.collection_name} 不存在")
                return []
            q = np.asarray(query_vectors, dtype=np.float32)
            if q.ndim == 1:
                q = q[None, :]
            _score, raw, ids = self.client.search_ranked(self.collection_name, q, top_k, filter=filter)
            return LazyBatch(self, raw, ids)
        except Exception as e:
            logger.error(f"搜索失败: {e}")
            return []

    def _candidate_of_row(self, row_id: int, distance: float) -> Dict[str, Any]:
        """The candidate dict of one (row, raw inner product): same arithmetic as _candidate (Python floats)."""
        f = lambda name: self.client.field(self.collection_name, name, row_id)   # noqa: E731
        level = f("level")
        base = float(distance)
        return {
            "code": f("code"),
            "title": f("preferred_zh"),
            "score": float(base * self._calculate_level_weight(level)),
            "original_score": float(base),
            "metadata": {
                "has_complication": f("has_complication"),
                "main_code": f("main_code"),
                "secondary_code": f("secondary_code"),
                "level": level,
                "parent_code": f("parent_code"),
                "category_path": f("category_path"),
                "semantic_text": f("semantic_text"),
            },
        }

    @staticmethod
    def _row_of_record(rec: Dict[str, Any]) -> Dict[str, Any]:
        """The scalar fields insert_records stores for one record (reference :233-244: None codes become '')."""
        main_code, secondary = rec.get("main_code"), rec.get("secondary_code")
        return {
            "code": rec["code"],
            "preferred_zh": rec.get("preferred_zh", ""),
            "has_complication": rec.get("has_complication", False),
            "main_code": "" if main_code is None else main_code,
            "secondary_code": "" if secondary is None else secondary,
            "level": rec.get("level", 1),
            "parent_code": rec.get("parent_code", ""),
            "category_path": rec.get("category_path", ""),
            "semantic_text": rec.get("semantic_text", ""),
        }

    # extension (SURVEY 8e / 8a-P): the build path hands over one [n, dim] float32 array (numpy, or a torch tensor
    # still on the GPU) instead of n Python lists; same validation and bool result as insert_records
    def insert_records_array(self, records: List[Dict[str, Any]], vectors) -> bool:
        if len(records) != int(vectors.shape[0]):
            raise ValueError("记录数量与向量数量不匹配")
        logger.info(f"准备插入 {len(records)} 条记录到集合 {self.collection_name}")
        try:
            rows = [self._row_of_record(rec) for rec in records]
            self.client.insert_arrays(self.collection_name, rows, vectors)
            logger.info(f"成功插入 {len(records)} 条记录")
            return True
        except Exception as e:
            logger.error(f"插入记录失败: {e}")
            return False

    # reference :322-342
    def get_collection_stats(self) -> Dict[str, Any]:
        try:
            stats = {
                "collection_name": self.collection_name,
                "exists": self.client.has_collection(collection_name=self.collection_name),
                "dimension": self.dimension,
            }
            if stats["exists"]:
                stats["num_entities"] = self.client.get_collection_stats(
                    collection_name=self.collection_name).get("row_count", 0)
            else:
                stats["num_entities"] = 0
            return stats
        except Exception as e:
            logger.error(f"获取统计信息失败: {e}")
            return {"error": str(e)}

    # reference :344-357
    def load_collection(self) -> bool:
        try:
            if not self.client.has_collection(collection_name=self.collection_name):
                logger.error(f"集合 {self.collection_name} 不存在")
                return False
            self.client.load_collection(collection_name=self.collection_name)
            logger.info(f"集合 {self.collection_name} 已加载到内存")
            return True
        except Exception as e:
            logger.error(f"加载集合失败: {e}")
            return False

    # reference :359-371
    def clear_collection(self) -> bool:
        try:
            if self.client.has_collection(collection_name=self.collection_name):
                self.client.drop_collection(collection_name=self.collection_name)
                logger.info(f"集合 {self.collection_name} 已删除")
            self._setup_collection()
            return True
        except Exception as e:
            logger.error(f"清空集合失败: {e}")
            return False

    # reference :373-409
    def test_connection(self) -> Dict[str, Any]:
        mode = self.config.get("milvus", {}).get("mode", "local")
        try:
            info = {"connected": True, "mode": mode, "collection_stats": self.get_collection_stats(),
                    "client_type": "MilvusClient"}
            cfg = self.config.get("milvus", {})
            if mode == "remote":
                info["remote_info"] = {"host": cfg.get("host"), "port": cfg.get("port"),
                                       "db_name": cfg.get("db_name"), "secure": cfg.get("secure")}
            else:
                info["local_info"] = {"db_path": cfg.get("db_path")}
            return info
        except Exception as e:
            logger.error(f"连接测试失败: {e}")
            return {"connected": False, "error": str(e), "mode": mode}

    # reference :411-435
    def release_collection(self) -> Dict[str, Any]:
        try:
            if not self.client:
                return {"success": False, "message": "客户端未连接"}
            if not self.client.has_collection(collection_name=self.collection_name):
                return {"success": False, "message": f"集合 {self.collection_name} 不存在"}
            self.client.release_collection(collection_name=self.collection_name)
            logger.info(f"✅ 集合 {self.collection_name} 内存已释放")
            return {"success": True, "message": f"集合 {self.collection_name} 内存已释放",
                    "collection_name": self.collection_name}
        except Exception as e:
            msg = f"释放集合内存失败: {e}"
            logger.error(msg)
            return {"success": False, "message": msg}

    # reference :437-459
    def get_collection_load_state(self) -> Dict[str, Any]:
        try:
            if not self.client:
                return {"loaded": False, "message": "客户端未连接"}
            if not self.client.has_collection(collection_name=self.collection_name):
                return {"loaded": False, "message": f"集合 {self.collection_name} 不存在"}
            state = self.client.get_load_state(collection_name=self.collection_name)
            return {"loaded": state == "Loaded", "state": state, "collection_name": self.collection_name}
        except Exception as e:
            msg = f"获取集合加载状态失败: {e}"
            logger.warning(msg)
            return {"loaded": False, "message": msg}

    # reference :461-497
    def disconnect(self) -> Dict[str, Any]:
        try:
            if not self.client:
                return {"success": True, "message": "客户端已经断开"}
            released = self.release_collection()
            try:
                if hasattr(self.client, "close"):
                    self.client.close()
                self.client = None
                logger.info("🔌 Milvus客户端连接已断开")
                return {"success": True, "message": "Milvus连接已断开，资源已清理", "release_result": released}
            except Exception as close_err:
                logger.warning(f"关闭Milvus客户端时出错: {close_err}")
                self.client = None
                return {"success": True, "message": "连接已断开（可能有警告）", "warning": str(close_err)}
        except Exception as e:
            msg = f"断开Milvus连接失败: {e}"
            logger.error(msg)
            return {"success": False, "message": msg}

    # reference :499-523
    def get_memory_usage(self) -> Dict[str, Any]:
        try:
            if not self.client:
                return {"memory_usage": 0, "message": "客户端未连接"}
            if not self.client.has_collection(collection_name=self.collection_name):
                return {"memory_usage": 0, "message": f"集合 {self.collection_name} 不存在"}
            stats = self.get_collection_stats()
            state = self.get_collection_load_state()
            return {
                "collection_name": self.collection_name,
                "loaded": state.get("loaded", False),
                "load_state": state.get("state", "Unknown"),
                "num_entities": stats.get("num_entities", 0),
                "estimated_memory_mb": stats.get("num_entities", 0) * self.dimension * 4 / (1024 * 1024),
                "message": "内存使用为估算值（基于向量维度和实体数量）",
            }
        except Exception as e:
            msg = f"获取内存使用情况失败: {e}"
            logger.warning(msg)
            return {"memory_usage": 0, "message": msg}

    # reference :525-548
    def health_check(self) -> Dict[str, Any]:
        try:
            conn = self.test_connection()
            state = self.get_collection_load_state()
            mem = self.get_memory_usage()
            return {"healthy": conn.get("connected", False) and state.get("loaded", False), "connection": conn,
                    "load_state": state, "memory_usage": mem, "timestamp": datetime.datetime.now().isoformat()}
        except Exception as e:
            return {"healthy": False, "error": str(e), "timestamp": datetime.datetime.now().isoformat()}

    def _calculate_level_weight(self, level: int) -> float:
        return _LEVEL_WEIGHTS.get(level, 1.0)
