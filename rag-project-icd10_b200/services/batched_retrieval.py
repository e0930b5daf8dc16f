"""Batched serve path (SURVEY 8f-1): the retrieval step of a whole request in one encoder pass and one scan.

The reference retrieves per extracted diagnosis, one after the other
(/root/reference/services/multi_diagnosis_service.py:98-103 loop; :152-153 ``encode_query`` then
``milvus_service.search(query_vector, top_k * 2)``; :156-158 hierarchical re-scoring): n batch-1 encoder forwards and
n single-query scans per request.  ``retrieve`` does the same work as 1 encode + 1 scan; element i of its result is
what the reference's two calls return for diagnoses[i].
"""
from __future__ import annotations

from typing import Any, Dict, List, Optional, Sequence


class BatchedRetrieval:
    def __init__(self, embedding_service, milvus_service, hierarchical_similarity=None):
        self.embedding_service = embedding_service
        self.milvus_service = milvus_service
        self.hierarchical_similarity = hierarchical_similarity

    def retrieve(self, diagnoses: Sequence[str], top_k: int = 10, filter: str = "") -> List[List[Dict[str, Any]]]:
        """base_search_results of every diagnosis (multi_diagnosis_service.py:152-153, limit top_k * 2); `filter` restricts
        every diagnosis's candidates to the rows a scalar expression allows (MilvusService.search_batch)."""
        diagnoses = list(diagnoses)
        if not diagnoses:
            return []
        vectors = self.embedding_service.encode_queries(diagnoses)
        if filter:
            return self.milvus_service.search_batch(vectors, top_k * 2, filter=filter)
        return self.milvus_service.search_batch(vectors, top_k * 2)

    def retrieve_enhanced(self, diagnoses: Sequence[str], query_entities: Sequence[Dict[str, Any]], top_k: int = 10):
        """...followed by the hierarchical re-scoring of every candidate list (:156-158), cut to top_k (:162)."""
        if self.hierarchical_similarity is None:
            raise RuntimeError("no hierarchical similarity service")
        base = [list(c) for c in self.retrieve(diagnoses, top_k)]
        many = getattr(self.hierarchical_similarity, "batch_calculate_similarities_many", None)
        if many is not None:
            enhanced = many(list(zip(diagnoses, query_entities, base)))
        else:
            enhanced = [self.hierarchical_similarity.batch_calculate_similarities(d, e, b)
                        for d, e, b in zip(diagnoses, query_entities, base)]
        return [e[:top_k] for e in enhanced]
