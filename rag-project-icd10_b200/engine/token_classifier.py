"""TokenClassifierEngine -- the object MedicalNERService holds where the reference holds
``pipeline("ner", model=AutoModelForTokenClassification..., aggregation_strategy="simple")``
(/root/reference/services/medical_ner_service.py:76-90, called as ``self.ner_pipeline(text)`` at :182).

Same call shape and result layout -- a list of ``{"entity_group", "score", "word", "start", "end"}`` per
text -- with the BERT forward and the classifier head running in libicdrag.so on the GPU
(icd_encoder_set_token_head / icd_encoder_token_logits).  Tokenisation, the softmax over <= 64 labels and
the "simple" grouping of adjacent tokens stay on the host, as they do inside the transformers pipeline
(third party, transformers TokenClassificationPipeline: postprocess / gather_pre_entities / aggregate /
group_entities; restated here, checked against the pipeline itself in tests/test_ner_*.py).

Long texts.  The encoder takes sequences of up to 512 tokens (S <= 128 is one tile of the tensor-core attention kernel,
longer ones run it split over 128-key tiles with a combine pass, csrc/attention_tc.cu), so a model with a 512-token position table reads a text in ONE
pass truncated at 512 tokens, exactly like the reference pipeline.  When the window is shorter than the horizon (an
encoder built with a smaller max_seq_length), a text that does not fit is cut into overlapping windows (the
tokenizer's own overflow mechanism, `stride` tokens of overlap) that go through the GPU as one batch, and the windows'
entities are merged with the pipeline's rule for exactly this case (aggregate_overlapping_entities: of two
overlapping entities the longer wins, then the higher score) -- the algorithm of ``pipeline(..., stride=n)``.  Tokens
beyond the reference's 512-token horizon are dropped, as they are there.
"""
from __future__ import annotations

import json
import os
from typing import Dict, List, Optional, Sequence, Union

import numpy as np

from .. import _native as N
from . import weights as W
from .encoder import EncoderEngine, load_tokenizer


def _get_tag(entity_name: str):
    if entity_name.startswith("B-"):
        return "B", entity_name[2:]
    if entity_name.startswith("I-"):
        return "I", entity_name[2:]
    return "I", entity_name  # not in B-/I- format: continuation


def softmax_rows(logits: np.ndarray) -> np.ndarray:
    maxes = np.max(logits, axis=-1, keepdims=True)
    e = np.exp(logits - maxes)
    return e / e.sum(axis=-1, keepdims=True)


def merge_overlapping(entities: List[dict]) -> List[dict]:
    """transformers' aggregate_overlapping_entities: entities of all windows sorted by start; of two that overlap
    the longer one survives, at equal length the higher score."""
    if not entities:
        return entities
    entities = sorted(entities, key=lambda x: x["start"])
    out = []
    prev = entities[0]
    for ent in entities:
        if prev["start"] <= ent["start"] < prev["end"]:
            cur_len, prev_len = ent["end"] - ent["start"], prev["end"] - prev["start"]
            if cur_len > prev_len or (cur_len == prev_len and ent["score"] > prev["score"]):
                prev = ent
        else:
            out.append(prev)
            prev = ent
    out.append(prev)
    return out


def aggregate_simple(tokenizer, id2label: Dict[int, str], sentence: str, input_ids: Sequence[int],
                     scores: np.ndarray, offsets: Sequence[Sequence[int]], special_mask: Sequence[int],
                     ignore_labels=("O",)) -> List[dict]:
    """aggregation_strategy="simple": per token argmax label, adjacent tokens with the same tag (and no new
    "B-") merge into one group whose score is the mean of its tokens' scores."""
    entities = []
    for idx in range(len(input_ids)):
        if special_mask[idx]:
            continue
        word = tokenizer.convert_ids_to_tokens(int(input_ids[idx]))
        start, end = int(offsets[idx][0]), int(offsets[idx][1])
        if int(input_ids[idx]) == tokenizer.unk_token_id:
            word = sentence[start:end]
        k = int(scores[idx].argmax())
        entities.append({"entity": id2label[k], "score": scores[idx][k], "index": idx, "word": word,
                         "start": start, "end": end})
    groups, cur = [], []

    def flush():
        tag = cur[0]["entity"].split("-", 1)[-1]
        groups.append({"entity_group": tag, "score": np.mean(np.nanmean([e["score"] for e in cur])),
                       "word": tokenizer.convert_tokens_to_string([e["word"] for e in cur]),
                       "start": cur[0]["start"], "end": cur[-1]["end"]})

    for ent in entities:
        if not cur:
            cur.append(ent)
            continue
        bi, tag = _get_tag(ent["entity"])
        _, last_tag = _get_tag(cur[-1]["entity"])
        if tag == last_tag and bi != "B":
            cur.append(ent)
        else:
            flush()
            cur = [ent]
    if cur:
        flush()
    return [g for g in groups if g["entity_group"] not in ignore_labels]


class TokenClassifierEngine:
    """Callable like the reference's ``ner_pipeline``: ``engine(text)`` -> list of entity groups,
    ``engine([t1, t2, ...])`` -> list of lists (one GPU batch per length bucket)."""

    def __init__(self, model_name_or_path: Optional[str] = None, device: Union[str, int, None] = None, *,
                 encoder: Optional[EncoderEngine] = None, head_weight: Optional[np.ndarray] = None,
                 head_bias: Optional[np.ndarray] = None, id2label: Optional[Dict[int, str]] = None,
                 tokenizer=None, max_tokens: int = 1024 * 128, stride: int = 16, horizon: int = 512):
        if encoder is None:
            path = W.resolve_model_dir(model_name_or_path, allow_env_override=False)
            cfg, blob, _meta = W.load_model_dir(path)
            if _meta["position_offset"]:
                raise ValueError(f"{path}: token classification is served for BERT models only (XLM-RoBERTa position "
                                 "numbering is supported by the sentence encoder)")
            state = W.load_state(path)
            head_weight = np.asarray(state["classifier.weight"], np.float32)
            head_bias = np.asarray(state["classifier.bias"], np.float32)
            with open(os.path.join(path, "config.json"), encoding="utf-8") as fh:
                id2label = {int(k): v for k, v in json.load(fh).get("id2label", {}).items()}
            tokenizer = tokenizer or load_tokenizer(path)
            encoder = EncoderEngine(cfg=cfg, blob=blob, tokenizer=tokenizer, device=device,
                                    max_seq_length=min(512, cfg.max_position), max_tokens=max_tokens)
        if head_weight is None or head_bias is None:
            raise ValueError("a classifier head (weight, bias) is required")
        self.encoder = encoder
        self.tokenizer = tokenizer or encoder.tokenizer
        self.encoder.set_token_head(head_weight, head_bias)
        n = int(np.asarray(head_weight).shape[0])
        self.id2label = id2label or {i: f"LABEL_{i}" for i in range(n)}
        if len(self.id2label) != n:
            raise ValueError("id2label does not match the classifier head")
        self.max_seq_length = self.encoder.max_seq_length   # tokens per window (<= 512, the kernel limit)
        self.stride = int(stride)                            # overlap of the windows of a long text, in tokens
        self.horizon = int(horizon)                          # the reference pipeline truncates at model_max_length

    def __call__(self, inputs, **_ignored):
        single = isinstance(inputs, str)
        texts = [inputs] if single else list(inputs)
        out = self.extract(texts)
        return out[0] if single else out

    def extract(self, texts: Sequence[str]) -> List[List[dict]]:
        if not texts:
            return []
        enc = self.tokenizer(list(texts), padding=False, truncation=True, max_length=self.max_seq_length,
                             stride=self.stride, return_overflowing_tokens=True,
                             return_special_tokens_mask=True, return_offsets_mapping=True,
                             return_attention_mask=False, return_token_type_ids=False)
        ids = enc["input_ids"]                                   # one entry per WINDOW
        owner = enc["overflow_to_sample_mapping"]                # window -> text
        # windows that start beyond the reference's 512-token horizon are dropped (it never sees those tokens)
        step = max(1, self.max_seq_length - 2 - self.stride)
        seen, keep = {}, []
        for w, t in enumerate(owner):
            k = seen.get(t, 0)
            seen[t] = k + 1
            # a model that reads the whole horizon in one pass (max_seq_length >= 512) sees exactly the reference's
            # single truncated window; shorter windows tile the horizon with `stride` tokens of overlap
            if (k == 0) if self.max_seq_length >= self.horizon else (k * step < max(1, self.horizon - 2)):
                keep.append(w)
        per_window: Dict[int, List[dict]] = {}
        order = sorted(keep, key=lambda w: -len(ids[w]))
        lo = 0
        while lo < len(order):
            S = max(1, len(ids[order[lo]]))
            B = max(1, min(len(order) - lo, self.encoder.max_tokens // S))
            idx = order[lo:lo + B]
            mat = np.zeros((B, S), np.int32)
            lens = np.zeros((B,), np.int32)
            for r, w in enumerate(idx):
                mat[r, :len(ids[w])] = ids[w]
                lens[r] = len(ids[w])
            logits = self.encoder.token_logits(mat, lens)
            for r, w in enumerate(idx):
                n = int(lens[r])
                scores = softmax_rows(logits[r, :n].astype(np.float32))
                per_window[w] = aggregate_simple(self.tokenizer, self.id2label, texts[owner[w]], ids[w], scores,
                                                 enc["offset_mapping"][w], enc["special_tokens_mask"][w])
            lo += B
        results: List[List[dict]] = [[] for _ in texts]
        windows_of: Dict[int, int] = {}
        for w in keep:
            results[owner[w]].extend(per_window[w])
            windows_of[owner[w]] = windows_of.get(owner[w], 0) + 1
        for t, n_win in windows_of.items():
            if n_win > 1:
                results[t] = merge_overlapping(results[t])
        return results

    def close(self) -> None:
        self.encoder.close()
