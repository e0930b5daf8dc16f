"""Weight blob for icd_encoder_create: HF BertModel tensors flattened to fp32 in the canonical
order documented in csrc/api_encoder.cu.  Loads an HF / sentence-transformers model directory
(config.json + model.safetensors | pytorch_model.bin + vocab.txt | tokenizer.json), the layout
SentenceTransformer(model_name) resolves in the reference (services/embedding_service.py:61).

Two encoder shapes are served: hidden 768 with 12 heads (BERT-base, text2vec-base-chinese) and hidden 1024 with 16
heads (BERT-large, XLM-RoBERTa-large: intfloat/multilingual-e5-large(-instruct), the reference's code default).
XLMRobertaModel has BertModel's tensors and arithmetic; it differs in two embedding conventions, which `meta` carries:
positions of real tokens start at pad_token_id + 1, and <unk> is id 3.
"""
from __future__ import annotations

import json
import os
from typing import Dict, Optional, Tuple

import numpy as np

from .. import _native as N


MODEL_TYPES = ("bert", "xlm-roberta")
SHAPES = {768: 12, 1024: 16}      # hidden size -> attention heads (head dim 64)


def config_from_dict(cfg: dict) -> N.BertCfg:
    mt = cfg.get("model_type", "bert")
    if mt not in MODEL_TYPES:
        raise ValueError(f"model_type {mt!r} is not supported: BERT and XLM-RoBERTa encoders only (hidden 768 / 12 heads "
                         "or 1024 / 16 heads)")
    if cfg.get("hidden_act", "gelu") != "gelu":
        raise ValueError("only erf-GELU ('gelu') is supported")
    if cfg.get("position_embedding_type", "absolute") != "absolute":
        raise ValueError("only absolute position embeddings are supported")
    hidden, heads = int(cfg["hidden_size"]), int(cfg["num_attention_heads"])
    if heads * 64 != hidden:
        raise ValueError(f"head dim must be 64: hidden {hidden} with {heads} heads is not supported (supported shapes: "
                         "hidden 768 with 12 heads, hidden 1024 with 16 heads)")
    if hidden not in SHAPES:
        raise ValueError(f"hidden size {hidden} is not supported (supported shapes: hidden 768 with 12 heads, hidden 1024 "
                         "with 16 heads)")
    return N.BertCfg(vocab_size=int(cfg["vocab_size"]), hidden=int(cfg["hidden_size"]),
                     layers=int(cfg["num_hidden_layers"]), heads=int(cfg["num_attention_heads"]),
                     intermediate=int(cfg["intermediate_size"]), max_position=int(cfg["max_position_embeddings"]),
                     type_vocab=int(cfg.get("type_vocab_size", 2)), ln_eps=float(cfg.get("layer_norm_eps", 1e-12)))


def tensor_order(layers: int):
    names = ["embeddings.word_embeddings.weight", "embeddings.position_embeddings.weight",
             "embeddings.token_type_embeddings.weight", "embeddings.LayerNorm.weight", "embeddings.LayerNorm.bias"]
    for l in range(layers):
        p = f"encoder.layer.{l}."
        names += [p + "attention.self.query.weight", p + "attention.self.key.weight", p + "attention.self.value.weight",
                  p + "attention.self.query.bias", p + "attention.self.key.bias", p + "attention.self.value.bias",
                  p + "attention.output.dense.weight", p + "attention.output.dense.bias",
                  p + "attention.output.LayerNorm.weight", p + "attention.output.LayerNorm.bias",
                  p + "intermediate.dense.weight", p + "intermediate.dense.bias",
                  p + "output.dense.weight", p + "output.dense.bias",
                  p + "output.LayerNorm.weight", p + "output.LayerNorm.bias"]
    return names


def pack_state_dict(state: Dict[str, "np.ndarray"], cfg: N.BertCfg) -> np.ndarray:
    """state: name -> array-like (torch tensors accepted); names may carry a 'bert.', 'roberta.' or '0.auto_model.'
    prefix."""
    def get(name):
        for cand in (name, "bert." + name, "roberta." + name, "0.auto_model." + name):
            if cand in state:
                t = state[cand]
                if hasattr(t, "detach"):
                    t = t.detach().float().cpu().numpy()
                return np.ascontiguousarray(t, dtype=np.float32).reshape(-1)
        raise KeyError(f"missing tensor {name}")
    parts = [get(n) for n in tensor_order(cfg.layers)]
    blob = np.concatenate(parts)
    want = int(N.lib().icd_encoder_weight_count(cfg)) if os.path.exists(N.LIB_PATH) else blob.size
    if blob.size != want:
        raise ValueError(f"weight blob has {blob.size} values, the config needs {want}")
    return blob


def resolve_model_dir(name_or_path: str, allow_env_override: bool = True) -> str:
    """A directory, $ICD_B200_MODEL_DIR (the EMBEDDING model's directory: callers loading any other model pass
    allow_env_override=False), or an entry of the local HF cache (no network)."""
    env = os.environ.get("ICD_B200_MODEL_DIR") if allow_env_override else None
    for cand in (name_or_path, env):
        if cand and os.path.isdir(cand) and os.path.exists(os.path.join(cand, "config.json")):
            return cand
    try:
        from huggingface_hub import snapshot_download
        return snapshot_download(name_or_path, local_files_only=True)
    except Exception as e:
        raise FileNotFoundError(
            f"model '{name_or_path}' is not a local directory and not in the local HF cache "
            f"(set ICD_B200_MODEL_DIR to a directory with config.json, model.safetensors, vocab.txt)") from e


def load_state(path: str) -> dict:
    """name -> tensor of an HF model directory (model.safetensors, else pytorch_model.bin)."""
    st = os.path.join(path, "model.safetensors")
    if os.path.exists(st):
        from safetensors.numpy import load_file
        return load_file(st)
    import torch
    state = torch.load(os.path.join(path, "pytorch_model.bin"), map_location="cpu", weights_only=True)
    return {k: v.float().numpy() for k, v in state.items()}


def position_offset(cfg: dict) -> int:
    """First position row of a sequence's real tokens: XLM-R numbers them from pad_token_id + 1 (create_position_ids_
    from_input_ids on a right-padded batch), BERT from 0."""
    if cfg.get("model_type", "bert") == "xlm-roberta":
        return int(cfg.get("pad_token_id", 1)) + 1
    return 0


def unk_id(path: str) -> Optional[int]:
    """The unknown-token id of the directory's tokenizer (tokenizer.json, else vocab.txt); None if neither says."""
    tj = os.path.join(path, "tokenizer.json")
    if os.path.exists(tj):
        with open(tj, encoding="utf-8") as fh:
            model = json.load(fh).get("model") or {}
        if model.get("type") == "Unigram" and model.get("unk_id") is not None:
            return int(model["unk_id"])
        vocab = model.get("vocab")
        if isinstance(vocab, dict) and model.get("unk_token") in vocab:
            return int(vocab[model["unk_token"]])
    vt = os.path.join(path, "vocab.txt")
    if os.path.exists(vt):
        with open(vt, encoding="utf-8") as fh:
            for i, line in enumerate(fh):
                if line.rstrip("\n") == "[UNK]":
                    return i
    return None


def load_model_dir(path: str) -> Tuple[N.BertCfg, np.ndarray, dict]:
    """(config, weight blob, meta); meta: max_seq_length, do_lower_case_text, pooling, position_offset, unk_id (None:
    the library's default rule)."""
    with open(os.path.join(path, "config.json"), encoding="utf-8") as fh:
        cfg_d = json.load(fh)
    cfg = config_from_dict(cfg_d)
    state = load_state(path)
    meta = {"max_seq_length": 128, "do_lower_case_text": False, "pooling": "mean",
            "position_offset": position_offset(cfg_d), "unk_id": unk_id(path)}
    sb = os.path.join(path, "sentence_bert_config.json")
    if os.path.exists(sb):
        with open(sb, encoding="utf-8") as fh:
            d = json.load(fh)
        meta["max_seq_length"] = int(d.get("max_seq_length", 128))
        meta["do_lower_case_text"] = bool(d.get("do_lower_case", False))
    # sentence-transformers pooling module (1_Pooling/config.json): this engine implements masked MEAN pooling only
    # (text2vec-base-chinese); a CLS- or max-pooled model would silently produce different embeddings
    pool = os.path.join(path, "1_Pooling", "config.json")
    if os.path.exists(pool):
        with open(pool, encoding="utf-8") as fh:
            pc = json.load(fh)
        modes = [k for k, v in pc.items() if k.startswith("pooling_mode_") and v is True]
        if modes != ["pooling_mode_mean_tokens"]:
            raise ValueError(f"{path}: pooling modes {modes} are not supported (masked mean pooling only, as in "
                             "shibing624/text2vec-base-chinese)")
    if meta["do_lower_case_text"]:
        raise ValueError(f"{path}: sentence_bert_config.json asks for text lower-casing before tokenisation, which this "
                         "engine does not apply")
    if meta["max_seq_length"] > 512:
        raise ValueError(f"{path}: max_seq_length {meta['max_seq_length']} exceeds this engine's 512-token limit")
    return cfg, pack_state_dict(state, cfg), meta
