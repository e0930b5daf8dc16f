"""Synthetic 1024-wide encoders for the tests and profiles: an XLM-RoBERTa-large-shaped model in the layout of
intfloat/multilingual-e5-large(-instruct) (config.json, model.safetensors, a SentencePiece-Unigram tokenizer.json,
sentence_bert_config.json, 1_Pooling/config.json in mean mode), built offline from a seed, and the fp32 reference the
engine stands in for: transformers XLMRobertaModel / BertModel -> masked mean -> L2 normalise.  Test infrastructure only.
"""
import json
import os
from typing import Dict, Sequence

import numpy as np
import torch

SPECIALS = ["<s>", "<pad>", "</s>", "<unk>"]       # XLM-R ids 0..3: pad_token_id = 1, unk = 3
PAD_ID, UNK_ID = 1, 3


def xlmr_config(layers=4, vocab_size=4000, hidden=1024, heads=16, intermediate=4096, max_position=514):
    from transformers import XLMRobertaConfig
    return XLMRobertaConfig(vocab_size=vocab_size, hidden_size=hidden, num_hidden_layers=layers,
                            num_attention_heads=heads, intermediate_size=intermediate, hidden_act="gelu",
                            max_position_embeddings=max_position, type_vocab_size=1, layer_norm_eps=1e-5,
                            pad_token_id=PAD_ID, bos_token_id=0, eos_token_id=2, hidden_dropout_prob=0.0,
                            attention_probs_dropout_prob=0.0)


def bert_large_config(layers=4, vocab_size=4000, max_position=512):
    from transformers import BertConfig
    return BertConfig(vocab_size=vocab_size, hidden_size=1024, num_hidden_layers=layers, num_attention_heads=16,
                      intermediate_size=4096, hidden_act="gelu", max_position_embeddings=max_position, type_vocab_size=2,
                      layer_norm_eps=1e-12, hidden_dropout_prob=0.0, attention_probs_dropout_prob=0.0)


def _model(cfg):
    from transformers import BertModel, XLMRobertaModel
    cls = XLMRobertaModel if cfg.model_type == "xlm-roberta" else BertModel
    return cls(cfg, add_pooling_layer=False)


def state_dict(cfg, seed=0) -> Dict[str, torch.Tensor]:
    """Seeded HF-named fp32 weights (HF init), LayerNorm gains / offsets and biases perturbed so every fused epilogue
    is exercised (as oracle.encoder.synthetic_state_dict does for BERT-base)."""
    torch.manual_seed(seed)
    model = _model(cfg)
    g = torch.Generator().manual_seed(seed + 1)
    sd = {}
    for name, p in model.state_dict().items():
        t = p.detach().clone().float()
        if name.endswith("LayerNorm.weight"):
            t = 1.0 + 0.1 * torch.randn(t.shape, generator=g)
        elif name.endswith("LayerNorm.bias") or name.endswith(".bias"):
            t = 0.05 * torch.randn(t.shape, generator=g)
        sd[name] = t.contiguous()
    return sd


class Reference:
    """fp32 CPU forward of the HF model on `state`, then masked mean and L2 normalise (SentenceTransformer's mean
    pooling + Normalize).  ids [B, S] right-padded, lens [B]."""

    def __init__(self, cfg, state):
        self.cfg = cfg
        self.model = _model(cfg)
        missing = self.model.load_state_dict(state, strict=False)
        assert not [m for m in missing.missing_keys if "position_ids" not in m and "token_type_ids" not in m], missing
        self.model.eval()

    @torch.no_grad()
    def __call__(self, ids, lens) -> np.ndarray:
        ids = torch.as_tensor(np.asarray(ids), dtype=torch.int64).clone()
        lens = np.asarray(lens)
        S = ids.shape[1]
        mask = torch.from_numpy((np.arange(S)[None, :] < lens[:, None]).astype(np.int64))
        if self.cfg.model_type == "xlm-roberta":
            ids[mask == 0] = PAD_ID          # XLM-R derives positions from the pad id: pad the way its tokenizer does
        h = self.model(input_ids=ids, attention_mask=mask).last_hidden_state.float()
        m = mask.unsqueeze(-1).float()
        pooled = (h * m).sum(1) / m.sum(1).clamp(min=1e-9)
        return torch.nn.functional.normalize(pooled, p=2, dim=1).numpy().astype(np.float32)


def unigram_tokenizer(texts: Sequence[str]):
    """A SentencePiece-Unigram tokenizer.json (tokenizers library) over the characters of `texts`: Metaspace
    pre-tokenizer, <s> $A </s> template, ids 0..3 = <s> <pad> </s> <unk> as in XLM-R; wrapped as XLMRobertaTokenizerFast."""
    from tokenizers import Tokenizer, decoders, models, pre_tokenizers, processors
    from transformers import XLMRobertaTokenizerFast
    chars = sorted({c for t in texts for c in t if not c.isspace()} | set("abcdefghijklmnopqrstuvwxyz0123456789:.,"))
    pieces = [(s, 0.0) for s in SPECIALS] + [("▁", -2.0)]
    pieces += [("▁" + c, -3.0) for c in chars] + [(c, -4.0) for c in chars]
    pieces += [("▁query", -1.0), ("▁passage", -1.0), (":", -2.5)]
    seen, vocab = set(), []
    for p, s in pieces:
        if p not in seen:
            seen.add(p)
            vocab.append((p, s))
    tok = Tokenizer(models.Unigram(vocab, unk_id=UNK_ID))
    tok.pre_tokenizer = pre_tokenizers.Metaspace(replacement="▁", prepend_scheme="always")
    tok.decoder = decoders.Metaspace(replacement="▁", prepend_scheme="always")
    tok.post_processor = processors.TemplateProcessing(single="<s> $A </s>", pair="<s> $A </s> </s> $B </s>",
                                                       special_tokens=[("<s>", 0), ("</s>", 2)])
    return XLMRobertaTokenizerFast(tokenizer_object=tok, bos_token="<s>", eos_token="</s>", unk_token="<unk>",
                                   pad_token="<pad>", cls_token="<s>", sep_token="</s>", mask_token="<unk>")


def save_e5_dir(path: str, cfg, state, tokenizer, max_seq_length=512) -> str:
    """The files SentenceTransformer('intfloat/multilingual-e5-large') resolves, with synthetic contents."""
    from safetensors.torch import save_file
    os.makedirs(os.path.join(path, "1_Pooling"), exist_ok=True)
    d = cfg.to_dict()
    d["model_type"] = cfg.model_type
    with open(os.path.join(path, "config.json"), "w") as fh:
        json.dump(d, fh)
    save_file({k: v.contiguous() for k, v in state.items()}, os.path.join(path, "model.safetensors"))
    tokenizer.save_pretrained(path)
    with open(os.path.join(path, "sentence_bert_config.json"), "w") as fh:
        json.dump({"max_seq_length": max_seq_length, "do_lower_case": False}, fh)
    with open(os.path.join(path, "1_Pooling", "config.json"), "w") as fh:
        json.dump({"word_embedding_dimension": cfg.hidden_size, "pooling_mode_cls_token": False,
                   "pooling_mode_mean_tokens": True, "pooling_mode_max_tokens": False,
                   "pooling_mode_mean_sqrt_len_tokens": False}, fh)
    return path
