"""The 1024-wide encoder without a GPU: which configs load, the weight blob of prefixed state dicts, a synthetic
multilingual-e5-large directory (XLM-R config, Unigram tokenizer.json, sentence-transformers files), the fp64
references at hidden 1024 / 16 heads against torch and transformers, planted defects the bounds must reject, and the
compile of the wide kernel shim."""
import importlib
import os
import subprocess

import numpy as np
import pytest
import torch
import torch.nn.functional as F

import wide_model as WM
from wide_encoder_ref import ref as R

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
W = importlib.import_module("rag-project-icd10_b200.engine.weights")
H, HEADS = 1024, 16


def _cfg(**kw):
    d = {"model_type": "bert", "vocab_size": 1000, "hidden_size": 1024, "num_hidden_layers": 2,
         "num_attention_heads": 16, "intermediate_size": 4096, "max_position_embeddings": 512, "type_vocab_size": 2,
         "layer_norm_eps": 1e-12, "hidden_act": "gelu"}
    d.update(kw)
    return d


# ------------------------------------------------------------------------------------------------ configs
def test_config_accepts_bert_large_and_xlmr_large():
    c = W.config_from_dict(_cfg())
    assert (c.hidden, c.heads, c.intermediate) == (1024, 16, 4096)
    x = W.config_from_dict(_cfg(model_type="xlm-roberta", max_position_embeddings=514, type_vocab_size=1, pad_token_id=1))
    assert (x.hidden, x.heads, x.max_position, x.type_vocab) == (1024, 16, 514, 1)
    assert W.position_offset({"model_type": "xlm-roberta", "pad_token_id": 1}) == 2
    assert W.position_offset({"model_type": "bert"}) == 0
    b = W.config_from_dict(_cfg(hidden_size=768, num_attention_heads=12, intermediate_size=3072))
    assert (b.hidden, b.heads) == (768, 12)


@pytest.mark.parametrize("kw,match", [
    (dict(hidden_size=896, num_attention_heads=14), "hidden size 896"),
    (dict(num_attention_heads=12), "head dim must be 64"),
    (dict(position_embedding_type="rotary"), "absolute position"),
    (dict(hidden_act="gelu_new"), "erf-GELU"),
    (dict(model_type="roberta"), "model_type 'roberta'"),
])
def test_config_rejections_name_the_reason(kw, match):
    with pytest.raises(ValueError, match=match):
        W.config_from_dict(_cfg(**kw))


def _write_dir(tmp_path, pooling="mean", max_seq=512, lower=False):
    tok = WM.unigram_tokenizer(["急性胃肠炎 发热", "cholera A00.0"])
    cfg = WM.xlmr_config(layers=1, vocab_size=600, intermediate=1024)
    state = WM.state_dict(cfg, seed=2)
    d = str(tmp_path / "e5")
    WM.save_e5_dir(d, cfg, state, tok, max_seq_length=max_seq)
    import json
    with open(os.path.join(d, "sentence_bert_config.json"), "w") as fh:
        json.dump({"max_seq_length": max_seq, "do_lower_case": lower}, fh)
    if pooling != "mean":
        with open(os.path.join(d, "1_Pooling", "config.json"), "w") as fh:
            json.dump({"pooling_mode_cls_token": True, "pooling_mode_mean_tokens": False}, fh)
    return d, cfg, state, tok


@pytest.mark.parametrize("kw,match", [(dict(pooling="cls"), "pooling modes"), (dict(lower=True), "lower-casing"),
                                      (dict(max_seq=1024), "512-token limit")])
def test_model_dir_rejections_are_kept(tmp_path, kw, match):
    d = _write_dir(tmp_path, **kw)[0]
    with pytest.raises(ValueError, match=match):
        W.load_model_dir(d)


# ------------------------------------------------------------------------------------------------ packing
def _c_count(cfg):
    Hh, Ii = cfg.hidden, cfg.intermediate
    n = cfg.vocab_size * Hh + cfg.max_position * Hh + cfg.type_vocab * Hh + 2 * Hh
    return n + cfg.layers * (3 * Hh * Hh + 3 * Hh + Hh * Hh + Hh + 2 * Hh + Ii * Hh + Ii + Hh * Ii + Hh + 2 * Hh)


@pytest.mark.parametrize("prefix", ["roberta.", "0.auto_model.", ""])
def test_pack_prefixed_state_dicts(prefix):
    cfg = WM.xlmr_config(layers=2, vocab_size=300, intermediate=1024)
    state = {prefix + k: v for k, v in WM.state_dict(cfg, seed=1).items()}
    ncfg = W.config_from_dict(dict(cfg.to_dict(), model_type="xlm-roberta"))
    blob = W.pack_state_dict(state, ncfg)
    assert blob.size == _c_count(ncfg)
    assert np.array_equal(blob[:1024], state[prefix + "embeddings.word_embeddings.weight"][0].numpy())


# ------------------------------------------------------------------------------------------------ e5 directory
def test_e5_directory_loads_with_offset_unk_and_hf_tokenizer(tmp_path):
    d, cfg, state, tok = _write_dir(tmp_path)
    c, blob, meta = W.load_model_dir(d)
    assert (c.hidden, c.heads) == (1024, 16)
    assert meta["position_offset"] == 2 and meta["unk_id"] == 3 and meta["max_seq_length"] == 512
    assert blob.size == _c_count(c)
    E = importlib.import_module("rag-project-icd10_b200.engine.encoder")
    T = importlib.import_module("rag-project-icd10_b200.engine.tokenizer")
    loaded = E.load_tokenizer(d)
    assert T._plain_bert_pipeline(loaded) is None
    assert not T.NativeTokenizer(loaded).native
    from oracle import text as otext
    recs = otext.load_records(os.path.join(ROOT, "data", "ICD_10v601.csv"))[:50]
    texts = [otext.query_text(r["semantic_text"]) for r in recs] + ["query: 急性胃肠炎", "Ω unknown ☃"]
    a = loaded(texts, add_special_tokens=True)["input_ids"]
    b = tok(texts, add_special_tokens=True)["input_ids"]
    assert a == b
    assert all(r[0] == 0 and r[-1] == 2 for r in a)
    assert 3 in loaded("☃")["input_ids"]


# ------------------------------------------------------------------------------------------------ references
def _gen(s):
    return torch.Generator().manual_seed(s)


def test_layernorm_reference_matches_torch():
    x = torch.randn((50, H), generator=_gen(1), dtype=torch.float64) * 3 + 1
    g, b = 1 + 0.1 * torch.randn(H, generator=_gen(2), dtype=torch.float64), 0.1 * torch.randn(H, generator=_gen(3), dtype=torch.float64)
    ref, _ = R.layernorm(x, g, b, 1e-12)
    assert torch.allclose(ref, F.layer_norm(x, (H,), g, b, 1e-12), atol=1e-10)


def _qkv(B, S, seed):
    return torch.randn((B * S, 3 * H), generator=_gen(seed), dtype=torch.float32).to(torch.bfloat16)


def test_attention_reference_matches_sdpa_with_16_heads():
    B, S = 3, 40
    lens = torch.tensor([40, 17, 1])
    qkv = _qkv(B, S, 4)
    ref, _ = R.attention(qkv, lens, B, S)
    x = R.f64(qkv).reshape(B, S, 3, HEADS, 64).permute(2, 0, 3, 1, 4)
    mask = (torch.arange(S)[None, :] < lens[:, None])[:, None, None, :]
    o = F.scaled_dot_product_attention(x[0], x[1], x[2], attn_mask=mask)
    o = o.permute(0, 2, 1, 3).reshape(B * S, H)
    live = (torch.arange(B * S) % S) < lens.repeat_interleave(S)
    assert torch.allclose(ref[live], o[live], atol=1e-10)


def test_embed_ln_reference_matches_xlmr_embeddings():
    from transformers.models.xlm_roberta.modeling_xlm_roberta import XLMRobertaEmbeddings
    cfg = WM.xlmr_config(layers=1, vocab_size=300)
    cfg.layer_norm_eps = 1e-5
    emb = XLMRobertaEmbeddings(cfg).double().eval()
    with torch.no_grad():
        emb.LayerNorm.weight.copy_(1 + 0.1 * torch.randn(H, generator=_gen(5)))
        emb.LayerNorm.bias.copy_(0.1 * torch.randn(H, generator=_gen(6)))
    B, S = 2, 30
    ids = torch.randint(4, 300, (B, S), generator=_gen(7))
    with torch.no_grad():
        hf = emb(input_ids=ids)
    p = {k: v.detach() for k, v in emb.named_parameters()}
    ref, _ = R.embed_ln(ids.reshape(-1).to(torch.int32), S, 300, 3, p["word_embeddings.weight"], p["position_embeddings.weight"],
                        p["token_type_embeddings.weight"][0], p["LayerNorm.weight"], p["LayerNorm.bias"], 1e-5, pos_offset=2)
    assert torch.allclose(ref, hf.reshape(B * S, H), atol=1e-9)
    off_by_one, tol = R.embed_ln(ids.reshape(-1).to(torch.int32), S, 300, 3, p["word_embeddings.weight"],
                                 p["position_embeddings.weight"], p["token_type_embeddings.weight"][0],
                                 p["LayerNorm.weight"], p["LayerNorm.bias"], 1e-5, pos_offset=1)
    # planted defect: positions off by one (BERT numbering shifted) -- rejected by >= 100x its own bound
    assert R.worst(off_by_one, ref, tol) >= 100


def test_one_xlmr_layer_matches_the_reference_chain():
    from transformers.models.xlm_roberta.modeling_xlm_roberta import XLMRobertaLayer
    cfg = WM.xlmr_config(layers=1, vocab_size=300)
    layer = XLMRobertaLayer(cfg).double().eval()
    B, S = 2, 20
    x = torch.randn((B, S, H), generator=_gen(8), dtype=torch.float64)
    with torch.no_grad():
        hf = layer(x)[0] if isinstance(layer(x), tuple) else layer(x)
    sd = {k: v for k, v in layer.state_dict().items()}
    lin = lambda a, n: a @ sd[n + ".weight"].T + sd[n + ".bias"]
    h = x.reshape(B * S, H)
    qkv = torch.cat([lin(h, "attention.self.query"), lin(h, "attention.self.key"), lin(h, "attention.self.value")], 1)
    ctx, _ = R.attention(qkv, torch.tensor([S, S]), B, S)
    t = R.layernorm(lin(ctx, "attention.output.dense") + h, sd["attention.output.LayerNorm.weight"],
                    sd["attention.output.LayerNorm.bias"], cfg.layer_norm_eps)[0]
    f = R.gelu_erf(lin(t, "intermediate.dense"))
    y = R.layernorm(lin(f, "output.dense") + t, sd["output.LayerNorm.weight"], sd["output.LayerNorm.bias"],
                    cfg.layer_norm_eps)[0]
    assert torch.allclose(y, hf.reshape(B * S, H), atol=1e-9)


# ------------------------------------------------------------------------------------------------ planted defects
def test_bounds_reject_12_of_16_heads():
    B, S = 2, 33
    lens = torch.tensor([33, 20])
    qkv = _qkv(B, S, 9)
    ref, tol = R.attention(qkv, lens, B, S)
    bad = ref.clone()
    bad[:, 12 * 64:] = 0                     # a kernel that walks 12 heads (the 768 head count) leaves 4 unwritten
    live = (torch.arange(B * S) % S) < lens.repeat_interleave(S)
    assert R.worst(bad[live], ref[live], tol[live]) >= 100


def test_bounds_reject_six_of_eight_statistics_slots():
    M = 64
    a = (torch.randn((M, H), generator=_gen(10)) + 0.5).to(torch.bfloat16)
    w = (0.02 * torch.randn((256, H), generator=_gen(11))).to(torch.bfloat16)
    bias = 0.05 * torch.randn(256, generator=_gen(12))
    stats = R.row_partials(R.f64(a)).to(torch.float32)
    assert stats.shape[0] == 8
    c = R.f64(w).sum(1)
    ref, tol = R.linear(a, w, bias, "bias", lnin=(c, stats), eps=1e-12)[:2]
    mu, rs, _, _ = R.row_stats(a, 1e-12, stats, slots=slice(0, 6))   # the 768 slot count
    got = (R.f64(a) - mu[:, None]) * rs[:, None] @ R.f64(w).T + R.f64(bias)
    assert R.worst(got, ref, tol) >= 100


def test_bounds_reject_a_qkv_stride_of_2304():
    B, S = 1, 64
    lens = torch.tensor([64])
    qkv = _qkv(B, S, 13)
    ref, tol = R.attention(qkv, lens, B, S)
    # rows read with the 768 stride (2304 elements): row r starts at 2304 r instead of 3072 r
    strided = qkv.reshape(-1)
    wrong = torch.stack([strided[r * 2304: r * 2304 + 3 * H] for r in range(B * S)])
    got, _ = R.attention(wrong, lens, B, S)
    assert R.worst(got, ref, tol) >= 100


def test_bounds_reject_the_bert_unk_id():
    vocab, S = 300, 16
    ids = torch.randint(4, vocab, (S,), generator=_gen(14), dtype=torch.int64)
    ids[3] = vocab + 5
    word = torch.randn((vocab, H), generator=_gen(15), dtype=torch.float64)
    pos = torch.randn((514, H), generator=_gen(16), dtype=torch.float64) * 0.5
    ty = torch.zeros(H, dtype=torch.float64)
    g, b = torch.ones(H, dtype=torch.float64), torch.zeros(H, dtype=torch.float64)
    ref, tol = R.embed_ln(ids, S, vocab, 3, word, pos, ty, g, b, 1e-5, pos_offset=2)
    got, _ = R.embed_ln(ids, S, vocab, 100, word, pos, ty, g, b, 1e-5, pos_offset=2)
    assert R.worst(got, ref, tol) >= 100


# ------------------------------------------------------------------------------------------------ shim compile
def test_wide_shim_compiles_for_sm100a(tmp_path):
    nvcc = R.nvcc_path()
    if nvcc is None:
        pytest.skip("no CUDA compiler")
    csrc = os.path.join(ROOT, "rag-project-icd10_b200", "csrc")
    r = subprocess.run([nvcc, "-gencode", "arch=compute_100a,code=sm_100a", "-std=c++17", "-Xcompiler", "-fPIC",
                        "-I", csrc, "-I", os.path.join(ROOT, "include"), "-c",
                        os.path.join(ROOT, "tests", "encoder_kernel_shim_wide.cu"), "-o", str(tmp_path / "w.o")],
                       capture_output=True, text=True)
    assert r.returncode == 0, r.stderr
