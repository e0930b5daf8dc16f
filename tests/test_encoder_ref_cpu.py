"""The fp64 encoder references of tests/encoder_ref.py, without a GPU: each reference agrees with an independent
torch implementation (F.layer_norm, F.scaled_dot_product_attention, F.gelu, one transformers BertLayer), and the
comparator's bounds are tight enough to reject the kernel defects they exist to catch.  Also compiles the test shim
over the encoder launchers (compile only), so a header change that breaks it shows without a GPU."""
import os
import subprocess

import pytest
import torch
import torch.nn.functional as F

import encoder_ref as R

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CSRC = os.path.join(ROOT, "rag-project-icd10_b200", "csrc")
D = torch.float64


def _gen(seed):
    return torch.Generator().manual_seed(seed)


def _bf(shape, g, scale=1.0, shift=0.0):
    return R.bf16_round(torch.randn(shape, generator=g, dtype=D) * scale + shift)


def _close(a, b, tol=1e-9):
    assert torch.allclose(a, b, rtol=tol, atol=tol), float((a - b).abs().max())


# ------------------------------------------------------------------------------------------------ references vs torch
def test_linear_epilogues_match_torch():
    g = _gen(0)
    a, w, b = _bf((37, 768), g), _bf((512, 768), g, 0.02), torch.randn(512, generator=g, dtype=D) * 0.05
    _close(R.linear(a, w, b)[0], F.linear(a, w, b))
    _close(R.linear(a, w, b, "gelu")[0], F.gelu(F.linear(a, w, b), approximate="none"))
    res = _bf((37, 512), g)
    _close(R.linear(a, w, b, "residual", res=res)[0], F.linear(a, w, b) + res)


def test_deferred_layernorm_references_match_torch():
    g = _gen(1)
    eps = 1e-12
    x = _bf((40, 768), g, 2.0, 0.7)
    gamma, beta = 1 + 0.1 * torch.randn(768, generator=g, dtype=D), 0.05 * torch.randn(768, generator=g, dtype=D)
    w, b = _bf((256, 768), g, 0.02), 0.05 * torch.randn(256, generator=g, dtype=D)
    c = w.sum(1)
    want = F.linear(F.layer_norm(x, (768,), eps=eps), w, b)
    for stats in (R.row_partials(x), "row"):
        _close(R.linear(x, w, b, lnin=(c, stats), eps=eps)[0], want)
    # residual through LayerNorm: beta rides in the bias
    a, wo = _bf((40, 768), g), _bf((768, 768), g, 0.02)
    bo = 0.05 * torch.randn(768, generator=g, dtype=D)
    want = F.linear(a, wo, bo) + F.layer_norm(x, (768,), gamma, beta, eps=eps)
    for stats in (R.row_partials(x), "row"):
        got = R.linear(a, wo, bo + beta, "residual", res=x, res_gamma=gamma, res_stats=stats, eps=eps)[0]
        _close(got, want)


def test_row_partials_cover_each_128_column_slot():
    x = _bf((5, 768), _gen(2))
    p = R.row_partials(x)
    assert p.shape == (6, 5, 2)
    for j in range(6):
        _close(p[j, :, 0], x[:, 128 * j:128 * (j + 1)].sum(1))
        _close(p[j, :, 1], (x[:, 128 * j:128 * (j + 1)] ** 2).sum(1))


def test_gelu_is_the_erf_form():
    x = torch.linspace(-12, 12, 4801, dtype=D)
    _close(R.gelu_erf(x), F.gelu(x, approximate="none"), 1e-12)
    # the derivative bound used to propagate the pre-activation error
    xs = torch.linspace(-12, 12, 240001, dtype=D, requires_grad=True)
    (d,) = torch.autograd.grad(R.gelu_erf(xs).sum(), xs)
    assert float(d.abs().max()) <= R.GELU_DERIV_MAX


@pytest.mark.parametrize("S,split", [(1, False), (7, False), (64, False), (128, False), (200, True), (512, True)])
def test_attention_matches_sdpa(S, split):
    g = _gen(S)
    B = 3
    qkv = _bf((B * S, 2304), g)
    lens = torch.tensor([S, max(1, S // 2), 1])
    got, tol = R.attention(qkv, lens, B, S, split_kv=split)
    x = qkv.reshape(B, S, 3, 12, 64).permute(2, 0, 3, 1, 4)
    t = torch.arange(S)
    mask = (t[None, :] < lens[:, None])[:, None, None, :]
    want = F.scaled_dot_product_attention(x[0], x[1], x[2], attn_mask=mask, scale=0.125)
    want = want.permute(0, 2, 1, 3).reshape(B * S, 768)
    live = (t[None, :] < lens[:, None]).reshape(-1)
    _close(got[live], want[live])
    assert (got[~live] == 0).all() and (tol[~live] == 0).all()


def test_layernorm_and_embedding_references_match_torch():
    g = _gen(4)
    eps = 1e-12
    x = _bf((33, 768), g, 3.0, 5.0)
    gamma, beta = 1 + 0.1 * torch.randn(768, generator=g, dtype=D), 0.05 * torch.randn(768, generator=g, dtype=D)
    _close(R.layernorm(x, gamma, beta, eps)[0], F.layer_norm(x, (768,), gamma, beta, eps=eps))
    vocab, S = 50, 7
    word, pos, ty = (torch.randn(s, generator=g, dtype=D) for s in ((vocab, 768), (512, 768), (768,)))
    ids = torch.tensor([3, -1, vocab, 2 ** 31 - 1, 0, 49, 5, 6, 7, 8])
    got = R.embed_ln(ids, S, vocab, 1, word, pos, ty, gamma, beta, eps)[0]
    idc = torch.tensor([3, 1, 1, 1, 0, 49, 5, 6, 7, 8])
    want = F.layer_norm(word[idc] + pos[torch.arange(10) % S] + ty, (768,), gamma, beta, eps=eps)
    _close(got, want)


def test_pool_and_token_head_references():
    g = _gen(5)
    B, S = 4, 9
    h = _bf((B * S, 768), g)
    lens = torch.tensor([1, 9, 20, 0])          # > S clamps, 0 gives zeros
    got, tol = R.pool_normalise(h, lens, B, S)
    x = h.reshape(B, S, 768)
    for b, n in enumerate([1, 9, 9]):
        _close(got[b], F.normalize(x[b, :n].mean(0), dim=0))
    assert (got[3] == 0).all() and torch.isfinite(tol).all()
    raw = R.pool_normalise(h, lens, B, S, normalise=False)[0]
    _close(raw[1], x[1].mean(0))
    w, bb = torch.randn(9, 768, generator=g, dtype=D), torch.randn(9, generator=g, dtype=D)
    _close(R.token_head(h, w, bb)[0], F.linear(h, w, bb))


def test_composed_references_match_one_bert_layer():
    """qkv -> attention -> O + residual -> LN -> FFN-up + GELU -> FFN-down + residual -> LN, composed from the
    references, against transformers' BertLayer in float64; and the deferred-LayerNorm dataflow the kernels run
    (un-normalised streams, gamma folded into W, beta into the bias, statistics from 128-column partials) gives the
    same layer."""
    from transformers.models.bert.modeling_bert import BertLayer
    from oracle import encoder as oenc
    cfg = oenc.bert_config(1, 100, 512)
    cfg._attn_implementation = "eager"
    torch.manual_seed(0)
    layer = BertLayer(cfg).to(D).eval()
    g = _gen(6)
    with torch.no_grad():
        for n, p in layer.named_parameters():
            if n.endswith("LayerNorm.weight"):
                p.copy_(1 + 0.1 * torch.randn(p.shape, generator=g, dtype=D))
            elif n.endswith("bias"):
                p.copy_(0.05 * torch.randn(p.shape, generator=g, dtype=D))
    P = dict(layer.named_parameters())
    att = "attention.self."
    wqkv = torch.cat([P[att + n + ".weight"] for n in ("query", "key", "value")]).detach()
    bqkv = torch.cat([P[att + n + ".bias"] for n in ("query", "key", "value")]).detach()
    wo, bo = P["attention.output.dense.weight"].detach(), P["attention.output.dense.bias"].detach()
    g1, be1 = P["attention.output.LayerNorm.weight"].detach(), P["attention.output.LayerNorm.bias"].detach()
    w1, b1 = P["intermediate.dense.weight"].detach(), P["intermediate.dense.bias"].detach()
    w2, b2 = P["output.dense.weight"].detach(), P["output.dense.bias"].detach()
    g2, be2 = P["output.LayerNorm.weight"].detach(), P["output.LayerNorm.bias"].detach()
    B, S, eps = 3, 20, 1e-12
    lens = torch.tensor([20, 11, 3])
    h = torch.randn(B * S, 768, generator=g, dtype=D)
    qkv = R.linear(h, wqkv, bqkv)[0]
    ctx = R.attention(qkv, lens, B, S)[0]
    t = R.linear(ctx, wo, bo, "residual", res=h)[0]
    t1 = R.layernorm(t, g1, be1, eps)[0]
    f = R.linear(t1, w1, b1, "gelu")[0]
    out = R.layernorm(R.linear(f, w2, b2, "residual", res=t1)[0], g2, be2, eps)[0]
    mask = (torch.arange(S)[None, :] < lens[:, None])
    ext = torch.zeros(B, 1, 1, S, dtype=D).masked_fill(~mask[:, None, None, :], torch.finfo(D).min)
    with torch.no_grad():
        want = layer(h.reshape(B, S, 768), attention_mask=ext)
    want = (want[0] if isinstance(want, tuple) else want).reshape(B * S, 768)
    live = mask.reshape(-1)
    _close(out[live], want[live])
    # deferred form: FFN-up reads the un-normalised t with its partials, FFN-down rebuilds LN1(t) in its residual
    w1f = w1 * g1[None, :]
    f2 = R.linear(t, w1f, b1 + w1 @ be1, "gelu", lnin=(w1f.sum(1), R.row_partials(t)), eps=eps)[0]
    _close(f2, f)
    x2 = R.linear(f2, w2, b2 + be1, "residual", res=t, res_gamma=g1, res_stats=R.row_partials(t), eps=eps)[0]
    _close(R.layernorm(x2, g2, be2, eps)[0][live], want[live])


# ------------------------------------------------------------------------------------------------ defects must fail
def _must_fail(bad, ref, tol, what):
    w = R.worst(bad, ref, tol)
    assert w > 1.0, f"the bound lets '{what}' through (worst ratio {w:.3g})"


def _production_attention(S, seed):
    g = _gen(seed)
    B = 8
    qkv = _bf((B * S, 2304), g)
    lens = torch.randint(2, S, (B,), generator=g)
    return qkv, lens, B


@pytest.mark.parametrize("S,split", [(128, False), (64, False), (384, True)])
def test_attention_bound_rejects_defects(S, split):
    qkv, lens, B = _production_attention(S, S)
    ref, tol = R.attention(qkv, lens, B, S, split_kv=split)
    _must_fail(R.attention(qkv, lens, B, S, split_kv=split, admit_key=True)[0], ref, tol, "admit key len")
    _must_fail(R.attention(qkv, lens, B, S, split_kv=split, drop_last_key=True)[0], ref, tol, "drop key len - 1")
    _must_fail(R.attention(qkv, lens, B, S, split_kv=split, no_scale=True)[0], ref, tol, "no 1/8 scale")
    sw = ref.clone()
    sw[:, 0:64], sw[:, 64:128] = ref[:, 64:128], ref[:, 0:64]
    _must_fail(sw, ref, tol, "two heads swapped")


def _production_linear(seed, M=256, N=768, K=768):
    g = _gen(seed)
    a = _bf((M, K), g)
    w = _bf((N, K), g, 0.02)
    b = 0.05 * torch.randn(N, generator=g, dtype=D)
    return g, a, w, b


def test_linear_bound_rejects_defects():
    g, a, w, b = _production_linear(7)
    res = _bf((256, 768), g)
    ref, tol = R.linear(a, w, b, "residual", res=res)[:2]
    bad = ref.clone()
    bad[128:256, 64:128] -= res[128:256, 64:128]
    _must_fail(bad, ref, tol, "residual omitted in one 128 x 64 box")
    # bias of the neighbouring 256-column tile
    bad = ref.clone()
    bad[:, 256:512] += b[512:768] - b[256:512]
    _must_fail(bad, ref, tol, "bias from the next tile")
    # FFN-up shape: GELU replaced by the identity
    _, a, w, b = _production_linear(8, 256, 3072, 768)
    ref, tol = R.linear(a, w, b, "gelu")[:2]
    _must_fail(R.linear(a, w, b)[0], ref, tol, "identity for GELU")


def test_deferred_layernorm_bound_rejects_five_of_six_slots():
    g, x, w, b = _production_linear(9)
    x = R.bf16_round(x * 1.5 + 0.3)
    part = R.row_partials(x)
    ref, tol = R.linear(x, w, b, lnin=(w.sum(1), part))[:2]
    five = part.clone()
    five[5] = 0
    _must_fail(R.linear(x, w, b, lnin=(w.sum(1), five))[0], ref, tol, "5 of 6 statistics slots (input side)")
    gamma = 1 + 0.1 * torch.randn(768, generator=g, dtype=D)
    ref, tol = R.linear(x, w, b, "residual", res=x, res_gamma=gamma, res_stats=part)[:2]
    bad = R.linear(x, w, b, "residual", res=x, res_gamma=gamma, res_stats=five)[0]
    _must_fail(bad, ref, tol, "5 of 6 statistics slots (residual side)")


@pytest.mark.parametrize("out_bf16", [False, True])
def test_pool_bound_rejects_one_token_short(out_bf16):
    g = _gen(10)
    B, S = 16, 128
    h = _bf((B * S, 768), g)
    lens = torch.randint(2, S + 1, (B,), generator=g)
    ref, tol = R.pool_normalise(h, lens, B, S, out_bf16=out_bf16)
    _must_fail(R.pool_normalise(h, lens, B, S, drop_last=True)[0], ref, tol, "pool over len - 1 tokens")


# ------------------------------------------------------------------------------------------------ the shim compiles
def test_shim_compiles_against_the_headers(tmp_path):
    nvcc = R.nvcc_path()
    if nvcc is None:
        pytest.skip("no nvcc")
    src = os.path.join(ROOT, "tests", "encoder_kernel_shim.cu")
    cmd = [nvcc, "-gencode", "arch=compute_100a,code=sm_100a", "-std=c++17", "-Xcompiler", "-fPIC,-Wall",
           "-I", CSRC, "-I", os.path.join(ROOT, "include"), "-c", src, "-o", str(tmp_path / "shim.o")]
    r = subprocess.run(cmd, capture_output=True, text=True)
    assert r.returncode == 0, r.stderr
