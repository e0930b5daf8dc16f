"""The 1024-wide encoder (hidden 1024, 16 heads of 64, FFN 4096: BERT-large, XLM-RoBERTa-large) on the GPU.

* Per-launch parity: every encoder launcher at hidden 1024 against the fp64 references of tests/wide_encoder_ref.py
  (tests/encoder_ref.py at H = 1024), through tests/encoder_kernel_shim_wide.cu, built into pytest's temporary
  directory as tests/test_encoder_kernels_gpu.py builds its shim.  Guard rows after every output stay untouched.
* Whole forwards against transformers XLMRobertaModel / BertModel (fp32) -> masked mean -> L2 normalise.
* Path agreement (few-token vs tile kernels), padding invariance, PDL on / off bitwise identical.
* End to end: EmbeddingService over a synthetic multilingual-e5-large directory, tools/build_database.py over 2 000
  rows of data/ICD_10v601.csv into a 1024-d collection, MilvusService.search / search_batch with and without filter=.
The worst |err| / bound per kernel family is printed at the end of the module."""
import ctypes as C
import importlib
import os
import subprocess

import numpy as np
import pytest
import torch

import wide_model as WM
from wide_encoder_ref import ref as R

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CSRC = os.path.join(ROOT, "rag-project-icd10_b200", "csrc")
H, I, HEADS = 1024, 4096, 16
EPI = {"bias": 0, "gelu": 1, "residual": 2}
EPS = 1e-12
GUARD = 64
SENTINEL = 12345.0
DEV = "cuda"


@pytest.fixture(scope="module")
def wshim(tmp_path_factory, native):
    nvcc = R.nvcc_path()
    assert nvcc, "nvcc is needed to build the encoder kernel shim"
    assert os.path.exists(os.path.join(CSRC, "libicdrag.so")), "build() first"
    out = str(tmp_path_factory.mktemp("wshim") / "libencshimwide.so")
    cmd = [nvcc, "-gencode", "arch=compute_100a,code=sm_100a", "-std=c++17", "-shared", "-Xcompiler", "-fPIC",
           "-cudart", "none", "-I", CSRC, "-I", os.path.join(ROOT, "include"),
           os.path.join(ROOT, "tests", "encoder_kernel_shim_wide.cu"), "-L", CSRC, "-licdrag",
           "-Xlinker", "-rpath," + CSRC, "-o", out]
    r = subprocess.run(cmd, capture_output=True, text=True)
    assert r.returncode == 0, r.stderr
    native.lib()
    L = C.CDLL(out)
    vp, i32, i64, f32 = C.c_void_p, C.c_int, C.c_long, C.c_float
    L.wshim_gemm.argtypes = [vp, i64, vp, vp, vp, vp, vp, i64, i32, i32, i32, i32, vp, vp, i32, i32, f32, vp]
    L.wshim_skinny_supported.argtypes = [i32, i32, i32, i32]
    L.wshim_skinny.argtypes = [vp, vp, vp, vp, vp, vp, i32, i32, i32, i32, i32, f32, i32, vp]
    L.wshim_attention.argtypes = [vp, i64, vp, i32, i32, vp, i64, i32, vp]
    L.wshim_attention_long_scratch.argtypes = [i32, i32, i32, C.POINTER(i64)]
    L.wshim_attention_long_scratch.restype = i64
    L.wshim_attention_long.argtypes = [vp, i64, vp, i32, i32, vp, vp, vp, i32, vp]
    L.wshim_embed_ln.argtypes = [vp, i32, i32, i32, i32, vp, vp, vp, vp, vp, f32, vp, i32, i32, vp]
    L.wshim_layernorm.argtypes = [vp, i32, vp, vp, f32, vp, i32, vp]
    L.wshim_pool_normalise.argtypes = [vp, vp, i32, i32, vp, i32, i32, vp]
    L.wshim_token_head.argtypes = [vp, i32, vp, vp, i32, vp, i32, vp]
    return L


@pytest.fixture(scope="module", autouse=True)
def _report(request):
    yield
    tr = request.config.pluginmanager.get_plugin("terminalreporter")
    capman = request.config.pluginmanager.get_plugin("capturemanager")
    if tr is None or capman is None or not R.RATIOS:
        return
    with capman.global_and_fixture_disabled():
        tr.write_line("")
        tr.write_line("hidden 1024: worst |err| / bound per kernel family (<= 1 passes):")
        for k in sorted(R.RATIOS):
            tr.write_line(f"  {k:<48s} {R.RATIOS[k]:.3f}")


def _stream():
    return C.c_void_p(torch.cuda.current_stream().cuda_stream)


def _p(t):
    return None if t is None else C.c_void_p(t.data_ptr())


def _ok(native, status, what):
    if status != 0:
        raise AssertionError(f"{what}: status {status}: {native.lib().icd_last_error().decode()}")


def _gen(seed):
    return torch.Generator().manual_seed(seed)


def _randn(shape, seed, scale=1.0, dtype=torch.bfloat16):
    return (torch.randn(shape, generator=_gen(seed), dtype=torch.float32) * scale).to(dtype).to(DEV)


def _round_up(x, m):
    return (x + m - 1) // m * m


def _with_guard(rows, cols, dtype, fill=float("nan")):
    t = torch.full((rows + GUARD, cols), fill, dtype=dtype, device=DEV)
    t[rows:] = SENTINEL
    return t


def _guard_intact(buf, rows, what):
    g = buf[rows:]
    assert bool((g == SENTINEL).all()), f"{what}: wrote {int((g != SENTINEL).sum())} elements past its mapped rows"


# ------------------------------------------------------------------------------------------------ GEMM
def _stream_rows(rows, K, seed, shift_sigma=0.0):
    z = torch.randn((rows, K), generator=_gen(seed), dtype=torch.float32)
    z = z + shift_sigma * z.std(-1, keepdim=True)
    return z.to(torch.bfloat16).to(DEV)


def _gemm_inputs(M, N, K, seed, a_shift=0.0):
    rows = _round_up(M, 128)
    A = _stream_rows(rows, K, seed, a_shift)
    A[M:] = 1000.0
    W = _randn((N, K), seed + 1, 0.02)
    bias = (torch.randn(N, generator=_gen(seed + 2)) * 0.05).to(DEV)
    res = _stream_rows(rows, N, seed + 3, a_shift)
    res[M:] = -1000.0
    gamma = (1.0 + 0.1 * torch.randn(N, generator=_gen(seed + 4))).to(DEV)
    return rows, A, W, bias, res, gamma


def _partials32(x):
    """fp32 partials [8, stride, 2] of x[:M] (exact fp64 sums rounded once)."""
    M = x.shape[0]
    stride = _round_up(M, 256)
    p = torch.zeros((H // 128, stride, 2), dtype=torch.float32, device=DEV)
    exact = R.row_partials(R.f64(x))
    p[:, :M] = exact.to(torch.float32)
    return p


def run_gemm(wshim, native, A, a_rows, W, bias, M, epi, res=None, vec2=None, stats_in=None, want_stats=False):
    N, K = W.shape
    out_rows = _round_up(M, 128)
    out = _with_guard(out_rows, N, torch.bfloat16)
    stride = _round_up(M, 256)
    stats_out = torch.full((N // 128, stride, 2), float("nan"), dtype=torch.float32, device=DEV) if want_stats else None
    if stats_in is not None:
        stride = stats_in.shape[1]
    st = wshim.wshim_gemm(_p(A), a_rows, _p(W), _p(bias), _p(vec2), _p(res), _p(out), out_rows, M, N, K, EPI[epi],
                          _p(stats_in), _p(stats_out), stride if (stats_in is not None or want_stats) else 0, H, EPS,
                          _stream())
    _ok(native, st, f"gemm M={M} N={N} K={K} {epi}")
    torch.cuda.synchronize()
    _guard_intact(out, out_rows, f"gemm M={M} N={N} K={K} {epi} out")
    return out[:M], stats_out


# the four layer shapes at hidden 1024: (N, K, epilogue, lnin, residual through LayerNorm, emit statistics)
GEMM_CASES = {
    "qkv": (3 * H, H, "bias", False, False, False),
    "qkv_lnin": (3 * H, H, "bias", True, False, False),
    "o_residual_stats": (H, H, "residual", False, False, True),
    "o_residual_ln_stats": (H, H, "residual", False, True, True),
    "up_gelu_lnin": (I, H, "gelu", True, False, False),
    "down_residual_ln": (H, I, "residual", False, True, False),
    "down_residual_ln_stats": (H, I, "residual", False, True, True),
}
GEMM_M = [1, 127, 128, 129, 256, 257, 1000, 4097, 8192]


def gemm_case(wshim, native, case, M, seed):
    N, K, epi, lnin, res_ln, stats = GEMM_CASES[case]
    rows, A, W, bias, res, gamma = _gemm_inputs(M, N, K, seed, a_shift=0.5 if (lnin or res_ln) else 0.0)
    vec2 = stats_in = None
    if lnin:
        vec2 = R.f64(W).sum(1).to(torch.float32)
        stats_in = _partials32(A[:M])
    elif res_ln:
        vec2 = gamma
        stats_in = _partials32(res[:M])
    out, stats_out = run_gemm(wshim, native, A, rows, W, bias, M, epi, res=res if epi == "residual" else None,
                              vec2=vec2, stats_in=stats_in, want_stats=stats)
    ref_stats = stats_in[:, :M] if stats_in is not None else None
    ref, tol, pre, pre_tol = R.linear(A[:M], W, bias, epi, res=res[:M] if epi == "residual" else None,
                                      res_gamma=gamma if res_ln else None, res_stats=ref_stats,
                                      lnin=(vec2, ref_stats) if lnin else None, eps=EPS)
    fam = "gemm_tc " + case
    R.check(fam, out, ref, tol, f"M={M}")
    if stats:
        assert stats_out.shape[0] == 8
        R.check(fam + " stats_out", stats_out[:, :M].permute(1, 0, 2).reshape(M, -1),
                R.row_partials(pre).permute(1, 0, 2).reshape(M, -1),
                R.partials_tol(pre, pre_tol).permute(1, 0, 2).reshape(M, -1), f"M={M}")


@pytest.mark.parametrize("M", GEMM_M)
@pytest.mark.parametrize("case", list(GEMM_CASES))
def test_gemm_tc_1024_matches_fp64(wshim, native, case, M):
    gemm_case(wshim, native, case, M, seed=M + 17)


def test_gemm_tc_rejects_other_statistics_widths(wshim, native):
    M = 256
    rows, A, W, bias, res, gamma = _gemm_inputs(M, H, H, 1)
    out = torch.zeros((M, H), dtype=torch.bfloat16, device=DEV)
    st = torch.zeros((8, M, 2), device=DEV)
    c = torch.zeros(H, device=DEV)
    for cols in (512, 896, 1152):
        assert wshim.wshim_gemm(_p(A), M, _p(W), _p(bias), _p(c), None, _p(out), M, M, H, H, 0, _p(st), None, M, cols,
                                EPS, _stream()) == -1
    torch.cuda.synchronize()


# ------------------------------------------------------------------------------------------------ skinny_linear
SKINNY_CASES = {
    "qkv": (3 * H, H, "bias", 0, False),
    "qkv_lnin": (3 * H, H, "bias", 1, False),
    "o_residual": (H, H, "residual", 0, False),
    "o_residual_ln": (H, H, "residual", 0, True),
    "up_gelu_lnin": (I, H, "gelu", 1, False),
    "down_residual_ln": (H, I, "residual", 0, True),
}


@pytest.mark.parametrize("M", [1, 2, 12, 16, 17, 32, 33, 63, 64])
@pytest.mark.parametrize("case", list(SKINNY_CASES))
def test_skinny_linear_1024_matches_fp64_and_the_tile_kernel(wshim, native, case, M):
    N, K, epi, lnin, res_ln = SKINNY_CASES[case]
    assert wshim.wshim_skinny_supported(M, N, K, H) == 1
    rows, A, W, bias, res, gamma = _gemm_inputs(M, N, K, seed=700 + M, a_shift=0.5 if (lnin or res_ln) else 0.0)
    vec2 = R.f64(W).sum(1).to(torch.float32) if lnin else (gamma if res_ln else None)
    out = _with_guard(M, N, torch.bfloat16)
    r = res[:M].contiguous() if epi == "residual" else None
    st = wshim.wshim_skinny(_p(A), _p(W), _p(bias), _p(vec2), _p(r), _p(out), M, N, K, EPI[epi], lnin, EPS, H, _stream())
    _ok(native, st, f"skinny {case} M={M}")
    torch.cuda.synchronize()
    _guard_intact(out, M, f"skinny {case} M={M}")
    ref, tol = R.linear(A[:M], W, bias, epi, res=r, res_gamma=gamma if res_ln else None, res_stats="row",
                        lnin=(vec2, "row") if lnin else None, eps=EPS)[:2]
    R.check("skinny_linear " + case, out[:M], ref, tol, f"M={M}")
    again = torch.empty_like(out)
    _ok(native, wshim.wshim_skinny(_p(A), _p(W), _p(bias), _p(vec2), _p(r), _p(again), M, N, K, EPI[epi], lnin, EPS, H,
                                   _stream()), "skinny rerun")
    torch.cuda.synchronize()
    assert torch.equal(out[:M].view(torch.int16), again[:M].view(torch.int16)), "skinny_linear is not deterministic"
    stats_in = _partials32(A[:M] if lnin else res[:M]) if (lnin or res_ln) else None
    ref_stats = stats_in[:, :M] if stats_in is not None else None
    tile, _ = run_gemm(wshim, native, A, rows, W, bias, M, epi, res=res if epi == "residual" else None, vec2=vec2,
                       stats_in=stats_in)
    ttol = R.linear(A[:M], W, bias, epi, res=r, res_gamma=gamma if res_ln else None, res_stats=ref_stats,
                    lnin=(vec2, ref_stats) if lnin else None, eps=EPS)[1]
    R.check("skinny_linear vs gemm_tc " + case, out[:M], R.f64(tile), tol + ttol, f"M={M}")


def test_skinny_linear_1024_rejections(wshim, native):
    A, W = _randn((65, I), 1), _randn((I, I), 2)
    bias, c = torch.zeros(I, device=DEV), torch.zeros(I, device=DEV)
    out = torch.zeros((65, I), dtype=torch.bfloat16, device=DEV)
    s = _stream()
    assert wshim.wshim_skinny(_p(A), _p(W), _p(bias), None, None, _p(out), 65, H, H, 0, 0, EPS, H, s) == -1      # 65 tokens
    assert wshim.wshim_skinny(_p(A), _p(W), _p(bias), _p(c), None, _p(out), 8, H, I, 0, 1, EPS, H, s) == -1      # lnin, K != H
    assert wshim.wshim_skinny(_p(A), _p(W), _p(bias), _p(c), None, _p(out), 8, H, H, 0, 1, EPS, 896, s) == -1    # width
    torch.cuda.synchronize()


# ------------------------------------------------------------------------------------------------ attention
def _qkv(B, S, lens, seed, rows=None):
    """qkv [rows, 3072]; keys / values of positions t >= len and of rows past B*S are poisoned (K x 30, V = +-1e3)."""
    n = B * S
    rows = rows or _round_up(n, 128)
    x = torch.randn((rows, 3 * H), generator=_gen(seed), dtype=torch.float32)
    t = torch.arange(rows)
    seq = t // S
    L = torch.as_tensor(lens).to(torch.int64)
    dead = (seq >= B) | (t % S >= L[seq.clamp(max=B - 1)])
    x[dead, H:2 * H] *= 30.0
    x[dead, 2 * H:] = torch.where(torch.rand((int(dead.sum()), H), generator=_gen(seed + 1)) < 0.5, -1e3, 1e3)
    return x.to(torch.bfloat16).to(DEV), rows


def _check_attention(fam, got, qkv, lens, B, S, split):
    ref, tol = R.attention(qkv, lens, B, S, split_kv=split)
    t = torch.arange(B * S, device=DEV) % S
    padded = t >= lens.to(DEV).to(torch.int64).repeat_interleave(S)
    assert bool((got[padded] == 0).all()), f"{fam}: query rows at t >= len are not exactly 0"
    R.check(fam, got, ref, tol, f"B={B} S={S}")


@pytest.mark.parametrize("S", [1, 2, 7, 31, 33, 64, 65, 127, 128])
def test_attention_tc_1024_matches_fp64(wshim, native, S):
    G = 128 // S
    for B in sorted({1, G, G + 1, 10 * G + 3}):
        lens = torch.randint(1, S + 1, (B,), generator=_gen(S * 31 + B), dtype=torch.int32)
        lens[0] = S
        qkv, rows = _qkv(B, S, lens, seed=S + B)
        ctx_rows = _round_up(B * S, 128)
        ctx = _with_guard(ctx_rows, H, torch.bfloat16)
        _ok(native, wshim.wshim_attention(_p(qkv), rows, _p(lens.to(DEV)), B, S, _p(ctx), ctx_rows, H, _stream()),
            f"attention B={B} S={S}")
        torch.cuda.synchronize()
        _guard_intact(ctx, ctx_rows, f"attention B={B} S={S}")
        _check_attention("attention_tc", ctx[:B * S], qkv, lens, B, S, split=False)


@pytest.mark.parametrize("S", [129, 200, 256, 257, 384, 511, 512])
def test_attention_tc_long_1024_matches_fp64(wshim, native, S):
    lens = torch.tensor(sorted({min(v, S) for v in (1, 127, 128, 129, 256, 257, S)}), dtype=torch.int32)
    B = len(lens)
    qkv, rows = _qkv(B, S, lens, seed=S)
    sb = C.c_long(0)
    pb = wshim.wshim_attention_long_scratch(B, S, H, C.byref(sb))
    QT = (S + 127) // 128
    assert pb == QT * B * QT * 128 * H * 2 and sb.value == QT * HEADS * B * QT * 128 * 8
    part = torch.empty(pb // 2, dtype=torch.bfloat16, device=DEV)
    stats = torch.empty(sb.value // 4, dtype=torch.float32, device=DEV)
    ctx = _with_guard(B * S, H, torch.bfloat16)
    _ok(native, wshim.wshim_attention_long(_p(qkv), rows, _p(lens.to(DEV)), B, S, _p(part), _p(stats), _p(ctx), H,
                                           _stream()), f"attention_long S={S}")
    torch.cuda.synchronize()
    _guard_intact(ctx, B * S, f"attention_long S={S}")
    _check_attention("attention_tc_long", ctx[:B * S], qkv, lens, B, S, split=True)


# ------------------------------------------------------------------------------------------------ smaller kernels
@pytest.mark.parametrize("S", [1, 7, 128, 512])
def test_embed_ln_1024_with_position_offset_and_unk(wshim, native, S):
    vocab, unk, off = 1000, 3, 2
    B = max(1, 600 // S)
    M = B * S
    g = _gen(S)
    ids = torch.randint(0, vocab, (M,), generator=g, dtype=torch.int64)
    ids[::5] = -1
    ids[1::7] = vocab
    ids[2::11] = 2 ** 31 - 1
    ids = ids.to(torch.int32)
    word = _randn((vocab, H), 1, dtype=torch.float32)
    word[unk] = 3.0 * word[unk] + 1.0
    pos = _randn((514, H), 2, 0.5, dtype=torch.float32)
    ty = _randn((H,), 3, 0.1, dtype=torch.float32)
    gamma = (1 + 0.1 * torch.randn(H, generator=g)).to(DEV)
    beta = (0.05 * torch.randn(H, generator=g)).to(DEV)
    out = _with_guard(M, H, torch.bfloat16)
    _ok(native, wshim.wshim_embed_ln(_p(ids.to(DEV)), M, S, vocab, unk, _p(word), _p(pos), _p(ty), _p(gamma), _p(beta),
                                     EPS, _p(out), off, H, _stream()), "embed_ln")
    torch.cuda.synchronize()
    _guard_intact(out, M, "embed_ln")
    ref, tol = R.embed_ln(ids, S, vocab, unk, word, pos, ty, gamma, beta, EPS, pos_offset=off)
    R.check("embed_ln offset 2 unk 3", out[:M], ref, tol, f"S={S}")


@pytest.mark.parametrize("M", [1, 9, 1000])
def test_layernorm_pool_and_token_head_1024(wshim, native, M):
    x = _stream_rows(M, H, M, shift_sigma=3.0)
    gamma = (1 + 0.1 * torch.randn(H, generator=_gen(M))).to(DEV)
    beta = (0.05 * torch.randn(H, generator=_gen(M + 1))).to(DEV)
    y = _with_guard(M, H, torch.bfloat16)
    _ok(native, wshim.wshim_layernorm(_p(x), M, _p(gamma), _p(beta), EPS, _p(y), H, _stream()), "layernorm")
    torch.cuda.synchronize()
    _guard_intact(y, M, "layernorm")
    ref, tol = R.layernorm(x, gamma, beta, EPS)
    R.check("layernorm", y[:M], ref, tol, f"M={M}")
    # pooling over sequences of S = M tokens, B = 3 with lengths S, 1, S // 2 (padding rows poisoned)
    S, B = M, 3
    h = _stream_rows(B * S, H, M + 5)
    lens = torch.tensor([S, 1, max(1, S // 2)], dtype=torch.int32)
    for b in range(B):
        h[b * S + int(lens[b]):(b + 1) * S] = 1e4
    for flags, norm in ((0, True), (0x100, False)):
        out = _with_guard(B, H, torch.float32)
        _ok(native, wshim.wshim_pool_normalise(_p(h), _p(lens.to(DEV)), B, S, _p(out), flags, H, _stream()), "pool")
        torch.cuda.synchronize()
        _guard_intact(out, B, "pool")
        ref, tol = R.pool_normalise(h, lens, B, S, normalise=norm)
        R.check("pool_normalise", out[:B], ref, tol, f"S={S} norm={norm}")
    # token head, 9 labels
    w = (0.03 * torch.randn((9, H), generator=_gen(M + 7))).to(DEV)
    bb = (0.1 * torch.randn(9, generator=_gen(M + 8))).to(DEV)
    lo = _with_guard(M, 9, torch.float32)
    _ok(native, wshim.wshim_token_head(_p(x), M, _p(w), _p(bb), 9, _p(lo), H, _stream()), "token_head")
    torch.cuda.synchronize()
    _guard_intact(lo, M, "token_head")
    ref, tol = R.token_head(x, w, bb)
    R.check("token_head", lo[:M], ref, tol, f"M={M}")


# ------------------------------------------------------------------------------------------------ whole forwards
VOCAB = 4000


@pytest.fixture(scope="module")
def xlmr4():
    cfg = WM.xlmr_config(layers=4, vocab_size=VOCAB)
    return cfg, WM.state_dict(cfg, seed=11)


def _engine(pkg_native, cfg, state, layers=None, offset=0, unk=None):
    E = importlib.import_module("rag-project-icd10_b200.engine.encoder")
    W = importlib.import_module("rag-project-icd10_b200.engine.weights")
    ncfg = W.config_from_dict(dict(cfg.to_dict(), model_type=cfg.model_type))
    return E.EncoderEngine(cfg=ncfg, blob=W.pack_state_dict(state, ncfg), tokenizer=object(), device=0,
                           max_tokens=64 * 512, position_offset=offset, unk_id=unk, max_seq_length=512)


def _batch(B, S, seed, vocab=VOCAB):
    rng = np.random.default_rng(seed)
    lens = rng.integers(1, S + 1, size=B).astype(np.int32)
    lens[0] = S
    ids = np.zeros((B, S), np.int32)
    for b in range(B):
        ids[b, :lens[b]] = rng.integers(4, vocab, size=lens[b])
        ids[b, 0], ids[b, lens[b] - 1] = 0, 2
    return ids, lens


def _cos(a, b):
    return (a * b).sum(1) / (np.linalg.norm(a, axis=1) * np.linalg.norm(b, axis=1))


@pytest.mark.parametrize("S", [1, 12, 64, 127, 128, 129, 300, 512])
def test_xlmr_large_forward_matches_hf(native, xlmr4, S):
    cfg, state = xlmr4
    eng = _engine(native, cfg, state, offset=2, unk=3)
    try:
        B = 1 if S == 512 else (3 if S > 128 else 6)
        ids, lens = _batch(B, S, seed=S)
        got = eng.forward_ids(ids, lens)
        ref = WM.Reference(cfg, state)(ids, lens)
        cos = _cos(got, ref)
        assert cos.min() >= 0.999, (S, cos)
        assert eng.position_offset == 2 and eng.max_seq_length == 512
    finally:
        eng.close()


def test_xlmr_large_24_layers_matches_hf(native):
    cfg = WM.xlmr_config(layers=24, vocab_size=VOCAB)
    state = WM.state_dict(cfg, seed=24)
    eng = _engine(native, cfg, state, offset=2, unk=3)
    ref = WM.Reference(cfg, state)
    try:
        for S in (12, 64, 128):
            ids, lens = _batch(4, S, seed=100 + S)
            cos = _cos(eng.forward_ids(ids, lens), ref(ids, lens))
            assert cos.min() >= 0.999, (S, cos)
    finally:
        eng.close()


@pytest.mark.parametrize("S", [12, 128, 300])
def test_bert_large_forward_matches_hf(native, S):
    cfg = WM.bert_large_config(layers=4, vocab_size=VOCAB)
    state = WM.state_dict(cfg, seed=5)
    eng = _engine(native, cfg, state)
    try:
        ids, lens = _batch(4, S, seed=S + 1)
        cos = _cos(eng.forward_ids(ids, lens), WM.Reference(cfg, state)(ids, lens))
        assert cos.min() >= 0.999, (S, cos)
    finally:
        eng.close()


def test_xlmr_paths_padding_and_pdl(native, xlmr4):
    cfg, state = xlmr4
    eng = _engine(native, cfg, state, offset=2, unk=3)
    try:
        ids, lens = _batch(1, 40, seed=9)
        few = eng.forward_ids(ids, lens)                       # 40 tokens: the skinny kernels
        native.tune(enc_skinny=0)
        tile = eng.forward_ids(ids, lens)
        native.tune(enc_skinny=1)
        assert _cos(few, tile).min() >= 0.9999
        # padding invariance: the same sentence inside a batch padded to 128
        big = np.zeros((3, 128), np.int32)
        big[0, :40] = ids[0]
        big[1:, :100] = 5
        padded = eng.forward_ids(big, np.array([40, 100, 100], np.int32))
        assert _cos(padded[:1], tile).min() >= 0.99999
        # out-of-range ids read <unk> = 3
        bad = ids.copy()
        bad[0, 5] = VOCAB + 7
        unk = ids.copy()
        unk[0, 5] = 3
        assert np.array_equal(eng.forward_ids(bad, lens), eng.forward_ids(unk, lens))
        for S in (12, 64, 200):
            ids2, lens2 = _batch(5, S, seed=S + 50)
            a = eng.forward_ids(ids2, lens2)
            native.tune(enc_pdl=0)
            b = eng.forward_ids(ids2, lens2)
            native.tune(enc_pdl=1)
            assert np.array_equal(a.view(np.int32), b.view(np.int32)), S
    finally:
        native.tune(enc_skinny=1, enc_pdl=1)
        eng.close()


def test_create_rejects_other_shapes(native, xlmr4):
    cfg, state = xlmr4
    N = native
    W = importlib.import_module("rag-project-icd10_b200.engine.weights")
    good = W.config_from_dict(dict(cfg.to_dict(), model_type="xlm-roberta"))
    blob = W.pack_state_dict(state, good)
    for hidden, heads in ((1024, 12), (768, 16)):
        bad = N.BertCfg(vocab_size=good.vocab_size, hidden=hidden, layers=good.layers, heads=heads,
                        intermediate=good.intermediate, max_position=good.max_position, type_vocab=good.type_vocab,
                        ln_eps=good.ln_eps)
        h = C.c_void_p()
        assert N.lib().icd_encoder_create(N.buf_ptr(blob), blob.size, C.byref(bad), 0, C.byref(h)) == -1
        assert b"hidden=1024 with heads=16" in N.lib().icd_last_error()
    eng = _engine(native, cfg, state, offset=2, unk=3)
    try:
        # S + offset <= max_position (514): 512 tokens pass at offset 2 and are refused at offset 3
        ids = np.full((1, 512), 5, np.int32)
        assert eng.forward_ids(ids, np.array([512], np.int32)).shape == (1, 1024)
        assert N.lib().icd_encoder_set_embedding_ids(eng._h, 3, 3) == 0
        with pytest.raises(N.NativeError, match="position offset exceeds max_position"):
            eng.forward_ids(ids, np.array([512], np.int32))
        assert N.lib().icd_encoder_set_embedding_ids(eng._h, 0, VOCAB) == -1          # unk outside the vocabulary
    finally:
        eng.close()


# ------------------------------------------------------------------------------------------------ end to end
@pytest.fixture(scope="module")
def e5_dir(tmp_path_factory):
    from oracle import text as otext
    recs = otext.load_records(os.path.join(ROOT, "data", "ICD_10v601.csv"))
    texts = [otext.query_text(r["semantic_text"]) for r in recs[:2000]] + ["query: 急性胃肠炎 发热 霍乱 伤寒"]
    tok = WM.unigram_tokenizer(texts)
    cfg = WM.xlmr_config(layers=4, vocab_size=VOCAB)
    state = WM.state_dict(cfg, seed=3)
    d = str(tmp_path_factory.mktemp("e5large"))
    WM.save_e5_dir(d, cfg, state, tok)
    return d, cfg, state


def test_e5_large_service_build_and_search(tmp_path, monkeypatch, e5_dir):
    from oracle import text as otext
    from parity import check_topk
    d, cfg, state = e5_dir
    src = open(os.path.join(ROOT, "data", "ICD_10v601.csv"), encoding="utf-8-sig").read().splitlines()
    sub_csv = tmp_path / "subset.csv"
    sub_csv.write_text("﻿" + "\n".join(src[:2001]) + "\n", encoding="utf-8")
    monkeypatch.setenv("EMBEDDING_MODEL_NAME", d)
    monkeypatch.setenv("EMBEDDING_DEVICE", "auto")
    monkeypatch.setenv("MILVUS_DB_PATH", str(tmp_path / "db" / "icd.db"))
    monkeypatch.setenv("MILVUS_COLLECTION_NAME", "icd10")
    monkeypatch.chdir(tmp_path)
    B = importlib.import_module("rag-project-icd10_b200.tools.build_database")
    assert B.main(["--input", str(sub_csv), "--rebuild"]) is True
    builder = B.DatabaseBuilder()
    builder.initialize_services()
    es, ms = builder.embedding_service, builder.milvus_service
    assert es.get_model_info()["embedding_dimension"] == 1024 and ms.dimension == 1024
    assert es.model.position_offset == 2 and es.model.unk_id == 3 and es.model.max_seq_length == 512
    assert not es.model._ntok.native                         # Unigram: the HF fast tokenizer feeds the engine
    recs = otext.load_records(str(sub_csv))
    n = len(recs)
    stored = ms.client.cols["icd10"].index.read(0, n)
    assert stored.shape == (n, 1024)
    # encode_query / encode_queries / encode_batch against the HF reference on the tokenizer's own ids
    ref = WM.Reference(cfg, state)
    probes = ["急性胃肠炎", "霍乱", "伤寒", recs[700]["preferred_zh"]]
    for p in probes:
        enc = es.model.tokenizer([f"query: {p}"])["input_ids"][0]
        r = ref(np.array([enc]), np.array([len(enc)]))[0]
        assert float(es.encode_query(p) @ r) >= 0.999
    qs = np.asarray(es.encode_queries(probes), np.float32)
    assert qs.shape == (4, 1024)
    eb = np.asarray(es.encode_batch(probes, show_progress=False), np.float32)
    assert eb.shape == (4, 1024)
    # searches against an exact numpy search over the stored 1024-d vectors
    codes = [r["code"] for r in recs]
    level = np.array([int(r["level"]) for r in recs])
    for filt in ("", "level == 3"):
        allowed = np.ones(n, bool) if not filt else (level == 3)
        batch = ms.search_batch(qs, top_k=10, filter=filt)
        for qi, q in enumerate(qs):
            full = stored.astype(np.float64) @ q.astype(np.float64)
            full[~allowed] = -np.inf
            order = np.argsort(-full, kind="stable")[:10]
            single = ms.search(q, top_k=10, filter=filt)
            for hits in (single, batch[qi]):
                got = sorted(hits, key=lambda h: -h["original_score"])
                gi = np.array([[codes.index(h["code"]) for h in got]])
                gs = np.array([[h["original_score"] for h in got]], np.float32)
                check_topk(gi, gs, order[None, :], full[order][None, :].astype(np.float32),
                           exact_scores_of=lambda b, ids: full[ids])
                assert all(allowed[codes.index(h["code"])] for h in hits)
    ms.disconnect()
