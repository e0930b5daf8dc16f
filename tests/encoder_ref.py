"""fp64 references of the encoder kernels, with per-element error bounds derived from each kernel's arithmetic.

Every reference is computed in float64 from the exact bf16 (or fp32) values the kernel reads, and returns
(ref, tol): the exact result and, per element, how far the kernel's output may lie from it.  The bounds are built
from these pieces and nothing else:

* bf16 storage of an output: one bf16 ulp of |reference| + pre-rounding bound (round-to-nearest moves the
  computed value by half of its own ulp, and that value may sit one binade above the reference).
* fp32 accumulation of a K-term dot product: 2 * K * 2^-24 * sum|a*w| (the classical gamma_K bound; the factor 2
  allows truncating rather than rounding adders, which tensor cores may use).
* fp32 epilogue arithmetic: a few units of 2^-24 on the magnitude of each term it adds.
* GELU: the documented fit of csrc/common.cuh, 2.6e-5 + 2^-11 * |x / 2| (tanh.approx.f32), on top of the
  propagated pre-activation error (|gelu'| <= 1.13).
* attention: P is packed to bf16 before P.V (bf16 unit roundoff 2^-8, times sum p|v| / sum p); the split-KV
  path adds its bf16 partial outputs (another 2^-8 of the same).
* LayerNorm statistics summed in fp32: 8 * 2^-24 of the magnitudes summed, per quantity, propagated through
  mu and 1 / sigma.

No bound is fitted to an observed error.  `check` reports the worst |got - ref| / tol, so the margin shows in the
test log.  Works on CPU or CUDA tensors (all math is float64 torch).
"""
import math
import os
import shutil

import torch

U = 2.0 ** -24          # fp32 unit roundoff
H = 768                 # hidden size: the row length of every LayerNorm
HEADS, HD = 12, 64
GELU_FIT_ABS = 2.6e-5   # max |fit - gelu_erf| with exact tanh (csrc/common.cuh)
GELU_TANH_REL = 2.0 ** -11
GELU_DERIV_MAX = 1.13   # max |d gelu / dx| = Phi(x) + x phi(x) at x = sqrt(2)


def nvcc_path():
    """The CUDA compiler that builds the test shim over the encoder launchers, or None."""
    for cand in (os.environ.get("NVCC"), shutil.which("nvcc"), "/usr/local/cuda/bin/nvcc"):
        if cand and os.path.exists(cand):
            return cand
    return None


def f64(t):
    return t.to(torch.float64)


def bf16_round(t):
    return t.to(torch.bfloat16).to(torch.float64)


def bf16_ulp(x):
    """bf16 ulp of |x| (8 significant bits); 0 for x == 0."""
    a = x.abs()
    e = torch.floor(torch.log2(torch.where(a > 0, a, torch.ones_like(a))))
    return torch.where(a > 0, torch.exp2(e - 7), torch.zeros_like(a))


def stored(ref, tol):
    """Bound of a bf16-stored result: the pre-rounding bound plus one ulp of the largest value the pre-rounding result
    can take (round-to-nearest moves it by half of its own ulp)."""
    return tol + bf16_ulp(ref.abs() + tol)


def gelu_erf(x):
    return 0.5 * x * (1.0 + torch.erf(x / math.sqrt(2.0)))


# ------------------------------------------------------------------------------------------------ LayerNorm statistics
def row_partials(x):
    """[H/128, M, 2] per-row (sum, sum of squares) of each 128-column slot of x [M, 768] (fp64)."""
    M = x.shape[0]
    s = x.reshape(M, H // 128, 128)
    return torch.stack([s.sum(-1), (s * s).sum(-1)], -1).transpose(0, 1).contiguous()


def _stats_bounds(mu, var, ss, e_s, e_ss, eps):
    """(rs, dmu, drs) of the one-pass fp32 form mu = s / 768, var = ss / 768 - mu^2, rs = rsqrt(var + eps), given
    bounds e_s, e_ss on the fp32 error of the sums s and ss."""
    rs = 1.0 / torch.sqrt(var.clamp(min=0.0) + eps)
    dmu = e_s / H + 2 * U * mu.abs()
    dvar = e_ss / H + 2 * U * ss / H + 2 * mu.abs() * dmu + 2 * U * mu * mu
    drs = rs * (dvar / (2 * (var.clamp(min=0.0) + eps)) + 4 * U)
    return rs, dmu, drs


def row_stats(x, eps, stats, slots=None):
    """Row (mu, rs, dmu, drs) a kernel applies to the stream x [M, 768]: mu and rs in fp64, dmu and drs bounds on the
    kernel's fp32 evaluation.  stats = fp32 partials [6, M, 2] as the GEMM reads them (six values summed, then the
    one-pass form), or "row": the kernel sums the row itself in one fp32 pass (skinny_linear: 96 sequential terms per
    lane, 3 shuffle levels).  `slots` restricts which partials are summed (a defect model)."""
    if isinstance(stats, str):
        assert stats == "row"
        x = f64(x)
        s, ss = x.sum(-1), (x * x).sum(-1)
        e_s, e_ss = 100 * U * x.abs().sum(-1), 100 * U * ss
    else:
        p = f64(stats)
        if slots is not None:
            p = p[slots]
        s, ss = p[..., 0].sum(0), p[..., 1].sum(0)
        # six fp32 partials summed with 5 adds (and their own rounding to fp32)
        e_s, e_ss = 8 * U * p[..., 0].abs().sum(0), 8 * U * p[..., 1].sum(0)
    mu = s / H
    var = ss / H - mu * mu
    rs, dmu, drs = _stats_bounds(mu, var, ss, e_s, e_ss, eps)
    return mu, rs, dmu, drs


def exact_stats(x, eps):
    """Two-pass (mu, rs) of rows of x in fp64 (what LayerNorm means)."""
    mu = x.mean(-1)
    var = ((x - mu[:, None]) ** 2).mean(-1)
    return mu, 1.0 / torch.sqrt(var + eps)


# ------------------------------------------------------------------------------------------------ linear layers
def linear(a, w, bias, epi="bias", res=None, res_gamma=None, res_stats=None, lnin=None, eps=1e-12, strict_norm=False):
    """Reference of one launch of gemm_tc / skinny_linear, out = epi(A' W^T + bias):

    a [M, K], w [N, K] bf16 values; bias [N].
    lnin = (c, stats): A is an un-normalised stream, A' = (A - mu) * rs with mu, rs from `stats` (see row_stats:
        the fp32 partials the GEMM reads, or "row").  c is the kernel's column vector (row sums of W); it enters the
        bound only: the reference never uses the folding identity.
    epi = "bias" | "gelu" | "residual"; res [M, N]; res_gamma [N]: the residual goes through a LayerNorm,
        res' = (res - mu) * rs * gamma with (mu, rs) from res_stats (as lnin's stats).
    strict_norm: bound the accumulation by sum |A' w| (the error an fp32 GEMM on the normalised input would make)
        instead of the raw stream's sum |A w|: the bf16 bound the deferred LayerNorm is held to in the row-mean sweep.
    Returns (ref, tol, pre, pre_tol): the stored output and its bound, and the value before the epilogue's final
    rounding (what the statistics of stats_out are taken over) and its bound.
    """
    a, w, bias = f64(a), f64(w), f64(bias)
    K = a.shape[1]
    if lnin is not None:
        c, stats = lnin
        mu, rs, dmu, drs = row_stats(a, eps, stats)
        an = (a - mu[:, None]) * rs[:, None]
        pre = an @ w.T + bias
        raw = a @ w.T                                     # what the tensor cores accumulate
        c = f64(c)
        if strict_norm:
            pre_tol = 2 * K * U * (an.abs() @ w.abs().T) + 4 * U * (pre.abs() + bias.abs())
        else:
            acc = rs[:, None] * 2 * K * U * (a.abs() @ w.abs().T)
            acc = acc + 2 * U * rs[:, None] * mu.abs()[:, None] * c.abs()      # c rounded to fp32
            # rs * raw - rs * mu * c + b with perturbed rs, mu (the kernel's fp32 statistics)
            stat = (drs[:, None] * (raw - mu[:, None] * c).abs() + rs[:, None] * dmu[:, None] * c.abs())
            epi_r = 4 * U * (rs[:, None] * raw.abs() + (rs * mu).abs()[:, None] * c.abs() + bias.abs())
            pre_tol = acc + stat + epi_r
    else:
        pre = a @ w.T + bias
        pre_tol = 2 * K * U * (a.abs() @ w.abs().T) + 2 * U * (pre.abs() + bias.abs())
    if epi == "gelu":
        out = gelu_erf(pre)
        out_tol = GELU_DERIV_MAX * pre_tol + GELU_FIT_ABS + GELU_TANH_REL * pre.abs() / 2 + 4 * U * pre.abs()
    elif epi == "residual":
        r = f64(res)
        if res_gamma is not None:
            mu, rs, dmu, drs = row_stats(r, eps, res_stats)
            g = f64(res_gamma)[None, :]
            rn = (r - mu[:, None]) * rs[:, None]
            rterm = rn * g
            rtol = g.abs() * ((r - mu[:, None]).abs() * drs[:, None] + rs[:, None] * dmu[:, None]) \
                + 4 * U * g.abs() * (r.abs() * rs[:, None] + (mu * rs).abs()[:, None])
        else:
            rterm, rtol = r, torch.zeros_like(r)
        out = pre + rterm
        out_tol = pre_tol + rtol + 2 * U * (pre.abs() + rterm.abs())
    else:
        out, out_tol = pre, pre_tol
    return out, stored(out, out_tol), out, out_tol


def partials_tol(pre, pre_tol):
    """Bound on the kernel's fp32 (sum, sum sq) of 128 pre-rounding values per slot: their own error, plus a
    sequential fp32 sum of 128 terms (gamma_128)."""
    M = pre.shape[0]
    v = pre.reshape(M, -1, 128)
    t = pre_tol.reshape(M, -1, 128)
    ds = t.sum(-1) + 130 * U * v.abs().sum(-1)
    dss = (2 * v.abs() * t + t * t).sum(-1) + 130 * U * (v * v).sum(-1)
    return torch.stack([ds, dss], -1).transpose(0, 1).contiguous()


# ------------------------------------------------------------------------------------------------ attention
def attention(qkv, lens, B, S, split_kv=False, drop_last_key=False, admit_key=False, no_scale=False):
    """ctx [B*S, 768] = softmax(Q K^T / 8 + mask) V per (sequence, head); query rows t >= len are exactly 0.
    qkv [>= B*S, 2304] bf16 values; lens [B] (clamped to S).  The keyword defects exist for the comparator's tests."""
    x = f64(qkv[: B * S]).reshape(B, S, 3, HEADS, HD).permute(2, 0, 3, 1, 4)   # [3, B, heads, S, 64]
    q, k, v = x[0], x[1], x[2]
    L = torch.as_tensor(lens, device=qkv.device).to(torch.int64).clamp(0, S)
    scale = 1.0 if no_scale else 0.125
    logits = (q @ k.transpose(-1, -2)) * scale                                   # [B, h, S, S]
    t = torch.arange(S, device=qkv.device)
    kl = L - 1 if drop_last_key else (L + 1 if admit_key else L)
    keymask = t[None, :] < kl[:, None]                                           # [B, S]
    logits = logits.masked_fill(~keymask[:, None, None, :], float("-inf"))
    m = logits.amax(-1, keepdim=True)
    p = torch.exp(logits - torch.where(torch.isfinite(m), m, torch.zeros_like(m)))
    den = p.sum(-1, keepdim=True)
    den_safe = torch.where(den > 0, den, torch.ones_like(den))
    o = (p @ v) / den_safe
    pav = (p @ v.abs()) / den_safe                                               # sum p|v| / sum p
    # error of a logit (in nats): fp32 QK^T accumulation, the log2(e)/8 scaling and max subtraction, ex2.approx
    lq = torch.where(keymask[:, None, None, :], logits.abs(), torch.zeros_like(logits))
    dl = 2 * HD * U * (q.abs() @ k.abs().transpose(-1, -2)) * 0.125 + 4 * U * lq + 4 * U * m.abs().clamp(max=1e30)
    dl = torch.where(keymask[:, None, None, :], dl, torch.zeros_like(dl)).amax(-1, keepdim=True)
    # + P.V accumulated over 128 keys in fp32, the row sum (128 terms), 1 / sum and the scaling
    rel = 2.0 ** -8 + 2 * dl + 2 * 128 * U + 48 * U
    if split_kv:
        rel = rel + 2.0 ** -8 + 8 * U
    tol = pav * rel
    qmask = (t[None, :] < L[:, None])[:, None, :, None]                          # [B, 1, S, 1]
    o = torch.where(qmask, o, torch.zeros_like(o))
    tol = torch.where(qmask, tol, torch.zeros_like(tol))
    to_rows = lambda z: z.permute(0, 2, 1, 3).reshape(B * S, H)
    o = to_rows(o)
    return o, stored(o, to_rows(tol))


# ------------------------------------------------------------------------------------------------ small kernels
def _ln_rows(x, gamma, beta, eps, dx):
    """LayerNorm of rows x [M, 768] (fp64) and the bound of the kernel's fp32 two-pass evaluation, given an absolute
    error dx [M, 768] already in x."""
    mu, rs = exact_stats(x, eps)
    xc = x - mu[:, None]
    xh = xc * rs[:, None]
    g, b = f64(gamma)[None, :], f64(beta)[None, :]
    out = xh * g + b
    # sums of 768 terms as 24 sequential per lane + a 5-level butterfly: gamma_29
    dmu = dx.amax(-1) + 32 * U * x.abs().mean(-1)
    var = (xc * xc).mean(-1)
    dxc = dx + dmu[:, None]
    dvar = (2 * xc.abs() * dxc + dxc * dxc).mean(-1) + 32 * U * var
    drs_rel = dvar / (2 * (var + eps)) + 4 * U
    tol = g.abs() * (xh.abs() * drs_rel[:, None] + rs[:, None] * (dx + dmu[:, None])) \
        + 4 * U * (g.abs() * xh.abs() + b.abs())
    return out, stored(out, tol)


def embed_ln(ids, S, vocab, unk, word, pos, type0, gamma, beta, eps):
    """h0[m] = LN(word[id'] + pos[m % S] + type0), id' = unk for ids outside [0, vocab)."""
    ids = torch.as_tensor(ids).to(torch.int64).to(word.device)
    idc = torch.where((ids >= 0) & (ids < vocab), ids, torch.full_like(ids, unk))
    t = torch.arange(ids.numel(), device=word.device) % S
    w, p, ty = f64(word)[idc], f64(pos)[t], f64(type0)[None, :]
    x = w + p + ty
    dx = 2 * U * (w.abs() + p.abs() + ty.abs())
    return _ln_rows(x, gamma, beta, eps, dx)


def layernorm(x, gamma, beta, eps):
    x = f64(x)
    return _ln_rows(x, gamma, beta, eps, torch.zeros_like(x))


def pool_normalise(h, lens, B, S, normalise=True, out_bf16=False, drop_last=False):
    """Masked mean over the first min(len, S) tokens, then x / max(||x||, 1e-12); len <= 0 gives zeros."""
    x = f64(h[: B * S]).reshape(B, S, H)
    L = torch.as_tensor(lens, device=h.device).to(torch.int64).clamp(max=S)
    if drop_last:
        L = L - 1
    t = torch.arange(S, device=h.device)
    m = (t[None, :] < L[:, None]).to(torch.float64)[..., None]
    n = L.clamp(min=0).to(torch.float64)[:, None]
    nz = torch.where(n > 0, n, torch.ones_like(n))
    mean = (x * m).sum(1) / nz
    amean = (x.abs() * m).sum(1) / nz
    # sequential fp32 sum of len terms, a division
    d = (n + 2) * U * amean
    if normalise:
        nrm = mean.norm(dim=1, keepdim=True).clamp(min=1e-12)
        out = mean / nrm
        # |d(x/||x||)| <= 2 |dx| / ||x|| (dx the vector error); the fp32 norm (768-term sum) and the multiply
        dvec = d.norm(dim=1, keepdim=True)
        tol = 2 * dvec / nrm + 40 * U * out.abs() + 4 * U
    else:
        out, tol = mean, d + 2 * U * mean.abs()
    if out_bf16:
        tol = stored(out, tol)
    return out, tol


def token_head(h, w, b):
    """logits[m, l] = h[m] . w[l] + b[l] in fp32 (24-term FMA chains + a 5-level butterfly)."""
    h, w, b = f64(h), f64(w), f64(b)
    out = h @ w.T + b
    tol = 2 * 30 * U * (h.abs() @ w.abs().T) + 2 * U * (out.abs() + b.abs())
    return out, tol


# ------------------------------------------------------------------------------------------------ comparator
def ratio(got, ref, tol):
    """Per-element |got - ref| / tol (0 where both sides are equal, inf where tol is 0 and they differ; NaN -> inf)."""
    got, ref, tol = f64(got), f64(ref), f64(tol)
    err = (got - ref).abs()
    r = torch.where(err == 0, torch.zeros_like(err), err / tol)
    return torch.where(torch.isnan(r), torch.full_like(r, float("inf")), r)


def worst(got, ref, tol):
    return float(ratio(got, ref, tol).max()) if ref.numel() else 0.0


RATIOS = {}


def check(family, got, ref, tol, what=""):
    """Assert |got - ref| <= tol everywhere; record the worst ratio under `family` for the summary."""
    r = ratio(got, ref, tol)
    w = float(r.max()) if r.numel() else 0.0
    RATIOS[family] = max(RATIOS.get(family, 0.0), w)
    if not w <= 1.0:
        idx = tuple(int(i) for i in torch.nonzero(r == r.max())[0])
        raise AssertionError(f"{family} {what}: worst |err|/bound = {w:.3g} at {idx}: got {float(f64(got)[idx])!r} "
                             f"ref {float(f64(ref)[idx])!r} bound {float(f64(tol)[idx])!r}")
    return w
