"""fp64 references of the encoder kernels at hidden 1024 / 16 heads (BERT-large, XLM-RoBERTa-large).

tests/encoder_ref.py is written in terms of its module constants H and HEADS.  `ref` below is a second, independent
instance of that module with H = 1024 and HEADS = 16, so the 768 references and their recorded ratios are untouched.
Three bounds count the terms of a fp32 sum, which grow with the width; they are restated here:

* LayerNorm (a warp per row): H / 32 = 32 sequential terms per lane + a 5-level butterfly, gamma_37 (768: gamma_29);
* token head: 32-term FMA chains + a 5-level butterfly (768: 24 + 5);
* row statistics the skinny kernel sums itself: 16 x 8 = 128 sequential terms per lane + 3 shuffle levels (768: 96 + 3).

embed_ln takes the position offset of XLM-R (token t reads position row offset + t).
"""
import importlib.util
import os
import sys

import torch

_HERE = os.path.dirname(os.path.abspath(__file__))
if _HERE not in sys.path:
    sys.path.insert(0, _HERE)

_spec = importlib.util.spec_from_file_location("wide_encoder_ref_1024", os.path.join(_HERE, "encoder_ref.py"))
ref = importlib.util.module_from_spec(_spec)
_spec.loader.exec_module(ref)
ref.H, ref.HEADS = 1024, 16
U, f64, stored = ref.U, ref.f64, ref.stored


def _ln_rows(x, gamma, beta, eps, dx):
    mu, rs = ref.exact_stats(x, eps)
    xc = x - mu[:, None]
    xh = xc * rs[:, None]
    g, b = f64(gamma)[None, :], f64(beta)[None, :]
    out = xh * g + b
    dmu = dx.amax(-1) + 40 * U * x.abs().mean(-1)           # gamma_37
    var = (xc * xc).mean(-1)
    dxc = dx + dmu[:, None]
    dvar = (2 * xc.abs() * dxc + dxc * dxc).mean(-1) + 40 * U * var
    drs_rel = dvar / (2 * (var + eps)) + 4 * U
    tol = g.abs() * (xh.abs() * drs_rel[:, None] + rs[:, None] * (dx + dmu[:, None])) \
        + 4 * U * (g.abs() * xh.abs() + b.abs())
    return out, stored(out, tol)


def embed_ln(ids, S, vocab, unk, word, pos, type0, gamma, beta, eps, pos_offset=0):
    """h0[m] = LN(word[id'] + pos[pos_offset + m % S] + type0), id' = unk for ids outside [0, vocab)."""
    ids = torch.as_tensor(ids).to(torch.int64).to(word.device)
    idc = torch.where((ids >= 0) & (ids < vocab), ids, torch.full_like(ids, unk))
    t = torch.arange(ids.numel(), device=word.device) % S + pos_offset
    w, p, ty = f64(word)[idc], f64(pos)[t], f64(type0)[None, :]
    x = w + p + ty
    dx = 2 * U * (w.abs() + p.abs() + ty.abs())
    return _ln_rows(x, gamma, beta, eps, dx)


def token_head(h, w, b):
    h, w, b = f64(h), f64(w), f64(b)
    out = h @ w.T + b
    tol = 2 * 38 * U * (h.abs() @ w.abs().T) + 2 * U * (out.abs() + b.abs())
    return out, tol


_row_stats_768 = ref.row_stats


def row_stats(x, eps, stats, slots=None):
    if isinstance(stats, str):
        x = f64(x)
        s, ss = x.sum(-1), (x * x).sum(-1)
        e_s, e_ss = 140 * U * x.abs().sum(-1), 140 * U * ss
        mu = s / ref.H
        var = ss / ref.H - mu * mu
        rs, dmu, drs = ref._stats_bounds(mu, var, ss, e_s, e_ss, eps)
        return mu, rs, dmu, drs
    return _row_stats_768(x, eps, stats, slots)


# the module's own callers (layernorm -> _ln_rows, linear -> row_stats) resolve these names in `ref`
ref._ln_rows, ref.embed_ln, ref.token_head, ref.row_stats = _ln_rows, embed_ln, token_head, row_stats
