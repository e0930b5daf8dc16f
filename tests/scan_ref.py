"""fp64 reference, derived error bounds and an exactness certificate for the two scan kernels.

The index returns, per query, the top-k rows by the CANONICAL fp32 score: the dot of the fp32 query with the row the index
holds (the bf16 image, or the fp32 master with keep_f32) accumulated in the fixed lane order of `finalise_kernel`
(topk_merge.cu, warp_dot_row) and `scan_stream_kernel`.  This module checks a result against the exact (fp64) scores of
those same inputs, with a bound derived from that arithmetic, so that a kernel which loses a true top-k row fails even
when the row it returned instead is only a few 1e-5 worse -- far inside parity.py's TIE_TOL.

- exact_scores(rows, q):       fp64 scores [B, n] of what the index holds.
- canonical_bound(q, rows):    per (query, row) bound of the canonical fp32 dot's rounding error.
- certify(...):                the rule the exact-search tests apply; returns the worst error / bound.

Everything takes numpy arrays or torch tensors (CPU or CUDA) and computes in torch.float64 on the tensors' device.
"""
from __future__ import annotations

import math
from dataclasses import dataclass

import numpy as np
import torch

U = 2.0 ** -24                    # unit roundoff of fp32
WEIGHTS = (1.0, 1.2, 1.0, 0.8)    # level weights, common.cuh level_weight_d (services/milvus_service.py:550-558)
WEIGHT_RERANK, WEIGHT_PRE, WEIGHT_NONE = 0, 1, 2


def _t(x, device=None, dtype=torch.float64):
    if isinstance(x, np.ndarray):
        x = torch.from_numpy(np.ascontiguousarray(x))
    if device is not None:
        x = x.to(device)
    return x.to(dtype) if dtype is not None else x


def bf16_round(x):
    """Round-to-nearest-even to bf16, returned as fp32 (what f32_to_bf16_kernel stores)."""
    if isinstance(x, np.ndarray):
        return torch.from_numpy(np.ascontiguousarray(x, np.float32)).to(torch.bfloat16).float().numpy()
    return x.to(torch.bfloat16).float()


def held_rows(corpus_f32, keep_f32):
    """What an index built from fp32 rows holds and rescores against: the fp32 master, or the bf16 image."""
    return corpus_f32 if keep_f32 else bf16_round(corpus_f32)


def exact_scores(rows, q):
    """fp64 [B, n] = q . rows^T over the inputs the index holds (rows: [n, dim] master or bf16 values, q: [B, dim] fp32)."""
    q = _t(q)
    return q @ _t(rows, q.device).T


def lanes_fmas(dim, f32rows):
    """fmas per lane of the canonical dot: E elements per 16-byte chunk, chunk c on lane c % 32."""
    E = 4 if f32rows else 8
    return E * math.ceil(dim / (32 * E))


def canonical_bound(q, rows, f32rows=False):
    """Bound [B, n] of |canonical fp32 dot - exact dot|: each lane runs L = E * ceil(dim / 32E) fmas, then a 5-level
    xor butterfly adds the lanes; every fp32 operation contributes at most 2^-24 of a partial sum bounded by
    sum |q_i c_i|.  Derived from the arithmetic of warp_dot_row, not fitted."""
    q = _t(q)
    rows = _t(rows, q.device)
    L = lanes_fmas(q.shape[1], f32rows)
    return (L + 5) * U * (q.abs() @ rows.abs().T)


def weights_of(levels, device=None):
    lv = _t(levels, device, dtype=torch.int64)
    return torch.tensor(WEIGHTS, dtype=torch.float64, device=lv.device)[lv]


@dataclass
class Certificate:
    score_ratio: float      # max |raw - exact| / canonical bound over the returned ids
    gap_ratio: float        # max (exact(outside) - exact(returned)) / (combined bound), 0 when no outside row beats
    worst: float            # max of the two: <= 1 passes

    def __repr__(self):
        return f"Certificate(score {self.score_ratio:.3g}, gap {self.gap_ratio:.3g})"


def reference(rows, q, f32rows=False):
    """(exact scores, canonical bound) for one (rows, queries) pair, to reuse across several result sets."""
    return exact_scores(rows, q), canonical_bound(q, rows, f32rows)


def _np(x):
    return x.detach().cpu().numpy() if isinstance(x, torch.Tensor) else np.asarray(x)


def _check_order(ids, raw, score, levels, weight_mode):
    """Order and score rules of finalise_kernel, on the returned values themselves (host, numpy)."""
    B, k = ids.shape
    valid = ids >= 0
    lv = np.zeros_like(ids, dtype=np.int64)
    lv[valid] = levels[ids[valid]]
    w64 = np.asarray(WEIGHTS, np.float64)[lv]
    w32 = w64.astype(np.float32)
    big = np.iinfo(np.int64).max
    id_key = np.where(valid, ids, big)
    if weight_mode == WEIGHT_PRE:
        sel = np.where(valid, raw * w32, -np.inf).astype(np.float32)        # fp32 key = raw * level_weight_f
    else:
        sel = np.where(valid, raw, -np.inf).astype(np.float32)
    order = np.lexsort((id_key, -sel.astype(np.float64)), axis=-1)          # (key desc, id asc)
    if weight_mode == WEIGHT_RERANK:
        wsel = np.take_along_axis(np.where(valid, raw.astype(np.float64) * w64, -np.inf), order, -1)
        order = np.take_along_axis(order, np.argsort(-wsel, axis=-1, kind="stable"), -1)
        want_score = np.where(valid, (raw.astype(np.float64) * w64).astype(np.float32), -np.inf)
    elif weight_mode == WEIGHT_PRE:
        want_score = sel
    else:
        want_score = np.where(valid, raw, -np.inf).astype(np.float32)
    bad = np.nonzero((order != np.arange(k)[None, :]).any(1))[0]
    assert bad.size == 0, f"query {bad[0]}: order {ids[bad[0]]} is not the kernel's rule (want {ids[bad[0]][order[bad[0]]]})"
    bad = np.nonzero((score.view(np.uint32) != want_score.view(np.uint32)).any(1))[0]
    assert bad.size == 0, f"query {bad[0]}: scores {score[bad[0]]} != {want_score[bad[0]]}"


def certify(ids, raw, score, rows, q, k, weight_mode, levels, mask=None, f32rows=False, ref=None, strict=True,
            top_outside=32):
    """The exact-search rule.  ids/raw/score: [B, k] results; rows: what the index holds; q: the fp32 queries;
    levels: [n] uint8; mask: [n] bool of the allowed rows (None = all); ref: reference(rows, q, f32rows) to reuse.

    Structural rules (AssertionError whatever `strict`): count min(k, allowed), unique, allowed, -inf / -1 tail,
    order (raw desc, id asc), or (raw * w desc, id asc) with WEIGHT_PRE, or the stable re-rank by
    float(double(raw) * w) with WEIGHT_RERANK, and scores as finalise_kernel computes them; an outside row tied exactly
    with a returned one must have the larger id.
    Bounded rules: |raw - exact| <= canonical bound per returned id; no allowed outside row beats a returned row by
    more than the two rows' combined bounds.  strict: AssertionError when either ratio exceeds 1."""
    e, d = reference(rows, q, f32rows) if ref is None else ref
    dev = e.device
    B, n = e.shape
    ids_t = _t(ids, dev, torch.int64)
    raw_t = _t(raw, dev, torch.float64)
    assert ids_t.shape == (B, k), (tuple(ids_t.shape), (B, k))
    allowed = torch.ones(n, dtype=torch.bool, device=dev) if mask is None else _t(mask, dev, torch.bool)
    n_allowed = int(allowed.sum())
    want = min(k, n_allowed)
    valid = ids_t >= 0
    # count, prefix, tail
    assert bool((valid.sum(1) == want).all()), f"result counts {valid.sum(1).unique().tolist()} != min(k, allowed) = {want}"
    assert bool(valid[:, :want].all()), "empty slots before the end of the list"
    assert bool(torch.isneginf(raw_t[:, want:]).all()), "tail raw scores are not -inf"
    assert bool((ids_t[:, want:] == -1).all()), "tail ids are not -1"
    ids_h = _np(ids_t)
    raw_h = _np(_t(raw, None, torch.float32)).astype(np.float32)
    score_h = _np(_t(score, None, torch.float32)).astype(np.float32)
    lv_h = _np(levels).astype(np.int64)
    if want == 0:
        return Certificate(0.0, 0.0, 0.0)
    sel_ids = ids_t[:, :want]
    assert bool((sel_ids < n).all()), "id out of range"
    srt = sel_ids.sort(1).values
    assert bool((srt[:, 1:] != srt[:, :-1]).all()), "duplicate ids"
    assert bool(allowed[sel_ids].all()), "a masked-out row was returned"
    _check_order(ids_h, raw_h, score_h, lv_h, weight_mode)

    # |raw - exact| per returned id
    er = e.gather(1, sel_ids)
    dr = d.gather(1, sel_ids)
    score_ratio = float(((raw_t[:, :want] - er).abs() / dr.clamp_min(1e-300)).max())

    # selection key and its bound
    if weight_mode == WEIGHT_PRE:
        w = weights_of(levels, dev)[None, :]
        key = e * w
        dk = d * w + 2 * U * key.abs()        # + the fp32 rounding of raw * w
    else:
        key, dk = e, d
    inside = torch.zeros((B, n), dtype=torch.bool, device=dev)
    inside.scatter_(1, sel_ids, True)
    outside = allowed[None, :] & ~inside
    gap_ratio = 0.0
    if n_allowed > want:
        kj, dj = key.gather(1, sel_ids), dk.gather(1, sel_ids)
        lo = (key - dk).masked_fill(~outside, -math.inf)
        T = min(top_outside, n)
        top_v, top_i = lo.topk(T, dim=1)
        kr, drr = key.gather(1, top_i), dk.gather(1, top_i)
        live = torch.isfinite(top_v)
        # pairwise (outside r, returned j)
        diff = kr[:, :, None] - kj[:, None, :]
        ratio = (diff / (drr[:, :, None] + dj[:, None, :]).clamp_min(1e-300)).masked_fill(~live[:, :, None], -math.inf)
        gap_ratio = max(0.0, float(ratio.max()))
        # the separable form of the same rule: max_r (key_r - dk_r) <= min_j (key_j + dk_j)
        sep = (lo.max(1).values - (kj + dj).min(1).values)
        if bool((sep > 0).any()):
            gap_ratio = max(gap_ratio, 1.0 + 1e-12)
        # an exact tie broken the wrong way: an outside row with the same exact key and a lower id
        tie = (kr[:, :, None] == kj[:, None, :]) & (top_i[:, :, None] < sel_ids[:, None, :]) & live[:, :, None]
        bad = torch.nonzero(tie.any(2).any(1)).flatten()
        assert bad.numel() == 0, f"query {int(bad[0])}: an exactly tied row with a lower id was left out"
    cert = Certificate(score_ratio, gap_ratio, max(score_ratio, gap_ratio))
    if strict:
        assert cert.score_ratio <= 1.0, f"returned raw scores off the exact ones by {cert.score_ratio:.3g}x the bound"
        assert cert.gap_ratio <= 1.0, f"an allowed row left out beats a returned one by {cert.gap_ratio:.3g}x the bound"
    return cert


# ------------------------------------------------------------------------------------------------ probe corpora
BK = 64                                            # K block of the tensor scan (64 bf16 = one 128-byte swizzle row)
LANE_PROBES = (0, 31, 32, 63, 64, 95, 96, 127)     # query-tile lanes at TMEM lane-quarter and warp edges


def _unit(x):
    return x / np.linalg.norm(x, axis=-1, keepdims=True)


def probe_corpus(n, dim, B, seed, spare_rows=()):
    """Random unit rows and queries with planted answers that a subtly wrong scan loses.  Returns (rows [n, dim] fp32,
    q [B, dim] fp32, plants {query: row}), the planted row being the query's clear best:

    - K-block probes: a query whose signal lies in one 64-wide K block only, and a row that matches it element for
      element there and is random elsewhere -- a dropped, misplaced or mis-swizzled K block loses that row;
    - row probes: planted best rows at ids 0, 127, 128, a sample of 128 m tile boundaries, and n - 1 (in a partial last
      tile when n % 128 != 0);
    - query-lane probes: distinct planted rows for the queries at tile lanes 0, 31, 32, 63, 64, 95, 96, 127 and B - 1,
      so a lane or TMEM-quarter mix-up returns a wrong id rather than a near-tie.
    spare_rows: ids that stay random (a caller's own plants)."""
    rng = np.random.default_rng(seed)
    rows = _unit(rng.standard_normal((n, dim))).astype(np.float32)
    q = _unit(rng.standard_normal((B, dim))).astype(np.float32)
    bounds = [128 * m for m in range(1, (n - 1) // 128 + 1)]
    if len(bounds) > 6:
        bounds = bounds[:2] + sorted(rng.choice(bounds[2:], 4, replace=False).tolist())
    row_ids = [r for r in dict.fromkeys([0, 127, 128] + bounds + [n - 1]) if 0 <= r < n and r not in spare_rows]
    lanes = [l for l in dict.fromkeys(list(LANE_PROBES) + [B - 1]) if l < B]
    nkb = dim // BK
    kb_lanes = [l for l in range(B) if l not in lanes][:nkb]
    free = [r for r in rng.permutation(n).tolist() if r not in row_ids and r not in spare_rows]
    plants = {}
    # query-lane probes on the row-probe ids first, then on random rows
    for l in lanes:
        r = row_ids.pop(0) if row_ids else (free.pop() if free else None)
        if r is None:
            break
        rows[r] = _unit(q[l] + 0.2 * _unit(rng.standard_normal(dim)))
        plants[l] = r
    for b, l in enumerate(kb_lanes):
        r = row_ids.pop(0) if row_ids else (free.pop() if free else None)
        if r is None:
            break
        u = _unit(rng.standard_normal(BK)).astype(np.float32)
        q[l] = 0.0
        q[l, b * BK:(b + 1) * BK] = u
        row = _unit(rng.standard_normal(dim)) * 0.7
        row[b * BK:(b + 1) * BK] = 0.7 * u
        rows[r] = row
        plants[l] = r
    return rows.astype(np.float32), q.astype(np.float32), plants
