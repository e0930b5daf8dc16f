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
            top_outside=32, chunk_rows=None):
    """The exact-search rule.  ids/raw/score: [B, k] results; rows: what the index holds; q: the fp32 queries;
    levels: [n] uint8; mask: [n] bool of the allowed rows (None = all); ref: reference(rows, q, f32rows) to reuse.
    chunk_rows: build the rules' summary (summarise) over row chunks of this size in fp64 instead of from the whole
    [B, n] score matrix, so that tables of millions of rows certify in bounded memory; the verdict is the same.

    Structural rules (AssertionError whatever `strict`): count min(k, allowed), unique, allowed, -inf / -1 tail,
    order (raw desc, id asc), or (raw * w desc, id asc) with WEIGHT_PRE, or the stable re-rank by
    float(double(raw) * w) with WEIGHT_RERANK, and scores as finalise_kernel computes them; an outside row tied exactly
    with a returned one must have the larger id.
    Bounded rules: |raw - exact| <= canonical bound per returned id; no allowed outside row beats a returned row by
    more than the two rows' combined bounds.  strict: AssertionError when either ratio exceeds 1."""
    if chunk_rows is None:
        e, d = reference(rows, q, f32rows) if ref is None else ref
        dev, n = e.device, e.shape[1]
        chunks = [(0, e, d)]
    else:
        dev, n = _t(q).device, rows.shape[0]
        chunks = ((r0, *reference(rows[r0:r0 + chunk_rows], q, f32rows)) for r0 in range(0, n, chunk_rows))
    B = q.shape[0]
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

    s = summarise(sel_ids, chunks, weight_mode, levels, allowed, top_outside)
    # |raw - exact| per returned id
    score_ratio = float(((raw_t[:, :want] - s["er"]).abs() / s["dr"].clamp_min(1e-300)).max())
    gap_ratio = 0.0
    if n_allowed > want:
        kj, dj, kr, drr, top_v, top_i = s["kj"], s["dj"], s["key"], s["dk"], s["lo"], s["id"]
        live = torch.isfinite(top_v)
        # pairwise (outside r, returned j)
        diff = kr[:, :, None] - kj[:, None, :]
        ratio = (diff / (drr[:, :, None] + dj[:, None, :]).clamp_min(1e-300)).masked_fill(~live[:, :, None], -math.inf)
        gap_ratio = max(0.0, float(ratio.max()))
        # the separable form of the same rule: max_r (key_r - dk_r) <= min_j (key_j + dk_j)
        sep = (top_v[:, 0] - (kj + dj).min(1).values)
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


def summarise(sel_ids, chunks, weight_mode, levels, allowed, top_outside=32):
    """The compact summary certify's bounded rules run on, accumulated over (row0, exact [B, m], bound [B, m]) chunks:
    er / dr, the exact score and bound of each returned id; kj / dj, its selection key and key bound; and the running
    top `top_outside` allowed rows outside the result by key - bound (lo), with their key, key bound and id."""
    dev = sel_ids.device
    B, want = sel_ids.shape
    w_all = weights_of(levels, dev) if weight_mode == WEIGHT_PRE else None
    z = torch.zeros((B, want), dtype=torch.float64, device=dev)
    out = {"er": z, "dr": z, "kj": z, "dj": z}
    top = [torch.empty((B, 0), dtype=torch.float64, device=dev) for _ in range(3)] + \
          [torch.empty((B, 0), dtype=torch.int64, device=dev)]
    for r0, e, d in chunks:
        e, d = e.to(dev), d.to(dev)
        m = e.shape[1]
        if weight_mode == WEIGHT_PRE:
            w = w_all[r0:r0 + m][None, :]
            key = e * w
            dk = d * w + 2 * U * key.abs()        # + the fp32 rounding of raw * w
        else:
            key, dk = e, d
        loc = sel_ids - r0
        here = (loc >= 0) & (loc < m)
        locc = loc.clamp(0, m - 1)
        for name, src in (("er", e), ("dr", d), ("kj", key), ("dj", dk)):
            out[name] = torch.where(here, src.gather(1, locc), out[name])
        inside = torch.zeros((B, m), dtype=torch.int32, device=dev).scatter_add_(1, locc, here.int()) > 0
        lo = (key - dk).masked_fill(~(allowed[None, r0:r0 + m] & ~inside), -math.inf)
        v, i = lo.topk(min(top_outside, m), dim=1)
        cand = [torch.cat([top[0], v], 1), torch.cat([top[1], key.gather(1, i)], 1),
                torch.cat([top[2], dk.gather(1, i)], 1), torch.cat([top[3], i + r0], 1)]
        v, j = cand[0].topk(min(top_outside, cand[0].shape[1]), dim=1)
        top = [v] + [c.gather(1, j) for c in cand[1:]]
    out.update(lo=top[0], key=top[1], dk=top[2], id=top[3])
    return out


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


# ------------------------------------------------------------------------------------------------ scan-side premises
# The certificate of finalise_kernel (DESIGN.md, "Exact search") rests on three properties of the tensor scan's own
# scores, checked one launch at a time by tests/test_scan_kernels_gpu.py:
#   (a) the merged list is the top kc by scan score;
#   (b) the pruning bound never exceeds the kc-th scan score (the pre-pass sees the main pass's bits);
#   (c) a scan score is within A + T of the exact score.
# These helpers give the bounds and the pre-pass model those tests compare against.
TILE = 128             # rows per accumulator tile (MMA N) of the tensor scan
PRE_SLOTS, PRE_FOLDS = 32, 4
MIN_KEY = -2139062144  # 0x80808080 as int32: the very negative key of an empty bound


def tc_term(dim):
    """Factor of sum |bf16(q)_i * bf16(c)_i| that bounds the tensor core's fp32 accumulation (DESIGN.md: 2 dim 2^-24)."""
    return 2.0 * dim * U


def scan_bound(q, rows):
    """Bound [B, n] of |tensor-scan score - exact q . rows| per (query, row), in the certificate's own terms.  The scan
    multiplies bf16(q) with bf16(rows) on the tensor cores: T = 2 dim 2^-24 sum |bf16 q_i bf16 c_i|, plus, where the
    query or the rows are not bf16 values, the exact input-rounding terms sum |q_i - bf16 q_i| |c_i| and
    sum |bf16 q_i| |c_i - bf16 c_i| (both zero for bf16 inputs)."""
    q = _t(q)
    rows = _t(rows, q.device)
    bq, bc = bf16_round(q.float()).double(), bf16_round(rows.float()).double()
    bound = tc_term(q.shape[1]) * (bq.abs() @ bc.abs().T)
    dq, dc = (q - bq).abs(), (rows - bc).abs()
    if bool(dq.any()):
        bound += dq @ rows.abs().T
    if bool(dc.any()):
        bound += bq.abs() @ dc.T
    return bound


def colstat_slack(q, colstat, f32rows):
    """Per-query (A, T, C) of finalise_kernel's certificate in fp64, from a colstat [2 dim + 2] as launch_column_stats
    leaves it: each term the smaller of its column-maxima form and its row-norm (Cauchy-Schwarz) form."""
    q = _t(q)
    cs = _t(colstat, q.device)
    dim = q.shape[1]
    M, D, Rn, Rd = cs[:dim], cs[dim:2 * dim], float(cs[2 * dim]), float(cs[2 * dim + 1])
    bq = bf16_round(q.float()).double()
    dq = q - bq
    nd = dq.norm(dim=1) * (1 + 1e-6)
    nb = bq.norm(dim=1) * (1 + 1e-6)
    nq = q.norm(dim=1) * (1 + 1e-6)
    A = torch.minimum(dq.abs() @ M, nd * Rn) + torch.minimum(bq.abs() @ D, nb * Rd)
    T = tc_term(dim) * torch.minimum(bq.abs() @ M, nb * Rn)
    L = lanes_fmas(dim, f32rows)
    C = (L + 5) * U * torch.minimum(q.abs() @ (M + D), nq * (Rn + Rd))
    return A, T, C


def float_key(x):
    """common.cuh float_key: the order-preserving int32 key of fp32 values (numpy)."""
    i = np.ascontiguousarray(x, np.float32).view(np.int32)
    return np.where(i >= 0, i, i ^ np.int32(0x7fffffff)).astype(np.int32)


def sampled_tiles(n_rows, stride):
    """Row tiles a pass at tile stride `stride` scans: tile index t' of the pass covers rows [t' s 128, t' s 128 + 128)."""
    tiles = -(-n_rows // TILE)
    return -(-tiles // max(1, stride))


def tile_groups(n_tiles, G):
    """Row group of each of the n_tiles tiles of a pass: group g owns tiles [n_tiles g / G, n_tiles (g + 1) / G)."""
    g = np.arange(G)
    owner = np.empty(n_tiles, np.int64)
    for gi, (a, b) in enumerate(zip(n_tiles * g // G, n_tiles * (g + 1) // G)):
        owner[a:b] = gi
    return owner


def slot_sets(n_rows, stride, G):
    """The slot pre-pass's partition of the sampled rows: (rows, group, slot, class) for every sampled row r < n_rows;
    slot = r mod 32 (the accumulator column mod 32), class = group mod 4 (bound_from_slots_kernel's fold)."""
    nt = sampled_tiles(n_rows, stride)
    owner = tile_groups(nt, G)
    t = np.repeat(np.arange(nt), TILE)
    col = np.tile(np.arange(TILE), nt)
    rows = t * max(1, stride) * TILE + col
    keep = rows < n_rows
    rows, t, col = rows[keep], t[keep], col[keep]
    g = owner[t]
    return rows, g, col % PRE_SLOTS, g % PRE_FOLDS


def expected_slot_max(scores, n_rows, stride, G, allowed=None):
    """[B, G, 32] slot maxima the pre-pass must write, from the scores [B, n] (fp32, weights already applied) of every
    row; masked-out rows and empty sets give -inf."""
    s = np.asarray(scores, np.float32)
    rows, g, slot, _ = slot_sets(n_rows, stride, G)
    if allowed is not None:
        keep = np.asarray(allowed, bool)[rows]
        rows, g, slot = rows[keep], g[keep], slot[keep]
    out = np.full((s.shape[0], G * PRE_SLOTS), -np.inf, np.float32)
    idx = g * PRE_SLOTS + slot
    for b in range(s.shape[0]):
        np.maximum.at(out[b], idx, s[b, rows])
    return out.reshape(s.shape[0], G, PRE_SLOTS)


def bound_from_slots(slot_max, kc):
    """Keys [B] of bound_from_slots_kernel: the slot maxima folded over the row groups of each class g mod 4, and the
    kc-th largest of the 128 fold maxima (ties by fold index), or MIN_KEY when that is -inf."""
    sm = np.asarray(slot_max, np.float32)
    B, P, S = sm.shape
    folds = np.full((B, PRE_FOLDS, S), -np.inf, np.float32)
    for f in range(PRE_FOLDS):
        if f < P:
            folds[:, f] = sm[:, f::PRE_FOLDS].max(1)
    v = folds.reshape(B, PRE_FOLDS * S)
    o = np.lexsort((np.broadcast_to(np.arange(v.shape[1]), v.shape), -v.astype(np.float64)), axis=-1)
    kth = np.take_along_axis(v, o[:, kc - 1:kc], 1)[:, 0]
    return np.where(np.isneginf(kth), MIN_KEY, float_key(kth)).astype(np.int32)
