"""Reference model of icd_index_search_page (include/icdrag.h), and a numpy emulation of the algorithm of
csrc/topk_large.cu, for the paged-search tests.

page_ref states the contract directly: from the canonical fp32 scores [B, n], drop the rows the mask or the range
(radius, range_filter] on the raw score excludes, order the rest by (key desc, id asc) -- key = raw, or the fp32
raw * w(level) under WEIGHT_PRE -- keep the first K = offset + limit, re-sort them by double(raw) * w(level) stably under
WEIGHT_RERANK, and return [offset, offset + limit) with a (-inf, -1) tail.

page_emulate runs the kernels' steps instead: order-preserving uint32 keys with one key for -0.0 / +0.0 and 0 for
excluded rows, a four-pass 8-bit radix select of the K-th key, the gather of the rows above it plus the lowest-id ties,
a sort of (key, ~id), and the WEIGHT_RERANK merge of the three level runs by binary search.
"""
import numpy as np

WEIGHT_RERANK, WEIGHT_PRE, WEIGHT_NONE = 0, 1, 2
W64 = np.array([1.0, 1.2, 1.0, 0.8], np.float64)     # level 0 (unknown) weighs 1.0; common.cuh level_weight_d
W32 = W64.astype(np.float32)                          # level_weight_f
MAX_LIMIT = 16384


def _allowed(raw, mask, radius, range_filter):
    ok = np.ones(raw.shape, bool) if mask is None else np.broadcast_to(np.asarray(mask, bool), raw.shape).copy()
    if radius is not None:
        ok &= raw > np.float32(radius)
    if range_filter is not None:
        ok &= raw <= np.float32(range_filter)
    return ok


def _lv(levels):
    lv = np.asarray(levels).astype(np.int64)
    return np.where((lv >= 1) & (lv <= 3), lv, 0)


def _out(B, limit):
    return (np.full((B, limit), -np.inf, np.float32), np.full((B, limit), -np.inf, np.float32),
            np.full((B, limit), -1, np.int64))


def _write(out, b, page, raw_b, lv, weight_mode):
    score, raw, ids = out
    m = len(page)
    ids[b, :m] = page
    raw[b, :m] = raw_b[page]
    if weight_mode == WEIGHT_RERANK:
        score[b, :m] = (raw_b[page].astype(np.float64) * W64[lv[page]]).astype(np.float32)
    elif weight_mode == WEIGHT_PRE:
        score[b, :m] = raw_b[page] * W32[lv[page]]
    else:
        score[b, :m] = raw_b[page]


def page_ref(raw, levels, weight_mode, offset, limit, mask=None, radius=None, range_filter=None):
    """raw: [B, n] float32 canonical scores; levels [n]; mask [n] bool or None.  -> (score, raw, ids) [B, limit]."""
    raw = np.asarray(raw, np.float32)
    B, n = raw.shape
    lv = _lv(levels)
    ok = _allowed(raw, mask, radius, range_filter)
    K = offset + limit
    out = _out(B, limit)
    for b in range(B):
        ids = np.nonzero(ok[b])[0]
        r = raw[b, ids]
        key = r * W32[lv[ids]] if weight_mode == WEIGHT_PRE else r
        lst = ids[np.lexsort((ids, -key.astype(np.float64)))][:K]     # -0.0 == +0.0: the id decides
        if weight_mode == WEIGHT_RERANK:
            tw = raw[b, lst].astype(np.float64) * W64[lv[lst]]
            lst = lst[np.argsort(-tw, kind="stable")]
        _write(out, b, lst[offset:K], raw[b], lv, weight_mode)
    return out


def sel_key(raw, lv, pre, excluded):
    """topk_large.cu sel_key: uint32 keys ordered like the selection scores, -0.0 and +0.0 one key, 0 = excluded."""
    k = raw * W32[lv] if pre else raw.copy()
    k = np.where(k == 0, np.float32(0.0), k).astype(np.float32)
    u = k.view(np.uint32)
    u = np.where(u & np.uint32(0x80000000), ~u, u | np.uint32(0x80000000)).astype(np.uint32)
    u = np.maximum(u, np.uint32(1))
    return np.where(excluded, np.uint32(0), u).astype(np.uint32)


def radix_kth(keys, K):
    """The K-th largest key by four 8-bit passes (page_hist_kernel / page_choose_kernel); len(keys) > K."""
    prefix, krem = 0, K
    for p in range(4):
        shift = 24 - 8 * p
        hi = (0xffffffff << (shift + 8)) & 0xffffffff if p else 0
        grp = keys[(keys & np.uint32(hi)) == np.uint32(prefix)]
        h = np.bincount((grp >> np.uint32(shift)) & np.uint32(255), minlength=256)
        cum, b = 0, 255
        while b > 0:
            if cum + h[b] >= krem:
                break
            cum += h[b]
            b -= 1
        prefix |= b << shift
        krem -= cum
    return np.uint32(prefix)


def page_emulate(raw, levels, weight_mode, offset, limit, mask=None, radius=None, range_filter=None, block_rows=8192):
    raw = np.asarray(raw, np.float32)
    B, n = raw.shape
    lv = _lv(levels)
    ok = _allowed(raw, mask, radius, range_filter)
    K = offset + limit
    out = _out(B, limit)
    pre = weight_mode == WEIGHT_PRE
    for b in range(B):
        keys = sel_key(raw[b], lv, pre, ~ok[b])
        kth = radix_kth(keys, K) if n > K else np.uint32(0)
        # per-block counts, exclusive scan, block-ordered writes (page_count / page_scan / page_gather)
        gt_rows, eq_rows = [], []
        for r0 in range(0, n, block_rows):
            blk = keys[r0:r0 + block_rows]
            gt_rows.append(r0 + np.nonzero(blk > kth)[0])
            eq_rows.append(r0 + np.nonzero(blk == kth)[0] if kth > 0 else np.zeros(0, np.int64))
        gt = np.concatenate(gt_rows) if gt_rows else np.zeros(0, np.int64)
        eq = np.concatenate(eq_rows) if eq_rows else np.zeros(0, np.int64)
        gt = gt[:K]
        ties = eq[:K - len(gt)]
        cand = np.concatenate([gt, ties]).astype(np.int64)
        # sort of (key << 32 | ~id), descending
        packed = (keys[cand].astype(np.uint64) << np.uint64(32)) | (~cand.astype(np.uint32)).astype(np.uint64)
        lst = cand[np.argsort(packed)[::-1]]          # ids are distinct, so are the packed values
        if weight_mode == WEIGHT_RERANK:
            cls = np.where(lv[lst] == 1, 0, np.where(lv[lst] == 3, 2, 1))
            runs = [np.nonzero(cls == c)[0] for c in range(3)]         # list positions, in list order
            cw = (1.2, 1.0, 0.8)
            rank = np.empty(len(lst), np.int64)
            for c in range(3):
                for i, p in enumerate(runs[c]):
                    tw = np.float64(raw[b, lst[p]]) * cw[c]
                    rk = i
                    for c2 in range(3):
                        if c2 == c:
                            continue
                        t2 = raw[b, lst[runs[c2]]].astype(np.float64) * cw[c2]
                        before = (t2 > tw) | ((t2 == tw) & (runs[c2] < p))
                        m = int(before.sum())
                        assert before[:m].all(), "the rows of a run that precede an element are not a prefix"
                        rk += m                               # what the kernel's binary search finds
                    rank[p] = rk
            reordered = np.empty_like(lst)
            reordered[rank] = lst
            lst = reordered
        _write(out, b, lst[offset:K], raw[b], lv, weight_mode)
    return out
