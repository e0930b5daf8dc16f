"""Kernel-level parity of the scan side: the tensor scan, the pre-pass bound, the merge, the finalise certificate and
the column statistics, one launch at a time, against fp64 and numpy references (tests/scan_ref.py).

The exact-search tests (test_scan_exact_gpu.py) check final results; finalise_kernel rescores every candidate and the
kc - k margin hides a candidate lost below rank k, so those tests cannot see the premises the certificate rests on
(DESIGN.md, "Exact search"):
  (a) the merged list is the top kc by scan score;
  (b) the pruning bound never exceeds the kc-th scan score: the pre-pass sees the main pass's bits for every
      (query, row), whatever launch shape either picks;
  (c) a scan score is within A + T of the exact score, T = 2 dim 2^-24 sum |bf16(q) c|.
Here they are checked directly.  A group's rows fit its list when n <= 128 G and kc = 128, so an unpruned main scan
then writes EVERY (query, row) scan score into its partial lists.

The launchers are internal C++ functions; tests/scan_kernel_shim.cu exposes them as extern "C" entries.  The module
fixture compiles it into pytest's temporary directory (never into the checkout) and links it against the built
csrc/libicdrag.so.  The tensor scan's CTAs wait on each other through the drift-limiter counters, so only `Scan.run`
launches it, always with a zeroed counter region of tensor_scan_progress_ints() ints and P = tensor_scan_max_partials(),
as index_search_device does.  The worst error / bound per (kernel, case) is printed at the end of the module."""
import ctypes as C
import os
import subprocess

import numpy as np
import pytest
import torch

import encoder_ref
import scan_ref as R

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CSRC = os.path.join(ROOT, "rag-project-icd10_b200", "csrc")
DEV = "cuda"
TC_DIMS = list(range(64, 769, 64))
WORST = {}      # (kernel, case) -> worst error / bound
GUARD_F, GUARD_I = 12345.0, -7


@pytest.fixture(scope="module", autouse=True)
def _report(request):
    yield
    tr = request.config.pluginmanager.get_plugin("terminalreporter")
    capman = request.config.pluginmanager.get_plugin("capturemanager")
    if tr is None or capman is None or not WORST:
        return
    with capman.global_and_fixture_disabled():
        tr.write_line("")
        tr.write_line("worst error / bound per (kernel, case) (<= 1 passes):")
        for key in sorted(WORST):
            tr.write_line(f"  {key[0]:<22s} {key[1]:<28s} {WORST[key]:.3f}")


def _record(kernel, case, ratio):
    WORST[(kernel, case)] = max(WORST.get((kernel, case), 0.0), float(ratio))


# ------------------------------------------------------------------------------------------------ shim
@pytest.fixture(scope="module")
def shim(tmp_path_factory, native):
    nvcc = encoder_ref.nvcc_path()
    assert nvcc, "nvcc is needed to build the scan kernel shim"
    assert os.path.exists(os.path.join(CSRC, "libicdrag.so")), "build() first"
    out = str(tmp_path_factory.mktemp("scanshim") / "libscanshim.so")
    cmd = [nvcc, "-gencode", "arch=compute_100a,code=sm_100a", "-std=c++17", "-shared", "-Xcompiler", "-fPIC",
           "-cudart", "none", "-I", CSRC, "-I", os.path.join(ROOT, "include"),
           os.path.join(ROOT, "tests", "scan_kernel_shim.cu"), "-L", CSRC, "-licdrag",
           "-Xlinker", "-rpath," + CSRC, "-o", out]
    r = subprocess.run(cmd, capture_output=True, text=True)
    assert r.returncode == 0, r.stderr
    native.lib()                      # the shim binds to this already-loaded libicdrag (same file)
    L = C.CDLL(out)
    vp, i32, i64 = C.c_void_p, C.c_int, C.c_long
    L.shim_tensor_scan.argtypes = [vp, vp, i64, i32, vp, i32, i32, i32, vp, vp, i32, vp, vp, i32, i32, vp,
                                   C.POINTER(i32), vp]
    L.shim_bound_from_slots.argtypes = [vp, i32, i32, i32, i32, vp, vp]
    L.shim_merge.argtypes = [vp, vp, i32, i32, i32, i32, vp, vp, i64, vp, vp, vp]
    L.shim_finalise.argtypes = [vp, vp, i32, i32, i32, i64, i64, vp, vp, i32, i32, vp, i32, vp, vp, vp, vp, vp, vp,
                                vp, vp]
    L.shim_column_stats.argtypes = [vp, vp, i64, i64, i32, vp, vp]
    L.shim_tensor_scan_sample_stride.argtypes = [i64, i32]
    return L


def _p(t):
    return None if t is None else C.c_void_p(t.data_ptr())


def _stream():
    return C.c_void_p(torch.cuda.current_stream().cuda_stream)


def _ok(native, status, what):
    if status != 0:
        raise AssertionError(f"{what}: status {status}: {native.lib().icd_last_error().decode()}")


class Scan:
    """The tensor scan and the kernels around it, launched the way index_search_device launches them."""

    def __init__(self, shim, native):
        self.L, self.native = shim, native
        self.P = shim.shim_tensor_scan_max_partials()
        self.slots = shim.shim_tensor_scan_pre_slots()
        self.prog_ints = shim.shim_tensor_scan_progress_ints()

    def run(self, table, levels, qb, kc, weight_pre=0, bound=None, stride=1, pre_slots=0, mask=None):
        """One launch_tensor_scan.  bound: None = no pruning (gbound null), "fresh" = gbound preset to the very negative
        key, or an int32 [B] tensor of keys to start from (copied).  Returns (part_score, part_id, G, gbound) with the
        partial buffers viewed [B, G, kc] (the pre-pass with pre_slots: [B, G, 32] slot maxima)."""
        B = qb.shape[0]
        n, dim = table.shape
        width = self.slots if pre_slots else kc
        ps = torch.full((B * self.P * max(kc, self.slots),), GUARD_F, dtype=torch.float32, device=DEV)
        pi = torch.full((B * self.P * kc,), GUARD_I, dtype=torch.int32, device=DEV)
        progress = torch.zeros(self.prog_ints, dtype=torch.int32, device=DEV)
        gb = None
        if isinstance(bound, str):
            assert bound == "fresh"
            gb = torch.full((B,), R.MIN_KEY, dtype=torch.int32, device=DEV)
        elif bound is not None:
            gb = bound.to(torch.int32).clone()
        G = C.c_int(0)
        st = self.L.shim_tensor_scan(_p(table), _p(levels), n, dim, _p(qb), B, kc, weight_pre, _p(ps), _p(pi), self.P,
                                     _p(gb), _p(progress), stride, pre_slots, _p(mask), C.byref(G), _stream())
        _ok(self.native, st, "tensor scan")
        torch.cuda.synchronize()
        g = G.value
        assert 1 <= g <= self.P
        return ps[:B * g * width].view(B, g, width), pi[:B * g * kc].view(B, g, kc), g, gb

    def merge(self, ps, pi, k_out, P=None, row_offset=0, want_bound=True, count=None, out=None):
        B, G, k_in = pi.shape
        P = G if P is None else P
        o_s, o_i = out if out is not None else (torch.empty(B, k_out, dtype=torch.float32, device=DEV),
                                                 torch.empty(B, k_out, dtype=torch.int64, device=DEV))
        key = torch.full((B,), GUARD_I, dtype=torch.int32, device=DEV) if want_bound else None
        st = self.L.shim_merge(_p(ps.contiguous()), _p(pi.contiguous()), B, P, k_in, k_out, _p(o_s), _p(o_i),
                               row_offset, _p(key), _p(count), _stream())
        _ok(self.native, st, "merge")
        torch.cuda.synchronize()
        return o_s, o_i, key

    def bound_from_slots(self, slot_max, kc, out=None):
        B, P, S = slot_max.shape
        key = torch.full((B,), GUARD_I, dtype=torch.int32, device=DEV) if out is None else out
        st = self.L.shim_bound_from_slots(_p(slot_max.contiguous()), B, P, S, kc, _p(key), _stream())
        _ok(self.native, st, "bound_from_slots")
        torch.cuda.synchronize()
        return key

    def column_stats(self, table, master, row0, n, colstat):
        st = self.L.shim_column_stats(_p(table), _p(master), row0, n, table.shape[1], _p(colstat), _stream())
        _ok(self.native, st, "column_stats")
        torch.cuda.synchronize()


@pytest.fixture(scope="module")
def scan(shim, native):
    return Scan(shim, native)


def _reset(native):
    native.tune(scan_pair=-1, scan_qsplit=-1, scan_generic=0, scan_kbs=3, scan_kbs_pair=6)


def _bits(x):
    return x.contiguous().view(torch.int32)


def _weights32(levels):
    return torch.tensor(R.WEIGHTS, dtype=torch.float32, device=DEV)[levels.long()]


# ------------------------------------------------------------------------------------------------ adversarial tables
HALF_TIE = 1.0 + 2.0 ** -8 - 2.0 ** -20     # just under the bf16 half-ulp tie above 1: rounds down, error ~ half an ulp
PROBE_Q, PROBE_ROW = 5, 7                    # premise (c) probe: the input-rounding error reaches the colstat bound


def adversarial(n, dim, B, seed):
    """fp32 master rows [n, dim] and fp32 queries [B, dim] where the scan's error terms are large: columns scaled over
    2^-20 .. 2^4, large cancelling pairs, master values just under bf16 half-ulp ties, row norms from 1e-3 to 1e3, and a
    probe (query PROBE_Q, row PROBE_ROW) whose input-rounding error equals the certificate's A term to within T."""
    g = torch.Generator(device=DEV).manual_seed(seed)
    rows = torch.randn(n, dim, generator=g, device=DEV)
    rows /= rows.norm(dim=1, keepdim=True)
    q = torch.randn(B, dim, generator=g, device=DEV)
    q /= q.norm(dim=1, keepdim=True)
    a = n // 6
    scale = 2.0 ** torch.linspace(-20, 4, dim, device=DEV)[torch.randperm(dim, generator=g, device=DEV)]
    rows[a:2 * a] *= scale
    pairs = torch.arange(0, dim - 1, 2, device=DEV)
    rows[2 * a:3 * a, pairs] = 8.0
    rows[2 * a:3 * a, pairs + 1] = -8.0 * (1 + 2.0 ** -12)
    q[10:20, pairs + 1] = q[10:20, pairs]
    sgn = torch.sign(torch.randn(a, dim, generator=g, device=DEV))
    ex = torch.randint(-6, 3, (a, dim), generator=g, device=DEV).float()
    rows[3 * a:4 * a] = sgn * HALF_TIE * 2.0 ** ex
    rows[4 * a:5 * a] *= 10.0 ** (6 * torch.rand(a, 1, generator=g, device=DEV) - 3)
    q[20:30] = R.bf16_round(q[20:30] * HALF_TIE)
    q[30:40] *= 2.0 ** torch.linspace(-20, 4, dim, device=DEV)
    q[PROBE_Q] = 0.0
    q[PROBE_Q, 0] = HALF_TIE
    rows[PROBE_ROW] = 0.0
    rows[PROBE_ROW, 0] = 4096.0 * HALF_TIE
    return rows.contiguous(), q.contiguous()


@pytest.fixture(scope="module")
def visible_tables():
    """Per dim: n = 6 001 rows (46 full row tiles and a partial one: n <= 128 G for every launch shape used here)."""
    cache = {}

    def get(dim):
        if dim not in cache:
            cache.clear()
            n, B = 6001, 384
            rows, q = adversarial(n, dim, B, seed=dim)
            g = torch.Generator(device=DEV).manual_seed(dim + 1)
            levels = torch.randint(1, 4, (n,), generator=g, device=DEV).to(torch.uint8)
            allowed = torch.rand(n, generator=g, device=DEV) < 0.5
            cache[dim] = dict(n=n, rows=rows, table=rows.to(torch.bfloat16), q=q, qb=q.to(torch.bfloat16),
                              levels=levels, allowed=allowed)
        return cache[dim]
    return get


def pack_mask(allowed):
    n = allowed.shape[0]
    words = (n + 31) // 32
    bits = torch.zeros(words * 32, dtype=torch.int64, device=allowed.device)
    bits[:n] = allowed.long()
    w = (bits.view(words, 32) << torch.arange(32, device=allowed.device)).sum(1)
    return torch.where(w >= 2 ** 31, w - 2 ** 32, w).to(torch.int32).contiguous()


def visible_scores(ps, pi, n, allowed=None):
    """Scatter the partial lists of a scan whose lists hold every row into [B, n] (NaN where no score was written);
    asserts that the ids written are exactly the allowed rows, each once."""
    B = ps.shape[0]
    ids = pi.reshape(B, -1).long()
    sc = ps.reshape(B, -1)
    live = ids >= 0
    want = torch.ones(n, dtype=torch.bool, device=DEV) if allowed is None else allowed
    counts = torch.zeros(B, n, dtype=torch.int32, device=DEV)
    counts.scatter_add_(1, ids.clamp_min(0), live.int())
    assert bool((counts == want.int()[None, :]).all()), \
        "the partial lists do not hold every allowed row exactly once (the visible-score regime does not hold)"
    out = torch.full((B, n), float("nan"), dtype=torch.float32, device=DEV)
    b = torch.arange(B, device=DEV)[:, None].expand_as(ids)
    out[b[live], ids[live]] = sc[live]
    return out


def check_scan_bound(S, q, rows, what):
    """premise (c) in the scan's own terms: every visible score within scan_bound of the exact score of what the index
    holds; returns the worst ratio."""
    e = R.exact_scores(rows, q)
    d = R.scan_bound(q, rows)
    ratio = float(((S.double() - e).abs() / d.clamp_min(1e-300)).max())
    assert ratio <= 1.0, f"{what}: a scan score is off the exact one by {ratio:.3g}x scan_bound"
    return ratio


# ------------------------------------------------------------------------------------------------ every scan score
SHAPES = {"single B=128": (128, {}), "pair B=256": (256, {}), "single B=384": (384, {}),
          "single B=256": (256, {"scan_pair": 0}), "qsplit on B=256": (256, {"scan_qsplit": 1}),
          "qsplit off B=384": (384, {"scan_qsplit": 0}), "kbs 1 B=128": (128, {"scan_kbs": 1}),
          "kbs_pair 2 B=256": (256, {"scan_kbs_pair": 2}), "generic B=256": (256, {"scan_generic": 1}),
          "generic B=384": (384, {"scan_generic": 1})}


@pytest.mark.parametrize("dim", TC_DIMS)
def test_every_scan_score_is_within_the_scan_bound_and_shape_independent(scan, native, visible_tables, dim):
    """The unpruned main scan with kc = 128 writes every (query, row) score.  Each is within scan_bound of fp64 (bf16
    inputs: T alone; fp32 queries and master rows: plus the input-rounding terms), and the same (query, row) gets the
    same bits in every launch shape: CTA pairs and single CTAs, specialised and generic issue loops, query tails in
    shared memory or not, every stage size.  weight_pre scores are fp32(s w) of the same raw score; a masked row never
    appears."""
    t = visible_tables(dim)
    n, table, qb, levels = t["n"], t["table"], t["qb"], t["levels"]
    ref = None
    for name, (B, knobs) in SHAPES.items():
        native.tune(**knobs)
        try:
            ps, pi, G, _ = scan.run(table, levels, qb[:B], 128)
        finally:
            _reset(native)
        S = visible_scores(ps, pi, n)
        if ref is None:
            ref = scan.run(table, levels, qb, 128)
            ref = visible_scores(ref[0], ref[1], n)
            r_bf = check_scan_bound(ref, qb.float(), table.float(), "bf16 inputs")
            r_32 = check_scan_bound(ref, t["q"], t["rows"], "fp32 queries on master rows")
            _record("tensor scan bf16", f"dim {dim}", r_bf)
            _record("tensor scan fp32/master", f"dim {dim}", r_32)
        assert torch.equal(_bits(S), _bits(ref[:B])), f"{name}: scan scores differ from the B = 384 launch's bits"
    # weight_pre: fp32(s * w) of the same raw score
    ps, pi, _, _ = scan.run(table, levels, qb[:256], 128, weight_pre=1)
    W = visible_scores(ps, pi, n)
    assert torch.equal(_bits(W), _bits(ref[:256] * _weights32(levels)[None, :]))
    # a row mask: exactly the allowed rows, same bits
    ps, pi, _, _ = scan.run(table, levels, qb[:128], 128, mask=pack_mask(t["allowed"]))
    Sm = visible_scores(ps, pi, n, t["allowed"])
    assert torch.equal(_bits(Sm[:, t["allowed"]]), _bits(ref[:128, t["allowed"]]))


@pytest.mark.parametrize("dim", [64, 320, 576, 768])
def test_candidate_lists_below_cap_hold_the_same_bits(scan, native, visible_tables, dim):
    """kc = 36 (the fp32-query kc of k = 10): the query tail in shared memory is in play at dim > 512.  Every listed
    (query, row) carries the visible scan's bits, and each list is the group's top 36 by (score desc, id asc)."""
    t = visible_tables(dim)
    n, table, qb, levels = t["n"], t["table"], t["qb"], t["levels"]
    full = scan.run(table, levels, qb, 128)
    S = visible_scores(full[0], full[1], n)
    for B, knobs in ((256, {}), (256, {"scan_qsplit": 0}), (384, {}), (128, {"scan_generic": 1})):
        native.tune(**knobs)
        try:
            ps, pi, G, _ = scan.run(table, levels, qb[:B], 36)
        finally:
            _reset(native)
        ids = pi.long()
        got = ps
        want = S[:B].gather(1, ids.clamp_min(0).reshape(B, -1)).reshape(ids.shape)
        live = ids >= 0
        assert bool(live.all()), "a list of a group with 128 rows is short"
        assert torch.equal(_bits(got), _bits(want)), f"B={B} {knobs}: listed scores differ from the visible scan's"
        # each list is its group's top 36
        sc = got.cpu().numpy()
        ii = ids.cpu().numpy()
        Sh = S[:B].cpu().numpy()
        tiles = R.tile_groups(R.sampled_tiles(n, 1), G)
        for b in (0, B // 2, B - 1):
            for g in (0, G - 1):
                rows_g = np.nonzero(np.repeat(tiles == g, 128)[:n])[0]
                top = rows_g[np.lexsort((rows_g, -Sh[b, rows_g].astype(np.float64)))][:36]
                assert ii[b, g].tolist() == top.tolist(), (b, g)


STRIDES = (2, 3, 7, 64)


@pytest.mark.parametrize("dim", [64, 448, 768])
def test_sampled_passes_see_the_main_pass_bits(scan, native, visible_tables, dim):
    """premise (b): the list pre-pass at strides 2, 3, 7 and 64 scores every sampled (query, row) with the main pass's
    bits, and every slot maximum of the slot pre-pass equals, bit for bit, the maximum of its row set in the model of
    scan_ref.slot_sets (also with weight_pre and a mask), at CTA pairs and single CTAs."""
    t = visible_tables(dim)
    n, table, qb, levels, allowed = t["n"], t["table"], t["qb"], t["levels"], t["allowed"]
    full = scan.run(table, levels, qb, 128)
    S = visible_scores(full[0], full[1], n)
    W = S * _weights32(levels)[None, :]
    mask = pack_mask(allowed)
    for B in (128, 256):
        for s in STRIDES:
            ps, pi, G, _ = scan.run(table, levels, qb[:B], 128, stride=s)
            rows, _, _, _ = R.slot_sets(n, s, G)
            sampled = torch.zeros(n, dtype=torch.bool, device=DEV)
            sampled[torch.from_numpy(rows).to(DEV)] = True
            Ss = visible_scores(ps, pi, n, sampled)
            assert torch.equal(_bits(Ss[:, sampled]), _bits(S[:B, sampled])), f"list pre-pass stride {s} B={B}"
            for wp, al in ((0, None), (1, None), (0, allowed), (1, allowed)):
                sm, _, Gs, _ = scan.run(table, levels, qb[:B], 128, weight_pre=wp, stride=s, pre_slots=1,
                                        mask=None if al is None else mask)
                want = R.expected_slot_max((W if wp else S)[:B].cpu().numpy(), n, s, Gs,
                                           None if al is None else al.cpu().numpy())
                got = sm.cpu().numpy()
                bad = np.nonzero(got.view(np.int32) != want.view(np.int32))
                assert bad[0].size == 0, \
                    f"slot pre-pass stride {s} B={B} wp={wp} mask={al is not None}: slot maximum " \
                    f"{tuple(int(x[0]) for x in bad)} is {got[bad][0]}, the model says {want[bad][0]}"


def premise_c_ratio(scan, t, colstat):
    """Worst |scan - exact(q . master)| / (A + T) over every visible (query, row), A and T per query from colstat."""
    full = scan.run(t["table"], t["levels"], t["qb"], 128)
    S = visible_scores(full[0], full[1], t["n"])
    A, T, _ = R.colstat_slack(t["q"], colstat, True)
    e = R.exact_scores(t["rows"], t["q"])
    ratio = ((S.double() - e).abs() / (A + T)[:, None]).max(1).values
    return ratio


@pytest.mark.parametrize("dim", TC_DIMS)
def test_scan_error_is_within_the_certificates_slack(scan, visible_tables, dim, colstat_defect=None):
    """premise (c) with the library's own numbers: with fp32 queries and master rows every visible scan score is within
    the per-query A + T that finalise_kernel computes from the colstat launch_column_stats produced.  The probe query
    (one column, values just under half-ulp ties, the probe row holding that column's maximum) brings the error to
    within T of A, so a colstat that understates one column maximum fails here."""
    t = visible_tables(dim)
    colstat = torch.zeros(2 * dim + 2, dtype=torch.float32, device=DEV)
    scan.column_stats(t["table"], t["rows"], 0, t["n"], colstat)
    if colstat_defect == "halve column 0":
        colstat[0] *= 0.5
    ratio = premise_c_ratio(scan, t, colstat)
    worst = float(ratio.max())
    assert worst <= 1.0, f"a scan score is off the exact one by {worst:.3g}x the certificate's A + T"
    assert float(ratio[PROBE_Q]) > 0.9, f"the probe query reaches only {float(ratio[PROBE_Q]):.3g} of A + T"
    _record("premise (c) A+T", f"dim {dim}", worst)


# ------------------------------------------------------------------------------------------------ pruning
@pytest.fixture(scope="module")
def big_tables():
    """Tables of 20 011, 600 001 and 2 000 003 rows at dim 768 (the two larger exceed 64 MB: drift limiter on at
    B >= 256), random unit rows with near-duplicate clusters around the queries, built on the GPU; 4 096 queries."""
    cache = {}

    def get(n):
        if n not in cache:
            cache.clear()
            torch.cuda.empty_cache()
            dim, B = 768, 4096
            g = torch.Generator(device=DEV).manual_seed(n)
            q = torch.randn(B, dim, generator=g, device=DEV)
            q /= q.norm(dim=1, keepdim=True)
            table = torch.empty(n, dim, dtype=torch.bfloat16, device=DEV)
            for r0 in range(0, n, 1 << 19):
                r1 = min(n, r0 + (1 << 19))
                x = torch.randn(r1 - r0, dim, generator=g, device=DEV)
                table[r0:r1] = (x / x.norm(dim=1, keepdim=True)).to(torch.bfloat16)
            # 300 near-duplicates of each of 8 queries, spread over the table
            src = torch.arange(8, device=DEV).repeat_interleave(300)
            at = torch.randperm(n, generator=g, device=DEV)[:src.numel()]
            x = q[src] + 0.05 * torch.randn(src.numel(), dim, generator=g, device=DEV) / dim ** 0.5
            table[at] = (x / x.norm(dim=1, keepdim=True)).to(torch.bfloat16)
            levels = torch.randint(1, 4, (n,), generator=g, device=DEV).to(torch.uint8)
            allowed = torch.rand(n, generator=g, device=DEV) < 0.5
            cache[n] = dict(n=n, table=table, qb=q.to(torch.bfloat16), levels=levels, allowed=allowed)
        return cache[n]
    return get


def pruned_topk(scan, t, kc, mode, wp, mask, stride, bound_override=None):
    """The pruned search of index_search_device: pre-pass (slot maxima + bound_from_slots, or lists + merge) at tile
    stride `stride`, main scan admitting against that bound, merge.  bound_override replaces the pre-pass's bound (defect
    injection).  Returns (scores, ids, the pre-pass's bound keys, the bound keys after the main scan)."""
    table, levels, qb = t["table"], t["levels"], t["qb"]
    if bound_override is not None:
        gb = bound_override
    elif mode == "slots":
        sm, _, G, gb = scan.run(table, levels, qb, kc, weight_pre=wp, bound="fresh", stride=stride, pre_slots=1,
                                mask=mask)
        gb = scan.bound_from_slots(sm, kc, out=gb)
    else:
        ps, pi, G, gb = scan.run(table, levels, qb, kc, weight_pre=wp, bound="fresh", stride=stride, mask=mask)
        _, _, key = scan.merge(ps, pi, kc)
        gb = key
    pre = gb.clone()
    ps, pi, G, gb_after = scan.run(table, levels, qb, kc, weight_pre=wp, bound=gb, mask=mask)
    s, i, _ = scan.merge(ps, pi, kc)
    return s, i, pre, gb_after


def check_pruning(scan, t, kc, mode, wp, masked, stride, **defect):
    mask = pack_mask(t["allowed"]) if masked else None
    ps, pi, _, _ = scan.run(t["table"], t["levels"], t["qb"], kc, weight_pre=wp, mask=mask)
    s0, i0, key0 = scan.merge(ps, pi, kc)
    if defect.get("gbound_ulp_above"):
        defect = {"bound_override": key0 + 1}
    s1, i1, pre, after = pruned_topk(scan, t, kc, mode, wp, mask, stride, **defect)
    assert torch.equal(i1, i0), f"pruning changed the merged top-{kc} of {int((i1 != i0).any(1).sum())} queries"
    assert torch.equal(_bits(s1), _bits(s0))
    assert bool((pre <= key0).all()), \
        f"the pre-pass bound exceeds the unpruned kc-th key for {int((pre > key0).sum())} queries"
    assert bool((after <= key0).all()), "the published bound exceeds the unpruned kc-th key"


PRUNE_N = (20011, 600001, 2000003)
KCS = (1, 7, 16, 36, 66, 128)


@pytest.mark.parametrize("n", PRUNE_N)
def test_pruning_is_only_a_performance_device(scan, shim, big_tables, n):
    """premises (a) and (b) end to end: at the library's pre-pass stride (2, 4 and 8 here) the merged top kc of pre-pass
    + pruned scan equals the unpruned scan's bit for bit, and the bound key is <= the unpruned kc-th key for every
    query, for kc in 1..128, slot and list pre-passes, each with and without weight_pre and a mask.  B = 256 runs CTA
    pairs in one launch; on the two tables past 64 MB, B = 384 (single CTAs) and B = 4 096 (two launches, each with its
    own drift-limiter region) run as well."""
    t = big_tables(n)
    stride_of = {20011: 2, 600001: 4, 2000003: 8}
    for B, kcs in ((256, KCS), (384, (7, 66)), (4096, (16, 128))):
        if B != 256 and n == 20011:
            continue
        tb = dict(t, qb=t["qb"][:B])
        i = 0
        for kc in kcs:
            stride = shim.shim_tensor_scan_sample_stride(n, kc)
            assert stride == stride_of[n]
            for mode in ("slots", "lists"):
                wp, masked = (i // 2) % 2, (i // 4) % 2 == 1     # every (mode, weight_pre, mask) over the kc sweep
                i += 1
                check_pruning(scan, tb, kc, mode, wp, masked, stride)


# ------------------------------------------------------------------------------------------------ merge and bound
def merge_ref(ps, pi, k_out, row_offset=0):
    """numpy merge_kernel: every (score, id >= 0) entry of the P lists, sorted (score desc, id asc), cut to k_out."""
    B = ps.shape[0]
    s = ps.reshape(B, ps.shape[1] * ps.shape[2])
    i = pi.reshape(B, ps.shape[1] * ps.shape[2]).astype(np.int64)
    out_s = np.full((B, k_out), -np.inf, np.float32)
    out_i = np.full((B, k_out), -1, np.int64)
    key = np.full(B, R.MIN_KEY, np.int32)
    for b in range(B):
        live = i[b] >= 0
        ss, ii = s[b][live], i[b][live]
        o = np.lexsort((ii, -ss.astype(np.float64)))[:k_out]
        m = len(o)
        out_s[b, :m], out_i[b, :m] = ss[o], ii[o] + row_offset
        if m == k_out:
            key[b] = R.float_key(ss[o][-1:])[0]
    return out_s, out_i, key


def random_lists(B, P, k_in, seed, fill=0.7, ties=True):
    """Sorted (score desc, id asc) lists with -inf / -1 tails, distinct ids, scores on a coarse grid (ties across and
    within lists)."""
    rng = np.random.default_rng(seed)
    ps = np.full((B, P, k_in), -np.inf, np.float32)
    pi = np.full((B, P, k_in), -1, np.int32)
    for b in range(B):
        ids = rng.permutation(P * k_in * 2)[:P * k_in].reshape(P, k_in)
        for l in range(P):
            m = int(rng.binomial(k_in, fill))
            sc = (rng.integers(0, 40, m) / 8.0 if ties else rng.standard_normal(m)).astype(np.float32)
            o = np.lexsort((ids[l, :m], -sc.astype(np.float64)))
            ps[b, l, :m], pi[b, l, :m] = sc[o], ids[l, :m][o]
    return ps, pi


@pytest.mark.parametrize("P,k_in", [(1, 1), (1, 255), (31, 7), (32, 36), (33, 128), (148, 66), (1024, 16)])
def test_merge_matches_numpy(scan, P, k_in, defect=None):
    """merge_kernel against numpy: ties in score broken by id, -inf / -1 tails, row_offset, the bound key of the k_out-th
    score (the very negative key for short lists), bit for bit."""
    B = 9
    ps, pi = random_lists(B, P, k_in, seed=P * 1000 + k_in)
    ps[0] = -np.inf
    pi[0] = -1                                  # an empty query
    for k_out in sorted({1, max(1, k_in // 2), k_in}):
        want_s, want_i, want_k = merge_ref(ps, pi, k_out, row_offset=1 << 33)
        P_arg = P - 1 if defect == "P - 1 lists" else P
        got_s, got_i, got_k = scan.merge(torch.from_numpy(ps).to(DEV), torch.from_numpy(pi).to(DEV), k_out, P=P_arg,
                                         row_offset=1 << 33)
        assert np.array_equal(got_i.cpu().numpy(), want_i), f"k_out={k_out}: ids"
        assert np.array_equal(got_s.cpu().numpy().view(np.int32), want_s.view(np.int32)), f"k_out={k_out}: scores"
        assert np.array_equal(got_k.cpu().numpy(), want_k), f"k_out={k_out}: bound keys"
    assert want_k[0] == R.MIN_KEY


def test_merge_count_leaves_rows_past_the_count_untouched(scan, count_defect=0):
    """count mode (the exact fallback's merge): only the first *count lists are merged; rows past it keep their guard
    values."""
    B, P, k = 40, 148, 10
    ps, pi = random_lists(B, P, k, seed=3)
    for cnt in (0, 1, 17, B):
        o_s = torch.full((B, k), GUARD_F, dtype=torch.float32, device=DEV)
        o_i = torch.full((B, k), GUARD_I, dtype=torch.int64, device=DEV)
        count = torch.tensor([cnt + count_defect], dtype=torch.int32, device=DEV)
        scan.merge(torch.from_numpy(ps).to(DEV), torch.from_numpy(pi).to(DEV), k, count=count, out=(o_s, o_i),
                   want_bound=False)
        want_s, want_i, _ = merge_ref(ps[:cnt], pi[:cnt], k)
        got_s, got_i = o_s.cpu().numpy(), o_i.cpu().numpy()
        assert np.array_equal(got_i[:cnt], want_i) and np.array_equal(got_s[:cnt], want_s)
        assert (got_s[cnt:] == GUARD_F).all() and (got_i[cnt:] == GUARD_I).all(), f"count {cnt}: a row past it moved"


@pytest.mark.parametrize("P", [1, 2, 3, 4, 5, 7, 31, 32, 33, 35, 36, 37, 148])
def test_bound_from_slots_matches_numpy(scan, P, kc_defect=0):
    """bound_from_slots_kernel against the numpy fold (classes g mod 4, kc-th of 128 by (value desc, index asc)) for kc
    1..128: P < 4 (empty classes), P not a multiple of 4, P around the 8-way unroll edge (32 - 37), -inf slots and tied
    maxima."""
    rng = np.random.default_rng(P)
    B = 64
    sm = (rng.integers(0, 200, (B, P, 32)) / 16.0).astype(np.float32)   # ties
    sm[rng.random((B, P, 32)) < 0.2] = -np.inf
    sm[0] = -np.inf
    sm[1, :, :16] = -np.inf
    dev = torch.from_numpy(sm).to(DEV)
    for kc in list(range(1 + (kc_defect > 0), 129, 1 if P in (1, 5, 33) else 9)) + [128]:
        got = scan.bound_from_slots(dev, kc - kc_defect).cpu().numpy()
        want = R.bound_from_slots(sm, kc)
        bad = np.nonzero(got != want)[0]
        assert bad.size == 0, f"kc={kc} query {bad[:1]}: key {got[bad[:1]]} != {want[bad[:1]]}"


# ------------------------------------------------------------------------------------------------ column statistics
def colstat_ref(table, master):
    t = table.double()
    m = master.double() if master is not None else t
    M = torch.maximum(t.abs(), m.abs()).amax(0).float()
    D = (m - t).abs().amax(0).float() if master is not None else torch.zeros_like(M)
    Rn = torch.maximum(t.norm(dim=1), m.norm(dim=1)).max()
    Rd = (m - t).norm(dim=1).max() if master is not None else torch.zeros((), dtype=torch.float64, device=t.device)
    return M, D, float(Rn), float(Rd)


@pytest.mark.parametrize("dim", [8, 64, 264, 768, 1024])
@pytest.mark.parametrize("n", [1, 3001])
def test_column_stats(scan, dim, n):
    """launch_column_stats: column maxima bit-exact against torch, norms >= the fp64 norm and within 2e-6 of it, two
    appends fold to the same bits as one, adopt (no master) is the bf16 image's statistics; values include +-0,
    subnormals and 1e30."""
    g = torch.Generator(device=DEV).manual_seed(dim * 7 + n)
    master = torch.randn(n, dim, generator=g, device=DEV)
    if n > 10:
        master[1] = 0.0
        master[2] = -0.0
        master[3, ::2] = 1e-40
        master[3, 1::2] = -3e-39
        master[4, dim // 2] = 1e30
        master[5] *= 1e-30
        master[6:40] *= HALF_TIE * 4
    table = master.to(torch.bfloat16)
    for m in (master, None):
        one = torch.zeros(2 * dim + 2, dtype=torch.float32, device=DEV)
        scan.column_stats(table, m, 0, n, one)
        M, D, Rn, Rd = colstat_ref(table, m)
        assert torch.equal(_bits(one[:dim]), _bits(M)), "column maxima"
        assert torch.equal(_bits(one[dim:2 * dim]), _bits(D)), "rounding maxima"
        for got, want in ((float(one[2 * dim]), Rn), (float(one[2 * dim + 1]), Rd)):
            assert want <= got <= want * (1 + 2e-6) + 1e-300, (got, want)
        if n > 1:
            two = torch.zeros_like(one)
            h = n // 3
            scan.column_stats(table, m, 0, h, two)
            scan.column_stats(table, m, h, n - h, two)
            assert torch.equal(_bits(one), _bits(two)), "two appends differ from one"


# ------------------------------------------------------------------------------------------------ certificate
@pytest.mark.parametrize("wm", [R.WEIGHT_NONE, R.WEIGHT_PRE])
@pytest.mark.parametrize("f32rows", [False, True])
def test_finalise_certifies_only_what_the_formula_proves(scan, native, shim, wm, f32rows):
    """finalise_kernel with colstat, fed candidate lists of a real table with s_kc swept across the threshold: whenever
    it certifies, the DESIGN.md formula evaluated in fp64 holds (up to a relative band of 1e-12 for the kernel's own
    double summation order), and whenever the formula holds outside that band it certifies.  The fallback list holds each
    uncertified query once, and the fb_in pass writes list slot j into query fb[2 + j]'s rows only."""
    n, dim, B, k, kc = 20011, 768, 512, 10, 36
    g = torch.Generator(device=DEV).manual_seed(11)
    rows = torch.randn(n, dim, generator=g, device=DEV)
    rows /= rows.norm(dim=1, keepdim=True)
    q = rows[torch.randint(0, n, (B,), generator=g, device=DEV)] + 0.05 * torch.randn(B, dim, generator=g, device=DEV)
    q = (q / q.norm(dim=1, keepdim=True)).contiguous()
    table = rows.to(torch.bfloat16)
    held = rows if f32rows else table.float()
    levels = torch.randint(1, 4, (n,), generator=g, device=DEV).to(torch.uint8)
    colstat = torch.zeros(2 * dim + 2, dtype=torch.float32, device=DEV)
    scan.column_stats(table, rows if f32rows else None, 0, n, colstat)
    e = R.exact_scores(held, q)
    cand = e.topk(kc, dim=1).indices.sort(1).values.contiguous()    # any candidate order: finalise sorts
    cid = cand.to(torch.int64).contiguous()
    rows_arg = rows if f32rows else table

    def fin(cs, ci, colst, fb=None, fb_in=None, kcp=kc):
        outs = [torch.full((B, k), GUARD_F, dtype=torch.float32, device=DEV),
                torch.full((B, k), GUARD_F, dtype=torch.float32, device=DEV),
                torch.full((B, k), GUARD_I, dtype=torch.int64, device=DEV)]
        st = shim.shim_finalise(_p(cs), _p(ci), B, kcp, k, 0, n, _p(q), _p(rows_arg), int(f32rows), dim, _p(levels),
                                wm, _p(outs[0]), _p(outs[1]), _p(outs[2]), None, _p(colst), _p(fb), _p(fb_in),
                                _stream())
        _ok(native, st, "finalise")
        torch.cuda.synchronize()
        return outs

    base = fin(torch.zeros(B, kc, dtype=torch.float32, device=DEV), cid, None)
    kth = base[0][:, k - 1].double()                         # the k-th canonical key (score = key in NONE and PRE)
    A, T, Cc = R.colstat_slack(q, colstat, f32rows)
    slack = A + T + Cc
    wmax = 1.2 if wm == R.WEIGHT_PRE else 1.0
    # s_kc swept across the threshold, finer near it
    f = torch.linspace(-0.5, 0.5, B, device=DEV, dtype=torch.float64)
    f = torch.sign(f) * f.abs() ** 3 * 8
    s_kc = (kth - wmax * slack * (1 + f)).float()
    cs = torch.zeros(B, kc, dtype=torch.float32, device=DEV)
    cs[:, -1] = s_kc
    fb = torch.zeros(2 + B, dtype=torch.int32, device=DEV)
    out = fin(cs, cid, colstat, fb)
    certified = out[2][:, 0] != GUARD_I
    s = s_kc.double()
    margin = kth - (s + wmax * slack + 4 * R.U * (s.abs() + kth.abs()))
    band = 1e-12 * (s.abs() + kth.abs() + slack)
    assert not bool((certified & (margin <= -band)).any()), \
        f"certified {int((certified & (margin <= -band)).sum())} queries the formula does not prove"
    assert not bool((~certified & (margin > band)).any()), "left uncertified a query the formula proves"
    assert 0 < int(certified.sum()) < B, "the sweep must straddle the threshold"
    for o, b0 in zip(out, base):
        assert torch.equal(o[certified], b0[certified]), "a certified query's result differs from the plain finalise"
    # the fallback list
    fbh = fb.cpu().numpy()
    cnt = int(fbh[0])
    assert cnt == int(fbh[1]) == int((~certified).sum())
    listed = fbh[2:2 + cnt]
    assert len(set(listed.tolist())) == cnt
    assert set(listed.tolist()) == set(torch.nonzero(~certified).flatten().tolist())
    # the fb_in pass: candidates of list slot j in row j, written into query fb[2 + j]'s rows
    order = torch.from_numpy(listed.astype(np.int64)).to(DEV)
    ci2 = torch.full((B, kc), -1, dtype=torch.int64, device=DEV)
    ci2[:cnt] = cid[order]
    out2 = fin(torch.zeros(B, kc, dtype=torch.float32, device=DEV), ci2, None, fb_in=fb)
    for o, b0 in zip(out2, base):
        assert torch.equal(o[order], b0[order]), "the fb_in pass wrote another query's result"
        assert bool((o[certified] == (GUARD_I if o.dtype == torch.int64 else GUARD_F)).all()), \
            "the fb_in pass wrote the rows of a query it does not serve"


# ------------------------------------------------------------------------------------------------ the suite catches
DEFECTS = ["bound built with kc - 1", "gbound one ulp above the kc-th key", "merge of P - 1 lists",
           "colstat column maximum halved", "count one more than the list holds"]


@pytest.mark.parametrize("defect", DEFECTS)
def test_injected_defects_fail_their_checks(scan, shim, native, visible_tables, big_tables, defect):
    """Each defect is a wrong NUMBER passed through the shim (never a pointer or an unzeroed counter), and the check
    meant to see it fails."""
    with pytest.raises(AssertionError):
        if defect == "bound built with kc - 1":
            test_bound_from_slots_matches_numpy(scan, 33, kc_defect=1)
        elif defect == "gbound one ulp above the kc-th key":
            t = big_tables(20011)
            with pytest.raises(AssertionError, match="pruning changed"):    # the kernel-level check, not the bound's
                check_pruning(scan, dict(t, qb=t["qb"][:256]), 16, "slots", 0, False, 2, gbound_ulp_above=True)
            raise AssertionError("caught by the top-kc check")
        elif defect == "merge of P - 1 lists":
            test_merge_matches_numpy(scan, 33, 128, defect="P - 1 lists")
        elif defect == "colstat column maximum halved":
            test_scan_error_is_within_the_certificates_slack(scan, visible_tables, 768, colstat_defect="halve column 0")
        elif defect == "count one more than the list holds":
            test_merge_count_leaves_rows_past_the_count_untouched(scan, count_defect=1)
