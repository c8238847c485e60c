"""-m gpu: which keys the attention kernels attend, (row, key) pair by pair, against the oracle's mask.

With K = 0 every score is exactly 0 whatever Q and the RoPE tables are, so every visible key weighs exactly 1:
  forward   V one-hot windows V[b, j, h, d] = [j == base + 96h + d]: O[b, i, h, d] = bf16(1/n_i) if row i sees key
            base + 96h + d, exactly 0 otherwise; LSE = ln n_i.  One launch maps 3072 keys for every row.
  backward  dO one-hot probes dO[b, i, h, d] = [i == base + 96h + d]: dV[b, j, h, d] = bf16(P) ~ 1/n_i if probe row i
            sees key j, exactly 0 otherwise (3072 rows x every key per launch); dQ = 0 exactly; dK = 0 exactly on the keys
            the probe rows of a head do not see.
  decode    V windows in the cache: out[b, h, d] = bf16(1/L_b) or exactly 0 for every key of the cache.
A tolerance test cannot see one key attended wrongly among n ~ 100 or more (it moves O and the LSE by ~1/n); this census
resolves every single pair.  The references (helpers.MaskRef, allowed_slab, visible_counts, decode_visible) are built
from lang_x / attention_mask through the oracle, or from explicit validity masks and intervals, never from the
metadata tensors the kernels read -- except the end-to-end cache test, which hands the cache's own bookkeeping to the
kernels and builds the expected mask from the prompts' masks."""
import copy
import math

import numpy as np
import pytest
import torch

import helpers as Hp
from oracle import mma_oracle as O
import test_gpu_attention_numerics as numerics
from test_gpu_attention import CASES, _edge_prompt
from test_cpu_attention_census import EDGE_KINDS

pytestmark = pytest.mark.gpu
dev = "cuda"
H, D = 32, 96
SCALE = D ** -0.5
W = Hp.CENSUS_W
BF = torch.bfloat16


def _ops():
    from aki_b200 import ops
    return ops


def _tables(pos):
    """longrope cos / sin (B|1, T, 48) fp32 on the device for integer positions (B|1, T)."""
    return tuple(x.to(dev) for x in numerics._tables(pos))


def _queries(B, T, seed=0):
    """Positive, finite queries: the scores stay exactly 0 against K = 0, and a dK sum cannot cancel to 0."""
    g = torch.Generator().manual_seed(seed)
    return (0.5 + torch.rand(B, T, H, D, generator=g)).to(BF).to(dev)


def _lse_tol(n):
    """|LSE - ln n| bound of the kernels' logarithm (__logf: 2^-21.41 absolute on [0.5, 2], 3 ulp elsewhere) plus the
    fp32 rounding.  Below half of ln(n+1) - ln(n) for n <= 65536, so the LSE identifies n exactly."""
    ln = torch.log(n.double().clamp(min=1))
    return 2.0 ** -21.41 + 4.0 * Hp.ulp32(ln)


# ---------------------------------------------------------------------------------------------------------- census
def fwd_census(q, cos, sin, meta, R, simt=False, q_off=0, check_values=True, what=""):
    """Every (row, key) pair of attn_fwd_raw against allowed_slab(R).  Returns the pairs whose map disagrees (see
    helpers.census_diff); where the map agrees and check_values, O must be bf16(1/n_i) bit for bit and the LSE ln(n_i)
    (+inf on rows that see nothing)."""
    ops = _ops()
    B, T = q.shape[:2]
    Tk = q_off + T
    Rd = R.to(dev)
    n = Hp.visible_counts(Rd)[:, q_off:Tk]
    k = torch.zeros(B, Tk, H, D, dtype=BF, device=dev)
    v = torch.zeros(B, Tk, W, dtype=BF, device=dev)
    rows = torch.arange(q_off, Tk, device=dev)
    diffs = []
    for base in range(0, Tk, W):
        nc = min(W, Tk - base)
        c = torch.arange(nc, device=dev)
        v.zero_()
        v[:, base + c, c] = 1
        o, lse = ops.attn_fwd_raw(q, k, v.view(B, Tk, H, D), cos, sin, meta, SCALE, simt=simt, q_offset=q_off)
        got = o.view(B, T, W)[:, :, :nc]
        want = Hp.allowed_slab(Rd, (q_off, Tk), (base, base + nc))
        d = Hp.census_diff(got, want, rows, base + c)
        diffs.append(d)
        if check_values and d.shape[0] == 0:
            ref = Hp.recip_bf16(n)[:, :, None].expand_as(got)
            bad = want & (got.double() != ref)
            if bad.any():
                b, r, kk = bad.nonzero()[0].tolist()
                raise AssertionError(f"{what}: {int(bad.sum())} visible pairs are not bf16(1/n) (ex2(0) != 1?); first "
                                     f"b={b} row={q_off + r} key={base + kk}: {float(got[b, r, kk])!r} vs "
                                     f"{float(ref[b, r, kk])!r} (n={int(n[b, r])})")
            if base == 0:
                lt = lse.transpose(1, 2).double()                    # (B, T, H)
                dead = (n == 0)[:, :, None].expand_as(lt)
                assert bool((lt[dead] == math.inf).all()), f"{what}: rows that see nothing need LSE = +inf"
                err = (lt - torch.log(n.double().clamp(min=1))[:, :, None]).abs()
                tol = _lse_tol(n)[:, :, None].expand_as(lt)
                assert bool((err[~dead] <= tol[~dead]).all()), f"{what}: LSE != ln(n), max err {float(err[~dead].max())}"
    return torch.cat(diffs)


def bwd_census(q, cos, sin, meta, R, simt=False, check_values=True, what=""):
    """Every (row, key) pair of attn_bwd_raw's dV against allowed_slab(R); dQ = 0 and the per-head dK key map.  The
    LSE handed to the backward is the reference ln(n_i) in fp32, O is 0 (delta = 0) and V = 1, so dS = P on visible
    pairs.  The dV map mismatches are returned; the rest is asserted when the dV map agrees and check_values.
    Returns (diff, probe rows whose bf16(P) took the accepted neighbour of bf16(1/n), flip_bound of those rows)."""
    ops = _ops()
    B, T = q.shape[:2]
    Rd = R.to(dev)
    n = Hp.visible_counts(Rd)
    lse = torch.where(n > 0, torch.log(n.double().clamp(min=1)), torch.full_like(n, math.inf, dtype=torch.float64))
    lse = lse.to(torch.float32)[:, None, :].expand(B, H, T).contiguous()
    k = torch.zeros(B, T, H, D, dtype=BF, device=dev)
    v = torch.ones(B, T, H, D, dtype=BF, device=dev)
    o = torch.zeros_like(k)
    d_o = torch.zeros(B, T, W, dtype=BF, device=dev)
    keys = torch.arange(T, device=dev)
    diffs, flips, bound = [], 0, 0
    for base in range(0, T, W):
        nr = min(W, T - base)
        c = torch.arange(nr, device=dev)
        d_o.zero_()
        d_o[:, base + c, c] = 1
        dq = torch.full((B, T, H, D), float("nan"), dtype=BF, device=dev)
        dk, dv = dq.clone(), dq.clone()
        ops.attn_bwd_raw(d_o.view(B, T, H, D), q, k, v, o, lse, cos, sin, meta, SCALE, dq, dk, dv, simt=simt)
        got = dv.view(B, T, W)[:, :, :nr].transpose(1, 2)            # [b, probe row, key]
        want = Hp.allowed_slab(Rd, (base, base + nr), (0, T))
        d = Hp.census_diff(got, want, base + c, keys)
        diffs.append(d)
        if not check_values or d.shape[0]:
            continue
        assert bool((dq == 0).all()), f"{what}: dQ must be exactly 0 with K = 0"
        # dK[b, j, h] != 0 exactly where one of head h's 96 probe rows sees key j
        wk = torch.zeros(B, W, T, dtype=torch.bool, device=dev)
        wk[:, :nr] = want
        want_k = wk.view(B, H, D, T).any(2).transpose(1, 2)
        got_k = (dk != 0).any(-1)
        assert not torch.isnan(dk.float()).any(), what
        if not torch.equal(got_k, want_k):
            b, j, h = (got_k != want_k).nonzero()[0].tolist()
            raise AssertionError(f"{what}: dK key map wrong at b={b} key={j} head={h} (want nonzero: "
                                 f"{bool(want_k[b, j, h])}), {int((got_k != want_k).sum())} in all")
        # dV = bf16(P), P = exp2 of the folded LSE: tie-aware around 1/n
        nrow = n[:, base:base + nr].double()
        v64 = 1.0 / nrow.clamp(min=1)
        eps = 2.0 ** -20 * (1.0 + torch.log(nrow.clamp(min=1)))
        ref, alt, band = Hp.bf16_branches(v64, eps)
        sel = lambda x: x[:, :, None].expand_as(got)[want]
        fl = Hp.accept_branches(got[want], sel(ref), sel(alt), sel(band), what=f"{what} dV values")
        # every pair of a probe row takes the same P, so a row flips as a whole: flips and their bound count rows
        flm = torch.zeros_like(want)
        flm[want] = fl
        flips += int(flm.any(-1).sum())
        live = want.any(-1)
        bound += Hp.flip_bound(v64[live], eps[live]) if live.any() else 0
    return torch.cat(diffs), flips, bound


def decode_census(B, t_cap, kv_len, kv_start, valid, max_kv_len, what="", check_values=True, kernel=None):
    """Every key of the cache for decode_op: returns the map mismatches (rows are all 0).  The reference keys are
    decode_visible(kv_len, kv_start, valid) (lists / tensors; valid (B, t_cap) bool or None).  The kernel gets the same
    description unless `kernel` = (kv_len, kv_start, validity words) device tensors replaces it."""
    ops = _ops()
    from aki_b200.cache import bool_to_bits
    ref_start = None if kv_start is None else torch.as_tensor(kv_start).to(dev)
    vis = Hp.decode_visible(torch.as_tensor(kv_len).to(dev), ref_start, None if valid is None else valid.to(dev), t_cap)
    if kernel is None:
        bits = None
        if valid is not None:
            pad = torch.zeros(B, 32 * ((t_cap + 31) // 32), dtype=torch.bool, device=dev)
            pad[:, :t_cap] = valid.to(dev)
            bits = bool_to_bits(pad)
        kernel = (torch.as_tensor(kv_len, dtype=torch.int32).to(dev),
                  None if kv_start is None else torch.as_tensor(kv_start, dtype=torch.int32).to(dev), bits)
    kv_len_d, kv_start_d, bits = kernel
    L = vis.sum(1)
    g = torch.Generator().manual_seed(B * 7 + t_cap)
    q = torch.randn(B, H, D, generator=g).to(BF).to(dev)
    kc = torch.zeros(B, H, t_cap, D, dtype=BF, device=dev)
    vc = torch.zeros_like(kc)
    diffs = []
    for base in range(0, t_cap, W):
        nc = min(W, t_cap - base)
        c = torch.arange(nc, device=dev)
        vc.zero_()
        vc[:, c // D, base + c, c % D] = 1
        out = ops.decode_op(q, kc, vc, kv_len_d, max_kv_len, SCALE, kv_start_d, bits)
        got = out.view(B, 1, W)[:, :, :nc]
        want = vis[:, None, base:base + nc]
        d = Hp.census_diff(got, want, torch.zeros(1, dtype=torch.int64, device=dev), base + c)
        diffs.append(d)
        if check_values and d.shape[0] == 0:
            ref = Hp.recip_bf16(L)[:, None, None].expand_as(got)
            bad = want & (got.double() != ref)
            assert not bad.any(), f"{what}: {int(bad.sum())} visible keys are not bf16(1/L) (exp2f(0) != 1?)"
    return torch.cat(diffs)


def _assert_clean(diff, what):
    assert diff.shape[0] == 0, Hp.census_message(diff, what)


# ---------------------------------------------------------------------------------------------------------- geometry
def _ragged_b4():
    L, N = 700, 64
    g = np.random.default_rng(71)
    lang = g.integers(3, 31000, size=(4, L)).astype(np.int64); am = np.ones_like(lang)
    M, A, PAD = Hp.MEDIA_ID, Hp.ASST_ID, Hp.PAD_ID
    lang[0, 10] = M; lang[0, 300] = M; lang[0, 650] = A                        # full length, two images
    lang[1, 50] = M; lang[1, 500] = A; lang[1, 600:] = PAD; am[1, 600:] = 0    # right padding
    lang[2, :150] = PAD; am[2, :150] = 0; lang[2, 200] = M; lang[2, 400] = M; lang[2, 600] = A   # left padding
    lang[3, 5] = M; lang[3, 30] = A; lang[3, 50:] = PAD; am[3, 50:] = 0        # short sample
    return lang, am, N


GEOMS = (["causal-1", "causal-127", "causal-128", "causal-129", "causal-300", "causal-8192"]
         + [c[0] for c in CASES if not c[0].endswith("-norope")] + EDGE_KINDS
         + ["left-pad-tables", "ragged-b4", "cfg3-8192", "cfg3-32768"])


def geometry(name):
    """(B, T, kernel metadata (MMASegments or None), reference MaskRef, RoPE tables (cos, sin))."""
    ops = _ops()
    pos = None
    if name.startswith("causal-"):
        T = int(name.split("-")[1])
        return 1, T, None, Hp.MaskRef.causal(1, T), _tables(torch.arange(T)[None])
    text_only, t_cap = False, None
    if name.startswith("cfg3-"):
        import bench
        T = int(name.split("-")[1])
        lang, am = bench.make_prompt(1, T, 4)
        N, t_cap = 128, T
    elif name == "left-pad-tables":
        c = numerics.case_left_pad()
        lang, am, N = c["lang"], c["am"], c["N"]
        pos = c["cos"], c["sin"]
    elif name == "ragged-b4":
        lang, am, N = _ragged_b4()
    elif name in EDGE_KINDS:
        lang, am, N, text_only = _edge_prompt(name)
    else:
        _, B, L, N, n_img, _, pad = next(c for c in CASES if c[0] == name)
        lang, am = Hp.make_prompt(B, L, N, n_img, pad_right=pad, first_img=min(8, L // 3))
    S = O.segments_ref(lang, am, N, Hp.MEDIA_ID, text_only=text_only)
    segs = ops.build_segments(torch.from_numpy(lang).to(dev), torch.from_numpy(am).to(dev), N, Hp.MEDIA_ID,
                              text_only=text_only, t_cap=t_cap, exact_shape=t_cap is None)
    T = segs.T
    assert T == int(S.seq_len.max())
    R = Hp.MaskRef.from_segments(S, T, text_only)
    if pos is None:
        pos = _tables(torch.arange(T)[None])
    else:
        pos = tuple(x.to(dev).contiguous() for x in pos)
    return lang.shape[0], T, segs, R, pos


def _meta(segs, plan):
    ops = _ops()
    if segs is None:
        return None
    m = ops.meta_tuple(segs)
    return m if plan else m[:7] + (None,)


# ---------------------------------------------------------------------------------------------------------- tests
def test_ex2_of_zero_is_one():
    """The census' bit-exact values rest on ex2.approx(0) == 1 and exp2f(0) == 1: then l_i = n_i exactly, and the row
    with one visible key has LSE = log(1) = 0 exactly in the tcgen05 and SIMT forwards; every O value is bf16(1/n_i)
    and every decode output bf16(1/L)."""
    ops = _ops()
    T = 300
    q = _queries(1, T, seed=1)
    R = Hp.MaskRef.causal(1, T)
    for simt in (False, True):
        k = torch.zeros(1, T, H, D, dtype=BF, device=dev)
        _, lse = ops.attn_fwd_raw(q, k, torch.ones_like(k), None, None, None, SCALE, simt=simt)
        assert bool((lse[0, :, 0] == 0).all()), ("simt" if simt else "tcgen05", lse[0, :, 0])
        _assert_clean(fwd_census(q, None, None, None, R, simt=simt, what=f"causal-300 simt={simt}"), "causal-300")
    _assert_clean(decode_census(1, 700, [700], None, None, 700, what="decode 700"), "decode 700")


@pytest.mark.parametrize("name", GEOMS)
def test_forward_census(name):
    """tcgen05 forward with and without RoPE tables (both template instantiations), with the work plan and without it
    (per-query-tile key ends), and the SIMT forward, every (row, key) pair."""
    B, T, segs, R, (cos, sin) = geometry(name)
    q = _queries(B, T, seed=T)
    variants = [(True, True), (True, False), (False, True), (False, False)]
    if T > 8192:
        variants = variants[::3]
    for rope, plan in variants:
        if segs is None and not plan:
            continue                       # no metadata: there is no plan to leave out
        c, s = (cos, sin) if rope else (None, None)
        what = f"{name} tcgen05 rope={rope} plan={plan}"
        _assert_clean(fwd_census(q, c, s, _meta(segs, plan), R, what=what), what)
    if T <= 8192:
        _assert_clean(fwd_census(q, cos, sin, _meta(segs, True), R, simt=True, what=f"{name} simt"), f"{name} simt")


@pytest.mark.parametrize("name", GEOMS)
def test_backward_census(name):
    """tcgen05 and SIMT backward: the dV probe map over every row, dQ = 0 and the dK key map."""
    B, T, segs, R, (cos, sin) = geometry(name)
    q = _queries(B, T, seed=T + 1)
    runs = [(False, True)] + ([(True, False)] if T <= 8192 else [])
    for simt, rope in runs:
        c, s = (cos, sin) if rope else (None, None)
        what = f"{name} {'simt' if simt else 'tcgen05'} backward rope={rope}"
        diff, flips, bound = bwd_census(q, c, s, _meta(segs, True), R, simt=simt, what=what)
        _assert_clean(diff, what)
        print(f"{what}: {flips} probe rows with accepted bf16 flips (bound {bound})")
        assert flips <= bound, (what, flips, bound)


# ---- continuation chunks (forward only: the backward refuses q_offset)
def continuation_geometry(past, T=700, B=2):
    """Key-coordinate metadata of a chunk [past, past + T): invalid keys at word and tile edges and around past, an
    image span straddling past (its chunk rows see later keys up to past + 300), one inside the chunk, sample 1 shorter
    than the keys and with an invalid run.  Returns the kernel's tensors and the reference MaskRef."""
    from aki_b200.cache import bool_to_bits
    Tk = past + T
    valid = torch.ones(B, Tk, dtype=torch.bool)
    row_lo = torch.zeros(B, Tk, dtype=torch.int64); row_hi = torch.zeros(B, Tk, dtype=torch.int64)
    for b in range(B):
        for j in (31, 32, 63, 64, 127, 128, past - 1, past, past + 1):
            if 0 <= j < Tk and not (b == 0 and j == past):
                valid[b, j] = False
        spans = [(max(0, past - 20), 48, min(Tk, past + 300)),
                 (past + 100 + 26 * b, 64 + 66 * b, Tk if b else past + 600)]
        for s, ln, e in spans:
            row_lo[b, s:s + ln] = s + ln
            row_hi[b, s:s + ln] = e
    valid[1, past + 200:past + 260] = False
    seq_len = torch.tensor([Tk, Tk - 37])
    R = Hp.MaskRef(seq_len, valid, valid, row_lo, row_hi)
    words = (Tk + 31) // 32
    pad = torch.zeros(B, 32 * words, dtype=torch.bool)
    pad[:, :Tk] = valid
    vbits = bool_to_bits(pad)
    tensors = [x.to(dev).contiguous() for x in (seq_len.to(torch.int32), row_lo.to(torch.int32), row_hi.to(torch.int32),
                                                  vbits, vbits.clone())]
    return tensors, R


@pytest.mark.parametrize("past", [1, 127, 128, 129, 1000, 4095])
def test_continuation_census(past):
    ops = _ops()
    T = 700
    (seq_len, lo, hi, vb, mb), R = continuation_geometry(past, T)
    q = _queries(2, T, seed=past)
    cos, sin = _tables(past + torch.arange(T)[None])
    for plan in (True, False):
        meta = ops.continuation_meta(seq_len, lo, hi, vb, mb, T, past, plan=plan)
        c, s = (cos, sin) if plan else (None, None)
        what = f"continuation past={past} plan={plan}"
        _assert_clean(fwd_census(q, c, s, meta, R, q_off=past, what=what), what)
    what = f"continuation past={past} simt"
    _assert_clean(fwd_census(q, cos, sin, ops.continuation_meta(seq_len, lo, hi, vb, mb, T, past), R, simt=True,
                             q_off=past, what=what), what)


# ---- decode
KV_LENS = [1, 511, 512, 513, 4097, 4608]
STARTS = [0, 31, 32, 511, 512, 513, -1]                      # -1: kv_len - 1
RUNS = [[], [(30, 70)], [(500, 530)], [(1024, 1536)], None, [(0, 33), (4000, 4100)]]   # None: no valid key at all


def _decode_specs(t_cap):
    specs = []
    for r, runs in enumerate(RUNS):
        for ln in KV_LENS:
            for st in STARTS:
                ln_ = min(ln, t_cap)
                specs.append((ln_, ln_ - 1 if st < 0 else min(st, ln_ - 1), runs))
    return specs


def _decode_batch(specs, t_cap):
    valid = torch.ones(len(specs), t_cap, dtype=torch.bool)
    for b, (_, _, runs) in enumerate(specs):
        if runs is None:
            valid[b] = False
        else:
            for a, e in runs:
                valid[b, a:e] = False
    return [s[0] for s in specs], [s[1] for s in specs], valid


@pytest.mark.parametrize("B", [1, 8, 9, 64])
def test_decode_census(B):
    """kv_len at chunk edges, kv_start at word and chunk edges and at kv_len - 1, invalid runs across 32-bit words and
    512-key splits, a split with no valid key and samples with none at all; max_kv_len = max(kv_len) (eager steps) and
    = t_cap (graph steps, whose trailing splits are empty)."""
    t_cap = 4608
    specs = _decode_specs(t_cap)
    if B == 1:
        specs = specs[::9]
    for i in range(0, len(specs), B):
        batch = specs[i:i + B]
        kv_len, kv_start, valid = _decode_batch(batch, t_cap)
        for max_kv in (max(kv_len), t_cap):
            what = f"decode B={len(batch)} batch {i // B} max_kv_len={max_kv}"
            _assert_clean(decode_census(len(batch), t_cap, kv_len, kv_start, valid, max_kv, what=what), what)


@pytest.mark.parametrize("B,kv_len,kv_start", [(1, [131072], [0]), (2, [100001, 77777], [513, 0])])
def test_decode_census_long(B, kv_len, kv_start):
    t_cap = 131072
    valid = torch.ones(B, t_cap, dtype=torch.bool)
    valid[0, 65530:65600] = False
    valid[B - 1, 4096:4608] = False                          # one whole 512-key split
    valid[B - 1, 77700:77777] = False
    for max_kv in sorted({max(kv_len), t_cap}):
        what = f"decode t_cap={t_cap} B={B} max_kv_len={max_kv}"
        _assert_clean(decode_census(B, t_cap, kv_len, kv_start, valid, max_kv, what=what), what)


# ---- the KV cache's own bookkeeping, end to end
@pytest.fixture(scope="module")
def runner():
    from aki_b200.model import AkiPhi3Runner, phi35_mini_config
    return AkiPhi3Runner(phi35_mini_config(num_layers=2), device=dev, seed=0)


def test_cache_metadata_end_to_end(runner):
    """A left-padded first turn, a left-padded follow-up with an image, two eager and two graph decode steps on a
    2-layer runner; the cache's kv_len, kv_start, meta.kv_valid_bits and meta.attn_meta(past, T) then drive census
    launches.  Expected: keys cat(am1, the follow-up's spliced 2-D mask, ones) for the decode, plus the follow-up's
    mutual block for the continuation forward -- built from the prompts with the oracle."""
    ops = _ops()
    B, N = 3, 64
    g = np.random.default_rng(17)
    L1, pads1 = 200, [0, 17, 40]
    lang1 = g.integers(3, 31000, size=(B, L1)).astype(np.int64); am1 = np.ones_like(lang1)
    L2, pads2 = 120, [5, 0, 23]
    lang2 = g.integers(3, 31000, size=(B, L2)).astype(np.int64); am2 = np.ones_like(lang2)
    for b in range(B):
        lang1[b, :pads1[b]] = Hp.PAD_ID; am1[b, :pads1[b]] = 0
        lang2[b, :pads2[b]] = Hp.PAD_ID; am2[b, :pads2[b]] = 0
        lang2[b, pads2[b] + 10] = Hp.MEDIA_ID; lang2[b, 100] = Hp.ASST_ID
    segs1 = ops.build_segments(torch.from_numpy(lang1).to(dev), torch.from_numpy(am1).to(dev), N, Hp.MEDIA_ID)
    segs2 = ops.build_segments(torch.from_numpy(lang2).to(dev), torch.from_numpy(am2).to(dev), N, Hp.MEDIA_ID)
    S2 = O.segments_ref(lang2, am2, N, Hp.MEDIA_ID)
    T1, T2 = L1, int(S2.seq_len.max())
    Tk, n_steps = T1 + T2, 4
    t_cap = Tk + n_steps + 12
    torch.manual_seed(4)
    cache = runner.new_cache(B, t_cap)
    runner.prefill((torch.randn(B, T1, 3072, device=dev) * 0.05).to(BF), segs1, cache)
    l2 = runner.prefill((torch.randn(B, T2, 3072, device=dev) * 0.05).to(BF), segs2, cache)
    meta_c = cache.meta.attn_meta(T1, T2)
    # the follow-up chunk: causal over cat(am1, S2.valid), the chunk's mutual block in key coordinates
    R2 = Hp.MaskRef.from_segments(S2, T2)
    live = R2.row_hi > R2.row_lo
    z = torch.zeros(B, T1, dtype=torch.int64)
    valid_c = torch.cat([torch.from_numpy(am1).bool(), R2.valid], 1)
    shift = lambda x: torch.cat([z, torch.where(live, x + T1, 0)], 1)
    Rc = Hp.MaskRef(T1 + R2.seq_len, valid_c, torch.cat([z.bool(), R2.mutual], 1), shift(R2.row_lo), shift(R2.row_hi))
    q = _queries(B, T2, seed=5)
    _assert_clean(fwd_census(q, None, None, meta_c, Rc, q_off=T1, what="cache continuation"), "cache continuation")
    # decode steps, eager then graph-replayed
    tok = l2[:, -1].argmax(-1, keepdim=True)
    for step in range(n_steps):
        if step < 2:
            tok = runner.decode_step_fused(tok, cache)[:, -1].argmax(-1, keepdim=True)
        else:
            tok = runner.decode_step_graphed(tok, cache)
        kv = Tk + step + 1
        valid = torch.cat([valid_c, torch.ones(B, t_cap - Tk, dtype=torch.bool)], 1)
        assert cache.get_seq_length() == kv
        for max_kv in (kv, t_cap):
            what = f"cache decode step {step} max_kv_len={max_kv}"
            diff = decode_census(B, t_cap, [kv] * B, None, valid, max_kv, what=what,
                                 kernel=(cache.kv_len, cache.kv_start, cache.meta.kv_valid_bits))
            _assert_clean(diff, what)


# ---- negative controls: one pair group changed in the metadata given to the kernel, the reference left alone
def _mutated():
    """The cfg1 geometry and two single-point changes of its kernel metadata: one validity bit cleared (key 200, text
    after the image) and one image row's row_hi moved up by one; each with the reference it implies."""
    from aki_b200.cache import bits_to_bool, bool_to_bits
    ops = _ops()
    B, T, segs, R, tabs = geometry("cfg1")
    out = []
    s = copy.copy(segs)
    vb = bits_to_bool(segs.kv_valid_bits, 32 * segs.kv_valid_bits.shape[1])
    vb[0, 200] = False
    s.kv_valid_bits = bool_to_bits(vb)
    Rm = copy.copy(R)
    Rm.valid = R.valid.clone(); Rm.valid[0, 200] = False                   # mutual bits unchanged
    out.append(("cleared validity bit", ops.rebuild_tile_bounds(s), Rm))
    s = copy.copy(segs)
    i0 = 8 + 60                                              # an image row (span [8, 136), q_end > 137)
    s.row_hi = segs.row_hi.clone(); s.row_hi[0, i0] += 1
    Rm = copy.copy(R)
    Rm.row_hi = R.row_hi.clone(); Rm.row_hi[0, i0] += 1
    assert int(R.row_hi[0, i0]) > int(R.row_lo[0, i0])
    out.append(("row_hi + 1", ops.rebuild_tile_bounds(s), Rm))
    return B, T, R, tabs, out


def _expected_pairs(R, Rm, T):
    a, m = Hp.allowed_slab(R, (0, T), (0, T)), Hp.allowed_slab(Rm, (0, T), (0, T))
    idx = (a != m).nonzero()
    assert idx.shape[0] > 0
    return idx.tolist()


def test_negative_controls_forward_and_backward():
    B, T, R, (cos, sin), muts = _mutated()
    q = _queries(B, T, seed=9)
    for label, segs_m, Rm in muts:
        want = _expected_pairs(R, Rm, T)
        for plan in (True, False):
            d = fwd_census(q, cos, sin, _meta(segs_m, plan), R, check_values=False, what=label)
            assert d[:, :3].long().tolist() == want, (label, plan, d[:8].tolist(), want[:8])
        d, _, _ = bwd_census(q, cos, sin, _meta(segs_m, True), R, check_values=False, what=label)
        assert d[:, :3].long().tolist() == want, (label, "backward", d[:8].tolist(), want[:8])


def test_negative_control_decode():
    from aki_b200.cache import bool_to_bits
    B, t_cap = 3, 1100
    kv_len, kv_start = [1100, 700, 513], [0, 31, 0]
    valid = torch.ones(B, t_cap, dtype=torch.bool)
    valid[1, 500:530] = False
    pad = torch.zeros(B, 32 * ((t_cap + 31) // 32), dtype=torch.bool)
    pad[:, :t_cap] = valid
    pad[2, 511] = False                                      # the kernel loses key 511 of sample 2
    kernel = (torch.tensor(kv_len, dtype=torch.int32, device=dev), torch.tensor(kv_start, dtype=torch.int32, device=dev),
              bool_to_bits(pad).to(dev))
    d = decode_census(B, t_cap, kv_len, kv_start, valid, t_cap, check_values=False, kernel=kernel)
    assert d[:, :3].long().tolist() == [[2, 0, 511]], d.tolist()
