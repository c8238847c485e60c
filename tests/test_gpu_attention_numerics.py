"""-m gpu: the attention kernels at wide score ranges, against an fp64 reference.

The parity tests of test_gpu_attention.py draw q, k ~ N(0, 1) at scale 96^-0.5, so every score is about N(0, 1).  Paths
that only run, or only matter, outside that range are exercised here:
  * the forward's lazy rescale (attn_fwd_sm100.cu: O and l stay expressed against the running maximum until it grows by
    more than 2^8, and a row whose first visible key lies beyond its first key tile starts with alpha = 0);
  * the backward's fold of -LSE/scale into the S^T MMA as three bf16 terms (bwd_preprocess), whose precision only
    matters once |LSE/scale| reaches the hundreds;
  * the split-KV decode at 16 splits, kv_start across / on chunk boundaries, empty splits;
  * per-sample RoPE tables (left-padded batched generation), where rope_stride_b != 0.

Reference: fp64 on the host, explicit formulas (no autograd), computed from the bf16 operands the kernels consume (K read
back from rope_kv_write, Q rotated in fp32 and rounded to bf16 as the forward does).  Tolerance yardstick: a precision
model that evaluates the same formulas with bf16 rounding only where the kernels round (P before PV and before dV, dS
before dQ and dK, the outputs), so the bound keeps its teeth when the scores are wide:
    |kernel - exact| <= 2 * max|model - exact| + 1e-3 * max(RMS(exact), 1)   over live rows
and for the LSE |kernel - exact| <= 1e-3 + 1e-4 * |lse|."""
import math

import numpy as np
import pytest
import torch

import helpers as Hp
from oracle import mma_oracle as O

pytestmark = pytest.mark.gpu
dev = "cuda"
D = 96
SCALE = D ** -0.5
KEY_TILE = 128
RESCALE_LOG2 = 8.0        # attn_fwd_sm100.cu fwd::RESCALE_THRESHOLD (log2 units)
LOG2E = 1.0 / math.log(2.0)


def _ops():
    from aki_b200 import ops
    return ops


def _bf(x):
    """Round to bf16 and back (the kernels' rounding points)."""
    return x.to(torch.bfloat16).to(x.dtype)


# ------------------------------------------------------------------------------------------------ inputs
def _tables(positions, long_factors=False):
    """Phi-3 longrope cos / sin (B, T, 48) fp32 for integer positions (B, T)."""
    ext = (2.0 + 3.0 * np.arange(48, dtype=np.float32) / 48) if long_factors else (1.0 + np.arange(48, dtype=np.float32) / 48)
    cos, sin = O.rope_cos_sin(positions, O.longrope_inv_freq(D, 10000.0, ext), 1.1902)
    return cos[..., :48].contiguous(), sin[..., :48].contiguous()


def _rotate(x, cos, sin):
    """RoPE of x (B,T,H,D) with (B|1,T,48) fp32 tables, rounded to bf16 exactly as the forward rotates Q in shared
    memory.  The compiled rotation (attn_fwd_sm100.cu, rope_item) fuses the cos product and rounds the sin product:
    lo' = fma(lo, cos, -fp32(hi sin)), hi' = fma(hi, cos, fp32(lo sin)).  A plain fp32 evaluation differs from it in
    the last fp32 bit, which flips the bf16 rounding of a few elements per 10^5 -- at wide score ranges enough to move
    the LSE of a row whose dominant key meets such an element by more than its bound."""
    c, s = cos.double()[:, :, None, :], sin.double()[:, :, None, :]
    lo, hi = x.double()[..., :48], x.double()[..., 48:]           # bf16 x fp32 products are exact in fp64

    def f32(t):
        return t.float().double()

    return torch.cat([lo * c - f32(hi * s), hi * c + f32(lo * s)], -1).float().to(torch.bfloat16)


def _unrotate(g, cos, sin):
    """g = R^T g' for gradients (B,T,H,D) fp64 w.r.t. rotated operands."""
    c, s = cos.double()[:, :, None, :], sin.double()[:, :, None, :]
    lo, hi = g[..., :48], g[..., 48:]
    return torch.cat([lo * c + hi * s, hi * c - lo * s], -1)


def _allowed(S, T):
    """(B,T,T) bool mask of the reference (O.expand_segments_to_4d); plain causal without segments."""
    if S is None:
        return torch.tril(torch.ones(T, T, dtype=torch.bool))[None]
    return torch.from_numpy(O.expand_segments_to_4d(S, t_out=T)[:, 0] != 0)


def _segments(lang, am, N):
    ops = _ops()
    S = O.segments_ref(lang, am, N, Hp.MEDIA_ID)
    segs = ops.build_segments(torch.from_numpy(lang).to(dev), torch.from_numpy(am).to(dev), N, Hp.MEDIA_ID)
    return S, segs


def _randn(shape, seed, std=1.0):
    return (torch.randn(*shape, generator=torch.Generator().manual_seed(seed)) * std).to(torch.bfloat16)


# ------------------------------------------------------------------------------------------------ reference
def reference(q, k, v, allowed, scale, d_o=None, cos=None, sin=None, heads=None, row_block=256):
    """fp64 attention forward (+ backward when d_o is given) of the bf16 operands q (rotated), k (rotated), v (B,T,H,D).

    Returns (exact, model, tile_max): dicts of o (B,T,H,D), lse (B,H,T) [exact only], dq, dk, dv (B,T,H,D; w.r.t. the
    pre-RoPE q / k when tables are given), and the per-row maximum of the visible scaled scores in each aligned 128-key
    tile (B,H,T,n_tiles; -inf where a tile holds no visible key) for rescale_events().  The model rounds to bf16 where
    the kernels do: P (relative to the row maximum) before PV and dV, dS before dQ and dK, every output."""
    B, T, H, _ = q.shape
    heads = list(range(H)) if heads is None else list(heads)
    Hs = len(heads)
    qd, kd, vd = (x[:, :, heads].double() for x in (q, k, v))
    nt = (T + KEY_TILE - 1) // KEY_TILE
    ex = {"o": torch.zeros(B, T, Hs, D, dtype=torch.float64), "lse": torch.full((B, Hs, T), float("nan"), dtype=torch.float64)}
    md = {"o": torch.zeros(B, T, Hs, D, dtype=torch.float64)}
    tile_max = torch.full((B, Hs, T, nt), float("-inf"), dtype=torch.float64)
    bwd = d_o is not None
    if bwd:
        dod = d_o[:, :, heads].double()
        for r in (ex, md):
            for nm in ("dq", "dk", "dv"):
                r[nm] = torch.zeros(B, T, Hs, D, dtype=torch.float64)
    for b in range(B):
        kb, vb = kd[b].transpose(0, 1), vd[b].transpose(0, 1)               # (H,T,D)
        for r0 in range(0, T, row_block):
            r1 = min(T, r0 + row_block)
            m = allowed[b, r0:r1]
            vis = m.any(0).nonzero()
            if len(vis) == 0:
                continue
            kend = int(vis.max()) + 1                                          # keys beyond the block's reach are skipped
            m = m[:, :kend]
            qb = qd[b, r0:r1].transpose(0, 1)                                  # (H,R,D)
            s = scale * torch.matmul(qb, kb[:, :kend].transpose(1, 2))         # (H,R,K)
            s = s.masked_fill(~m, float("-inf"))
            pad = nt * KEY_TILE - kend
            tile_max[b, :, r0:r1] = torch.nn.functional.pad(s, (0, pad), value=float("-inf")).view(Hs, r1 - r0, nt, KEY_TILE).amax(-1)
            mx = s.amax(-1, keepdim=True)
            live = torch.isfinite(mx)
            e = torch.exp(s - torch.where(live, mx, torch.zeros_like(mx)))    # masked -> 0
            l = torch.where(live, e.sum(-1, keepdim=True), torch.ones_like(mx))
            p = e / l
            o_ex = torch.matmul(p, vb[:, :kend])                               # (H,R,D)
            o_md = _bf(torch.matmul(_bf(e), vb[:, :kend]) / l)                 # P rounded before PV, O normalised, rounded
            ex["o"][b, r0:r1] = o_ex.transpose(0, 1)
            md["o"][b, r0:r1] = o_md.transpose(0, 1)
            ex["lse"][b, :, r0:r1] = torch.where(live, mx + torch.log(l), torch.full_like(mx, float("nan")))[..., 0]
            if not bwd:
                continue
            dob = dod[b, r0:r1].transpose(0, 1)                                # (H,R,D)
            dp = torch.matmul(dob, vb[:, :kend].transpose(1, 2))               # (H,R,K)
            for r, o_r, rnd in ((ex, o_ex, lambda x: x), (md, o_md, _bf)):
                delta = (dob * o_r).sum(-1, keepdim=True)                      # the model's delta reads the bf16 O
                ds = rnd(p * (dp - delta))
                r["dq"][b, r0:r1] = (scale * torch.matmul(ds, kb[:, :kend])).transpose(0, 1)
                r["dk"][b, :kend] += (scale * torch.matmul(ds.transpose(1, 2), qb)).transpose(0, 1)
                r["dv"][b, :kend] += torch.matmul(rnd(p).transpose(1, 2), dob).transpose(0, 1)
    if bwd:
        for r in (ex, md):
            if cos is not None:
                r["dq"] = _unrotate(r["dq"], cos, sin)
                r["dk"] = _unrotate(r["dk"], cos, sin)
    for nm in ("dq", "dk", "dv") if bwd else ():
        md[nm] = _bf(md[nm])
    return ex, md, tile_max


def rescale_events(tile_max):
    """Replays the forward's lazy-rescale rule (attn_fwd_sm100.cu, softmax warps) per row over the aligned 128-key tiles:
    need = (m_new - m_used) * scale*log2(e) > 8  or  (m_used == -inf and m_new > -inf).  Returns per-row counts of the
    rescales at key tiles j > 0 (alpha = 2^((m_used - m_new) * scale*log2 e)) and of the late first-visible inits (the
    alpha = 0 branch: no visible key before tile j > 0), the smallest log2(alpha) of a rescale per row, and the number
    of rescales at each tile index."""
    tm = tile_max * LOG2E                                  # scores are already scaled: log2 units
    shape = tm.shape[:-1]
    m_used = torch.full(shape, float("-inf"), dtype=tm.dtype)
    rescales = torch.zeros(shape, dtype=torch.int64)
    late = torch.zeros(shape, dtype=torch.int64)
    min_alpha = torch.zeros(shape, dtype=tm.dtype)
    per_tile = []
    for j in range(tm.shape[-1]):
        m_new = torch.maximum(m_used, tm[..., j])
        fin_used, fin_new = torch.isfinite(m_used), torch.isfinite(m_new)
        grow = torch.where(fin_used & fin_new, m_new - m_used, torch.zeros_like(m_new))
        need = (grow > RESCALE_LOG2) | (~fin_used & fin_new)
        if j > 0:
            rs = need & fin_used
            rescales += rs
            late += need & ~fin_used
            min_alpha = torch.where(rs, torch.minimum(min_alpha, -grow), min_alpha)
            per_tile.append(int(rs.sum()))
        else:
            per_tile.append(0)
        m_used = torch.where(need, m_new, m_used)
    return {"rescales": rescales, "late": late, "min_log2_alpha": min_alpha, "per_tile": per_tile}


# ------------------------------------------------------------------------------------------------ checks
def check_close(name, got, exact, model, rows=None):
    """|kernel - exact| <= 2 max|model - exact| + 1e-3 max(RMS(exact), 1) over `rows` ((B,T) bool, None = all)."""
    got = got.detach().cpu().double()
    if rows is not None:
        got, exact, model = got[rows], exact[rows], model[rows]
    assert not torch.isnan(got).any(), f"{name}: NaN"
    err = float((got - exact).abs().max())
    yard = float((model - exact).abs().max())
    rms = float(exact.pow(2).mean().sqrt())
    tol = 2.0 * yard + 1e-3 * max(rms, 1.0)       # floor as in helpers.within_tolerance: saturated softmax -> ~0 gradients
    assert err <= tol, f"{name}: max err {err:.3e} > 2 x model err {yard:.3e} + 1e-3 x max(rms {rms:.3e}, 1)"
    return err, yard


def check_lse(got, exact, rows):
    """(B,H,T) LSE of live rows: |kernel - exact| <= 1e-3 + 1e-4 |lse|."""
    live = rows[:, None, :].expand_as(exact)
    got = got.detach().cpu().double()[live]
    ref = exact[live]
    bad = (got - ref).abs() > 1e-3 + 1e-4 * ref.abs()
    assert not bad.any(), f"lse: {int(bad.sum())} rows off, max err {float((got - ref).abs().max()):.3e}"


def run_kernels(q, k, v, cos, sin, segs, scale, d_o, simt=False):
    """q, k, v, d_o (B,T,H,D) bf16 on the host, pre-RoPE.  Returns o, lse, dq, dk, dv from the device kernels (gradients
    pre-filled with NaN) and the rotated K that rope_kv_write produced (B,T,H,D) when tables are given."""
    ops = _ops()
    B, T, H, _ = q.shape
    qd, kd, vd = q.to(dev), k.to(dev), v.to(dev)
    cd = sd = None
    k_in = kd
    if cos is not None:
        cd, sd = cos.to(dev), sin.to(dev)
        kr = torch.empty(B, H, T, D, dtype=torch.bfloat16, device=dev)
        packed = torch.cat([qd.reshape(B, T, -1), kd.reshape(B, T, -1), vd.reshape(B, T, -1)], -1).contiguous()
        ops.rope_kv_write(packed, cd, sd, kr, None, 0, H)
        k_in = kr.transpose(1, 2)
    meta = ops.meta_tuple(segs)
    o, lse = ops.attn_fwd_raw(qd, k_in, vd, cd, sd, meta, scale, simt=simt)
    dq = torch.full((B, T, H, D), float("nan"), dtype=torch.bfloat16, device=dev)
    dk, dv = dq.clone(), dq.clone()
    ops.attn_bwd_raw(d_o.to(dev), qd, k_in, vd, o, lse, cd, sd, meta, scale, dq, dk, dv, simt=simt)
    torch.cuda.synchronize()
    out = {"o": o.cpu(), "lse": lse.cpu(), "dq": dq.cpu(), "dk": dk.cpu(), "dv": dv.cpu()}
    return out, (k_in.cpu() if cos is not None else k)


def check_all(got, ex, md, rows):
    """o and lse over live rows; the gradients over every row (rows that see nothing have zero gradient)."""
    check_close("o", got["o"], ex["o"], md["o"], rows)
    check_lse(got["lse"], ex["lse"], rows)
    for nm in ("dq", "dk", "dv"):
        check_close(nm, got[nm], ex[nm], md[nm])
    if (~rows).any():
        assert float(got["o"].float()[~rows].abs().max()) == 0.0, "rows that see no key must be zero"


# ------------------------------------------------------------------------------------------------ case builders
def _unit(seed):
    """A fixed +-1 direction u (u.u = 96) for the constructed score patterns."""
    g = torch.Generator().manual_seed(seed)
    return (torch.randint(0, 2, (D,), generator=g) * 2 - 1).double()


def case_wide():
    """q, k ~ N(0, 3^2), causal: scaled scores ~ N(0, 9^2) -- the row maximum keeps growing from tile to tile."""
    B, T, H = 1, 1000, 8
    q, k, v = Hp.qkv_inputs(B, T, H, D, seed=101, std=3.0)
    v = _randn((B, T, H, D), 102)
    return dict(q=q, k=k, v=v, lang=None, N=None, cos=None, sin=None, scale=SCALE)


def case_scale_one():
    """The ABI's scale argument at 1.0 (no other test uses another value than 96^-0.5): scores ~ N(0, 96), two-image MMA
    prompt, RoPE."""
    lang, am = Hp.make_prompt(1, 600, 128, 2)
    T = int(O.segments_ref(lang, am, 128, Hp.MEDIA_ID).seq_len[0])
    q, k, v = Hp.qkv_inputs(1, T, 8, D, seed=111)
    cos, sin = _tables(torch.arange(T)[None])
    return dict(q=q, k=k, v=v, lang=lang, am=am, N=128, cos=cos, sin=sin, scale=1.0)


RAMP_SLOPES = [1.0, 1.25, 1.5, 2.0, 1.1, 1.2, -1.0, 1.4]    # per head; head 6 falls along the keys


def case_ramp():
    """A shared component along u: k_j = c_j u + noise with c_j rising linearly over the keys, q = a_h u + noise, so the
    scores rise along the keys by a_h * 20 * 96 * scale nats (283 log2 units at a_h = 1) over 8 key tiles; one head has
    a negative slope (its maximum sits in tile 0)."""
    B, T, H = 1, 1024, 8
    u = _unit(121)
    c = torch.linspace(-10.0, 10.0, T, dtype=torch.float64)
    a = torch.tensor(RAMP_SLOPES, dtype=torch.float64)
    q = (torch.randn(B, T, H, D, generator=torch.Generator().manual_seed(122), dtype=torch.float64) * 0.5
         + a[None, None, :, None] * u).to(torch.bfloat16)
    k = (torch.randn(B, T, H, D, generator=torch.Generator().manual_seed(123), dtype=torch.float64) * 0.5
         + c[None, :, None, None] * u).to(torch.bfloat16)
    v = _randn((B, T, H, D), 124)
    return dict(q=q, k=k, v=v, lang=None, N=None, cos=None, sin=None, scale=SCALE)


def _sink(q, k, pos, gap_nats, seed):
    """q += 3u for every row, the other keys made orthogonal to u, k[pos[h]] = c u: key pos[h] of head h scores
    gap_nats (+- 1.4) while the rest keep their N(0, 1) scores."""
    u = _unit(seed)
    c = gap_nats / (3 * D * SCALE)
    qd, kd = q.double() + 3 * u, k.double()
    kd -= (kd @ u)[..., None] * u / D
    for h, p in enumerate(pos):
        kd[:, p, h] = c * u
    return qd.to(torch.bfloat16), kd.to(torch.bfloat16)


def case_late_sink():
    """One key per (b, h) in key tile 2 or 3, +40 nats above the rest, in the text after the image span and before
    <|assistant|>: the image rows see it through the mutual block, after their own first key tile."""
    lang, am = Hp.make_prompt(1, 500, 128, 1)
    S = O.segments_ref(lang, am, 128, Hp.MEDIA_ID)
    T, H = int(S.seq_len[0]), 8
    q, k, v = Hp.qkv_inputs(1, T, H, D, seed=131)
    pos = [300 + 29 * h for h in range(H)]
    assert max(pos) < int(S.q_end[0]) and min(pos) >= int(np.nonzero(S.seg[0] == 1)[0][-1]) + 1
    q, k = _sink(q, k, pos, 40.0, 132)
    return dict(q=q, k=k, v=v, lang=lang, am=am, N=128, cos=None, sin=None, scale=SCALE, pos=pos)


def case_early_sink():
    """Key 0 +30 nats above the rest (the BOS-sink pattern): the maximum is set in tile 0 and never moves again, so the
    row sum spans e^0 .. e^-30 with no rescale."""
    B, T, H = 1, 700, 8
    q, k, v = Hp.qkv_inputs(B, T, H, D, seed=141)
    q, k = _sink(q, k, [0] * H, 30.0, 142)
    return dict(q=q, k=k, v=v, lang=None, N=None, cos=None, sin=None, scale=SCALE)


def case_very_negative():
    """Heads 0-3: q = -a u + noise, k = a u + noise, every visible score ~ -200 nats (LSE ~ -200, -LSE/scale ~ +1960 in
    the backward's fold).  Heads 4-7: N(0, 1) scores."""
    B, T, H = 1, 600, 8
    q, k, v = Hp.qkv_inputs(B, T, H, D, seed=151)
    u = _unit(152)
    a = math.sqrt(200.0 / (D * SCALE))
    qd, kd = q.double(), k.double()
    qd[:, :, :4] = qd[:, :, :4] * 0.3 - a * u
    kd[:, :, :4] = kd[:, :, :4] * 0.3 + a * u
    return dict(q=qd.to(torch.bfloat16), k=kd.to(torch.bfloat16), v=v, lang=None, N=None, cos=None, sin=None, scale=SCALE)


LEFT_PAD = 300


def case_left_pad():
    """AKI.generate style batch: padding_side="left", sample 0 starts with 300 pad tokens (> 2 key tiles), one image per
    sample, positions cumsum(mask) - 1 per sample -> per-sample RoPE tables (B,T,48)."""
    L, N = 500, 64
    g = np.random.default_rng(161)
    lang = g.integers(3, 31000, size=(2, L)).astype(np.int64)
    am = np.ones_like(lang)
    lang[0, :LEFT_PAD] = Hp.PAD_ID; am[0, :LEFT_PAD] = 0
    lang[0, LEFT_PAD + 5] = Hp.MEDIA_ID; lang[0, 450] = Hp.ASST_ID
    lang[1, 5] = Hp.MEDIA_ID; lang[1, 400] = Hp.ASST_ID
    S = O.segments_ref(lang, am, N, Hp.MEDIA_ID)
    T, H = int(S.seq_len.max()), 8
    valid = torch.from_numpy(S.valid.astype(np.int64))[:, :T]
    pos = (valid.cumsum(1) - 1).clamp(min=0)
    cos, sin = _tables(pos)
    assert not torch.equal(cos[0], cos[1])
    q, k, v = Hp.qkv_inputs(2, T, H, D, seed=162, std=1.5)
    return dict(q=q, k=k, v=v, lang=lang, am=am, N=N, cos=cos, sin=sin, scale=SCALE)


CASES = {"wide": case_wide, "scale-one": case_scale_one, "ramp": case_ramp, "late-sink": case_late_sink,
         "early-sink": case_early_sink, "very-negative": case_very_negative, "left-pad": case_left_pad}


def prepare(name):
    """Inputs, the host-side mask and the fp64 reference of a case (no device needed)."""
    c = CASES[name]()
    B, T, H, _ = c["q"].shape
    S = O.segments_ref(c["lang"], c["am"], c["N"], Hp.MEDIA_ID) if c["lang"] is not None else None
    allowed = _allowed(S, T)
    c["S"], c["allowed"] = S, allowed
    c["rows"] = allowed.any(-1)
    c["d_o"] = _randn((B, T, H, D), 9001)
    return c


def reference_for(c, k_rot):
    q_rot = _rotate(c["q"], c["cos"], c["sin"]) if c["cos"] is not None else c["q"]
    return reference(q_rot, k_rot, c["v"], c["allowed"], c["scale"], c["d_o"], c["cos"], c["sin"])


def assert_path_reached(name, c, ev):
    H = c["q"].shape[2]
    if name in ("wide", "scale-one"):
        assert int(ev["rescales"].sum()) > 0
    elif name == "ramp":
        up = [h for h in range(H) if RAMP_SLOPES[h] > 0]
        tm = c["tile_max"][0] * LOG2E
        # the maximum of the last row rises by > 200 log2 units from tile 0: unrescaled, P would overflow fp32 / bf16
        assert float((tm[up, -1, -1] - tm[up, -1, 0]).min()) > 200, "ramp too shallow"
        per_tile = rescale_events(c["tile_max"][:, up])["per_tile"]
        assert all(n > 0 for n in per_tile[1:]), per_tile        # a rescale at every key tile after the first
    elif name == "late-sink":
        img = torch.from_numpy(c["S"].seg[0] == 1)
        # image rows (before the sink) rescale with alpha ~ 2^-58 at the sink's tile
        assert float(ev["min_log2_alpha"][0][:, img].max()) < -45, float(ev["min_log2_alpha"][0][:, img].max())
    elif name == "early-sink":
        assert int(ev["rescales"].sum()) == 0 and int(ev["late"].sum()) == 0
    elif name == "very-negative":
        lse = c["ref"][0]["lse"][0, :4]
        assert float(lse.max()) < -150 and float(lse.min()) > -250
    elif name == "left-pad":
        late = ev["late"][0]                                      # sample 0: rows past the padding start in tile 2
        assert int(late.sum()) > 0 and int(late[:, LEFT_PAD:].min()) == 1


@pytest.mark.parametrize("name", list(CASES))
def test_wide_range_forward_backward(name):
    """Forward (o, lse) and backward (dq, dk, dv) of the tcgen05 kernels against the fp64 reference on constructed score
    patterns; each case first asserts that the forward path it targets is reached."""
    ops = _ops()
    c = prepare(name)
    B, T, H, _ = c["q"].shape
    segs = None
    if c["lang"] is not None:
        S, segs = _segments(c["lang"], c["am"], c["N"])
        assert segs.T == T
        assert np.array_equal(segs.expand_to_4d().cpu().numpy()[:, 0] != 0, c["allowed"].numpy())
    got, k_rot = run_kernels(c["q"], c["k"], c["v"], c["cos"], c["sin"], segs, c["scale"], c["d_o"])
    if c["cos"] is not None:        # rope_kv_write with these tables: K rotated in fp32, rounded once
        kr = _rotate(c["k"], c["cos"], c["sin"]).float()
        assert float((k_rot.float() - kr).abs().max()) <= float(kr.abs().max()) * 2 ** -7
    ex, md, c["tile_max"] = reference_for(c, k_rot)
    c["ref"] = (ex, md)
    assert_path_reached(name, c, rescale_events(c["tile_max"]))
    check_all(got, ex, md, c["rows"])
    if name == "left-pad":
        # fully padded key tiles of sample 0 (keys 0..255): no query sees them, the gradient is exactly zero
        for nm in ("dk", "dv"):
            assert float(got[nm][0, :2 * KEY_TILE].float().abs().max()) == 0.0, nm
        assert not c["rows"][0, :LEFT_PAD].any()


# ------------------------------------------------------------------------------------------------ full size
@pytest.fixture(scope="module")
def full_size():
    """BASELINE config 3 geometry (T = 8192, 4 image spans, long longrope factors), q, k ~ N(0, 2.5^2), 32 heads: the
    tcgen05 kernels, the SIMT verification kernels, and the fp64 reference of heads 0-1."""
    import bench
    ops = _ops()
    B, T, H = 1, 8192, 32
    lang, am = bench.make_prompt(B, T, 4)
    S = O.segments_ref(lang, am, 128, Hp.MEDIA_ID)
    segs = ops.build_segments(torch.from_numpy(lang).to(dev), torch.from_numpy(am).to(dev), 128, Hp.MEDIA_ID, t_cap=T,
                              exact_shape=False)
    assert segs.T == T
    q, k, v = Hp.qkv_inputs(B, T, H, D, seed=171, std=2.5)
    v = _randn((B, T, H, D), 172)
    d_o = _randn((B, T, H, D), 173)
    cos, sin = _tables(torch.arange(T)[None], long_factors=True)
    tc, k_rot = run_kernels(q, k, v, cos, sin, segs, SCALE, d_o)
    simt, _ = run_kernels(q, k, v, cos, sin, segs, SCALE, d_o, simt=True)
    heads = [0, 1]
    allowed = _allowed(S, T)
    ex, md, tile_max = reference(_rotate(q, cos, sin), k_rot, v, allowed, SCALE, d_o, cos, sin, heads=heads, row_block=512)
    return dict(tc=tc, simt=simt, ex=ex, md=md, tile_max=tile_max, heads=heads, rows=allowed.any(-1))


def test_full_size_wide_vs_fp64(full_size):
    """Heads 0-1 of the 32-head run at T = 8192 against the fp64 reference, with the precision-model yardstick."""
    f = full_size
    assert int(rescale_events(f["tile_max"])["rescales"].sum()) > 0
    got = {nm: (x[:, :, f["heads"]] if nm != "lse" else x[:, f["heads"]]) for nm, x in f["tc"].items()}
    check_all(got, f["ex"], f["md"], f["rows"])


def test_full_size_wide_tcgen05_vs_simt(full_size):
    """All 32 heads: the tcgen05 kernels against the SIMT kernels (fp32 throughout, no bf16 P or dS).  The bound is the
    fp64 yardstick of heads 0-1 taken relative to the tensor's maximum: the tcgen05 result may be 2 model errors off the
    exact value, the SIMT one a rounding of its output, so 3 x (max|model - exact| / max|exact|) x max|simt| + 1e-3 RMS."""
    f = full_size
    for nm in ("o", "dq", "dk", "dv"):
        a, b_ = f["tc"][nm].double(), f["simt"][nm].double()
        assert not torch.isnan(a).any() and not torch.isnan(b_).any(), nm
        rel = float((f["md"][nm] - f["ex"][nm]).abs().max()) / float(f["ex"][nm].abs().max())
        tol = 3.0 * rel * float(b_.abs().max()) + 1e-3 * float(b_.pow(2).mean().sqrt())
        err = float((a - b_).abs().max())
        assert err <= tol, f"{nm}: tcgen05 vs SIMT {err:.3e} > {tol:.3e}"
    lse_t, lse_s = f["tc"]["lse"].double(), f["simt"]["lse"].double()
    assert float(((lse_t - lse_s).abs() - 2e-3 - 2e-4 * lse_s.abs()).max()) <= 0


# ------------------------------------------------------------------------------------------------ decode
def _decode_exact(q, kc, vc, kv_len, kv_start, scale):
    """fp64 O.decode_attention over keys [kv_start, kv_len) of each sample.  Returns (B,H,D)."""
    outs = []
    for b in range(q.shape[0]):
        s0, n = int(kv_start[b]), int(kv_len[b])
        outs.append(O.decode_attention(q[b:b + 1].double()[:, :, None], kc[b:b + 1, :, s0:n].double(),
                                       vc[b:b + 1, :, s0:n].double(), [n - s0], scale)[:, 0])
    return torch.cat(outs)


def _decode_tol(got, exact):
    """The decode keeps P in fp32; only the output rounds: 2^-8 max|exact| (per sample and head) + 1e-3."""
    err = (got.double() - exact).abs().amax(-1)
    tol = 2 ** -8 * exact.abs().amax(-1) + 1e-3
    return bool((err <= tol).all()), float((err - tol).max())


def test_decode_long_split_kv():
    """16 splits at 8K, kv_start across a 512-key chunk boundary (1500) and exactly on one (1024), a single key, and
    max_kv_len above every kv_len (the graphed decode step passes the cache capacity): trailing splits are empty."""
    ops = _ops()
    B, H, tcap = 4, 32, 8192
    kv_len, kv_start = [8192, 4097, 1536, 1], [0, 1500, 1024, 0]
    q = _randn((B, H, D), 181, 3.0)
    kc = _randn((B, H, tcap, D), 182, 3.0)
    vc = _randn((B, H, tcap, D), 183)
    i32 = lambda x: torch.tensor(x, dtype=torch.int32, device=dev)   # noqa: E731
    out = ops.decode_op(q.to(dev), kc.to(dev), vc.to(dev), i32(kv_len), 8192 + 512, SCALE, i32(kv_start)).cpu()
    ok, worst = _decode_tol(out, _decode_exact(q, kc, vc, kv_len, kv_start, SCALE))
    assert ok, f"decode off by {worst:.3e} beyond the bound"


def test_decode_single_visible_key_is_that_value_row():
    """kv_start = kv_len - 1: one visible key, p = 1, so the output is that V row (exactly: l = 1 and A = V in fp32)."""
    ops = _ops()
    B, H, tcap = 4, 32, 4608
    kv_len = [1, 512, 513, 4097]
    q = _randn((B, H, D), 191, 3.0)
    kc = _randn((B, H, tcap, D), 192, 3.0)
    vc = _randn((B, H, tcap, D), 193)
    i32 = lambda x: torch.tensor(x, dtype=torch.int32, device=dev)   # noqa: E731
    out = ops.decode_op(q.to(dev), kc.to(dev), vc.to(dev), i32(kv_len), tcap, SCALE, i32([n - 1 for n in kv_len])).cpu()
    for b, n in enumerate(kv_len):
        assert torch.equal(out[b], vc[b, :, n - 1]), b


def test_decode_matches_prefill_last_row_wide():
    """Decode of token 4097 against the last row of the causal prefill over 4098 tokens, q, k ~ N(0, 3^2): both against
    the fp64 row (the prefill also rounds P to bf16: 2^-7), and each other."""
    ops = _ops()
    T, H = 4097, 32
    q, k, v = Hp.qkv_inputs(1, T + 1, H, D, seed=201, std=3.0)
    v = _randn((1, T + 1, H, D), 202)
    qd, kd, vd = q.to(dev), k.to(dev), v.to(dev)
    o_full, _ = ops.attn_fwd_raw(qd, kd, vd, None, None, None, SCALE)
    kcache, vcache = kd.transpose(1, 2).contiguous(), vd.transpose(1, 2).contiguous()
    o_dec = ops.decode_op(qd[:, T].contiguous(), kcache, vcache, torch.tensor([T + 1], dtype=torch.int32, device=dev),
                          T + 1, SCALE).cpu()
    exact = _decode_exact(q[:, T], k.transpose(1, 2), v.transpose(1, 2), [T + 1], [0], SCALE)
    ok, worst = _decode_tol(o_dec, exact)
    assert ok, f"decode off by {worst:.3e} beyond the bound"
    pre = o_full[:, T].cpu().double()
    bound = 2 ** -7 * exact.abs().amax(-1, keepdim=True) + 1e-3
    assert bool(((pre - exact).abs() <= bound).all())
    assert bool(((pre - o_dec.double()).abs() <= bound + 2 ** -8 * exact.abs().amax(-1, keepdim=True)).all())
