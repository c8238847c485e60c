"""Continuation onto a non-empty KV cache (follow-up turns, chunked prefill): the forward kernel with q_offset against
one forward over the whole sequence, the masked decode, and the module / runner / foreign-cache paths built on them."""
import numpy as np
import pytest
import torch

import helpers as Hp
from oracle import mma_oracle as O

pytestmark = pytest.mark.gpu
dev = torch.device("cuda", 0)
SCALE = 96 ** -0.5


def _abs_meta(B, Tk, spans, invalid, q_ends, device=dev):
    """Key-coordinate metadata of a Tk-row sequence: image spans (start, length) per sample whose rows see the later
    keys up to q_ends[b][k] (exclusive), keys listed in `invalid` masked out.  Returns the tensors and a (B,Tk,Tk)
    bool mask of the same predicate for the oracle."""
    row_lo = torch.zeros(B, Tk, dtype=torch.int32)
    row_hi = torch.zeros(B, Tk, dtype=torch.int32)
    valid = torch.ones(B, Tk, dtype=torch.bool)
    for b in range(B):
        for (s, n), e in zip(spans[b], q_ends[b]):
            row_lo[b, s:s + n] = s + n
            row_hi[b, s:s + n] = e
        for j in invalid[b]:
            valid[b, j] = False
    from aki_b200.cache import bool_to_bits
    W = (Tk + 31) // 32
    pad = torch.zeros(B, 32 * W, dtype=torch.bool)
    pad[:, :Tk] = valid
    vbits = bool_to_bits(pad)
    mbits = vbits.clone()
    i = torch.arange(Tk)[None, :, None]
    j = torch.arange(Tk)[None, None, :]
    allowed = ((j <= i) & valid[:, None, :]) | ((j >= row_lo[:, :, None]) & (j < row_hi[:, :, None]) & valid[:, None, :])
    seq_len = torch.full((B,), Tk, dtype=torch.int32)
    meta = [x.to(device).contiguous() for x in (seq_len, row_lo, row_hi, vbits, mbits)]
    return meta, allowed


def _geometry(past, T, B=2, seed=0, n_img=None):
    g = np.random.default_rng(seed)
    Tk = past + T
    spans, ends, invalid = [], [], []
    for b in range(B):
        sp, en = [], []
        n = (2 if Tk > 600 else 1) if n_img is None else n_img
        # one span in the prefix (when there is room) and one in the chunk
        cands = []
        if past > 80:
            cands.append(int(g.integers(0, past - 70)))
        if T > 80:
            cands.append(past + int(g.integers(0, T - 70)))
        for s in sorted(cands)[:max(n, 0)]:
            ln = int(g.integers(16, 65))
            top = Tk if s >= past else past
            sp.append((s, ln)); en.append(min(top, s + ln + int(g.integers(1, 200))))
        spans.append(sp); ends.append(en)
        invalid.append([int(x) for x in g.choice(Tk, size=min(5, Tk // 4), replace=False)] + list(range(b * 3)))
    return spans, ends, invalid


def _inputs(B, Tk, H, seed, rope):
    import aki_b200
    q, k, v = Hp.qkv_inputs(B, Tk, H, 96, seed=seed, device=dev)
    cos = sin = None
    if rope:
        r = aki_b200.LongRope(device=dev)
        cos, sin = r.tables(torch.arange(Tk, device=dev)[None], max_position=Tk - 1)
    return q, k, v, cos, sin


def _run_pair(past, T, rope, plan, seed=0, H=4, B=2, n_img=None):
    from aki_b200 import ops
    Tk = past + T
    spans, ends, invalid = _geometry(past, T, B, seed, n_img)
    (seq_len, lo, hi, vb, mb), allowed = _abs_meta(B, Tk, spans, invalid, ends)
    q, k, v, cos, sin = _inputs(B, Tk, H, seed, rope)
    full = ops.continuation_meta(seq_len, lo, hi, vb, mb, Tk, 0, plan=plan)
    o_full, lse_full = ops.attn_fwd_raw(q, k, v, cos, sin, full, SCALE)
    part = ops.continuation_meta(seq_len, lo, hi, vb, mb, T, past, plan=plan)
    c = None if cos is None else cos[:, past:].contiguous()
    s = None if sin is None else sin[:, past:].contiguous()
    o, lse = ops.attn_fwd_raw(q[:, past:], k, v, c, s, part, SCALE, q_offset=past)
    return o, lse, o_full, lse_full, (q, k, v, cos, sin, allowed, part, c, s)


@pytest.mark.parametrize("past,T", [(128, 896), (1000, 24), (777, 1271), (4096, 4096), (1, 383)])
@pytest.mark.parametrize("rope", [False, True])
@pytest.mark.parametrize("plan", [True, False])
def test_kernel_continuation_equals_one_shot(past, T, rope, plan):
    o, lse, o_full, lse_full, _ = _run_pair(past, T, rope, plan, seed=past + T)
    torch.cuda.synchronize()
    assert torch.equal(o, o_full[:, past:]), float((o.float() - o_full[:, past:].float()).abs().max())
    assert torch.equal(lse, lse_full[:, :, past:])


@pytest.mark.parametrize("past,T", [(1, 383), (128, 896), (1000, 24)])
def test_kernel_continuation_vs_fp32_oracle(past, T):
    o, _, _, _, (q, k, v, cos, sin, allowed, _, _, _) = _run_pair(past, T, True, True, seed=3)
    Tk = past + T
    c = torch.cat([cos, cos], -1).cpu(); s = torch.cat([sin, sin], -1).cpu()
    qf, kf, vf = (x.cpu().float().transpose(1, 2) for x in (q, k, v))
    qr, kr = O.apply_rope(qf, c, s), kf          # the kernel rotates Q only: k is its post-RoPE key input
    add = O.invert_4d_mask(allowed[:, None, past:].to(torch.int64), torch.float32)
    ref32 = O.eager_attention(qr[:, :, past:], kr, vf, add, SCALE)
    q16, k16, v16 = qr.to(torch.bfloat16), kr.to(torch.bfloat16), vf.to(torch.bfloat16)
    ref16 = O.eager_attention(q16[:, :, past:], k16, v16, add.to(torch.bfloat16), SCALE)
    rows = allowed[:, past:].any(-1)
    ok, ek, eb, _ = Hp.within_tolerance(o, ref16, ref32, rows=rows)
    assert ok, (ek, eb)
    assert Tk == q.shape[1]


def test_kernel_continuation_vs_simt_8k():
    from aki_b200 import ops
    past, T = 4096, 4096
    o, lse, _, _, (q, k, v, cos, sin, allowed, part, c, s) = _run_pair(past, T, True, True, seed=11, H=2, B=1)
    o_s, lse_s = ops.attn_fwd_raw(q[:, past:], k, v, c, s, part, SCALE, simt=True, q_offset=past)
    live = allowed[:, past:].any(-1).to(dev)
    err = float((o.float() - o_s.float()).abs()[live].max())
    assert err < 2e-2, err
    assert float((lse - lse_s).abs().transpose(1, 2)[live].max()) < 1e-2


@pytest.mark.parametrize("seed", [21, 22, 23, 24])
def test_kernel_continuation_random_geometries(seed):
    g = np.random.default_rng(seed)
    past, T = int(g.integers(1, 3000)), int(g.integers(2, 2000))
    o, lse, o_full, lse_full, (q, k, v, cos, sin, allowed, part, c, s) = _run_pair(
        past, T, bool(seed % 2), bool(seed % 3), seed=seed, n_img=int(g.integers(0, 3)))
    assert torch.equal(o, o_full[:, past:]) and torch.equal(lse, lse_full[:, :, past:]), (past, T)
    from aki_b200 import ops
    o2, lse2 = ops.attn_fwd_raw(q[:, past:], k, v, c, s, part, SCALE, q_offset=past)
    assert torch.equal(o, o2) and torch.equal(lse, lse2)


# ---------------------------------------------------------------------------------------------------------- decode
def test_masked_decode_skips_interior_rows():
    from aki_b200 import ops
    from aki_b200._lib import lib
    from aki_b200.cache import bool_to_bits
    B, H, t_cap = 3, 8, 2048
    g = torch.Generator().manual_seed(5)
    kc = torch.randn(B, H, t_cap, 96, generator=g).to(torch.bfloat16).to(dev)
    vc = torch.randn(B, H, t_cap, 96, generator=g).to(torch.bfloat16).to(dev)
    q = torch.randn(B, H, 96, generator=g).to(torch.bfloat16).to(dev)
    kv_len = torch.tensor([2048, 1500, 777], dtype=torch.int32, device=dev)
    valid = torch.ones(B, t_cap, dtype=torch.bool)
    valid[0, 600:613] = False; valid[1, 1000:1100] = False; valid[1, 31:33] = False; valid[2, 700:760] = False
    bits = bool_to_bits(valid).to(dev)
    out = ops.decode_op(q, kc, vc, kv_len, t_cap, SCALE, None, bits)
    for b in range(B):
        keep = valid[b, :int(kv_len[b])].nonzero().flatten().to(dev)
        kb, vb = kc[b:b + 1, :, keep].contiguous(), vc[b:b + 1, :, keep].contiguous()
        n = torch.tensor([keep.numel()], dtype=torch.int32, device=dev)
        ref = ops.decode_op(q[b:b + 1], kb, vb, n, keep.numel(), SCALE)
        assert float((out[b:b + 1].float() - ref.float()).abs().max()) < 1e-2, b
    plain = ops.decode_op(q, kc, vc, kv_len, t_cap, SCALE)
    ones = ops.decode_op(q, kc, vc, kv_len, t_cap, SCALE, None, torch.full_like(bits, -1))
    nb = lib.aki_mma_decode_workspace_bytes(B, H, 96, t_cap)
    ws = torch.empty(nb, dtype=torch.uint8, device=dev)
    null = torch.empty_like(q)
    assert lib.aki_mma_decode_masked(q.data_ptr(), kc.data_ptr(), vc.data_ptr(), kc.stride(0), kc.stride(1),
                                     kv_len.data_ptr(), None, None, 0, t_cap, B, H, 96, SCALE, null.data_ptr(),
                                     ws.data_ptr(), nb, torch.cuda.current_stream().cuda_stream) == 0
    assert torch.equal(null, plain) and torch.equal(ones, plain)


# ---------------------------------------------------------------------------------------------------------- runner
@pytest.fixture(scope="module")
def runner():
    from aki_b200.model import AkiPhi3Runner, phi35_mini_config
    return AkiPhi3Runner(phi35_mini_config(num_layers=2), device=dev, seed=0)


def _close(a, b, rel=3e-2):
    a, b = a.float(), b.float()
    err = float((a - b).abs().max())
    return err <= rel * max(1.0, float(b.abs().max())), err


@pytest.mark.parametrize("fused", [True, False])
def test_runner_chunked_prefill_then_decode(runner, fused):
    B, T1, T2 = 2, 700, 333
    torch.manual_seed(1)
    emb = (torch.randn(B, T1 + T2, 3072, device=dev) * 0.05).to(torch.bfloat16)
    c_one = runner.new_cache(B, T1 + T2 + 16)
    l_one = runner.prefill(emb, None, c_one, last_only=False, fused=fused)
    c_two = runner.new_cache(B, T1 + T2 + 16)
    runner.prefill(emb[:, :T1], None, c_two, fused=fused)
    l_two = runner.prefill(emb[:, T1:], None, c_two, last_only=False, fused=fused)
    ok, err = _close(l_two, l_one[:, T1:])
    assert ok, err
    tok = l_one[:, -1].argmax(-1, keepdim=True)
    for _ in range(8):
        a = runner.decode_step(tok, c_one)
        b = runner.decode_step(tok, c_two)
        ok, err = _close(b, a)
        assert ok, err
        tok = a[:, -1].argmax(-1, keepdim=True)


def test_runner_generate_continues_cache(runner):
    B, T1, T2 = 1, 300, 40
    torch.manual_seed(2)
    emb = (torch.randn(B, T1 + T2, 3072, device=dev) * 0.05).to(torch.bfloat16)
    _, cache = runner.generate(emb[:, :T1], None, 4, t_cap=T1 + T2 + 16)
    n = cache.get_seq_length()
    out, cache2 = runner.generate(emb[:, T1:], None, 4, cache=cache)
    assert cache2 is cache and cache.get_seq_length() == n + T2 + 4 and out.shape == (B, 4)


# ---------------------------------------------------------------------------------------------------------- module
def _module(seed=0):
    from aki_b200 import AkiMMAAttention
    from aki_b200.model import phi35_mini_config
    torch.manual_seed(seed)
    cfg = phi35_mini_config(num_layers=1)
    mod = AkiMMAAttention(cfg, layer_idx=0)
    with torch.no_grad():
        mod.qkv_proj.weight.normal_(0, 0.02); mod.o_proj.weight.normal_(0, 0.02)
    return cfg, mod.to(dev).to(torch.bfloat16).eval()


def _oracle_rows(mod, hidden, cos, sin, allowed, rows):
    """fp32 Phi3Attention over the whole sequence with the absolute (B,1,Tk,Tk) mask; rows [rows, Tk)."""
    add = O.invert_4d_mask(allowed[:, None].to(torch.int64), torch.float32)
    c = torch.cat([cos, cos], -1).cpu(); s = torch.cat([sin, sin], -1).cpu()
    out, _ = O.attention_module_forward(hidden.float().cpu(), mod.qkv_proj.weight.float().cpu(),
                                        mod.o_proj.weight.float().cpu(), c, s, add)
    return out[:, rows:]


def test_batched_follow_up_turn_with_image():
    import aki_b200
    from aki_b200 import ops
    cfg, mod = _module(1)
    B, T1, N = 3, 200, 64
    pads1 = [0, 17, 40]                              # left padding of the first turn's prompts
    pads2 = [5, 0, 23]                               # ... and of the follow-ups (interior rows of the cache)
    L2 = 120
    g = np.random.default_rng(7)
    lang2 = g.integers(3, 31000, size=(B, L2)).astype(np.int64)
    am2 = np.ones((B, L2), dtype=np.int64)
    for b in range(B):
        am2[b, :pads2[b]] = 0; lang2[b, :pads2[b]] = Hp.PAD_ID
        lang2[b, pads2[b] + 10] = Hp.MEDIA_ID; lang2[b, 100] = Hp.ASST_ID
    segs2 = ops.build_segments(torch.from_numpy(lang2).to(dev), torch.from_numpy(am2).to(dev), N, Hp.MEDIA_ID)
    T2 = segs2.T
    Tk = T1 + T2
    rope = aki_b200.LongRope(device=dev)
    cos, sin = rope.tables(torch.arange(Tk, device=dev)[None], max_position=Tk - 1)
    torch.manual_seed(3)
    hidden = (torch.randn(B, Tk, 3072, device=dev)).to(torch.bfloat16)
    am1 = torch.ones(B, T1, dtype=torch.int64, device=dev)
    for b in range(B):
        am1[b, :pads1[b]] = 0
    cache = aki_b200.AkiKVCache(1, B, 32, 96, t_cap=Tk + 8, device=dev)
    with torch.no_grad():
        mod(hidden[:, :T1], None, am1, past_key_values=cache, mma_rope=(cos[:, :T1].contiguous(), sin[:, :T1].contiguous()))
        out, _ = mod(hidden[:, T1:], None, None, past_key_values=cache, mma_segments=segs2,
                     mma_rope=(cos[:, T1:].contiguous(), sin[:, T1:].contiguous()))
    # the oracle's absolute mask: causal over valid keys + the chunk's mutual block
    S = O.segments_ref(lang2, am2, N, Hp.MEDIA_ID)
    m2 = torch.from_numpy(O.expand_segments_to_4d(S))[:, 0].bool()          # (B,T2,T2) chunk-relative
    valid = torch.cat([am1.cpu().bool(), torch.from_numpy(segs2.spliced_mask_2d().cpu().numpy()).bool()], 1)
    i = torch.arange(Tk)[:, None]; j = torch.arange(Tk)[None]
    allowed = (j <= i)[None] & valid[:, None, :]
    allowed[:, T1:, T1:] |= m2
    ref = _oracle_rows(mod, hidden, cos, sin, allowed, T1)
    live = allowed[:, T1:].any(-1)
    ok, err = _close(out.cpu()[live], ref[live])
    assert ok, err
    # the cache now holds the follow-ups' pad rows in its interior: their validity bit is 0
    from aki_b200.cache import bits_to_bool
    vb = bits_to_bool(cache.meta.kv_valid_bits, Tk).cpu()
    assert torch.equal(vb, valid)


def test_graph_decode_after_follow_up_skips_pad_rows(runner):
    B, T1, T2 = 3, 256, 96
    torch.manual_seed(4)
    emb = (torch.randn(B, T1 + T2, 3072, device=dev) * 0.05).to(torch.bfloat16)
    from aki_b200.cache import place_bits
    caches = []
    for _ in range(3):
        c = runner.new_cache(B, T1 + T2 + 16)
        runner.prefill(emb[:, :T1], None, c)
        l2 = runner.prefill(emb[:, T1:], None, c)
        inval = torch.zeros(B, T2, dtype=torch.bool, device=dev)
        inval[1, :30] = True; inval[2, :7] = True                           # left-padded follow-ups
        place_bits(c.meta.kv_valid_bits, ~inval, T1)
        caches.append(c)
    # garbage in the interior pad rows of one cache must not change the decode
    for li in range(2):
        caches[2].k[li][1, :, T1:T1 + 30] = 50.0
        caches[2].v[li][1, :, T1:T1 + 30] = -50.0
    tok = l2[:, -1].argmax(-1, keepdim=True)
    t_e = t_g = t_x = tok
    for _ in range(4):
        le = runner.decode_step_fused(t_e, caches[0])
        t_e = le[:, -1].argmax(-1, keepdim=True)
        t_g = runner.decode_step_graphed(t_g, caches[1])
        lx = runner.decode_step_fused(t_x, caches[2])
        t_x = lx[:, -1].argmax(-1, keepdim=True)
        assert torch.equal(t_g, t_e) and torch.equal(lx, le)


def test_foreign_caches_match_aki_cache():
    import aki_b200
    from aki_b200 import ops
    from transformers import DynamicCache
    cfg, mod = _module(2)
    B, T1, T2 = 2, 300, 150
    Tk = T1 + T2
    rope = aki_b200.LongRope(device=dev)
    cos, sin = rope.tables(torch.arange(Tk, device=dev)[None], max_position=Tk - 1)
    rp = lambda a, b_: (cos[:, a:b_].contiguous(), sin[:, a:b_].contiguous())
    torch.manual_seed(5)
    hidden = torch.randn(B, Tk, 3072, device=dev).to(torch.bfloat16)
    mask = torch.ones(B, Tk, dtype=torch.int64, device=dev)
    mask[1, :9] = 0
    ak = aki_b200.AkiKVCache(1, B, 32, 96, t_cap=Tk + 4, device=dev)
    try:
        dc = DynamicCache(config=cfg)
    except TypeError:
        dc = DynamicCache()
    with torch.no_grad():
        mod(hidden[:, :T1], None, mask[:, :T1], past_key_values=ak, mma_rope=rp(0, T1))
        a, _ = mod(hidden[:, T1:], None, mask, past_key_values=ak, mma_rope=rp(T1, Tk))
        mod(hidden[:, :T1], None, mask[:, :T1], past_key_values=dc, mma_rope=rp(0, T1))
        d, _ = mod(hidden[:, T1:], None, mask, past_key_values=dc, mma_rope=rp(T1, Tk))
        ok, err = _close(d, a)
        assert ok, err
        # 4-D additive mask of HF for the same continuation: reduced to key validity
        add = torch.zeros(B, 1, T2, Tk, device=dev)
        add[1, :, :, :9] = torch.finfo(torch.float32).min
        ak.reset()
        mod(hidden[:, :T1], None, mask[:, :T1], past_key_values=ak, mma_rope=rp(0, T1))
        a4, _ = mod(hidden[:, T1:], None, add, past_key_values=ak, mma_rope=rp(T1, Tk))
        assert torch.equal(a4, a)
        # plugin: rotated q / k / v with key.shape[2] > T > 1
        k_all = dc.layers[0].keys if hasattr(dc, "layers") else dc.key_cache[0]
        v_all = dc.layers[0].values if hasattr(dc, "layers") else dc.value_cache[0]
        q_rot = torch.empty(B, 32, T2, 96, dtype=torch.bfloat16, device=dev)
        qkv = mod.qkv_proj(hidden[:, T1:])
        kt, vt = torch.empty_like(q_rot), torch.empty_like(q_rot)
        ops.rope_kv_write(qkv, *rp(T1, Tk), kt, vt, 0, 32, q_rot=q_rot)
        o, w = aki_b200.aki_mma_attention(None, q_rot, k_all, v_all, mask, scaling=SCALE)
        ref = ops.attn_fwd_raw(q_rot.transpose(1, 2), k_all.transpose(1, 2), v_all.transpose(1, 2), None, None,
                               ak.meta.attn_meta(T1, T2), SCALE, need_lse=False, q_offset=T1)[0]
        assert w is None and o.shape == (B, T2, 32, 96) and torch.equal(o, ref)


def test_longrope_boundary_continuation():
    import aki_b200
    cfg, mod = _module(3)
    g = np.random.default_rng(9)
    sf, lf = (1.0 + g.random(48)).tolist(), (1.0 + 4 * g.random(48)).tolist()
    rope = aki_b200.LongRope(short_factor=sf, long_factor=lf, device=dev)
    B, T1, T2 = 1, 4000, 200
    Tk = T1 + T2
    c1, s1 = rope.tables(torch.arange(T1, device=dev)[None], max_position=T1 - 1)             # short factors
    c2, s2 = rope.tables(T1 + torch.arange(T2, device=dev)[None], max_position=Tk - 1)        # long: crosses 4096
    torch.manual_seed(6)
    hidden = torch.randn(B, Tk, 3072, device=dev).to(torch.bfloat16)
    cache = aki_b200.AkiKVCache(1, B, 32, 96, t_cap=Tk, device=dev)
    with torch.no_grad():
        mod(hidden[:, :T1], None, None, past_key_values=cache, mma_rope=(c1, s1))
        out, _ = mod(hidden[:, T1:], None, None, past_key_values=cache, mma_rope=(c2, s2))
    # oracle: the prefix's keys as its prefill rotated them (short set), the new rows with the long set
    cos = torch.cat([c1, c2], 1); sin = torch.cat([s1, s2], 1)
    c = torch.cat([cos, cos], -1).cpu(); s = torch.cat([sin, sin], -1).cpu()
    qkv = hidden.float().cpu() @ mod.qkv_proj.weight.float().cpu().t()
    q, k, v = (qkv[..., i * 3072:(i + 1) * 3072].view(B, Tk, 32, 96).transpose(1, 2) for i in range(3))
    q, k = O.apply_rope(q, c, s), O.apply_rope(k, c, s)
    add = O.invert_4d_mask(torch.tril(torch.ones(Tk, Tk, dtype=torch.int64))[None, None, T1:], torch.float32)
    o = O.eager_attention(q[:, :, T1:], k, v, add, SCALE)
    ref = o.reshape(B, T2, 3072) @ mod.o_proj.weight.float().cpu().t()
    ok, err = _close(out.cpu(), ref)
    assert ok, err
    assert rope.original_max == 4096 and T1 + T2 > 4096
