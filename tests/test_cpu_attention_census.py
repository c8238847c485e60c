"""The reference builders of the attention census (helpers.allowed_slab, visible_counts, decode_visible, census_diff)
against the oracle's own mask constructions, on CPU: what test_gpu_attention_census.py compares the kernels with."""
import numpy as np
import pytest
import torch

import helpers as Hp
from oracle import mma_oracle as O
from test_gpu_attention import CASES, _edge_prompt

EDGE_KINDS = ["left-pad-generate", "mixed-image-counts", "tile-edges", "assistant-before-image", "no-assistant",
              "text-only-variant", "span-straddles-tiles", "back-to-back-spans", "more-spans-than-plan-cuts"]


def _prompts():
    for name, B, L, N, n_img, _, pad in CASES:
        lang, am = Hp.make_prompt(B, L, N, n_img, pad_right=pad, first_img=min(8, L // 3))
        yield name, lang, am, N, False
    for kind in EDGE_KINDS:
        lang, am, N, text_only = _edge_prompt(kind)
        yield kind, lang, am, N, text_only


PROMPTS = list(_prompts())


@pytest.mark.parametrize("name,lang,am,N,text_only", PROMPTS, ids=[p[0] for p in PROMPTS])
def test_allowed_slab_equals_oracle_masks(name, lang, am, N, text_only):
    S = O.segments_ref(lang, am, N, Hp.MEDIA_ID, text_only=text_only)
    T = int(S.seq_len.max())
    R = Hp.MaskRef.from_segments(S, T, text_only)
    full = Hp.allowed_slab(R, (0, T), (0, T))
    assert torch.equal(full, torch.from_numpy(O.expand_segments_to_4d(S, t_out=T, text_only=text_only)[:, 0]).bool())
    # straight from lang_x / attention_mask, without the Segments description
    variant = "text_only" if text_only else "contiguous"
    for b in range(lang.shape[0]):
        m = torch.from_numpy(O._generalised_mask(lang[b], am[b], N, Hp.MEDIA_ID, Hp.ASST_ID, variant)[0]).bool()
        tb = m.shape[0]
        assert torch.equal(full[b, :tb, :tb], m), (name, b)
        assert not full[b, tb:].any() and not full[b, :, tb:].any()
    # row-blocked and offset slabs are pieces of the same matrix; rows / keys past Tk see / are seen by nothing
    for rows, cols in [((0, min(T, 37)), (5, T)), ((T // 3, T), (0, T // 2 + 1)), ((T - 1, T + 40), (T - 3, T + 100))]:
        s = Hp.allowed_slab(R, rows, cols)
        r1, c1 = min(rows[1], T), min(cols[1], T)
        assert torch.equal(s[:, :r1 - rows[0], :c1 - cols[0]], full[:, rows[0]:r1, cols[0]:c1])
        assert not s[:, r1 - rows[0]:].any() and not s[:, :, c1 - cols[0]:].any()
    assert torch.equal(Hp.visible_counts(R), full.sum(-1))


def test_pure_causal_and_explicit_validity():
    R = Hp.MaskRef.causal(2, 300, seq_len=[300, 129])
    a = Hp.allowed_slab(R, (0, 300), (0, 300))
    tril = torch.tril(torch.ones(300, 300, dtype=torch.bool))
    assert torch.equal(a[0], tril)
    assert torch.equal(a[1, :129, :129], tril[:129, :129]) and a[1].sum() == 129 * 130 // 2
    assert torch.equal(Hp.visible_counts(R)[1, :130], torch.cat([torch.arange(1, 130), torch.zeros(1, dtype=torch.int64)]))
    # an explicit 2-D validity mask plus intervals, the form of a continuation's key-coordinate metadata: the same
    # predicate written element by element
    g = np.random.default_rng(3)
    B, Tk = 2, 260
    valid = torch.from_numpy(g.random((B, Tk)) > 0.1)
    lo = torch.zeros(B, Tk, dtype=torch.int64); hi = torch.zeros(B, Tk, dtype=torch.int64)
    lo[0, 40:90] = 90; hi[0, 40:90] = 200
    lo[1, 120:140] = 140; hi[1, 120:140] = 400                       # interval past the sequence end
    R = Hp.MaskRef(torch.tensor([Tk, 230]), valid, valid, lo, hi)
    a = Hp.allowed_slab(R, (0, Tk), (0, Tk))
    for b in range(B):
        n = int(R.seq_len[b])
        for i in range(0, Tk, 7):
            want = [i < n and j < n and bool(valid[b, j]) and (j <= i or lo[b, i] <= j < hi[b, i]) for j in range(Tk)]
            assert a[b, i].tolist() == want, (b, i)
    assert torch.equal(Hp.visible_counts(R), a.sum(-1))


def test_decode_visible_and_values():
    valid = torch.ones(3, 600, dtype=torch.bool)
    valid[1, 30:70] = False
    vis = Hp.decode_visible(torch.tensor([1, 513, 600]), torch.tensor([0, 31, 599]), valid, 600)
    assert vis[0].nonzero().flatten().tolist() == [0]
    assert vis[1].nonzero().flatten().tolist() == list(range(70, 513))
    assert vis[2].nonzero().flatten().tolist() == [599]
    assert torch.equal(Hp.decode_visible(torch.tensor([4]), None, None, 6), torch.tensor([[1, 1, 1, 1, 0, 0]]).bool())
    n = torch.tensor([0, 1, 3, 257, 32768])
    r = Hp.recip_bf16(n)
    assert r[0] == 0 and r[1] == 1 and r[4] == 2.0 ** -15
    assert r[2] == float(torch.tensor(1 / 3, dtype=torch.float32).to(torch.bfloat16))


def test_census_diff_reports_first_pair_and_count():
    want = torch.zeros(2, 4, 5, dtype=torch.bool)
    want[:, :, :2] = True
    got = want.to(torch.float32) * 0.5
    assert Hp.census_diff(got, want, torch.arange(4), torch.arange(5)).shape == (0, 5)
    got[1, 2, 4] = 0.25                                               # one extra key
    got[0, 3, 1] = 0.0                                                # one missing key
    d = Hp.census_diff(got, want, torch.arange(100, 104), torch.arange(7, 12))
    assert d.tolist() == [[0, 103, 8, 0.0, 1.0], [1, 102, 11, 0.25, 0.0]]
    msg = Hp.census_message(d, "x")
    assert "2 (row, key) pairs" in msg and "(0, 103, 8, 0, True)" in msg
