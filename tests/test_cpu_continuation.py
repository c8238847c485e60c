"""CPU checks of the continuation (follow-up turn / chunked prefill) support: the key-coordinate metadata a KV cache
keeps for its rows, against a numpy restatement, and the argument validation of the offset entry points."""
import ctypes as C
import types

import numpy as np
import pytest
import torch

from aki_b200.cache import KeyMeta, bits_to_bool, bool_to_bits, place_bits, shift_rows


def _np_bits(words, n):
    w = words.astype(np.int64) & 0xFFFFFFFF
    return np.array([[(w[b, j // 32] >> (j % 32)) & 1 for j in range(n)] for b in range(w.shape[0])], dtype=bool)


@pytest.mark.parametrize("past,T", [(0, 77), (5, 40), (37, 300), (100, 29), (129, 1), (1000, 333), (4095, 130)])
def test_chunk_meta_shift_and_bit_placement(past, T):
    g = np.random.default_rng(past * 7 + T)
    B, t_cap = 3, past + T + int(g.integers(0, 70))
    lo = g.integers(0, T, size=(B, T)).astype(np.int32)
    hi = (lo + g.integers(-3, 50, size=(B, T))).astype(np.int32)          # empty (hi <= lo) and live intervals
    vchunk = g.random((B, T)) < 0.8
    mchunk = g.random((B, T)) < 0.5
    W = (T + 31) // 32
    pad = lambda x: np.concatenate([x, np.zeros((B, 32 * W - T), dtype=bool)], 1)
    segs = types.SimpleNamespace(row_lo=torch.from_numpy(lo), row_hi=torch.from_numpy(hi),
                                 kv_valid_bits=bool_to_bits(torch.from_numpy(pad(vchunk))),
                                 kv_mutual_bits=bool_to_bits(torch.from_numpy(pad(mchunk))),
                                 seq_len=torch.full((B,), T, dtype=torch.int32))
    km = KeyMeta(B, t_cap, "cpu")
    before_v = np.ones((B, t_cap), dtype=bool)
    before_v[:, : past // 2] = g.random((B, past // 2)) < 0.5              # some earlier rows already invalid
    place_bits(km.kv_valid_bits, torch.from_numpy(before_v[:, :t_cap]), 0)
    km.write_chunk(past, T, segs)
    # numpy restatement
    live = hi > lo
    exp_lo = np.zeros((B, t_cap), np.int32); exp_hi = np.zeros((B, t_cap), np.int32)
    exp_lo[:, past:past + T] = np.where(live, lo + past, 0); exp_hi[:, past:past + T] = np.where(live, hi + past, 0)
    exp_v = before_v.copy(); exp_v[:, past:past + T] = vchunk
    exp_m = np.zeros((B, t_cap), bool); exp_m[:, past:past + T] = mchunk
    assert np.array_equal(km.row_lo.numpy(), exp_lo) and np.array_equal(km.row_hi.numpy(), exp_hi)
    W_cap = (t_cap + 31) // 32
    bits_v = _np_bits(km.kv_valid_bits.numpy(), 32 * W_cap)
    assert np.array_equal(bits_v[:, :t_cap], exp_v)
    assert bits_v[:, t_cap:].all()                                         # words past t_cap untouched (initial ones)
    assert np.array_equal(_np_bits(km.kv_mutual_bits.numpy(), t_cap), exp_m)
    assert (km.seq_len.numpy() == past + T).all()
    # helpers on their own
    l2, h2 = shift_rows(torch.from_numpy(lo), torch.from_numpy(hi), past)
    assert np.array_equal(l2.numpy(), exp_lo[:, past:past + T]) and np.array_equal(h2.numpy(), exp_hi[:, past:past + T])
    assert torch.equal(bits_to_bool(km.kv_valid_bits, t_cap), torch.from_numpy(exp_v))
    km.reset()
    assert (km.kv_valid_bits == -1).all() and not km.kv_mutual_bits.any() and not km.row_hi.any()


def test_write_chunk_from_key_validity():
    km = KeyMeta(2, 100, "cpu")
    valid = torch.ones(2, 45, dtype=torch.bool)
    valid[1, :13] = False
    km.write_chunk(33, 45, None, valid)
    exp = torch.ones(2, 100, dtype=torch.bool)
    exp[1, 33:46] = False
    assert torch.equal(bits_to_bool(km.kv_valid_bits, 100), exp)
    assert not km.row_hi.any() and not km.kv_mutual_bits.any() and (km.seq_len == 78).all()


@pytest.fixture(scope="module")
def lib():
    from aki_b200 import _lib
    return _lib


def test_offset_argument_validation_without_gpu(lib):
    L = lib.lib
    p = lib.AttnParams()
    p.B, p.H, p.T, p.D = 1, 32, 128, 96
    p.q_offset = -1
    assert L.aki_mma_attn_fwd(C.byref(p), None) == -2
    assert L.aki_mma_attn_fwd_simt(C.byref(p), None) == -2
    p.q_offset = 2 ** 31 - 100                     # q_offset + T overflows int32
    assert L.aki_mma_attn_fwd(C.byref(p), None) == -2
    bp = lib.AttnBwdParams()
    bp.fwd.B, bp.fwd.H, bp.fwd.T, bp.fwd.D = 1, 32, 128, 96
    bp.fwd.q_offset = 64                           # training never continues onto a cache
    assert L.aki_mma_attn_bwd(C.byref(bp), None) == -3
    assert L.aki_mma_attn_bwd_simt(C.byref(bp), None) == -3
    buf = (C.c_int32 * 64)()
    assert L.aki_mma_fwd_plan_at(buf, buf, buf, None, 1, 128, -1, 256, 0, 4, 3, buf, None) == -2
    assert L.aki_mma_fwd_plan_at(buf, buf, buf, None, 1, 128, 200, 256, 0, 4, 3, buf, None) == -2    # pitch < 328
    assert L.aki_mma_fwd_plan_at(buf, buf, buf, buf, 1, 128, 100, 228, 7, 4, 3, buf, None) == -2     # 7*32 < 228
    assert L.aki_mma_tile_bounds_at(buf, buf, buf, 1, 128, 100, 200, buf, None, None) == -2          # t_cap < 228
    assert L.aki_mma_tile_bounds_at(buf, buf, buf, 1, 128, 100, 228, buf, buf, None) == -3           # backward mask
    assert L.aki_mma_decode_masked(buf, buf, buf, 96, 96, buf, None, buf, 1, 64, 1, 1, 96, 0.1, buf, buf, 1 << 20,
                                   None) == -2                                                      # 1 word < 64 keys
    assert L.aki_mma_decode_masked(None, buf, buf, 96, 96, buf, None, None, 0, 64, 1, 1, 96, 0.1, buf, buf, 1 << 20,
                                   None) == -1


def test_continuation_symbols_exported(lib):
    for name in ("aki_mma_fwd_plan_at", "aki_mma_tile_bounds_at", "aki_mma_decode_masked"):
        assert name in lib.EXPORTED_SYMBOLS and hasattr(lib.lib, name)
    assert [f[0] for f in lib.AttnParams._fields_][-1] == "q_offset"
