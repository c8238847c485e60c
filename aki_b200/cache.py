"""Preallocated KV cache honouring the HF past_key_values contract the reference relies on
(codes/open_flamingo/src/vlm.py:463-468 reads past_key_values[0][0].shape[2];
codes/open_flamingo/src/aki_generation.py:45-47,80): per layer (K, V), each (B, H, T_kv, D), K stored post-RoPE,
appended along dim 2.  Instead of DynamicCache's torch.cat per step, prefill and decode write rows in place into
(B, H, t_cap, D) buffers (layout chosen so one (b,h) stream is contiguous for TMA and for the decode kernel)."""
from __future__ import annotations

from typing import List, Optional, Tuple

import torch
from transformers.cache_utils import Cache, CacheLayerMixin


def bits_to_bool(words: torch.Tensor, n: int) -> torch.Tensor:
    """(B, W) int32 bit-vectors (bit j of word j // 32 = key j) -> (B, n) bool."""
    idx = torch.arange(n, device=words.device)
    return ((words[:, idx // 32] >> (idx % 32)) & 1).bool()


def bool_to_bits(flags: torch.Tensor) -> torch.Tensor:
    """(B, 32 W) bool -> (B, W) int32 bit-vectors (the uint32 bit pattern)."""
    B, n = flags.shape
    w = (flags.view(B, n // 32, 32).to(torch.int64) << torch.arange(32, device=flags.device)).sum(-1)
    return torch.where(w >= 1 << 31, w - (1 << 32), w).to(torch.int32)


def place_bits(dst: torch.Tensor, src: torch.Tensor, past: int) -> None:
    """Overwrite bits [past, past + T) of the (B, W) int32 bit-vectors `dst` with the (B, T) bool `src`, in place; the
    other bits of the words touched are kept.  Device ops only (no host read)."""
    T = src.shape[1]
    w0, w1 = past // 32, (past + T + 31) // 32
    cur = bits_to_bool(dst[:, w0:w1], 32 * (w1 - w0))
    cur[:, past - 32 * w0:past - 32 * w0 + T] = src
    dst[:, w0:w1] = bool_to_bits(cur)


def shift_rows(row_lo: torch.Tensor, row_hi: torch.Tensor, past: int) -> Tuple[torch.Tensor, torch.Tensor]:
    """Chunk-relative mutual intervals [row_lo, row_hi) -> key coordinates of a chunk that starts at row `past` (rows
    without an interval keep 0 / 0)."""
    live = row_hi > row_lo
    zero = torch.zeros_like(row_lo)
    return torch.where(live, row_lo + past, zero), torch.where(live, row_hi + past, zero)


class KeyMeta:
    """MMA description of the rows of a KV cache in absolute key coordinates (include/aki_mma.h, AkiMmaAttnParams):
    validity / mutual bits (B, ceil(t_cap/32)) and row_lo / row_hi (B, t_cap).  Validity starts as all ones, so rows
    appended by decode steps (eager or graph-replayed) are valid with no extra work; each prefill or continuation chunk
    writes its own rows (write_chunk).  A continuation attends over these with q_offset = past (attn_meta)."""

    def __init__(self, batch: int, t_cap: int, device):
        self.t_cap = int(t_cap)
        words = (self.t_cap + 31) // 32
        self.kv_valid_bits = torch.empty(batch, words, dtype=torch.int32, device=device)
        self.kv_mutual_bits = torch.empty_like(self.kv_valid_bits)
        self.row_lo = torch.empty(batch, self.t_cap, dtype=torch.int32, device=device)
        self.row_hi = torch.empty_like(self.row_lo)
        self.seq_len = torch.empty(batch, dtype=torch.int32, device=device)   # keys of the last chunk's attention
        self.reset()

    def reset(self) -> None:
        self.kv_valid_bits.fill_(-1)
        self.kv_mutual_bits.zero_()
        self.row_lo.zero_()
        self.row_hi.zero_()
        self.seq_len.zero_()

    def write_chunk(self, past: int, T: int, segs=None, key_valid: Optional[torch.Tensor] = None) -> None:
        """Rows [past, past + T) from the chunk's own (chunk-relative) segments, or from key_valid (B, T) bool alone
        (no MMA term; None = all valid)."""
        if past + T > self.t_cap:
            raise ValueError(f"KV cache capacity {self.t_cap} exceeded (need {past + T})")
        B = self.row_lo.shape[0]
        if segs is not None:
            lo, hi = shift_rows(segs.row_lo[:, :T], segs.row_hi[:, :T], past)
            self.row_lo[:, past:past + T] = lo
            self.row_hi[:, past:past + T] = hi
            place_bits(self.kv_valid_bits, bits_to_bool(segs.kv_valid_bits, T), past)
            place_bits(self.kv_mutual_bits, bits_to_bool(segs.kv_mutual_bits, T), past)
            self.seq_len.copy_(segs.seq_len.clamp(max=T) + past)
            return
        self.row_lo[:, past:past + T] = 0
        self.row_hi[:, past:past + T] = 0
        valid = (torch.ones(B, T, dtype=torch.bool, device=self.row_lo.device) if key_valid is None
                 else key_valid.to(device=self.row_lo.device, dtype=torch.bool))
        place_bits(self.kv_valid_bits, valid, past)
        place_bits(self.kv_mutual_bits, torch.zeros_like(valid), past)
        self.seq_len.fill_(past + T)

    def attn_meta(self, past: int, T: int, max_spans: int = 8, plan: bool = True):
        """Metadata tuple for ops.attn_fwd_raw(..., q_offset=past) of the chunk written last."""
        from . import ops
        return ops.continuation_meta(self.seq_len, self.row_lo, self.row_hi, self.kv_valid_bits, self.kv_mutual_bits, T,
                                     past, max_spans, plan)


class _AkiCacheLayer(CacheLayerMixin):
    """One layer's view of the preallocated buffers, so that AkiKVCache is a real transformers `Cache` (HF generate,
    masking utilities and model code only ever talk to `cache.layers[i]` / the Cache methods built on them)."""
    is_compileable = False
    is_sliding = False

    def __init__(self, owner: "AkiKVCache", idx: int):
        self._owner, self._idx = owner, idx
        super().__init__()
        self.is_initialized = True

    # the base class assigns keys / values = None in __init__; here they are live views of the owner's buffers
    keys = property(lambda self: self._owner.k[self._idx][:, :, :self._owner._len[self._idx]], lambda self, v: None)
    values = property(lambda self: self._owner.v[self._idx][:, :, :self._owner._len[self._idx]], lambda self, v: None)

    @property
    def device(self):
        return self._owner.k[self._idx].device

    def lazy_initialization(self, key_states, value_states) -> None:
        return None

    def update(self, key_states, value_states, *args, **kwargs):
        return self._owner._append(self._idx, key_states, value_states)

    def get_mask_sizes(self, query_length, *args) -> Tuple[int, int]:
        q = int(query_length.shape[0]) if isinstance(query_length, torch.Tensor) else int(query_length)
        return self._owner._len[self._idx] + q, 0

    def get_seq_length(self, *args) -> int:
        return self._owner._len[self._idx]

    def get_max_cache_shape(self) -> int:
        return self._owner.t_cap

    def reset(self) -> None:
        self._owner._len[self._idx] = 0

    def offload(self):
        raise NotImplementedError("AkiKVCache lives in HBM (180 GB per B200): offloading is not supported")

    prefetch = offload

    def reorder_cache(self, beam_idx) -> None:
        raise NotImplementedError("beam search is not part of the reference path (AKI.generate pops num_beams, aki.py:160)")


class AkiKVCache(Cache):
    def __init__(self, num_layers: int, batch: int, num_heads: int, head_dim: int, t_cap: int, device,
                 dtype=torch.bfloat16):
        super().__init__(layers=[_AkiCacheLayer(self, i) for i in range(num_layers)])
        self.t_cap = int(t_cap)
        self.k: List[torch.Tensor] = [torch.zeros(batch, num_heads, t_cap, head_dim, dtype=dtype, device=device)
                                      for _ in range(num_layers)]
        self.v: List[torch.Tensor] = [torch.zeros_like(self.k[0]) for _ in range(num_layers)]
        self._len = [0] * num_layers
        self.kv_len = torch.zeros(batch, dtype=torch.int32, device=device)   # device copy for the decode kernel
        # first visible key of every sequence: the leading pad rows of a left-padded prompt (AKI.generate pads on the
        # left, aki.py:172-182) stay in the cache but must not be attended by the decode steps.  A cheap lower bound: the
        # pad rows a follow-up turn leaves inside the cache are described by meta.kv_valid_bits.  Positions are uniform
        # across the batch (past + arange(T), as the decode steps use): pad rows inside a chunk still take a position.
        self.kv_start = torch.zeros(batch, dtype=torch.int32, device=device)
        # CUDA-graph decode: the step reads the write row / key count from these device tensors instead of host ints
        self.past_dev = torch.zeros(batch, dtype=torch.int32, device=device)
        self.device_driven = False
        # absolute MMA metadata of the cached rows (follow-up turns / chunked prefill attend over it; the decode steps
        # skip the rows whose validity bit is 0 -- interior pad rows of a batched follow-up turn)
        self.meta = KeyMeta(batch, t_cap, device)
        self._chunk_meta = None      # (past, T, meta tuple) of the chunk being prefilled, shared by all layers

    # ---- HF Cache surface --------------------------------------------------------------------------
    def get_seq_length(self, layer_idx: int = 0) -> int:
        return self._len[layer_idx]

    def get_max_cache_shape(self, layer_idx: int = 0) -> int:
        return self.t_cap

    def get_mask_sizes(self, query_length, layer_idx: int = 0):
        return self.layers[layer_idx].get_mask_sizes(query_length)

    def __len__(self) -> int:
        return len(self.k)

    def __getitem__(self, layer_idx: int) -> Tuple[torch.Tensor, torch.Tensor]:
        n = self._len[layer_idx]
        return self.k[layer_idx][:, :, :n], self.v[layer_idx][:, :, :n]

    def __iter__(self):
        for i in range(len(self.k)):
            yield self[i]

    def update(self, key_states: torch.Tensor, value_states: torch.Tensor, layer_idx: int, *args, **kwargs):
        """DynamicCache-compatible append of already rotated (B,H,T,D) states (used by foreign callers; the
        drop-in module writes through reserve()/commit() instead so RoPE and the copy are one kernel)."""
        return self._append(layer_idx, key_states, value_states)

    def _append(self, layer_idx: int, key_states: torch.Tensor, value_states: torch.Tensor):
        n, t = self._len[layer_idx], key_states.shape[2]
        self.reserve(layer_idx, t)
        self.k[layer_idx][:, :, n:n + t].copy_(key_states)
        self.v[layer_idx][:, :, n:n + t].copy_(value_states)
        self.commit(layer_idx, t)
        return self[layer_idx]

    # ---- in-place protocol used by AkiMMAAttention -------------------------------------------------
    def set_key_start(self, mask_2d: Optional[torch.Tensor]) -> None:
        """Number of leading invalid keys per sequence from the spliced 2-D mask (device arithmetic, no host read)."""
        if mask_2d is None:
            self.kv_start.zero_()
        else:
            self.kv_start.copy_((mask_2d.to(torch.int32).cumsum(1) == 0).sum(1).to(torch.int32))

    def write_prefill_meta(self, T: int, segs=None) -> None:
        """After a prefill onto the empty cache (and set_key_start): rows [0, T) are valid from kv_start on -- exactly
        the keys the decode steps attend -- and keep the prompt's mutual intervals."""
        valid = torch.arange(T, device=self.kv_start.device)[None] >= self.kv_start[:, None]
        self.meta.write_chunk(0, T, None, valid)
        if segs is not None:
            lo, hi = shift_rows(segs.row_lo[:, :T], segs.row_hi[:, :T], 0)
            self.meta.row_lo[:, :T] = lo
            self.meta.row_hi[:, :T] = hi
            place_bits(self.meta.kv_mutual_bits, bits_to_bool(segs.kv_mutual_bits, T), 0)

    def chunk_meta(self, past: int, T: int, segs=None, key_valid: Optional[torch.Tensor] = None, first: bool = True):
        """Metadata of a continuation chunk at row `past`: the first layer writes the chunk's rows and builds the plan,
        the other layers reuse it."""
        if first or self._chunk_meta is None or self._chunk_meta[:2] != (past, T):
            self.meta.write_chunk(past, T, segs, key_valid)
            self._chunk_meta = (past, T, self.meta.attn_meta(past, T, segs.max_spans if segs is not None else 8))
        return self._chunk_meta[2]

    def reserve(self, layer_idx: int, t: int) -> int:
        n = self._len[layer_idx]
        self._check(n + t)
        if layer_idx == 0:            # one tiny fill per step; every layer then reads the same device scalar(s)
            self.kv_len.fill_(n + t)
        return n

    def commit(self, layer_idx: int, t: int) -> None:
        self._len[layer_idx] += t

    def _check(self, need: int) -> None:
        if need > self.t_cap:
            raise ValueError(f"KV cache capacity {self.t_cap} exceeded (need {need})")

    def advance_host(self, t: int = 1) -> None:
        """Host-side bookkeeping after a device-driven (graph-replayed) step appended t rows to every layer."""
        self._check(self._len[0] + t)
        self._len = [n + t for n in self._len]

    def reset(self) -> None:
        """Forget the contents (buffers are reused; nothing is freed)."""
        self._len = [0] * len(self.k)
        self.kv_len.zero_()
        self.kv_start.zero_()
        self.past_dev.zero_()
        self.meta.reset()
        self._chunk_meta = None

    def to_legacy_cache(self):
        return tuple(self[i] for i in range(len(self.k)))
