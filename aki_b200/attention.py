"""Drop-in attention for AKI's Phi-3.5-mini decoder layers.

  AkiMMAAttention      nn.Module with Phi3Attention's constructor, parameters (state-dict keys
                       ``qkv_proj.weight`` (9216,3072), ``o_proj.weight`` (3072,3072)) and forward signature
                       (installed transformers/models/phi3/modeling_phi3.py:208-271).  The 4.41-era remote-code
                       call the reference's pinned transformers makes -- keywords ``attention_mask, position_ids,
                       past_key_value, output_attentions, use_cache``, no position_embeddings, no **kwargs, three
                       return values -- is served too: cos / sin come from ``position_ids`` through the module's own
                       LongRope and the MMA description from ``mma_context(segs)`` (the 4.41 decoder layer forwards
                       no extra kwargs).  Replaces the eager path the reference is forced onto by its 4-D mask
                       (codes/open_flamingo/src/aki.py:125-130).
  aki_mma_attention    AttentionInterface function (``config._attn_implementation = "aki_mma"``).
  replace_phi3_attention / register_attention_interface   installers.

The MMA description travels as ``mma_segments`` (ops.MMASegments) in the layer kwargs, which HF forwards
unchanged to every layer; without it the op is plain causal attention.  qkv_proj / o_proj stay cuBLAS GEMMs.
"""
from __future__ import annotations

import contextlib
import threading
from typing import Optional, Tuple

import torch
from torch import nn

from . import ops
from .cache import AkiKVCache, KeyMeta, place_bits
from .rope import LongRope, half_tables_from_hf

_ctx = threading.local()


def _key_valid(attention_mask: Optional[torch.Tensor], n_keys: int) -> Optional[torch.Tensor]:
    """(B, n_keys) bool validity of the keys of a continuation from HF's mask: 2-D (B, past+T) 0/1, or 4-D
    (B, 1, T, past+T) reduced to its last query row (bool: True = visible; integer: 1 = visible; floating: additive,
    0 = visible).  The MMA term of the chunk comes from mma_segments only.  None: every key is valid."""
    if attention_mask is None:
        return None
    m = attention_mask if attention_mask.dim() == 2 else attention_mask[:, 0, -1]
    m = m[:, :n_keys]
    if m.dtype == torch.bool:
        return m
    return (m == 0) if (attention_mask.dim() == 4 and m.is_floating_point()) else (m != 0)


def _foreign_continuation_meta(B: int, t_kv: int, T: int, segs: Optional[ops.MMASegments], attention_mask, device):
    """Key-coordinate metadata of a continuation onto a cache that keeps no MMA description (DynamicCache, the
    AttentionInterface plugin): causal over all t_kv keys, validity from the mask, the chunk's own segments shifted."""
    past = t_kv - T
    km = KeyMeta(B, t_kv, device)
    valid = _key_valid(attention_mask, t_kv)
    if valid is not None and past > 0:
        place_bits(km.kv_valid_bits, valid[:, :past], 0)
    km.write_chunk(past, T, segs, None if (segs is not None or valid is None) else valid[:, past:])
    return km.attn_meta(past, T, segs.max_spans if segs is not None else 8)


@contextlib.contextmanager
def mma_context(segs: Optional[ops.MMASegments]):
    """Carries the MMA description to every AkiMMAAttention called inside the block, for callers whose decoder layers
    forward no extra kwargs (transformers 4.41.2, the reference's pin: codes/setup.py:12).  Usage in the reference:
    ``with mma_context(new_inputs.pop("mma_segments")): output = self.lang_model(**new_inputs, ...)`` (aki.py:125-130)."""
    prev = getattr(_ctx, "segs", None)
    _ctx.segs = segs
    try:
        yield
    finally:
        _ctx.segs = prev


class AkiMMAAttention(nn.Module):
    def __init__(self, config, layer_idx: Optional[int] = None):
        super().__init__()
        self.config = config
        self.layer_idx = layer_idx
        self.num_heads = config.num_attention_heads
        self.head_dim = getattr(config, "head_dim", None) or config.hidden_size // config.num_attention_heads
        kv_heads = getattr(config, "num_key_value_heads", self.num_heads)
        if kv_heads != self.num_heads:
            raise ValueError("AkiMMAAttention implements Phi-3.5-mini's MHA (num_key_value_heads == num_attention_heads)")
        if self.head_dim != ops.HEAD_DIM:
            raise ValueError(f"head_dim {self.head_dim} unsupported: the sm_100a kernels are tiled for head_dim 96")
        self.num_key_value_heads = kv_heads
        self.num_key_value_groups = 1
        self.scaling = self.head_dim ** -0.5
        self.attention_dropout = getattr(config, "attention_dropout", 0.0)
        self.is_causal = True
        op_size = 3 * self.num_heads * self.head_dim
        self.o_proj = nn.Linear(self.num_heads * self.head_dim, config.hidden_size, bias=False)
        self.qkv_proj = nn.Linear(config.hidden_size, op_size, bias=False)

    def forward(self, hidden_states: torch.Tensor, position_embeddings: Optional[Tuple[torch.Tensor, torch.Tensor]] = None,
                attention_mask: Optional[torch.Tensor] = None, past_key_values=None, **kwargs):
        if self.training and self.attention_dropout > 0.0:
            raise NotImplementedError("attention dropout > 0 is not implemented (Phi-3.5-mini uses 0.0)")
        legacy = position_embeddings is None and "mma_rope" not in kwargs and kwargs.get("position_ids") is not None
        if legacy:
            out, _ = self._forward(hidden_states, None, attention_mask, kwargs.pop("past_key_value", past_key_values), **kwargs)
            return out, None, kwargs.get("past_key_value", past_key_values)       # 4.41: (out, attn_weights, past_key_value)
        return self._forward(hidden_states, position_embeddings, attention_mask, past_key_values, **kwargs)

    def _legacy_rope(self, position_ids: torch.Tensor):
        """cos / sin (B,T,48) fp32 from position_ids: what the 4.41-era Phi3 rotary embedding computes inside the
        attention module (the factor set follows the running maximum position, as there)."""
        if getattr(self, "_rope", None) is None:
            rp = getattr(self.config, "rope_parameters", None) or getattr(self.config, "rope_scaling", None) or {}
            self._rope = LongRope(self.head_dim, rp.get("rope_theta", getattr(self.config, "rope_theta", 10000.0)),
                                  rp.get("short_factor"), rp.get("long_factor"), self.config.max_position_embeddings,
                                  rp.get("original_max_position_embeddings",
                                         getattr(self.config, "original_max_position_embeddings", 4096)),
                                  device=position_ids.device)
        return self._rope.tables(position_ids)

    def _forward(self, hidden_states, position_embeddings, attention_mask, past_key_values, **kwargs):
        past_key_values = kwargs.pop("past_key_value", past_key_values)           # 4.41-era keyword
        segs: Optional[ops.MMASegments] = kwargs.get("mma_segments")
        if segs is None:
            segs = getattr(_ctx, "segs", None)                                    # mma_context()
        rope = kwargs.get("mma_rope")                                             # (cos, sin) (B|1,T,48) fp32
        if rope is None:
            if position_embeddings is not None:
                rope = half_tables_from_hf(position_embeddings)
            elif kwargs.get("position_ids") is not None:
                rope = self._legacy_rope(kwargs["position_ids"])
            else:
                raise ValueError("pass position_embeddings=(cos, sin), mma_rope=(cos48, sin48) or position_ids")
        cos, sin = rope
        if segs is not None and hidden_states.shape[1] == 1:
            segs = None          # decode step: the generate loop's mask is all ones (aki_generation.py:56-62)
        continuing = hasattr(past_key_values, "get_seq_length") and past_key_values.get_seq_length(self.layer_idx or 0) > 0
        if (attention_mask is not None and attention_mask.dim() == 4 and segs is None and hidden_states.shape[1] > 1
                and not continuing):
            # (a continuation reduces a 4-D mask to key validity, see _key_valid)
            # (a one-token step gets HF's (B,1,1,T_kv) row, all visible by the generate contract: nothing to describe)
            raise ValueError("a materialised 4-D mask was passed without mma_segments: build the compact description "
                             "with aki_b200.prepare_inputs_for_forward / ops.build_segments instead")
        B, T, _ = hidden_states.shape
        H, D = self.num_heads, self.head_dim
        qkv = self.qkv_proj(hidden_states)
        if qkv.dtype != torch.bfloat16:
            raise TypeError("AkiMMAAttention computes in bf16: run the module in bf16 or under autocast(bfloat16)")
        meta = ops.meta_tuple(segs)

        if past_key_values is None:
            # training / cache-less prefill: autograd-capable fused op
            o, _, _ = ops.attn_packed_op(qkv, cos, sin, H, self.scaling, *(meta or ()))
        elif isinstance(past_key_values, AkiKVCache):
            cache = past_key_values
            if T == 1 and cache.device_driven:
                # CUDA-graph decode step: write row and key count come from device memory, nothing host-dependent
                q_rot = torch.empty(B, H, 1, D, dtype=torch.bfloat16, device=qkv.device)
                ops.rope_kv_write(qkv, cos, sin, cache.k[self.layer_idx], cache.v[self.layer_idx], 0, H, q_rot=q_rot,
                                  past_len_dev=cache.past_dev)
                o = ops.decode_op(q_rot.view(B, H, D), cache.k[self.layer_idx], cache.v[self.layer_idx], cache.kv_len,
                                  cache.t_cap, self.scaling, cache.kv_start, cache.meta.kv_valid_bits).view(B, 1, H * D)
                return self.o_proj(o), None
            past = cache.reserve(self.layer_idx, T)
            if T == 1 and past > 0:
                q_rot = torch.empty(B, H, 1, D, dtype=torch.bfloat16, device=qkv.device)
                ops.rope_kv_write(qkv, cos, sin, cache.k[self.layer_idx], cache.v[self.layer_idx], past, H, q_rot=q_rot)
                cache.commit(self.layer_idx, 1)
                o = ops.decode_op(q_rot.view(B, H, D), cache.k[self.layer_idx], cache.v[self.layer_idx], cache.kv_len,
                                  past + 1, self.scaling, cache.kv_start, cache.meta.kv_valid_bits).view(B, 1, H * D)
            elif past > 0:
                # follow-up turn / chunked prefill: the chunk's queries are key rows [past, past + T) of the cache.  The
                # chunk's mutual intervals come from its own segments (an image row sees the later keys of its chunk up
                # to that chunk's <|assistant|>: the single-turn rule applied per turn).
                ops.rope_kv_write(qkv, cos, sin, cache.k[self.layer_idx], cache.v[self.layer_idx], past, H)
                cache.commit(self.layer_idx, T)
                valid = None if segs is not None else _key_valid(attention_mask, past + T)
                meta = cache.chunk_meta(past, T, segs, None if valid is None else valid[:, past:],
                                        first=self.layer_idx in (0, None))
                k4 = cache.k[self.layer_idx][:, :, :past + T].transpose(1, 2)
                v4 = cache.v[self.layer_idx][:, :, :past + T].transpose(1, 2)
                q4 = qkv[..., : H * D].unflatten(-1, (H, D))
                o, _ = ops.attn_fwd_raw(q4, k4, v4, cos, sin, meta, self.scaling, need_lse=False, q_offset=past)
                o = o.view(B, T, H * D)
            else:
                ops.rope_kv_write(qkv, cos, sin, cache.k[self.layer_idx], cache.v[self.layer_idx], 0, H)
                cache.commit(self.layer_idx, T)
                if self.layer_idx in (0, None):      # decode steps skip the leading pad rows of a left-padded prompt
                    cache.set_key_start(segs.spliced_mask_2d() if segs is not None else
                                        (attention_mask if attention_mask is not None and attention_mask.dim() == 2 else None))
                    cache.write_prefill_meta(T, segs)
                k4 = cache.k[self.layer_idx][:, :, :T].transpose(1, 2)
                v4 = cache.v[self.layer_idx][:, :, :T].transpose(1, 2)
                q4 = qkv[..., : H * D].unflatten(-1, (H, D))
                o, _ = ops.attn_fwd_raw(q4, k4, v4, cos, sin, meta, self.scaling, need_lse=False)
                o = o.view(B, T, H * D)
        else:
            # foreign HF Cache (DynamicCache): honour update(); K/V come back as (B,H,T_kv,D)
            k_new = torch.empty(B, H, T, D, dtype=torch.bfloat16, device=qkv.device)
            v_new = torch.empty_like(k_new)
            q_rot = torch.empty_like(k_new)
            ops.rope_kv_write(qkv, cos, sin, k_new, v_new, 0, H, q_rot=q_rot)
            k_all, v_all = past_key_values.update(k_new, v_new, self.layer_idx)
            t_kv = k_all.shape[2]
            if t_kv == T:
                o, _ = ops.attn_fwd_raw(q_rot.transpose(1, 2), k_all.transpose(1, 2), v_all.transpose(1, 2), None, None,
                                        meta, self.scaling, need_lse=False)
                o = o.view(B, T, H * D)
            elif T == 1:
                k_all, v_all = k_all.contiguous(), v_all.contiguous()
                kv_len = torch.full((B,), t_kv, dtype=torch.int32, device=qkv.device)
                o = ops.decode_op(q_rot.view(B, H, D), k_all, v_all, kv_len, t_kv, self.scaling).view(B, 1, H * D)
            else:
                meta = _foreign_continuation_meta(B, t_kv, T, segs, attention_mask, qkv.device)
                o, _ = ops.attn_fwd_raw(q_rot.transpose(1, 2), k_all.transpose(1, 2), v_all.transpose(1, 2), None, None,
                                        meta, self.scaling, need_lse=False, q_offset=t_kv - T)
                o = o.view(B, T, H * D)
        return self.o_proj(o), None


def aki_mma_attention(module, query, key, value, attention_mask, scaling: Optional[float] = None, dropout: float = 0.0,
                      **kwargs):
    """AttentionInterface plugin: query/key/value (B,H,T,D) post-RoPE; returns ((B,T,H,D) contiguous, None).
    Same contract as eager_attention_forward (modeling_phi3.py:153-175)."""
    if dropout:
        raise NotImplementedError("dropout > 0 not implemented")
    if scaling is None:
        scaling = query.shape[-1] ** -0.5
    segs = kwargs.get("mma_segments")
    if segs is None:
        segs = getattr(_ctx, "segs", None)          # mma_context(): HF generate() rejects unknown model kwargs
    B, H, T, D = query.shape
    if T == 1:
        segs = None                                 # decode step: all cached keys visible (aki_generation.py:56-62)
    if key.shape[2] != T and T > 1:
        # continuation: the queries are the last T of key.shape[2] keys
        t_kv = key.shape[2]
        meta = _foreign_continuation_meta(B, t_kv, T, segs, attention_mask, query.device)
        o, _ = ops.attn_fwd_raw(query.transpose(1, 2), key.transpose(1, 2), value.transpose(1, 2), None, None, meta,
                                float(scaling), need_lse=False, q_offset=t_kv - T)
        return o, None
    if key.shape[2] != T:
        kv_len = torch.full((B,), key.shape[2], dtype=torch.int32, device=query.device)
        o = ops.decode_op(query.reshape(B, H, D), key.contiguous(), value.contiguous(), kv_len, key.shape[2], scaling)
        return o.view(B, 1, H, D), None
    meta = ops.meta_tuple(segs)
    o, _ = ops.attn_op(query.transpose(1, 2), key.transpose(1, 2), value.transpose(1, 2), float(scaling), *(meta or ()))
    return o, None


def register_attention_interface(name: str = "aki_mma") -> str:
    from transformers import AttentionInterface
    AttentionInterface.register(name, aki_mma_attention)
    return name


def replace_phi3_attention(model: nn.Module, layers_attr: str = "model.layers") -> int:
    """Swap every decoder layer's self_attn for AkiMMAAttention, re-using the existing parameters (the same
    `decoder_layers_attr_name` the reference uses, codes/open_flamingo/src/factory.py:182)."""
    layers = model
    for part in layers_attr.split("."):
        layers = getattr(layers, part)
    n = 0
    for idx, layer in enumerate(layers):
        old = layer.self_attn
        new = AkiMMAAttention(old.config, layer_idx=getattr(old, "layer_idx", idx))
        new.qkv_proj, new.o_proj = old.qkv_proj, old.o_proj
        new.train(old.training)
        layer.self_attn = new
        n += 1
    return n
