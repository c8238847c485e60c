"""PyTorch custom ops over the C ABI (include/aki_mma.h).  PyTorch supplies device memory, streams and autograd
plumbing only; every computation below is a CUDA kernel in libaki_mma.so.  There is no fallback path: a CPU
tensor or a missing library raises.

Ops (torch.library, namespace ``aki_mma``):
  aki_mma::attn_packed   fused-QKV entry used by the drop-in module: RoPE(K)->cache write, RoPE(Q) at load,
                         MMA attention; autograd returns the gradient of the packed projection.
  aki_mma::attn          plugin-level entry on already rotated q/k/v (AttentionInterface function).
  aki_mma::decode        single-query attention against the KV cache.
"""
from __future__ import annotations

import ctypes as C
from dataclasses import dataclass
from typing import Optional, Tuple

import torch

from . import _lib
from ._lib import AttnBwdParams, AttnParams, Tensor4, check, lib

HEAD_DIM = _lib.HEAD_DIM
TILE = _lib.TILE


def _stream() -> C.c_void_p:
    return C.c_void_p(torch.cuda.current_stream().cuda_stream)


def _ptr(t: Optional[torch.Tensor]) -> Optional[int]:
    return None if t is None else t.data_ptr()


def _require_cuda(*ts):
    for t in ts:
        if t is not None and not t.is_cuda:
            raise _lib.AkiMmaError("aki_mma ops run on CUDA tensors only (no CPU fallback)")


# --------------------------------------------------------------------------------------------------
# segment metadata
# --------------------------------------------------------------------------------------------------
@dataclass
class MMASegments:
    """Compact description of the reference's (B,1,T,T) mask (vlm.py:410-443, utils.py:99-108)."""
    seq_len: torch.Tensor          # (B,) int32
    q_end: torch.Tensor            # (B,) int32
    seg: torch.Tensor              # (B,T) int32
    row_lo: torch.Tensor           # (B,T) int32
    row_hi: torch.Tensor           # (B,T) int32
    src: torch.Tensor              # (B,T) int32
    kv_valid_bits: torch.Tensor    # (B,ceil(T/32)) int32 (bit pattern of uint32)
    kv_mutual_bits: torch.Tensor   # (B,ceil(T/32)) int32
    q_tile_kv_end: torch.Tensor    # (B,ceil(T/128)) int32
    kv_tile_q_mask: torch.Tensor   # (B,ceil(T/128),ceil(ceil(T/128)/32)) int32 (bit pattern of uint32)
    T: int
    fwd_plan: Optional[torch.Tensor] = None   # (B, 1 + pairs, 4) int32: forward work plan (aki_mma_fwd_plan)
    max_spans: int = 8                        # image spans per sample that may start a query tile of their own
    status: Optional[torch.Tensor] = None     # (1,) int32 device flag of aki_mma_segments: 1 = some sample exceeded t_cap

    def check(self) -> "MMASegments":
        """Raises if a sample was longer than t_cap.  build_segments(t_cap=..., exact_shape=False) does no host read
        (nothing on the prefill path synchronises); call this where a read is affordable."""
        if self.status is not None and int(self.status.item()):
            raise _lib.AkiMmaError(f"t_cap={self.T} is smaller than the longest spliced sample ({int(self.seq_len.max())})")
        return self

    @property
    def B(self) -> int:
        return self.seq_len.shape[0]

    def expand_to_4d(self) -> torch.Tensor:
        """The reference's attention_mask: (B,1,T,T) int64 in {0,1} (debug / parity only; O(T^2))."""
        out = torch.empty(self.B, 1, self.T, self.T, dtype=torch.int64, device=self.seg.device)
        check(lib.aki_mma_expand_mask(_ptr(self.seq_len), _ptr(self.row_lo), _ptr(self.row_hi),
                                      _ptr(self.kv_valid_bits), _ptr(self.kv_mutual_bits), self.B, self.T, self.T,
                                      _ptr(out), _stream()), "aki_mma_expand_mask")
        return out

    def spliced_mask_2d(self) -> torch.Tensor:
        """(B,T) int64 2-D key-validity mask after splicing (ones on vision tokens), mask coordinates."""
        idx = torch.arange(self.T, device=self.seg.device)
        words = self.kv_valid_bits[:, idx // 32]
        return ((words >> (idx % 32)[None]) & 1).to(torch.int64)

    def truncated(self, T: int) -> "MMASegments":
        if T == self.T:
            return self
        return rebuild_tile_bounds(MMASegments(
            self.seq_len, self.q_end, self.seg[:, :T].contiguous(), self.row_lo[:, :T].contiguous(),
            self.row_hi[:, :T].contiguous(), self.src[:, :T].contiguous(),
            self.kv_valid_bits[:, :(T + 31) // 32].contiguous(), self.kv_mutual_bits[:, :(T + 31) // 32].contiguous(),
            self.q_tile_kv_end, self.kv_tile_q_mask, T, None, self.max_spans))


def rebuild_tile_bounds(s: MMASegments) -> MMASegments:
    nt = (s.T + TILE - 1) // TILE
    dev = s.seq_len.device
    s.q_tile_kv_end = torch.empty(s.B, nt, dtype=torch.int32, device=dev)
    s.kv_tile_q_mask = torch.empty(s.B, nt, (nt + 31) // 32, dtype=torch.int32, device=dev)
    check(lib.aki_mma_tile_bounds(_ptr(s.seq_len), _ptr(s.row_lo), _ptr(s.row_hi), s.B, s.T, s.T,
                                  _ptr(s.q_tile_kv_end), _ptr(s.kv_tile_q_mask), _stream()), "aki_mma_tile_bounds")
    s.fwd_plan = build_fwd_plan(s.seq_len, s.row_lo, s.row_hi, s.kv_valid_bits, s.T, s.max_spans)
    return s


def build_fwd_plan(seq_len, row_lo, row_hi, vbits, T: int, max_spans: int = 8, q_offset: int = 0) -> torch.Tensor:
    """Forward work plan (include/aki_mma.h, aki_mma_fwd_plan_at): (B, 1 + pairs, 4) int32 for the T query rows
    [q_offset, q_offset + T) of metadata in key coordinates."""
    B = seq_len.shape[0]
    nt = (T + TILE - 1) // TILE
    pairs = (nt + max_spans + 2) // 2
    plan = torch.empty(B, 1 + pairs, 4, dtype=torch.int32, device=seq_len.device)
    mp, bp = (row_lo.shape[1] if row_lo is not None else 0), (vbits.shape[1] if vbits is not None else 0)
    fl = 3   # cut at span starts, rank and pair by key-tile count
    if q_offset:
        check(lib.aki_mma_fwd_plan_at(_ptr(seq_len), _ptr(row_lo), _ptr(row_hi), _ptr(vbits), B, T, int(q_offset), mp, bp,
                                      pairs, fl, _ptr(plan), _stream()), "aki_mma_fwd_plan_at")
    else:
        check(lib.aki_mma_fwd_plan(_ptr(seq_len), _ptr(row_lo), _ptr(row_hi), _ptr(vbits), B, T, mp, bp, pairs, fl,
                                   _ptr(plan), _stream()), "aki_mma_fwd_plan")
    return plan


def continuation_meta(seq_len, row_lo, row_hi, vbits, mbits, T: int, q_offset: int, max_spans: int = 8,
                      plan: bool = True):
    """Metadata tuple (see meta_tuple) for attn_fwd_raw(..., q_offset=q_offset) from key-coordinate arrays
    (row_lo / row_hi (B, >= q_offset + T), bits (B, >= ceil((q_offset + T)/32))).  plan=False: per-query-tile key ends
    (aki_mma_tile_bounds_at) and aligned tiles instead of the work plan."""
    if plan:
        return (seq_len, row_lo, row_hi, vbits, mbits, None, None,
                build_fwd_plan(seq_len, row_lo, row_hi, vbits, T, max_spans, q_offset=q_offset))
    nt = (T + TILE - 1) // TILE
    kv_end = torch.empty(seq_len.shape[0], nt, dtype=torch.int32, device=seq_len.device)
    check(lib.aki_mma_tile_bounds_at(_ptr(seq_len), _ptr(row_lo), _ptr(row_hi), seq_len.shape[0], T, int(q_offset),
                                     row_lo.shape[1], _ptr(kv_end), None, _stream()), "aki_mma_tile_bounds_at")
    return (seq_len, row_lo, row_hi, vbits, mbits, kv_end, None, None)


def build_segments(lang_x: torch.Tensor, attention_mask: torch.Tensor, num_tokens_per_vis: int, media_token_id: int,
                   assistant_token_id: int = 32001, t_cap: Optional[int] = None, text_only: bool = False,
                   exact_shape: bool = True, max_spans: int = 8) -> MMASegments:
    """Device replacement of the mask half of _prepare_inputs_for_forward (vlm.py:486-577).

    t_cap: row pitch / upper bound of the spliced length; default L + (#<image> in the widest row)*(N-1) needs one
    small host read.  exact_shape=True trims T to max_b T_b exactly like the reference's stack (one more read)."""
    _require_cuda(lang_x, attention_mask)
    lang_x = lang_x.contiguous().to(torch.int64)
    attention_mask = attention_mask.contiguous().to(torch.int64)
    B, L = lang_x.shape
    N = int(num_tokens_per_vis)
    dev = lang_x.device
    seq_len = torch.empty(B, dtype=torch.int32, device=dev)
    if t_cap is None:
        # size pass: only seq_len is produced
        status = torch.zeros(1, dtype=torch.int32, device=dev)
        check(lib.aki_mma_segments(_ptr(lang_x), _ptr(attention_mask), B, L, N, media_token_id, assistant_token_id,
                                   1 << 30, int(text_only), _ptr(seq_len), None, None, None, None, None, None, None,
                                   None, _stream()), "aki_mma_segments(size)")
        t_cap = int(seq_len.max().item())
        exact_shape = False
    T = int(t_cap)
    words = (T + 31) // 32
    q_end = torch.empty(B, dtype=torch.int32, device=dev)
    seg = torch.empty(B, T, dtype=torch.int32, device=dev)
    row_lo = torch.empty_like(seg); row_hi = torch.empty_like(seg); src = torch.empty_like(seg)
    vbits = torch.empty(B, words, dtype=torch.int32, device=dev); mbits = torch.empty_like(vbits)
    status = torch.zeros(1, dtype=torch.int32, device=dev)
    check(lib.aki_mma_segments(_ptr(lang_x), _ptr(attention_mask), B, L, N, media_token_id, assistant_token_id, T,
                               int(text_only), _ptr(seq_len), _ptr(q_end), _ptr(seg), _ptr(row_lo), _ptr(row_hi),
                               _ptr(src), _ptr(vbits), _ptr(mbits), _ptr(status), _stream()), "aki_mma_segments")
    s = MMASegments(seq_len, q_end, seg, row_lo, row_hi, src, vbits, mbits, None, None, T, None, int(max_spans))
    s.status = status          # (1,) int32: 1 if some sample was longer than t_cap (outputs truncated); see check()
    if exact_shape:
        t_max, overflow = torch.stack([seq_len.max(), status[0]]).tolist()      # ONE host read for both
        if overflow or t_max > T:
            raise _lib.AkiMmaError(f"t_cap={T} is smaller than the longest spliced sample ({t_max})")
        if t_max < T:
            return s.truncated(t_max)
    return rebuild_tile_bounds(s)


def splice(lang_embeds: torch.Tensor, vision_tokens: Optional[torch.Tensor], labels: Optional[torch.Tensor],
           segs: MMASegments, pad_value: float, padding_side: str = "right"):
    """inputs_embeds / labels of vlm.py:516-588 as one gather kernel."""
    _require_cuda(lang_embeds, vision_tokens, labels)
    B, L, E = lang_embeds.shape
    lang_embeds = lang_embeds.contiguous()
    if lang_embeds.dtype != torch.bfloat16:
        raise _lib.AkiMmaError("splice expects bf16 embeddings")
    n_img_max, N = 0, 1
    if vision_tokens is not None:
        vision_tokens = vision_tokens.contiguous().to(torch.bfloat16)
        n_img_max, N = vision_tokens.shape[1], vision_tokens.shape[2]
    out = torch.empty(B, segs.T, E, dtype=torch.bfloat16, device=lang_embeds.device)
    labels_out = None
    if labels is not None:
        labels = labels.contiguous().to(torch.int64)
        labels_out = torch.empty(B, segs.T, dtype=torch.int64, device=lang_embeds.device)
    check(lib.aki_mma_splice(_ptr(lang_embeds), _ptr(vision_tokens), _ptr(labels), _ptr(segs.src), _ptr(segs.seq_len),
                             B, L, N, max(n_img_max, 1), E, segs.T, segs.T, float(pad_value),
                             int(padding_side == "left"), _ptr(out), _ptr(labels_out), _stream()), "aki_mma_splice")
    return out, labels_out


class _SpliceFn(torch.autograd.Function):
    """splice() with a backward pass: the gather is one-to-one, so the gradient of the embeddings / vision tokens is
    a scatter-add of the output gradient through `src` (training path, padding_side="right" only)."""

    @staticmethod
    def forward(ctx, lang_embeds, vision_tokens, segs, pad_value):
        out, _ = splice(lang_embeds, vision_tokens, None, segs, pad_value, "right")
        ctx.save_for_backward(segs.src)
        ctx.shapes = (lang_embeds.shape, None if vision_tokens is None else vision_tokens.shape)
        return out

    @staticmethod
    def backward(ctx, d_out):
        (src,) = ctx.saved_tensors
        (B, L, E), vshape = ctx.shapes
        src = src[:, : d_out.shape[1]].to(torch.int64)
        is_text = src >= 0
        is_vis = (src < 0) & (src > -(1 << 31))
        d_lang = torch.zeros(B, L, E, dtype=d_out.dtype, device=d_out.device)
        d_lang.scatter_add_(1, src.clamp(min=0)[..., None].expand(-1, -1, E), d_out * is_text[..., None])
        d_vis = None
        if vshape is not None:
            n_tok = vshape[1] * vshape[2]
            d_vis = torch.zeros(B, n_tok, E, dtype=d_out.dtype, device=d_out.device)
            d_vis.scatter_add_(1, (-1 - src).clamp(0, n_tok - 1)[..., None].expand(-1, -1, E), d_out * is_vis[..., None])
            d_vis = d_vis.view(vshape)
        return d_lang, d_vis, None, None


def splice_trainable(lang_embeds: torch.Tensor, vision_tokens: Optional[torch.Tensor], segs: MMASegments,
                     pad_value: float) -> torch.Tensor:
    """Differentiable splice for the SFT step (bf16 in, bf16 out; right padding)."""
    return _SpliceFn.apply(lang_embeds, vision_tokens, segs, pad_value)


# --------------------------------------------------------------------------------------------------
# rope
# --------------------------------------------------------------------------------------------------
def rope_table(position_ids: torch.Tensor, inv_freq: torch.Tensor, attention_factor: float):
    """cos, sin (B,T,D/2) fp32 = cos/sin(pos * inv_freq) * attention_factor (Phi-3 longrope)."""
    _require_cuda(position_ids, inv_freq)
    position_ids = position_ids.contiguous().to(torch.int64)
    inv_freq = inv_freq.contiguous().to(torch.float32)
    B, T = position_ids.shape
    half = inv_freq.numel()
    cos = torch.empty(B, T, half, dtype=torch.float32, device=position_ids.device)
    sin = torch.empty_like(cos)
    check(lib.aki_mma_rope_table(_ptr(position_ids), _ptr(inv_freq), float(attention_factor), B, T, half, _ptr(cos),
                                 _ptr(sin), _stream()), "aki_mma_rope_table")
    return cos, sin


def rope_kv_write(qkv: torch.Tensor, cos: torch.Tensor, sin: torch.Tensor, k_cache: torch.Tensor,
                  v_cache: Optional[torch.Tensor], past_len: int, num_heads: int, q_rot: Optional[torch.Tensor] = None,
                  past_len_dev: Optional[torch.Tensor] = None):
    """qkv (B,T,3*H*D) bf16 -> K (post-RoPE) / V rows [past_len, past_len+T) of (B,H,t_cap,D) caches.
    past_len_dev (B,) int32 on the device replaces the host integer (CUDA-graph decode)."""
    _require_cuda(qkv, cos, sin, k_cache, v_cache, q_rot, past_len_dev)
    B, T, _ = qkv.shape
    if qkv.stride(2) != 1:
        qkv = qkv.contiguous()
    rope_sb = 0 if cos.shape[0] == 1 else cos.stride(0)
    if past_len_dev is not None:
        assert past_len_dev.dtype == torch.int32 and past_len_dev.numel() == B
        check(lib.aki_mma_rope_kv_write_dev(_ptr(qkv), qkv.stride(0), qkv.stride(1), _ptr(cos), _ptr(sin), rope_sb, B, T,
                                            num_heads, HEAD_DIM, _ptr(k_cache), _ptr(v_cache), k_cache.stride(0),
                                            k_cache.stride(1), _ptr(past_len_dev), k_cache.shape[2], _ptr(q_rot),
                                            _stream()),
              "aki_mma_rope_kv_write_dev")
        return
    check(lib.aki_mma_rope_kv_write(_ptr(qkv), qkv.stride(0), qkv.stride(1), _ptr(cos), _ptr(sin), rope_sb, B, T,
                                    num_heads, HEAD_DIM, _ptr(k_cache), _ptr(v_cache), k_cache.stride(0),
                                    k_cache.stride(1), int(past_len), k_cache.shape[2], _ptr(q_rot), _stream()),
          "aki_mma_rope_kv_write")


# --------------------------------------------------------------------------------------------------
# attention
# --------------------------------------------------------------------------------------------------
def _t4(t: torch.Tensor) -> Tensor4:
    """t is a (B,T,H,D) logical view with contiguous last dim."""
    assert t.dim() == 4 and t.stride(3) == 1 and t.dtype == torch.bfloat16, (t.shape, t.stride(), t.dtype)
    return Tensor4(t.data_ptr(), t.stride(0), t.stride(1), t.stride(2))


def _fill_params(p: AttnParams, q, k, v, o, lse, cos, sin, meta, scale, q_offset=0):
    B, T, H, D = q.shape
    assert k.shape[1] >= q_offset + T and v.shape[1] >= q_offset + T, (k.shape, q.shape, q_offset)
    p.B, p.H, p.T, p.D = B, H, T, D
    p.q_offset = int(q_offset)
    p.scale = float(scale)
    p.q, p.k, p.v, p.o = _t4(q), _t4(k), _t4(v), _t4(o)
    p.lse = _ptr(lse)
    if cos is not None:
        assert cos.dtype == torch.float32 and cos.is_contiguous() and sin.is_contiguous() and cos.shape[-1] == D // 2
        assert cos.shape[1] == T
        p.rope_cos, p.rope_sin = cos.data_ptr(), sin.data_ptr()
        p.rope_stride_b = 0 if cos.shape[0] == 1 else cos.stride(0)
    if meta is not None:
        seq_len, row_lo, row_hi, vbits, mbits, qkv_end, kvq_start, *rest = meta
        plan = rest[0] if rest else None
        if plan is not None:
            assert plan.dtype == torch.int32 and plan.is_contiguous() and plan.shape[0] == B and plan.shape[2] == 4
            p.fwd_plan, p.plan_pairs = plan.data_ptr(), plan.shape[1] - 1
        p.seq_len, p.row_lo, p.row_hi = _ptr(seq_len), _ptr(row_lo), _ptr(row_hi)
        p.kv_valid_bits, p.kv_mutual_bits = _ptr(vbits), _ptr(mbits)
        p.q_tile_kv_end, p.kv_tile_q_mask = _ptr(qkv_end), _ptr(kvq_start)
        p.meta_pitch = row_lo.shape[1] if row_lo is not None else 0
        p.bits_pitch = vbits.shape[1] if vbits is not None else 0
        if row_lo is not None:
            assert row_lo.shape[1] >= q_offset + T and row_lo.is_contiguous() and row_hi.is_contiguous()
        if qkv_end is not None:
            assert qkv_end.shape[1] == (T + TILE - 1) // TILE and qkv_end.is_contiguous()


def meta_tuple(segs: Optional[MMASegments]):
    if segs is None:
        return None
    return (segs.seq_len, segs.row_lo, segs.row_hi, segs.kv_valid_bits, segs.kv_mutual_bits, segs.q_tile_kv_end,
            segs.kv_tile_q_mask, segs.fwd_plan)


def attn_fwd_raw(q, k, v, cos, sin, meta, scale, need_lse=True, simt=False, q_offset=0):
    """q: (B,T,H,D), k,v: (B,q_offset+T,H,D) logical bf16 views; the queries are key rows [q_offset, q_offset+T) and
    the metadata is in key coordinates (a continuation chunk onto a KV cache; 0 = prefill).  cos/sin have T rows.
    Returns o (B,T,H,D) contiguous bf16, lse (B,H,T) fp32 or None."""
    _require_cuda(q, k, v)
    B, T, H, D = q.shape
    o = torch.empty(B, T, H, D, dtype=torch.bfloat16, device=q.device)
    lse = torch.empty(B, H, T, dtype=torch.float32, device=q.device) if need_lse else None
    p = AttnParams()
    _fill_params(p, q, k, v, o, lse, cos, sin, meta, scale, q_offset)
    fn = lib.aki_mma_attn_fwd_simt if simt else lib.aki_mma_attn_fwd
    check(fn(C.byref(p), _stream()), "aki_mma_attn_fwd" + ("_simt" if simt else ""))
    return o, lse


def attn_bwd_raw(d_o, q, k, v, o, lse, cos, sin, meta, scale, d_q, d_k, d_v, simt=False):
    """Writes gradients into the (B,T,H,D) views d_q, d_k, d_v (w.r.t. pre-RoPE q/k when cos/sin are given)."""
    _require_cuda(d_o, q, k, v, o, lse)
    B, T, H, D = q.shape
    p = AttnBwdParams()
    _fill_params(p.fwd, q, k, v, o, lse, cos, sin, meta, scale)
    if d_o.stride(3) != 1:
        d_o = d_o.contiguous()
    p.d_o, p.d_q, p.d_k, p.d_v = _t4(d_o), _t4(d_q), _t4(d_k), _t4(d_v)
    nbytes = lib.aki_mma_attn_bwd_workspace_bytes(B, H, T, D)
    ws = torch.empty(nbytes, dtype=torch.uint8, device=q.device)
    p.workspace, p.workspace_bytes = ws.data_ptr(), nbytes
    fn = lib.aki_mma_attn_bwd_simt if simt else lib.aki_mma_attn_bwd
    check(fn(C.byref(p), _stream()), "aki_mma_attn_bwd" + ("_simt" if simt else ""))


_OT = Optional[torch.Tensor]


@torch.library.custom_op("aki_mma::attn", mutates_args=())
def attn_op(q: torch.Tensor, k: torch.Tensor, v: torch.Tensor, scale: float, seq_len: _OT = None, row_lo: _OT = None,
            row_hi: _OT = None, vbits: _OT = None, mbits: _OT = None, q_tile_kv_end: _OT = None,
            kv_tile_q_mask: _OT = None, fwd_plan: _OT = None) -> Tuple[torch.Tensor, torch.Tensor]:
    """q,k,v (B,T,H,D) logical, already rotated.  Returns o (B,T,H,D), lse (B,H,T)."""
    meta = None if seq_len is None else (seq_len, row_lo, row_hi, vbits, mbits, q_tile_kv_end, kv_tile_q_mask, fwd_plan)
    return attn_fwd_raw(q, k, v, None, None, meta, scale)


@attn_op.register_fake
def _(q, k, v, scale, seq_len=None, row_lo=None, row_hi=None, vbits=None, mbits=None, q_tile_kv_end=None,
      kv_tile_q_mask=None, fwd_plan=None):
    B, T, H, D = q.shape
    return q.new_empty(B, T, H, D), q.new_empty(B, H, T, dtype=torch.float32)


def _attn_setup(ctx, inputs, output):
    q, k, v, scale, *meta = inputs
    o, lse = output
    ctx.save_for_backward(q, k, v, o, lse, *[m for m in meta if m is not None])
    ctx.scale = scale
    ctx.has_meta = meta[0] is not None


def _attn_backward(ctx, d_o, d_lse):
    q, k, v, o, lse, *meta = ctx.saved_tensors
    meta = tuple(meta) if ctx.has_meta else None
    B, T, H, D = q.shape
    dqkv = torch.empty(3, B, T, H, D, dtype=torch.bfloat16, device=q.device)
    attn_bwd_raw(d_o, q, k, v, o, lse, None, None, meta, ctx.scale, dqkv[0], dqkv[1], dqkv[2])
    return (dqkv[0], dqkv[1], dqkv[2], None) + (None,) * 8


attn_op.register_autograd(_attn_backward, setup_context=_attn_setup)


@torch.library.custom_op("aki_mma::attn_packed", mutates_args=())
def attn_packed_op(qkv: torch.Tensor, cos: torch.Tensor, sin: torch.Tensor, num_heads: int, scale: float,
                   seq_len: _OT = None, row_lo: _OT = None, row_hi: _OT = None, vbits: _OT = None, mbits: _OT = None,
                   q_tile_kv_end: _OT = None, kv_tile_q_mask: _OT = None, fwd_plan: _OT = None
                   ) -> Tuple[torch.Tensor, torch.Tensor, torch.Tensor]:
    """qkv (B,T,3*H*D) bf16 straight from qkv_proj; cos/sin (B|1,T,D/2) fp32.
    Returns o (B,T,H*D), lse (B,H,T), k_rot (B,H,T,D) (post-RoPE keys, kept for backward)."""
    B, T, _ = qkv.shape
    H, D = num_heads, HEAD_DIM
    k_rot = torch.empty(B, H, T, D, dtype=torch.bfloat16, device=qkv.device)
    rope_kv_write(qkv, cos, sin, k_rot, None, 0, H)
    q4 = qkv[..., : H * D].unflatten(-1, (H, D))
    v4 = qkv[..., 2 * H * D:].unflatten(-1, (H, D))
    meta = None if seq_len is None else (seq_len, row_lo, row_hi, vbits, mbits, q_tile_kv_end, kv_tile_q_mask, fwd_plan)
    o, lse = attn_fwd_raw(q4, k_rot.transpose(1, 2), v4, cos, sin, meta, scale)
    return o.view(B, T, H * D), lse, k_rot


@attn_packed_op.register_fake
def _(qkv, cos, sin, num_heads, scale, seq_len=None, row_lo=None, row_hi=None, vbits=None, mbits=None,
      q_tile_kv_end=None, kv_tile_q_mask=None, fwd_plan=None):
    B, T, _ = qkv.shape
    return (qkv.new_empty(B, T, num_heads * HEAD_DIM), qkv.new_empty(B, num_heads, T, dtype=torch.float32),
            qkv.new_empty(B, num_heads, T, HEAD_DIM))


def _packed_setup(ctx, inputs, output):
    qkv, cos, sin, num_heads, scale, *meta = inputs
    o, lse, k_rot = output
    ctx.save_for_backward(qkv, cos, sin, o, lse, k_rot, *[m for m in meta if m is not None])
    ctx.num_heads, ctx.scale, ctx.has_meta = num_heads, scale, meta[0] is not None


def _packed_backward(ctx, d_o, d_lse, d_krot):
    qkv, cos, sin, o, lse, k_rot, *meta = ctx.saved_tensors
    meta = tuple(meta) if ctx.has_meta else None
    B, T, _ = qkv.shape
    H, D = ctx.num_heads, HEAD_DIM
    d_qkv = torch.empty(B, T, 3 * H * D, dtype=torch.bfloat16, device=qkv.device)
    q4 = qkv[..., : H * D].unflatten(-1, (H, D))
    v4 = qkv[..., 2 * H * D:].unflatten(-1, (H, D))
    views = [d_qkv[..., i * H * D:(i + 1) * H * D].unflatten(-1, (H, D)) for i in range(3)]
    attn_bwd_raw(d_o.reshape(B, T, H, D), q4, k_rot.transpose(1, 2), v4, o.view(B, T, H, D), lse, cos, sin, meta,
                 ctx.scale, views[0], views[1], views[2])
    return (d_qkv, None, None, None, None) + (None,) * 8


attn_packed_op.register_autograd(_packed_backward, setup_context=_packed_setup)


# --------------------------------------------------------------------------------------------------
# decode
# --------------------------------------------------------------------------------------------------
@torch.library.custom_op("aki_mma::decode", mutates_args=())
def decode_op(q: torch.Tensor, k_cache: torch.Tensor, v_cache: torch.Tensor, kv_len: torch.Tensor, max_kv_len: int,
              scale: float, kv_start: _OT = None, kv_valid_bits: _OT = None) -> torch.Tensor:
    """q (B,H,D) bf16 post-RoPE; caches (B,H,t_cap,D) bf16; kv_len (B,) int32; kv_start (B,) int32 or None (first
    visible key: the leading pad rows of a left-padded prompt); kv_valid_bits (B, >= ceil(max_kv_len/32)) int32 or None
    (keys whose bit is 0 are skipped: interior pad rows of a batched follow-up turn).  Returns (B,H,D) bf16."""
    _require_cuda(q, k_cache, v_cache, kv_len, kv_start, kv_valid_bits)
    B, H, D = q.shape
    q = q.contiguous()
    out = torch.empty_like(q)
    nbytes = lib.aki_mma_decode_workspace_bytes(B, H, D, int(max_kv_len))
    ws = torch.empty(nbytes, dtype=torch.uint8, device=q.device)
    assert k_cache.stride(3) == 1 and k_cache.stride(2) == D and k_cache.stride() == v_cache.stride()
    if kv_valid_bits is None:
        check(lib.aki_mma_decode(_ptr(q), _ptr(k_cache), _ptr(v_cache), k_cache.stride(0), k_cache.stride(1),
                                 _ptr(kv_len), _ptr(kv_start), int(max_kv_len), B, H, D, float(scale), _ptr(out), _ptr(ws),
                                 nbytes, _stream()),
              "aki_mma_decode")
        return out
    assert kv_valid_bits.dtype == torch.int32 and kv_valid_bits.is_contiguous() and kv_valid_bits.shape[0] == B
    check(lib.aki_mma_decode_masked(_ptr(q), _ptr(k_cache), _ptr(v_cache), k_cache.stride(0), k_cache.stride(1),
                                    _ptr(kv_len), _ptr(kv_start), _ptr(kv_valid_bits), kv_valid_bits.shape[1],
                                    int(max_kv_len), B, H, D, float(scale), _ptr(out), _ptr(ws), nbytes, _stream()),
          "aki_mma_decode_masked")
    return out


@decode_op.register_fake
def _(q, k_cache, v_cache, kv_len, max_kv_len, scale, kv_start=None, kv_valid_bits=None):
    return torch.empty_like(q)


# --------------------------------------------------------------------------------------------------
# decode-sized linear layers around the attention op (SURVEY 8 f-1)
# --------------------------------------------------------------------------------------------------
def skinny_linear(x: torch.Tensor, weight: torch.Tensor, rms_weight: _OT = None, rms_eps: float = 1e-5,
                  residual: _OT = None, swiglu: bool = False, out: _OT = None) -> torch.Tensor:
    """y = epilogue(rmsnorm?(x) @ weight.T) for x (B<=64, K) bf16, weight (N or 2N, K) bf16 row-major:
    residual -> y = residual + (.), swiglu -> y = up * silu(gate) (gate_up_proj layout).  One weight-streaming kernel
    instead of Phi3RMSNorm + nn.Linear + activation / residual add (modeling_phi3.py:49-64, 295-335):
    aki_mma_skinny_linear for B <= 8, aki_mma_batch_linear (tcgen05) for 9 <= B <= 64."""
    _require_cuda(x, weight, rms_weight, residual)
    assert x.dim() == 2 and x.dtype == torch.bfloat16 and weight.dtype == torch.bfloat16 and x.stride(1) == 1
    assert weight.is_contiguous() and weight.shape[1] == x.shape[1] and not (swiglu and residual is not None)
    B, K = x.shape
    if B > 64:
        raise ValueError(f"skinny_linear takes at most 64 tokens, got {B}")
    N = weight.shape[0] // (2 if swiglu else 1)
    if out is None:
        out = torch.empty(B, N, dtype=torch.bfloat16, device=x.device)
    mode = 2 if swiglu else (1 if residual is not None else 0)
    fn = lib.aki_mma_skinny_linear if B <= 8 else lib.aki_mma_batch_linear
    check(fn(_ptr(x), x.stride(0), _ptr(weight), _ptr(rms_weight), float(rms_eps), _ptr(residual),
             residual.stride(0) if residual is not None else 0, _ptr(out), out.stride(0), B, N, K, mode, _stream()),
          fn.__name__)
    return out


def add_rmsnorm(x: torch.Tensor, weight: torch.Tensor, eps: float, residual: _OT = None, inplace_residual: bool = True):
    """(h, y) with h = residual + x (h = x when residual is None) and y = Phi3RMSNorm(h), for (..., K) bf16 rows at prefill
    size: one pass over HBM instead of the ATen kernels of the eager residual add + Phi3RMSNorm.forward
    (modeling_phi3.py:49-64, 317-335).  With inplace_residual the sum overwrites `residual`."""
    _require_cuda(x, weight, residual)
    K = x.shape[-1]
    x2 = x.reshape(-1, K)
    assert x2.dtype == torch.bfloat16 and x2.stride(1) == 1 and weight.dtype == torch.bfloat16 and weight.is_contiguous()
    y = torch.empty(x2.shape, dtype=torch.bfloat16, device=x.device)
    h = None
    r2 = None
    if residual is not None:
        r2 = residual.reshape(-1, K)
        assert r2.shape == x2.shape and r2.dtype == torch.bfloat16 and r2.stride(1) == 1
        h = r2 if (inplace_residual and r2.data_ptr() == residual.data_ptr()) else torch.empty_like(y)
    check(lib.aki_mma_add_rmsnorm(_ptr(x2), x2.stride(0), _ptr(r2), r2.stride(0) if r2 is not None else 0, _ptr(weight),
                                  float(eps), _ptr(h), h.stride(0) if h is not None else 0, _ptr(y), y.stride(0),
                                  x2.shape[0], K, _stream()), "aki_mma_add_rmsnorm")
    return (h.view(x.shape) if h is not None else x), y.view(x.shape)


def swiglu(gate_up: torch.Tensor) -> torch.Tensor:
    """up * silu(gate) for gate_up (..., 2N) bf16 = [gate | up] as Phi3MLP's gate_up_proj produces it (modeling_phi3.py:
    295-306): one pass instead of chunk + silu + mul on strided views."""
    _require_cuda(gate_up)
    N = gate_up.shape[-1] // 2
    g2 = gate_up.reshape(-1, 2 * N)
    assert g2.dtype == torch.bfloat16 and g2.stride(1) == 1
    y = torch.empty(g2.shape[0], N, dtype=torch.bfloat16, device=gate_up.device)
    check(lib.aki_mma_swiglu(_ptr(g2), g2.stride(0), _ptr(y), y.stride(0), g2.shape[0], N, _stream()), "aki_mma_swiglu")
    return y.view(*gate_up.shape[:-1], N)


class _ShiftedCrossEntropy(torch.autograd.Function):
    @staticmethod
    def forward(ctx, logits, labels, ignore_index):
        B, T, V = logits.shape
        row_loss = torch.empty(B, T, dtype=torch.float32, device=logits.device)
        row_lse = torch.empty_like(row_loss)
        check(lib.aki_mma_cross_entropy_fwd(_ptr(logits), logits.stride(0), logits.stride(1), _ptr(labels), labels.stride(0),
                                            B, T, V, int(ignore_index), _ptr(row_loss), _ptr(row_lse), _stream()),
              "aki_mma_cross_entropy_fwd")
        tgt = labels[:, 1:]
        n_valid = ((tgt != ignore_index) & (tgt >= 0) & (tgt < V)).sum().clamp_(min=1).to(torch.float32)
        ctx.save_for_backward(logits, labels, row_lse, n_valid)
        ctx.ignore_index = int(ignore_index)
        return row_loss.sum() / n_valid

    @staticmethod
    def backward(ctx, g):
        logits, labels, row_lse, n_valid = ctx.saved_tensors
        B, T, V = logits.shape
        scale = (g.to(torch.float32) / n_valid).reshape(1).contiguous()
        d = torch.empty(B, T, V, dtype=torch.bfloat16, device=logits.device)
        check(lib.aki_mma_cross_entropy_bwd(_ptr(logits), logits.stride(0), logits.stride(1), _ptr(labels), labels.stride(0),
                                            B, T, V, ctx.ignore_index, _ptr(row_lse), _ptr(scale), _ptr(d), d.stride(0),
                                            d.stride(1), _stream()), "aki_mma_cross_entropy_bwd")
        return d, None, None


def cross_entropy_shifted(logits: torch.Tensor, labels: torch.Tensor, ignore_index: int = -100) -> torch.Tensor:
    """Mean next-token cross-entropy of logits (B,T,V) bf16 against labels (B,T) int64 (row t pairs with labels[:, t+1];
    ignore_index rows skipped) = the loss Phi3ForCausalLM(labels=...) returns to AKI.forward (aki.py:125-130), without the
    fp32 copy of the logits; differentiable w.r.t. logits (gradient in bf16)."""
    _require_cuda(logits, labels)
    assert logits.dim() == 3 and logits.dtype == torch.bfloat16 and logits.stride(2) == 1
    assert labels.shape == logits.shape[:2] and labels.dtype == torch.int64 and labels.stride(1) == 1
    return _ShiftedCrossEntropy.apply(logits, labels, ignore_index)


# ---- training layout (amp_bf16: fp32 residual stream and norm weights, bf16 GEMM operands) ------------------------------
class _AddRmsNormAmp(torch.autograd.Function):
    """(h, a, w) -> (h + a, bf16(w * rmsnorm(h + a))); a may be None (then the first output is None too)."""

    @staticmethod
    def forward(ctx, h, a, w, eps):
        K = h.shape[-1]
        h2 = h.reshape(-1, K)
        M = h2.shape[0]
        a2 = a.reshape(-1, K) if a is not None else None
        h_new = torch.empty_like(h2) if a is not None else None
        x = torch.empty(M, K, dtype=torch.bfloat16, device=h.device)
        r = torch.empty(M, dtype=torch.float32, device=h.device)
        check(lib.aki_mma_add_rmsnorm_amp_fwd(_ptr(h2), _ptr(a2), _ptr(w), float(eps), _ptr(h_new), _ptr(x), _ptr(r), M, K,
                                              _stream()), "aki_mma_add_rmsnorm_amp_fwd")
        ctx.save_for_backward(h_new if a is not None else h2, r, w)
        ctx.has_a, ctx.shape = a is not None, h.shape
        if a is None:
            return None, x.view(h.shape)
        return h_new.view(h.shape), x.view(h.shape)

    @staticmethod
    def backward(ctx, d_h_new, d_x):
        h, r, w = ctx.saved_tensors
        M, K = h.shape
        if d_x is None:
            d_x = torch.zeros(M, K, dtype=torch.bfloat16, device=h.device)
        d_x = d_x.reshape(M, K).contiguous()
        dh_out = d_h_new.reshape(M, K).contiguous() if d_h_new is not None else None
        n_part = lib.aki_mma_rmsnorm_amp_bwd_partials(M)
        dw_p = torch.empty(n_part, K, dtype=torch.float32, device=h.device)
        dh = torch.empty(M, K, dtype=torch.float32, device=h.device)
        check(lib.aki_mma_rmsnorm_amp_bwd(_ptr(d_x), _ptr(dh_out), _ptr(h), _ptr(r), _ptr(w), _ptr(dh), _ptr(dw_p), M, K,
                                          _stream()), "aki_mma_rmsnorm_amp_bwd")
        dh = dh.view(ctx.shape)
        return dh, (dh.to(torch.bfloat16) if ctx.has_a else None), dw_p.sum(0), None


def add_rmsnorm_amp(h: torch.Tensor, a: _OT, weight: torch.Tensor, eps: float):
    """Training-layout residual add + Phi3RMSNorm + autocast cast: h (..., K) fp32 residual stream, a (..., K) bf16 branch
    output or None, weight (K) fp32.  Returns (h + a [None without a], x bf16) -- differentiable w.r.t. h, a and weight."""
    _require_cuda(h, a, weight)
    assert h.dtype == torch.float32 and weight.dtype == torch.float32 and h.is_contiguous() and weight.is_contiguous()
    assert a is None or (a.dtype == torch.bfloat16 and a.shape == h.shape and a.is_contiguous())
    return _AddRmsNormAmp.apply(h, a, weight, eps)


class _SwiGLUTrain(torch.autograd.Function):
    @staticmethod
    def forward(ctx, gate_up):
        ctx.save_for_backward(gate_up)
        return swiglu(gate_up)

    @staticmethod
    def backward(ctx, d_out):
        (gate_up,) = ctx.saved_tensors
        N = gate_up.shape[-1] // 2
        g2 = gate_up.reshape(-1, 2 * N)
        d2 = d_out.reshape(-1, N).contiguous()
        d_gu = torch.empty_like(g2)
        check(lib.aki_mma_swiglu_bwd(_ptr(d2), _ptr(g2), _ptr(d_gu), g2.shape[0], N, _stream()), "aki_mma_swiglu_bwd")
        return d_gu.view(gate_up.shape)


def swiglu_train(gate_up: torch.Tensor) -> torch.Tensor:
    """Differentiable ops.swiglu (bf16 in / out, eager autograd's rounding points in the backward)."""
    assert gate_up.dtype == torch.bfloat16 and gate_up.is_contiguous()
    return _SwiGLUTrain.apply(gate_up)
