"""Minimal Phi-3.5-mini runner around the drop-in attention: prefill that writes the KV cache in place and a greedy
decode loop ("next" rows f-1 / f-4 of SURVEY section 8 in their simplest form).  The decoder layers are the installed
transformers' Phi3DecoderLayer objects with `self_attn` swapped for AkiMMAAttention (same parameters / state-dict
keys); everything except the attention stays cuBLAS / ATen.  Calling the layers directly avoids HF's (B,1,T,T) mask
construction -- the MMA description travels as `mma_segments`."""
from __future__ import annotations

from typing import Optional

import torch
from torch import nn

from . import ops
from .attention import replace_phi3_attention
from .cache import AkiKVCache
from .rope import LongRope


def phi35_mini_config(num_layers: int = 32, short_factor=None, long_factor=None, vocab_size: int = 32064):
    """microsoft/Phi-3.5-mini-instruct geometry (hidden 3072, 32 heads x 96, MLP 8192, longrope 4096 -> 131072).
    The hub config.json is not available offline: the 48 longrope factors default to 1.0 unless given."""
    from transformers import Phi3Config
    half = 48
    sf = [1.0] * half if short_factor is None else [float(x) for x in short_factor]
    lf = [1.0] * half if long_factor is None else [float(x) for x in long_factor]
    return Phi3Config(hidden_size=3072, num_attention_heads=32, num_key_value_heads=32, intermediate_size=8192,
                      vocab_size=vocab_size, num_hidden_layers=num_layers, max_position_embeddings=131072,
                      original_max_position_embeddings=4096, rms_norm_eps=1e-5, attention_dropout=0.0, pad_token_id=0,
                      rope_parameters={"rope_type": "longrope", "rope_theta": 10000.0, "short_factor": sf,
                                       "long_factor": lf, "original_max_position_embeddings": 4096},
                      attn_implementation="eager")


class AkiPhi3Runner(nn.Module):
    def __init__(self, config, device="cuda", dtype=torch.bfloat16, seed: int = 0):
        super().__init__()
        from transformers import Phi3ForCausalLM
        torch.manual_seed(seed)
        with torch.device(device):
            self.lm = Phi3ForCausalLM(config).to(dtype)
        replace_phi3_attention(self.lm)
        self.config = config
        rp = config.rope_parameters
        self.rope = LongRope(96, rp["rope_theta"], rp["short_factor"], rp["long_factor"], config.max_position_embeddings,
                             rp["original_max_position_embeddings"], device=device)

    def new_cache(self, batch: int, t_cap: int) -> AkiKVCache:
        p = next(self.lm.parameters())
        return AkiKVCache(self.config.num_hidden_layers, batch, 32, 96, t_cap, p.device, p.dtype)

    def _run_layers(self, h, cos, sin, segs, cache):
        for layer in self.lm.model.layers:
            h = layer(h, attention_mask=None, position_ids=None, past_key_values=cache, use_cache=cache is not None,
                      position_embeddings=None, mma_segments=segs, mma_rope=(cos, sin))
            if isinstance(h, tuple):
                h = h[0]
        return self.lm.model.norm(h)

    def _run_layers_fused(self, h, cos, sin, segs, cache):
        """Inference-only pass through the decoder layers with the element-wise work fused ("next" row f-1 of SURVEY 8):
        residual add + RMSNorm in one kernel, SiLU gate in one kernel (ops.add_rmsnorm / ops.swiglu) instead of the ~12
        ATen kernels per layer of Phi3DecoderLayer.forward (modeling_phi3.py:295-335), which took 42 % of the prefill's
        kernel time (tools/prefill_profile.py).  The GEMMs stay cuBLAS; attention is the drop-in module.  Same rounding
        points as the eager layers.  Returns the final-norm output."""
        F = torch.nn.functional
        eps = self.config.rms_norm_eps
        layers = self.lm.model.layers
        res, x = ops.add_rmsnorm(h, layers[0].input_layernorm.weight, eps)        # res is the caller's tensor: not ours yet
        ours = False
        for li, layer in enumerate(layers):
            a = layer.self_attn(x, position_embeddings=None, attention_mask=None, past_key_values=cache,
                                mma_segments=segs, mma_rope=(cos, sin))[0]
            res, x = ops.add_rmsnorm(a, layer.post_attention_layernorm.weight, eps, residual=res, inplace_residual=ours)
            ours = True
            d = F.linear(ops.swiglu(F.linear(x, layer.mlp.gate_up_proj.weight)), layer.mlp.down_proj.weight)
            nxt = layers[li + 1].input_layernorm if li + 1 < len(layers) else self.lm.model.norm
            res, x = ops.add_rmsnorm(d, nxt.weight, eps, residual=res)
        return x

    @torch.no_grad()
    def prefill(self, inputs_embeds: torch.Tensor, segs: Optional[ops.MMASegments], cache: Optional[AkiKVCache],
                last_only: bool = True, fused: bool = True):
        """inputs_embeds (B,T,3072); positions arange(T) as AKI.generate passes them (aki.py:184-191).  fused=False runs
        HF's Phi3DecoderLayer objects (the parity reference of the fused pass).  Onto a non-empty cache (follow-up turn,
        chunked prefill) the chunk takes positions past + arange(T), the same for every sequence, with the longrope
        factor set of the running maximum past + T - 1 (the rule of the decode steps); `segs` then describes the chunk
        alone (chunk-relative, e.g. build_segments on the chunk's own tokens)."""
        B, T, _ = inputs_embeds.shape
        past = cache.get_seq_length() if cache is not None else 0
        cos, sin = self.rope.tables(past + torch.arange(T, device=inputs_embeds.device)[None], max_position=past + T - 1)
        fused = fused and inputs_embeds.dtype == torch.bfloat16 and inputs_embeds.shape[-1] <= 4096
        h = (self._run_layers_fused if fused else self._run_layers)(inputs_embeds.contiguous() if fused else inputs_embeds,
                                                                      cos, sin, segs, cache)
        return self.lm.lm_head(h[:, -1:] if last_only else h)

    @torch.no_grad()
    def decode_step(self, token_ids: torch.Tensor, cache: AkiKVCache):
        """One greedy step for every sequence: position id = past length (aki_generation.py:72-84)."""
        past = cache.get_seq_length()
        h = self.lm.model.embed_tokens(token_ids)            # (B,1,3072)
        pos = torch.full((1, 1), past, device=h.device, dtype=torch.long)
        cos, sin = self.rope.tables(pos, max_position=past)
        h = self._run_layers(h, cos, sin, None, cache)
        return self.lm.lm_head(h)

    # ---- fused decode layers ("next" row f-1 of SURVEY 8): 7 launches per layer instead of ~15 --------------------------
    @torch.no_grad()
    def _fused_layers(self, h: torch.Tensor, cos, sin, cache: AkiKVCache, past: Optional[int]):
        """One decode step through all decoder layers for h (B<=8, 3072): RMSNorm->qkv_proj, RoPE + KV write, decode
        attention, o_proj + residual, RMSNorm->gate_up_proj->SiLU gate, down_proj + residual -- each GEMM one
        weight-streaming kernel (ops.skinny_linear) with the norm / activation / residual fused in.  past=None: the write
        row and key count come from device memory (CUDA-graph replay).  Returns the last-layer hidden state (B,3072)."""
        B = h.shape[0]
        H, D, eps = 32, 96, self.config.rms_norm_eps
        for li, layer in enumerate(self.lm.model.layers):
            attn = layer.self_attn
            qkv = ops.skinny_linear(h, attn.qkv_proj.weight, layer.input_layernorm.weight, eps)
            q_rot = torch.empty(B, H, 1, D, dtype=torch.bfloat16, device=h.device)
            if past is None:
                ops.rope_kv_write(qkv.view(B, 1, -1), cos, sin, cache.k[li], cache.v[li], 0, H, q_rot=q_rot,
                                  past_len_dev=cache.past_dev)
                max_kv = cache.t_cap
            else:
                ops.rope_kv_write(qkv.view(B, 1, -1), cos, sin, cache.k[li], cache.v[li], past, H, q_rot=q_rot)
                max_kv = past + 1
            o = ops.decode_op(q_rot.view(B, H, D), cache.k[li], cache.v[li], cache.kv_len, max_kv, attn.scaling, cache.kv_start,
                              cache.meta.kv_valid_bits)
            h = ops.skinny_linear(o.view(B, H * D), attn.o_proj.weight, residual=h)
            act = ops.skinny_linear(h, layer.mlp.gate_up_proj.weight, layer.post_attention_layernorm.weight, eps, swiglu=True)
            h = ops.skinny_linear(act, layer.mlp.down_proj.weight, residual=h)
        return h

    @torch.no_grad()
    def decode_step_fused(self, token_ids: torch.Tensor, cache: AkiKVCache):
        """decode_step through the fused layers (host-driven cache bookkeeping); returns logits (B,1,vocab)."""
        past = cache.get_seq_length()
        cache._check(past + 1)
        B = token_ids.shape[0]
        if B > 8:
            return self.decode_step(token_ids, cache)
        h = self.lm.model.embed_tokens(token_ids).view(B, -1)
        pos = torch.full((1, 1), past, device=h.device, dtype=torch.long)
        cos, sin = self.rope.tables(pos, max_position=past)
        cache.kv_len.fill_(past + 1)
        h = self._fused_layers(h, cos, sin, cache, past)
        cache._len = [n + 1 for n in cache._len]
        logits = ops.skinny_linear(h, self.lm.lm_head.weight, self.lm.model.norm.weight, self.config.rms_norm_eps)
        return logits.view(B, 1, -1)

    # ---- CUDA-graph decode ("next" row f-4 of SURVEY 8): the whole 32-layer step is one graph launch -----------------
    @torch.no_grad()
    def _graph_body(self, cache: AkiKVCache):
        st = self._g
        cache.kv_len.copy_(cache.past_dev + 1)                       # keys visible to this step (incl. the new one)
        st["pos"].copy_(cache.past_dev[:1].to(torch.int64).view(1, 1))   # position id = past length (aki_generation.py:72-84)
        h = self.lm.model.embed_tokens(st["tok"])
        inv = self.rope.inv_freq_long if st["capturing_long"] else self.rope.inv_freq_short
        cos, sin = ops.rope_table(st["pos"], inv, self.rope.attention_factor)
        if st["fused"]:
            hf = self._fused_layers(h.view(h.shape[0], -1), cos, sin, cache, None)
            logits = ops.skinny_linear(hf, self.lm.lm_head.weight, self.lm.model.norm.weight, self.config.rms_norm_eps)
            st["next"].copy_(logits.argmax(-1, keepdim=True))
        else:
            h = self._run_layers(h, cos, sin, None, cache)
            st["next"].copy_(self.lm.lm_head(h)[:, -1].argmax(-1, keepdim=True))
        cache.past_dev.add_(1)

    @torch.no_grad()
    def decode_step_graphed(self, token_ids: torch.Tensor, cache: AkiKVCache, fused: bool = True) -> torch.Tensor:
        """Greedy decode step replayed from a CUDA graph: returns the next token ids (B,1).  fused (default, B <= 8): the
        layers run through the weight-streaming kernels of _fused_layers.  A graph is captured on first
        use for this cache and for each longrope factor set; the write row, the key count and the position id live in
        device memory (cache.past_dev), so replays need no host-side arguments.  The factor set follows the running
        maximum position exactly as the eager step and the reference do (modeling_rope_utils.py:47-80): short factors
        while past + 1 <= original_max, long factors afterwards -- the step switches graphs when the boundary is crossed."""
        past = cache.get_seq_length()
        cache._check(past + 1)                                       # BEFORE anything is enqueued: the row must exist
        fused = bool(fused) and token_ids.shape[0] <= 8
        g = getattr(self, "_g", None)
        if g is None or g["cache"] is not cache or g["fused"] != fused:
            B = token_ids.shape[0]
            dev = token_ids.device
            self._g = g = {"cache": cache, "tok": token_ids.clone(), "next": torch.zeros(B, 1, dtype=torch.int64, device=dev),
                           "pos": torch.zeros(1, 1, dtype=torch.int64, device=dev), "capturing_long": False, "graphs": {},
                           "fused": fused}
        use_long = (past + 1) > self.rope.original_max
        if use_long not in g["graphs"]:
            # warm-up (2 steps) + capture (1 step) write rows past .. past+2: they must exist, and they are restored below
            if past + 3 > cache.t_cap:
                raise ValueError(f"capturing the decode graph needs 3 free cache rows (have {cache.t_cap - past}): "
                                 f"allocate the cache with t_cap >= prompt + new tokens + 2")
            g["capturing_long"] = use_long
            cache.device_driven = True
            cache.past_dev.fill_(past)
            keep = (cache.past_dev.clone(), [k[:, :, past:past + 3].clone() for k in cache.k],
                    [v[:, :, past:past + 3].clone() for v in cache.v])
            dev = token_ids.device
            side = torch.cuda.Stream(device=dev)
            side.wait_stream(torch.cuda.current_stream())
            with torch.cuda.stream(side):
                for _ in range(2):                                   # warm-up outside capture (lazy inits, autotune)
                    self._graph_body(cache)
            torch.cuda.current_stream().wait_stream(side)
            graph = torch.cuda.CUDAGraph()
            with torch.cuda.graph(graph):
                self._graph_body(cache)
            g["graphs"][use_long] = graph
            # undo the side effects of warm-up + capture: three rows written past the end, counters advanced
            cache.past_dev.copy_(keep[0])
            for k, v, k0, v0 in zip(cache.k, cache.v, keep[1], keep[2]):
                k[:, :, past:past + 3].copy_(k0); v[:, :, past:past + 3].copy_(v0)
        cache.device_driven = True
        if g.get("expected_past") != past:                           # eager steps (or a reset) happened in between
            cache.past_dev.fill_(past)
        g["tok"].copy_(token_ids)
        g["graphs"][use_long].replay()
        g["expected_past"] = past + 1
        cache.advance_host(1)
        cache.device_driven = False
        return g["next"].clone()

    @torch.no_grad()
    def generate(self, inputs_embeds, segs, max_new_tokens: int, t_cap: Optional[int] = None,
                 cache: Optional[AkiKVCache] = None):
        """Greedy generation; with `cache` the prompt is a follow-up turn appended to that cache's contents."""
        B, T, _ = inputs_embeds.shape
        if cache is None:
            cache = self.new_cache(B, t_cap or (T + max_new_tokens))
        logits = self.prefill(inputs_embeds, segs, cache)
        out = []
        tok = logits[:, -1].argmax(-1, keepdim=True)
        for _ in range(max_new_tokens):
            out.append(tok)
            logits = self.decode_step(tok, cache)
            tok = logits[:, -1].argmax(-1, keepdim=True)
        return torch.cat(out, dim=1), cache


class AkiPhi3SFT(nn.Module):
    """Training-side counterpart of the LM half of AKI.forward (codes/open_flamingo/src/aki.py:125-130) with the
    reference's `amp_bf16` precision (configs/sft.yaml:55): fp32 master parameters, bf16 autocast compute.  Returns
    the shifted next-token cross-entropy HF computes for `labels` (-100 = ignored).  Wrap it in torch DDP for the
    data-parallel SFT step (train/instruction_finetune.py:128-130); the attention op itself has no collective."""

    def __init__(self, config, device="cuda", seed: int = 0):
        super().__init__()
        from transformers import Phi3ForCausalLM
        torch.manual_seed(seed)
        with torch.device(device):
            self.lm = Phi3ForCausalLM(config)           # fp32 master weights
        replace_phi3_attention(self.lm)
        self.config = config
        self.fused_ce = True
        self.fused_layers = True          # False: HF's Phi3DecoderLayer objects (the parity reference of the fused pass)
        rp = config.rope_parameters
        self.rope = LongRope(96, rp["rope_theta"], rp["short_factor"], rp["long_factor"], config.max_position_embeddings,
                             rp["original_max_position_embeddings"], device=device)

    def forward(self, inputs_embeds: torch.Tensor, segs: Optional[ops.MMASegments], labels: torch.Tensor):
        B, T, _ = inputs_embeds.shape
        cos, sin = self.rope.tables(torch.arange(T, device=inputs_embeds.device)[None], max_position=T - 1)
        layers = self.lm.model.layers
        fused = (self.fused_layers and inputs_embeds.dtype == torch.float32 and inputs_embeds.shape[-1] % 256 == 0
                 and inputs_embeds.shape[-1] <= 3072 and layers[0].input_layernorm.weight.dtype == torch.float32)
        with torch.autocast("cuda", dtype=torch.bfloat16):
            if fused:
                # SURVEY 8 f-1 for the SFT step: residual add + RMSNorm + operand cast, and the SiLU gate, as fused forward /
                # backward kernels in the amp layout (fp32 residual stream, bf16 GEMM operands) around the same Linears
                eps = self.config.rms_norm_eps
                h = inputs_embeds.contiguous()
                _, x = ops.add_rmsnorm_amp(h, None, layers[0].input_layernorm.weight, eps)
                for li, layer in enumerate(layers):
                    a = layer.self_attn(x, position_embeddings=None, attention_mask=None, past_key_values=None,
                                        mma_segments=segs, mma_rope=(cos, sin))[0]
                    h, x = ops.add_rmsnorm_amp(h, a.contiguous(), layer.post_attention_layernorm.weight, eps)
                    d = layer.mlp.down_proj(ops.swiglu_train(layer.mlp.gate_up_proj(x)))
                    nxt = layers[li + 1].input_layernorm if li + 1 < len(layers) else self.lm.model.norm
                    h, x = ops.add_rmsnorm_amp(h, d.contiguous(), nxt.weight, eps)
                logits = self.lm.lm_head(x)
            else:
                h = inputs_embeds
                for layer in layers:
                    h = layer(h, attention_mask=None, position_ids=None, past_key_values=None, use_cache=False,
                              position_embeddings=None, mma_segments=segs, mma_rope=(cos, sin))
                    if isinstance(h, tuple):
                        h = h[0]
                logits = self.lm.lm_head(self.lm.model.norm(h))
        if self.fused_ce and logits.dtype == torch.bfloat16 and logits.shape[-1] % 8 == 0:
            # SURVEY 8 f-2: one kernel forward, one backward, no fp32 copy of the (B,T,32064) logits
            return ops.cross_entropy_shifted(logits, labels.contiguous())
        logits = logits[:, :-1].float()
        return nn.functional.cross_entropy(logits.reshape(-1, logits.shape[-1]), labels[:, 1:].reshape(-1),
                                           ignore_index=-100)
