"""Fused optimizer step for the SFT loop (include/aki_mma.h section (10)).

The reference's training step (train_utils.py:143-158) runs `clip_grad_norm_` and `torch.optim.AdamW.step`, and
autocast casts every fp32 Linear weight to bf16 in each forward.  `AkiAdamW` does the clipping and the update in two
passes over HBM (a deterministic squared-norm pass, then one update pass that applies the clip factor on load), and
`use_bf16_weights` lets the update write a bf16 copy of each Linear weight that the forward reads instead of
autocast's cast.  The copy is rounded to nearest even like autocast's cast, so the forward and every gradient stay
bit-identical to the plain autocast step; only the optimizer arithmetic is this library's (torch.optim.AdamW's fused
formula in the same fp32 operations, with the clip factor computed from the norm on the device).

Differences from `clip_grad_norm_` + `torch.optim.AdamW`: `.grad` is not rescaled in place (the clip factor is applied
while the update reads it), and the global norm is summed in a different order (the same bits on every run)."""
from __future__ import annotations

import types
from typing import Optional

import numpy as np
import torch
import torch.nn.functional as F
from torch import nn

from . import _lib

_ENTRY = np.dtype([("param", np.uint64), ("grad", np.uint64), ("exp_avg", np.uint64), ("exp_avg_sq", np.uint64),
                   ("param_bf16", np.uint64), ("numel", np.int64)])
assert _ENTRY.itemsize == _lib.C.sizeof(_lib.AdamWTensor)


def _entries(rows) -> np.ndarray:
    """rows: (param, grad, exp_avg, exp_avg_sq, param_bf16 or None) tensors -> host array of AkiAdamWTensor."""
    a = np.zeros(len(rows), dtype=_ENTRY)
    for i, (p, g, m, v, w16) in enumerate(rows):
        a[i] = (p.data_ptr() if p is not None else 0, g.data_ptr(), m.data_ptr() if m is not None else 0,
                v.data_ptr() if v is not None else 0, w16.data_ptr() if w16 is not None else 0, g.numel())
    return a


def grad_sq_norm(grads, out: Optional[torch.Tensor] = None, workspace: Optional[torch.Tensor] = None) -> torch.Tensor:
    """sum(g^2) over the fp32 CUDA tensors `grads` into a one-element fp32 device tensor (aki_mma_grad_sq_norm)."""
    grads = list(grads)
    if not grads:
        raise ValueError("grad_sq_norm needs at least one tensor")
    for g in grads:
        if not (g.is_cuda and g.dtype == torch.float32 and g.is_contiguous()):
            raise ValueError("grad_sq_norm takes contiguous fp32 CUDA tensors")
    ent = _entries([(None, g, None, None, None) for g in grads])
    need = _lib.lib.aki_mma_grad_sq_norm_workspace_bytes(ent.ctypes.data, len(grads))
    dev = grads[0].device
    if workspace is None or workspace.numel() < need:
        workspace = torch.empty(need, dtype=torch.uint8, device=dev)
    if out is None:
        out = torch.empty(1, dtype=torch.float32, device=dev)
    _lib.check(_lib.lib.aki_mma_grad_sq_norm(ent.ctypes.data, len(grads), workspace.data_ptr(), workspace.numel(),
                                             out.data_ptr(), torch.cuda.current_stream(dev).cuda_stream),
               "aki_mma_grad_sq_norm")
    return out


class AkiAdamW(torch.optim.Optimizer):
    """torch.optim.AdamW for fp32 CUDA parameters, with `clip_grad_norm_(params, max_grad_norm)` folded in.

    `step()` launches the squared-norm pass (when `max_grad_norm` is set) and one update pass per parameter group
    (and per step count within a group), and never synchronises with the device.  The norm covers every parameter with
    a gradient in every group, as clip_grad_norm_(model.parameters()) does; `last_grad_norm` is that norm as a device
    tensor (what clip_grad_norm_ returns).  `group["lr"]` is read on every step, so LR schedulers work.  State keys and
    layout are torch.optim.AdamW's (`step`, `exp_avg`, `exp_avg_sq`; `step` a CPU fp32 tensor as in its non-fused
    modes), so state dicts load into either optimizer both ways.  Parameters registered with `use_bf16_weights` get
    their bf16 copy written by the same pass."""

    def __init__(self, params, lr: float = 1e-3, betas=(0.9, 0.999), eps: float = 1e-8, weight_decay: float = 1e-2,
                 max_grad_norm: Optional[float] = None, *, amsgrad: bool = False, maximize: bool = False):
        if amsgrad:
            raise ValueError("AkiAdamW does not implement amsgrad")
        if maximize:
            raise ValueError("AkiAdamW does not implement maximize")
        if not 0.0 <= lr:
            raise ValueError(f"Invalid learning rate: {lr}")
        if not 0.0 <= eps:
            raise ValueError(f"Invalid epsilon value: {eps}")
        if not (0.0 <= betas[0] < 1.0 and 0.0 <= betas[1] < 1.0):
            raise ValueError(f"Invalid betas: {betas}")
        if not 0.0 <= weight_decay:
            raise ValueError(f"Invalid weight_decay value: {weight_decay}")
        if max_grad_norm is not None and not max_grad_norm > 0.0:
            raise ValueError(f"Invalid max_grad_norm: {max_grad_norm}")
        # fused=True: a checkpoint of this optimizer loads into torch.optim.AdamW as its fused implementation, whose
        # arithmetic this update reproduces (without the key torch would fall back to its foreach path)
        super().__init__(params, dict(lr=lr, betas=betas, eps=eps, weight_decay=weight_decay, amsgrad=False,
                                      maximize=False, fused=True))
        self.max_grad_norm = max_grad_norm
        self.last_grad_norm: Optional[torch.Tensor] = None
        self._bf16: dict = {}          # fp32 parameter -> its bf16 copy (use_bf16_weights)
        self._workspace: Optional[torch.Tensor] = None
        self._sq: Optional[torch.Tensor] = None

    def add_param_group(self, param_group):
        params = param_group["params"]
        for p in ([params] if isinstance(params, torch.Tensor) else list(params)):
            if not isinstance(p, torch.Tensor):
                continue                                   # torch's own check reports it
            if not p.is_leaf:
                raise ValueError("can't optimize a non-leaf Tensor")
            if p.layout != torch.strided:
                raise ValueError("AkiAdamW takes dense parameters (got a sparse one)")
            if p.dtype != torch.float32:
                raise ValueError(f"AkiAdamW takes fp32 parameters (got {p.dtype})")
            if not p.is_cuda:
                raise ValueError("AkiAdamW takes CUDA parameters (got a CPU one)")
            if not p.is_contiguous():
                raise ValueError("AkiAdamW takes contiguous parameters")
        super().add_param_group(param_group)

    def load_state_dict(self, state_dict):
        super().load_state_dict(state_dict)
        # torch's fused / capturable AdamW keeps `step` on the device; the update takes it as a host integer
        for st in self.state.values():
            if "step" in st and torch.is_tensor(st["step"]) and st["step"].device.type != "cpu":
                st["step"] = st["step"].to("cpu", torch.float32)

    @torch.no_grad()
    def step(self, closure=None):
        loss = None
        if closure is not None:
            with torch.enable_grad():
                loss = closure()
        work = []
        for group in self.param_groups:
            if group.get("amsgrad") or group.get("maximize"):
                raise ValueError("AkiAdamW does not implement amsgrad or maximize")
            for p in group["params"]:
                g = p.grad
                if g is None:
                    continue
                if g.is_sparse or g.dtype != torch.float32 or not g.is_contiguous() or g.shape != p.shape:
                    raise RuntimeError("AkiAdamW needs dense contiguous fp32 gradients of the parameter's shape")
                st = self.state[p]
                if len(st) == 0:
                    st["step"] = torch.tensor(0.0, dtype=torch.float32)
                    st["exp_avg"] = torch.zeros_like(p, memory_format=torch.preserve_format)
                    st["exp_avg_sq"] = torch.zeros_like(p, memory_format=torch.preserve_format)
                work.append((group, p, g, st))
        if not work:
            return loss
        dev = work[0][1].device
        stream = torch.cuda.current_stream(dev).cuda_stream
        sq_ptr = None
        if self.max_grad_norm is not None:
            ent = _entries([(None, g, None, None, None) for _, _, g, _ in work])
            need = _lib.lib.aki_mma_grad_sq_norm_workspace_bytes(ent.ctypes.data, len(work))
            if self._workspace is None or self._workspace.numel() < need or self._workspace.device != dev:
                self._workspace = torch.empty(need, dtype=torch.uint8, device=dev)
                self._sq = torch.empty(1, dtype=torch.float32, device=dev)
            _lib.check(_lib.lib.aki_mma_grad_sq_norm(ent.ctypes.data, len(work), self._workspace.data_ptr(),
                                                     self._workspace.numel(), self._sq.data_ptr(), stream),
                       "aki_mma_grad_sq_norm")
            sq_ptr = self._sq.data_ptr()
            self.last_grad_norm = self._sq[0].sqrt()
        buckets: dict = {}
        for group, p, g, st in work:
            st["step"] += 1
            buckets.setdefault((id(group), int(st["step"].item())), (group, []))[1].append(
                (p, g, st["exp_avg"], st["exp_avg_sq"], self._bf16.get(p)))
        for (_, step), (group, rows) in buckets.items():
            ent = _entries(rows)
            b1, b2 = group["betas"]
            _lib.check(_lib.lib.aki_mma_adamw_step(ent.ctypes.data, len(rows), sq_ptr,
                                                   float(self.max_grad_norm or 0.0), float(group["lr"]), float(b1),
                                                   float(b2), float(group["eps"]), float(group["weight_decay"]), step,
                                                   stream),
                       "aki_mma_adamw_step")
        return loss


# ---- the bf16 weight copy read by the forward ---------------------------------------------------------------------
class _Bf16Weight(torch.autograd.Function):
    """Hands the Linear the bf16 copy in place of autocast's cast of the fp32 weight; the backward widens the bf16
    weight gradient to fp32 exactly as the cast's backward (ToCopyBackward) does.  The Linear itself is the same ATen
    op on the same operands as under plain autocast, so y, dx and dW keep their bits."""

    @staticmethod
    def forward(ctx, w, w16):
        return w16.detach()

    @staticmethod
    def backward(ctx, g16):
        return g16.to(torch.float32), None


def _bf16_linear_forward(self, x):
    w = self.weight
    if not (torch.is_autocast_enabled("cuda") and torch.get_autocast_dtype("cuda") == torch.bfloat16
            and w.dtype == torch.float32 and x.is_cuda):
        return self._aki_bf16_orig_forward(x)
    w16 = self._aki_weight_bf16
    if self._aki_bf16_version != w._version:
        # the master changed outside the optimizer's update (load_state_dict, copy_, nn.init): refresh the copy first
        with torch.no_grad():
            w16.copy_(w)
        self._aki_bf16_version = w._version
    return F.linear(x, _Bf16Weight.apply(w, w16))


def use_bf16_weights(model: nn.Module, optimizer: AkiAdamW) -> int:
    """For every bias-free nn.Linear under `model` whose fp32 CUDA weight `optimizer` updates: allocate a bf16 copy of
    the weight (2 bytes per element), register it with the optimizer, which rewrites it after each update, and rebind
    the module's forward (per instance, idempotent) so that under torch.autocast("cuda", torch.bfloat16) the Linear
    reads the copy instead of casting the weight.  Outside autocast the original forward runs.  The copy is a plain
    attribute, not a buffer: state-dict keys are unchanged, and DDP does not broadcast it.  A copy whose master was
    changed by anything but the optimizer (its `_version` moved) is rebuilt before the next forward; a write that
    bypasses the version counter (a raw-pointer kernel) is not seen.  Returns the number of modules rebound;
    `unuse_bf16_weights` restores them."""
    if not isinstance(optimizer, AkiAdamW):
        raise TypeError("use_bf16_weights needs the AkiAdamW that updates the weights")
    managed = {id(p) for g in optimizer.param_groups for p in g["params"]}
    n = 0
    for m in model.modules():
        if not isinstance(m, nn.Linear) or m.bias is not None or hasattr(m, "_aki_bf16_orig_forward"):
            continue
        w = m.weight
        if id(w) not in managed or w.dtype != torch.float32 or not w.is_cuda:
            continue
        m._aki_weight_bf16 = torch.empty_like(w, dtype=torch.bfloat16, memory_format=torch.contiguous_format)
        m._aki_bf16_version = -1
        m._aki_bf16_optimizer = optimizer
        optimizer._bf16[w] = m._aki_weight_bf16
        m._aki_bf16_orig_forward = m.forward
        m.forward = types.MethodType(_bf16_linear_forward, m)
        n += 1
    return n


def unuse_bf16_weights(model: nn.Module) -> int:
    """Restores the forwards `use_bf16_weights` rebound and frees the copies (the optimizer stops writing them)."""
    n = 0
    for m in model.modules():
        if hasattr(m, "_aki_bf16_orig_forward"):
            m.forward = m._aki_bf16_orig_forward
            m._aki_bf16_optimizer._bf16.pop(m.weight, None)
            for a in ("_aki_bf16_orig_forward", "_aki_weight_bf16", "_aki_bf16_version", "_aki_bf16_optimizer"):
                delattr(m, a)
            n += 1
    return n
