"""Kernel-only time of attn_bwd_sm100_kernel (T=8192, B=2, H=32; pure causal and 4 image spans) through the timing hook.
Used with AKI_MMA_LIB=<variant> for same-box A/B and knockout runs (tools/build_variant.sh); no result check here."""
import os, sys, statistics
import numpy as np, torch
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import bench
import aki_b200
from aki_b200 import ops
from aki_b200._lib import lib
dev = torch.device("cuda", 0)
H, D, T, B = 32, 96, 8192, 2
rope = aki_b200.LongRope(device=dev)
out = []
for n_img in (0, 4):
    lang, am = bench.make_prompt(B, T, n_img) if n_img else (np.random.default_rng(0).integers(3, 31000, size=(B, T)).astype(np.int64), np.ones((B, T), dtype=np.int64))
    segs = ops.build_segments(torch.from_numpy(lang).to(dev), torch.from_numpy(am).to(dev), 128, bench.MEDIA_ID, t_cap=T, exact_shape=False)
    meta = ops.meta_tuple(segs)
    g = torch.Generator(device=dev).manual_seed(0)
    qkv = torch.randn(B, T, 3 * H * D, generator=g, device=dev).to(torch.bfloat16)
    d_o = torch.randn(B, T, H, D, generator=g, device=dev).to(torch.bfloat16)
    cos, sin = rope.tables(torch.arange(T, device=dev)[None], max_position=T - 1)
    q4 = qkv[..., :H * D].unflatten(-1, (H, D)); v4 = qkv[..., 2 * H * D:].unflatten(-1, (H, D))
    k_rot = torch.empty(B, H, T, D, dtype=torch.bfloat16, device=dev)
    dq = torch.empty_like(q4.contiguous()); dk = torch.empty_like(dq); dv = torch.empty_like(dq)
    ops.rope_kv_write(qkv, cos, sin, k_rot, None, 0, H)
    o, lse = ops.attn_fwd_raw(q4, k_rot.transpose(1, 2), v4, cos, sin, meta, D ** -0.5)
    tb = []
    for it in range(7):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(); e1.record()      # torch creates the CUDA event lazily
        lib.aki_mma_set_timing_events(e0.cuda_event, e1.cuda_event)
        ops.attn_bwd_raw(d_o, q4, k_rot.transpose(1, 2), v4, o, lse, cos, sin, meta, D ** -0.5, dq, dk, dv)
        torch.cuda.synchronize()
        if it >= 2:
            tb.append(e0.elapsed_time(e1))
    out.append(statistics.median(tb))
print(f"{os.path.basename(os.environ.get('AKI_MMA_LIB', 'default')):28s} causal {out[0]:.3f} ms   4-images {out[1]:.3f} ms")
