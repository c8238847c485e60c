"""Kernel time of a continuation chunk (follow-up turn / chunked prefill): T = 512 and 2048 new query rows onto a
6K-token cache, B = 2, H = 32, 4 image spans of 128 tokens in the prefix, causal + the chunk's own validity.  CUDA
events around the tcgen05 forward kernel (timing hook); TFLOP/s over the chunk's exact number of visible (query, key)
pairs (4 * D flops each: QK^T and PV).  Prints the card name and power limit next to the numbers.
usage: python tools/continuation_time.py"""
import os, statistics, subprocess, sys
import torch
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import aki_b200
from aki_b200 import ops
from aki_b200._lib import lib
from aki_b200.cache import KeyMeta

dev = torch.device("cuda", 0)
H, D, B, PAST, N_IMG, N = 32, 96, 2, 6144, 4, 128
card = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                      capture_output=True, text=True).stdout.strip().splitlines()[0]
print(f"card: {card}")
for T in (512, 2048):
    Tk = PAST + T
    km = KeyMeta(B, Tk, dev)
    # prefix: 4 image spans whose rows see the later keys up to the prompt's <|assistant|> (row 5000)
    starts = [200 + k * 1000 for k in range(N_IMG)]
    for s in starts:
        km.row_lo[:, s:s + N] = s + N
        km.row_hi[:, s:s + N] = 5000
    km.kv_mutual_bits.fill_(-1)
    km.write_chunk(PAST, T, None, None)
    meta = km.attn_meta(PAST, T)
    # exact visible pairs of the chunk's rows (causal over all keys: every key is valid here)
    nnz = B * sum(PAST + r + 1 for r in range(T))
    g = torch.Generator(device=dev).manual_seed(0)
    q = torch.randn(B, T, H, D, generator=g, device=dev).to(torch.bfloat16)
    k = torch.randn(B, Tk, H, D, generator=g, device=dev).to(torch.bfloat16)
    v = torch.randn(B, Tk, H, D, generator=g, device=dev).to(torch.bfloat16)
    rope = aki_b200.LongRope(device=dev)
    cos, sin = rope.tables(PAST + torch.arange(T, device=dev)[None], max_position=Tk - 1)
    ts = []
    for it in range(25):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(); e1.record()
        lib.aki_mma_set_timing_events(e0.cuda_event, e1.cuda_event)
        o, _ = ops.attn_fwd_raw(q, k, v, cos, sin, meta, D ** -0.5, need_lse=False, q_offset=PAST)
        torch.cuda.synchronize()
        if it >= 5:
            ts.append(e0.elapsed_time(e1))
    ms = statistics.median(ts)
    tflops = 4 * D * nnz * H / (ms * 1e-3) / 1e12
    print(f"continuation B={B} H={H} past={PAST} T={T} ({N_IMG} images in the prefix): {ms * 1e3:.1f} us "
          f"(min {min(ts) * 1e3:.1f}), {tflops:.0f} TFLOP/s over nnz={nnz} per head", flush=True)
