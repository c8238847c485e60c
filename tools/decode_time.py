"""Decode step of the AKI-4B language model (32 layers): graph-replayed step through HF's decoder layers vs through the
fused layers (ops.skinny_linear: aki_mma_skinny_linear for B <= 8, aki_mma_batch_linear for 9 - 64 sequences), and the
weight-streaming kernels alone on the five projection shapes (GB/s against the measured copy bandwidth), with weight
sets larger than L2.  Prints the GPU name and power limit first.  usage: python tools/decode_time.py"""
import ctypes as C
import os, sys, json, subprocess
import torch
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import aki_b200
from aki_b200 import ops
from aki_b200._lib import lib
from aki_b200.model import AkiPhi3Runner, phi35_mini_config
dev = torch.device("cuda", 0)
ev = lambda: torch.cuda.Event(enable_timing=True)
peak = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))["hbm_gbs"] if os.path.exists(os.path.join(ROOT, "MEASURED_PEAKS.json")) else 6650.0
try:
    smi = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                         capture_output=True, text=True, timeout=30).stdout.strip().splitlines()[0]
except Exception as e:  # noqa: BLE001  (the numbers below still stand; say what is missing)
    smi = f"nvidia-smi unavailable ({e})"
print(f"GPU: {torch.cuda.get_device_name(0)} | name, power limit, max SM clock: {smi} | copy bandwidth {peak:.0f} GB/s", flush=True)

SHAPES = [(3072, 9216, {}), (3072, 3072, {"res": 1}), (3072, 8192, {"swiglu": 1}), (8192, 3072, {"res": 1}), (3072, 32064, {})]


def batch_linear(x, w, gamma, res, swiglu):
    """aki_mma_batch_linear directly (any B, also B <= 8, which ops.skinny_linear routes to skinny)."""
    B, K = x.shape
    N = w.shape[0] // (2 if swiglu else 1)
    y = torch.empty(B, N, dtype=torch.bfloat16, device=x.device)
    p = lambda t: None if t is None else C.c_void_p(t.data_ptr())
    mode = 2 if swiglu else (1 if res is not None else 0)
    rc = lib.aki_mma_batch_linear(p(x), x.stride(0), p(w), p(gamma), 1e-5, p(res), res.stride(0) if res is not None else 0,
                                  p(y), y.stride(0), B, N, K, mode, C.c_void_p(torch.cuda.current_stream().cuda_stream))
    assert rc == 0, rc
    return y


def time_projection(name, fn, B, K, N, kw):
    x = torch.randn(B, K, device=dev).to(torch.bfloat16)
    ws = [torch.randn((2 * N if kw.get("swiglu") else N), K, device=dev).to(torch.bfloat16) for _ in range(8)]   # > L2 in total
    res = torch.randn(B, N, device=dev).to(torch.bfloat16) if kw.get("res") else None
    gamma = torch.ones(K, device=dev, dtype=torch.bfloat16) if not kw.get("res") else None
    for w in ws: fn(x, w, gamma, res, bool(kw.get("swiglu")))
    torch.cuda.synchronize()
    graph = torch.cuda.CUDAGraph()                      # replayed: the launch path of 40 ctypes calls is not the subject
    with torch.cuda.graph(graph):
        for rep in range(5):
            for w in ws: fn(x, w, gamma, res, bool(kw.get("swiglu")))
    graph.replay(); torch.cuda.synchronize()
    a, b_ = ev(), ev(); a.record()
    graph.replay()
    b_.record(); torch.cuda.synchronize()
    ms = a.elapsed_time(b_) / 40
    gb = ws[0].numel() * 2 / 1e9
    split = lib.aki_mma_batch_linear_split(B, N, K, 2 if kw.get("swiglu") else (1 if kw.get("res") else 0))
    print(f"{name} B={B} K={K} N={N} {kw} (batch split {split}): {ms * 1e3:.1f} us, {gb / (ms * 1e-3):.0f} GB/s = "
          f"{gb / (ms * 1e-3) / peak:.2f} of {peak:.0f}", flush=True)
    del ws


skinny = lambda x, w, g, r, s: ops.skinny_linear(x, w, g, 1e-5, r, s)
for (K, N, kw) in SHAPES:
    time_projection("skinny_linear", skinny, 8, K, N, kw)
    time_projection("batch_linear ", batch_linear, 8, K, N, kw)
for B in (16, 32, 64):
    for (K, N, kw) in SHAPES:
        time_projection("batch_linear ", batch_linear, B, K, N, kw)

runner = AkiPhi3Runner(phi35_mini_config(), device=dev, seed=0)
n_dec = 16


def step_ms(B, T, fused):
    emb = (torch.randn(B, T, 3072, device=dev) * 0.05).to(torch.bfloat16)
    cache = runner.new_cache(B, T + n_dec + 4)
    tok = runner.prefill(emb, None, cache)[:, -1].argmax(-1, keepdim=True)
    tok = runner.decode_step_graphed(tok, cache, fused=fused)
    torch.cuda.synchronize()
    a, b_ = ev(), ev(); a.record()
    for _ in range(n_dec - 1):
        tok = runner.decode_step_graphed(tok, cache, fused=fused)
    b_.record(); torch.cuda.synchronize()
    del cache, emb
    runner._g = None
    torch.cuda.empty_cache()
    return a.elapsed_time(b_) / (n_dec - 1)


for (B, T) in [(8, 655), (16, 655), (32, 655), (64, 655)]:
    floor = (7.44e9 + 2 * B * 32 * (T + n_dec / 2) * 96 * 2 * 32) / (peak * 1e9) * 1e3
    for rnd in range(2):                               # the two paths alternated, twice, in one process
        for fused in (False, True):
            ms = step_ms(B, T, fused)
            print(f"decode B={B} T={T} round {rnd} {'fused layers' if fused else 'HF layers  '}: {ms:.2f} ms per step "
                  f"({B / ms * 1e3:.0f} tokens/s; HBM floor {floor:.2f} ms: 7.44 GB weights + K/V)", flush=True)
