"""bench.py -- headline benchmark of the MMA hot path (BASELINE.json: "MMA attn fwd+bwd TFLOP/s vs BF16 peak").

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--workload attn|sft|longctx]
                    [--dump-outputs DIR]

Workload (config.workload): BASELINE config 3 at the north-star point -- T=8192 context, B=2 per GPU, 32 heads x 96,
4 interleaved image spans of 128 vision tokens, <|assistant|> 64 tokens before the end, Phi-3 longrope on Q/K,
bf16, synthetic N(0,1) q/k/v/dO (seeded).  One step = one forward + one backward of the attention core over the
batch.  value = algorithmic FLOPs / time with FLOPs = 43008 * nnz (fwd 4*H*D*nnz, bwd 10*H*D*nnz; nnz = exact
number of visible (query,key) pairs, SURVEY 8d) -- masked work that the kernels skip is not counted.

Keys beyond the base contract:
  roofline      dominant kernel call (backward), tensor-bound, against MEASURED_PEAKS.json bf16_tflops
  cpu_baseline  the oracle (oracle/mma_oracle.py, fp32 eager with the materialised 4-D mask = the reference's CPU
                path) on the host cores, bounded sample, rank 0 only
  e2e           the same metric through the public module API (AkiMMAAttention fwd+bwd incl. qkv/o projections)
                with pinned HOST inputs copied in and the loss read back inside the timed region
N>1: one process per GPU (torchrun), batch-sharded, no data-path collective ("weak" scaling: B=2 per GPU).
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys
import threading
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

H, D, N_VIS = 32, 96, 128
MEDIA_ID, ASST_ID = 32012, 32001


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=50)
    ap.add_argument("--warmup", type=int, default=10)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="attn", choices=["attn", "sft", "longctx"],
                    help="attn: the headline line (+ AKI-4B prefill/decode section); sft: BASELINE config 4, DDP step")
    ap.add_argument("--sft-layers", type=int, default=32)
    ap.add_argument("--sft-bf16-reduce", action="store_true",
                    help="all-reduce gradients in bf16 (DDP compress hook) instead of fp32; measured SLOWER on 2 B200s over "
                         "NVLink (158.3 vs 145.4 ms per step: the casts cost more than the halved transfer saves)")
    ap.add_argument("--seq", type=int, default=8192)
    ap.add_argument("--batch", type=int, default=2)
    ap.add_argument("--images", type=int, default=4)
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-cpu", action="store_true")
    ap.add_argument("--no-prefill", action="store_true", help="skip the AKI-4B prefill/decode section")
    ap.add_argument("--no-longctx", action="store_true", help="skip the config-5 section (8K multi-image prefill + decode)")
    ap.add_argument("--no-sft", action="store_true", help="skip the config-4 section (SFT step, DDP when N > 1)")
    ap.add_argument("--prefill-batch", type=int, default=8)
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write what the last one returned (attention output, LSE, dQ/dK/dV, "
                         "post-RoPE K) as float32 DIR/<name>.npy, on a fixed sample of token rows")
    args = ap.parse_args()
    if args.steps < 1 or args.warmup < 0:
        ap.error("--steps must be >= 1 and --warmup >= 0")
    if args.dump_outputs and (args.impl != "ours" or args.workload != "attn"):
        ap.error("--dump-outputs covers the attention workload of --impl ours")
    return args


def init_nccl(dev):
    """One process per GPU over NCCL.  The communicator's kernels run on HIGH-PRIORITY streams: DDP's bucket all-reduces
    are launched while backward GEMMs fill every SM, and without priority their CTAs wait for whole GEMM waves to drain
    (measured on 2 B200s: the 27 ms of all-reduce left 17.5 ms exposed behind an 85 ms backward)."""
    import torch.distributed as dist
    try:
        opts = dist.ProcessGroupNCCL.Options(is_high_priority_stream=True)
        dist.init_process_group("nccl", device_id=dev, pg_options=opts)
    except Exception:
        dist.init_process_group("nccl", device_id=dev)


def make_prompt(B, T, n_img, seed=0):
    """lang_x (B,L) whose spliced length is exactly T: n_img <image> tokens evenly spaced (first at 8),
    <|assistant|> so that q_end = T - 64."""
    L = T - n_img * (N_VIS - 1)
    g = np.random.default_rng(seed)
    lang = g.integers(3, 31000, size=(B, L)).astype(np.int64)
    step = (L - 64 - 8) // max(n_img, 1)
    for k in range(n_img):
        lang[:, 8 + k * step] = MEDIA_ID
    lang[:, L - 65] = ASST_ID            # post-splice index T-65 -> q_end = T-64
    return lang, np.ones_like(lang)


DUMP_ROWS = 1024    # 1024 token rows x 61.6 KB (o, lse, dq, dk, dv, k_rot in float32) = 63.0 MB per dump


def dump_rows(B, T):
    """The token rows (b * T + t, ascending) --dump-outputs writes: drawn with a fixed seed, the same for the same B and
    T, so that two builds compare row for row."""
    return np.sort(np.random.default_rng(0).choice(B * T, size=min(B * T, DUMP_ROWS), replace=False))


def dump_outputs(out_dir, B, T, outputs):
    """Writes each (B, T, ...) array of `outputs`, restricted to the rows of dump_rows(), as float32 out_dir/<name>.npy."""
    rows = torch.from_numpy(dump_rows(B, T))
    os.makedirs(out_dir, exist_ok=True)
    for name, x in outputs.items():
        sample = x.flatten(0, 1)[rows.to(x.device)]
        np.save(os.path.join(out_dir, name + ".npy"), sample.float().cpu().numpy())


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return d, "measured (MEASURED_PEAKS.json)"
    return {"bf16_tflops": 1590.0, "bf16_tflops_sustained": 1400.0, "hbm_gbs": 6650.0}, "fallback (B200_PROFILING.md)"


class ClockSampler:
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.samples, self.proc, self.index = [], None, index

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-i", str(self.index), "-lms", "50"], stdout=subprocess.PIPE,
                                         stderr=subprocess.STDOUT, text=True)
            self.thread = threading.Thread(target=self._read, daemon=True)
            self.thread.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.samples.append((time.time(), line.strip()))

    def mark_begin(self):
        """Start of the timed region: the sampler itself is started earlier (nvidia-smi needs up to a second to
        produce its first line on an 8-GPU box); only samples that arrive inside the marked window are used."""
        self.t0 = time.time()

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        t1 = time.time()
        time.sleep(0.12)
        self.proc.terminate()
        try:
            self.thread.join(timeout=2.0)
        except Exception:
            pass
        t0 = getattr(self, "t0", 0.0)
        window = [s for (ts, s) in self.samples if t0 <= ts <= t1 + 0.1]
        if not window:                      # region shorter than one sampling period: take the nearest samples
            window = [s for (ts, s) in self.samples][-3:]
        self.samples = window
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for s in self.samples:
            f = [x.strip() for x in s.split(",")]
            if len(f) < 7:
                continue
            try:
                sm.append(float(f[0])); mx.append(float(f[1]))
            except ValueError:
                continue
            for n, v in zip(names, f[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(n)
        sm_hot = [x for x in sm if x > 0.3 * max(sm)] if sm else []
        out = {"sm_mhz": statistics.median(sm_hot) if sm_hot else None, "sm_max_mhz": max(mx) if mx else None,
               "reasons": sorted(reasons), "samples": len(sm)}
        if not sm and self.samples:
            out["raw"] = self.samples[:2]
        return out


# ------------------------------------------------------------------------------------------------ CPU arm
def cpu_reference_run(T, B, n_img, steps, warmup, threads=None, row_block=1024, budget_s=None):
    """The reference's CPU path for this workload: materialised (B,1,T,T) 0/1 mask -> additive fp32 mask -> eager
    softmax(QK^T*scale + mask) V and its autograd backward, fp32, all host threads (oracle/mma_oracle.py).  The T x T
    score tensors of the reference do not fit host RAM at 8K x 32 heads in one piece, so the same arithmetic runs in
    query-row blocks, each block doing its forward and backward (gradients accumulate).  Returns TFLOP/s, ms per step,
    threads, nnz and the number of steps actually timed (budget_s bounds the run on slow hosts)."""
    from oracle import mma_oracle as O
    threads = threads or os.cpu_count()
    torch.set_num_threads(threads)
    lang, am = make_prompt(B, T, n_img)
    S = O.segments_ref(lang, am, N_VIS, MEDIA_ID)
    nnz = O.count_allowed(S)
    g = torch.Generator().manual_seed(0)
    q, k, v = (torch.randn(B, H, T, D, generator=g) for _ in range(3))
    d_o = torch.randn(B, T, H, D, generator=torch.Generator().manual_seed(1))
    inv = O.longrope_inv_freq(D, 10000.0, np.ones(D // 2, dtype=np.float32))
    cos, sin = O.rope_cos_sin(torch.arange(T)[None].expand(B, -1), inv, 1.19)
    times = []
    t_begin = time.perf_counter()
    for it in range(warmup + steps):
        t0 = time.perf_counter()
        mask = torch.from_numpy(O.expand_segments_to_4d(S))                 # the (B,1,T,T) int64 tensor (a1-a3)
        add = O.invert_4d_mask(mask, torch.float32)                          # a7
        del mask
        qq = q.clone().requires_grad_(True); kk = k.clone().requires_grad_(True); vv = v.clone().requires_grad_(True)
        for r0 in range(0, T, row_block):
            r1 = min(T, r0 + row_block)
            qr = O.apply_rope(qq[:, :, r0:r1], cos[:, r0:r1], sin[:, r0:r1])
            out = O.eager_attention(qr, O.apply_rope(kk, cos, sin), vv, add[:, :, r0:r1], D ** -0.5)
            out.backward(d_o[:, r0:r1])
        dt = time.perf_counter() - t0
        if it >= warmup:
            times.append(dt)
        if budget_s is not None and it >= warmup and time.perf_counter() - t_begin > budget_s:
            break
    ms = statistics.median(times) * 1e3
    return 43008.0 * nnz / (ms * 1e-3) / 1e12, ms, threads, nnz, len(times)


def cpu_cfg1_layer_ms(threads=None):
    """BASELINE config 1 (SURVEY 8d): ONE AKI MMA attention layer forward, Phi-3.5-mini shape, batch 1, 128 image + 256
    text tokens (T = 384), fp32 on the host cores via the reference's eager 4-D mask path.  Returns ms (median of 5)."""
    from oracle import mma_oracle as O
    torch.set_num_threads(threads or os.cpu_count())
    g = np.random.default_rng(0)
    L, N = 257, 128
    lang = g.integers(3, 31000, size=(1, L)).astype(np.int64)
    lang[0, 8] = MEDIA_ID; lang[0, 224] = ASST_ID
    S = O.segments_ref(lang, np.ones_like(lang), N, MEDIA_ID)
    T = L - 1 + N
    torch.manual_seed(0)
    w_qkv = torch.randn(3 * H * D, H * D) * 0.02; w_o = torch.randn(H * D, H * D) * 0.02
    hidden = torch.randn(1, T, H * D, generator=torch.Generator().manual_seed(1))
    inv = O.longrope_inv_freq(D, 10000.0, np.ones(D // 2, dtype=np.float32))
    cos, sin = O.rope_cos_sin(torch.arange(T)[None], inv, 1.19)
    ts = []
    for it in range(7):
        t0 = time.perf_counter()
        add = O.invert_4d_mask(torch.from_numpy(O.expand_segments_to_4d(S)), torch.float32)
        O.attention_module_forward(hidden, w_qkv, w_o, cos, sin, add)
        if it >= 2:
            ts.append((time.perf_counter() - t0) * 1e3)
    return statistics.median(ts)


# ------------------------------------------------------------------------------------------------ AKI-4B prefill
def prefill_section(dev, rank, world, steps, warmup, longctx=None):
    """BASELINE config 2: random-init AKI-4B language model (Phi-3.5-mini geometry, 32 layers, bf16), batch 8 per
    GPU, 1 image (144 vision tokens, AKI default) + 511 text tokens -> T = 655; prefill writes the KV cache in place,
    then 32 greedy decode steps.  LM only: the vision tower is replaced by N(0,0.02) vision tokens (SURVEY 8d).
    e2e: host token ids + host vision tokens -> device -> segments + splice kernels -> prefill -> argmax -> host.
    longctx=(B, T, n_img, n_dec): BASELINE config 5 instead -- n_img x 128 image tokens interleaved in a T-token
    context (the prompt of the attention benchmark), then n_dec greedy decode steps against the long cache.
    Timed: `steps` prefills (resident, then e2e) after max(3, warmup // 3) warm-up prefills of each."""
    import aki_b200
    from aki_b200 import ops
    from aki_b200.model import AkiPhi3Runner, phi35_mini_config
    import torch.distributed as dist
    if longctx:
        B, T, n_img, n_dec = longctx
        N = N_VIS
        lang, am = make_prompt(B, T, n_img, seed=100 + rank)
        L = lang.shape[1]
    else:
        B, L, N, n_img, n_dec = parse().prefill_batch, 512, 144, 1, 32
        g = np.random.default_rng(100 + rank)
        lang = g.integers(3, 31000, size=(B, L)).astype(np.int64)
        lang[:, 8] = MEDIA_ID; lang[:, L - 40] = ASST_ID
        am = np.ones_like(lang)
        T = L - 1 + N
    runner = AkiPhi3Runner(phi35_mini_config(), device=dev, seed=0)
    host_ids = torch.from_numpy(lang).pin_memory(); host_am = torch.from_numpy(am).pin_memory()
    host_vis = (torch.randn(B, n_img, N, 3072) * 0.02).to(torch.bfloat16).pin_memory()
    host_out = torch.empty(B, dtype=torch.int64).pin_memory()
    me = type("M", (), {})()
    me.lang_model = runner.lm; me.media_token_id = MEDIA_ID; me.num_tokens_per_vis = N; me.pad_token_id = 32000
    cache = runner.new_cache(B, T + n_dec + 1)
    ev = lambda: torch.cuda.Event(enable_timing=True)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    ids_d, am_d, vis_d = host_ids.to(dev), host_am.to(dev), host_vis.to(dev)
    prep = aki_b200.prepare_inputs_for_forward(me, vis_d, ids_d, am_d, padding_side="left", exact_shape=False)
    embeds, segs = prep["inputs_embeds"], prep["mma_segments"]

    def prefill_resident():
        cache.reset()
        return runner.prefill(embeds, segs, cache)

    def prefill_e2e():
        cache.reset()
        i_d = host_ids.to(dev, non_blocking=True); a_d = host_am.to(dev, non_blocking=True)
        v_d = host_vis.to(dev, non_blocking=True)
        pr = aki_b200.prepare_inputs_for_forward(me, v_d, i_d, a_d, padding_side="left", exact_shape=False)
        logits = runner.prefill(pr["inputs_embeds"], pr["mma_segments"], cache)
        host_out.copy_(logits[:, -1].argmax(-1), non_blocking=True)
        torch.cuda.current_stream().synchronize()

    from aki_b200._lib import lib as _clib
    res = {}
    for name, fn in (("resident", prefill_resident), ("e2e", prefill_e2e)):
        for _ in range(max(3, warmup // 3)):
            fn()
        barrier()
        a, b_ = ev(), ev()
        launches0 = _clib.aki_mma_launch_count()
        a.record()
        for _ in range(steps):
            fn()
        b_.record()
        res[name + "_launches"] = int(_clib.aki_mma_launch_count() - launches0)
        barrier()
        res[name] = a.elapsed_time(b_) / steps
    # decode: n_dec steps on top of the last prefill
    logits = prefill_resident()
    tok = logits[:, -1].argmax(-1, keepdim=True)
    for _ in range(3):
        runner.decode_step(tok, cache)
    cache.reset(); prefill_resident()
    barrier()
    a, b_ = ev(), ev()
    a.record()
    for _ in range(n_dec):
        tok = runner.decode_step(tok, cache)[:, -1].argmax(-1, keepdim=True)
    b_.record()
    barrier()
    dec_eager_ms = a.elapsed_time(b_) / n_dec
    # the same steps replayed from a CUDA graph (device-resident write row / key count / position id)
    cache.reset(); logits = prefill_resident()
    tok = logits[:, -1].argmax(-1, keepdim=True)
    tok = runner.decode_step_graphed(tok, cache)          # captures the graph
    barrier()
    a, b_ = ev(), ev()
    a.record()
    for _ in range(n_dec - 1):
        tok = runner.decode_step_graphed(tok, cache)
    b_.record()
    barrier()
    dec_ms = a.elapsed_time(b_) / (n_dec - 1)
    kv_bytes = 2 * B * 32 * (T + n_dec / 2) * 96 * 2 * 32          # K+V read per step, all layers
    w_bytes = 2.0 * (32 * (9216 * 3072 + 3072 * 3072 + 16384 * 3072 + 3072 * 8192) + 32064 * 3072)   # bf16 weights streamed once per step
    stats = torch.tensor([res["resident"], res["e2e"], dec_ms, dec_eager_ms], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(stats, op=dist.ReduceOp.MAX)
    r_ms, e_ms, d_ms, de_ms = (float(x) for x in stats)
    del runner, cache
    torch.cuda.empty_cache()
    return {"workload": f"AKI-4B LM (Phi-3.5-mini geometry, 32 layers, random init, bf16) prefill B={B}/gpu T={T} "
                        f"({n_img} image(s) x {N} + {L - n_img} text), KV cache written in place, residual + RMSNorm and SiLU gate as fused kernels of this "
                        f"library around cuBLAS GEMMs, last-token logits; "
                        f"{n_dec} greedy decode steps",
            "prefill_tokens_per_s": world * B * T / (r_ms * 1e-3), "prefill_ms": r_ms, "prefill_steps": steps,
            "prefill_gpu_launches": res["resident_launches"],
            "prefill_e2e_tokens_per_s": world * B * T / (e_ms * 1e-3), "prefill_e2e_ms": e_ms,
            "e2e_h2d_bytes": int(host_ids.numel() * 8 * 2 + host_vis.numel() * 2), "e2e_d2h_bytes": B * 8,
            "decode_tokens_per_s": world * B / (d_ms * 1e-3), "decode_ms_per_step": d_ms,
            "decode_note": "greedy step for all 32 layers replayed from one CUDA graph; per layer 7 kernels of this "
                           "library chained by programmatic dependent launch (aki_mma_skinny_linear x4 with RMSNorm / "
                           "residual / SwiGLU fused, rope_kv_write, decode attention + combine)",
            "decode_eager_ms_per_step": de_ms,
            "decode_attn_kv_bytes_per_step": kv_bytes,
            "decode_attn_kv_gbs_floor": kv_bytes / (d_ms * 1e-3) / 1e9,
            "decode_weight_bytes_per_step": w_bytes,
            "decode_hbm_gbs": (kv_bytes + w_bytes) / (d_ms * 1e-3) / 1e9,
            "decode_hbm_floor_ms": (kv_bytes + w_bytes) / (peaks()[0]["hbm_gbs"] * 1e9) * 1e3}


# ------------------------------------------------------------------------------------------------ SFT step (config 4)
def sft_section(args, dev, rank, world, local, steps, warmup):
    """BASELINE config 4: AKI-4B language model (random init, Phi-3.5-mini geometry) instruction-finetune step in the
    reference's amp_bf16 precision, per-GPU batch 4, L = 513 tokens with one <image> (144 vision tokens) -> T = 656,
    labels -100 up to <|assistant|> (sft.yaml:19-21, base.py:81-87), AdamW, grad-norm clip 1.0 every step
    (train_utils.py:143-158); torch DDP over NCCL is the only collective (train/instruction_finetune.py:128-130).
    Vision tokens are synthetic N(0,0.02).  Besides the step time: the same step on the bare module (no gradient
    all-reduce) in the same run -> the all-reduce time that backward did NOT hide, and NCCL's bus bandwidth at 1 GiB."""
    import torch.distributed as dist
    from torch.nn.parallel import DistributedDataParallel as DDP
    import aki_b200
    from aki_b200.model import AkiPhi3SFT, phi35_mini_config
    Bp, L, N = 4, 513, 144
    T = L - 1 + N
    model = AkiPhi3SFT(phi35_mini_config(num_layers=args.sft_layers), device=dev, seed=0)
    n_params = sum(p.numel() for p in model.parameters())
    bucket_mb = int(os.environ.get("AKI_DDP_BUCKET_MB", "256"))
    # 15.3 GB of fp32 gradients per step: large buckets (NCCL reaches its NVLink bandwidth only on >= 100 MB messages;
    # DDP's 25 MB default left 16.7 ms exposed on 2 GPUs), bucket views instead of copies, static graph
    net = model            # wrapped in DDP below, AFTER the compute-only timing of the bare module
    opt = torch.optim.AdamW(model.parameters(), lr=2e-5, weight_decay=1e-4, fused=True)
    g = np.random.default_rng(1000 + rank)
    me = type("M", (), {})()
    me.lang_model = model.lm; me.media_token_id = MEDIA_ID; me.num_tokens_per_vis = N; me.pad_token_id = 32000
    host = []
    for _ in range(4):                      # a few distinct pinned host batches, cycled
        lang = g.integers(3, 31000, size=(Bp, L)).astype(np.int64)
        lang[:, 10] = MEDIA_ID; lang[:, 120] = ASST_ID
        labels = lang.copy(); labels[:, :121] = -100
        host.append((torch.from_numpy(lang).pin_memory(), torch.ones(Bp, L, dtype=torch.int64).pin_memory(),
                     torch.from_numpy(labels).pin_memory(),
                     (torch.randn(Bp, 1, N, 3072) * 0.02).to(torch.bfloat16).pin_memory()))
    host_loss = torch.empty(1, dtype=torch.float32).pin_memory()

    def step(i, sync=True):
        ids, am, lab, vis = (x.to(dev, non_blocking=True) for x in host[i % len(host)])
        pr = aki_b200.prepare_inputs_for_forward(me, vis, ids, am, labels=lab, padding_side="right")
        # sync=False: the same step on the bare module (no DDP hooks, no all-reduce): this rank's compute-only time
        loss = (net if sync else model)(pr["inputs_embeds"].float(), pr["mma_segments"], pr["labels"])
        loss.backward()
        torch.nn.utils.clip_grad_norm_(model.parameters(), 1.0)
        opt.step(); opt.zero_grad(set_to_none=True)
        host_loss.copy_(loss.detach().reshape(1), non_blocking=True)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def timed(n, sync):
        barrier()
        a, b_ = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        for i in range(n):
            step(i, sync)
        b_.record()
        barrier()
        return a.elapsed_time(b_) / n

    ms_nosync = None
    if world > 1:
        # this rank's compute-only step first, on the bare module (DDP's reducer hooks do not exist yet, so nothing of the
        # all-reduce machinery is in the way), then the data-parallel step
        for i in range(3):
            step(i, False)
        ms_nosync = timed(max(3, steps // 2), False)
        net = DDP(model, device_ids=[local], gradient_as_bucket_view=True, bucket_cap_mb=bucket_mb, static_graph=True)
        if args.sft_bf16_reduce:
            # gradients cross NVLink in bf16, as the reference's FSDP mixed-precision config reduces them
            # (train/distributed.py:163-167); halves the 15.3 GB fp32 all-reduce but adds two cast passes per bucket
            from torch.distributed.algorithms.ddp_comm_hooks import default_hooks
            net.register_comm_hook(None, default_hooks.bf16_compress_hook)
    for i in range(max(3, warmup)):
        step(i)
    ms = timed(steps, True)
    if ms_nosync is None:
        ms_nosync = ms
    # NCCL all-reduce alone on a 1 GiB fp32 buffer (the pool's measured reference: 725 GB/s bus bandwidth at 8 ranks)
    busbw = None
    if world > 1:
        buf = torch.zeros(256 * 1024 * 1024, dtype=torch.float32, device=dev)
        for _ in range(2):
            dist.all_reduce(buf)
        barrier()
        a, b_ = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        for _ in range(5):
            dist.all_reduce(buf)
        b_.record()
        barrier()
        ar_ms = a.elapsed_time(b_) / 5
        busbw = 2.0 * (world - 1) / world * buf.numel() * 4 / (ar_ms * 1e-3) / 1e9
        del buf
    t = torch.tensor([ms, ms_nosync], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms, ms_nosync = float(t[0]), float(t[1])
    loss_val = float(host_loss[0])
    grad_bytes = n_params * (2 if args.sft_bf16_reduce else 4)
    del model, net, opt
    torch.cuda.empty_cache()
    return {"workload": f"AKI-4B LM SFT step ({args.sft_layers} layers, {n_params / 1e9:.2f} B params, random init) B={Bp}/gpu "
                        f"L={L} 1 image x {N} -> T={T}, amp_bf16 (fp32 master weights), AdamW(fused), clip 1.0, host batches "
                        "copied in and loss read back every step",
            "parallelism": f"DDP x{world} (NCCL gradient all-reduce, {grad_bytes / 1e9:.1f} GB "
                           f"{'bf16' if args.sft_bf16_reduce else 'fp32'} per step, buckets of {bucket_mb} MB, static graph)",
            "step_ms": ms, "tokens_per_s": world * Bp * T / (ms * 1e-3), "n_params": n_params, "loss": loss_val,
            "step_ms_without_allreduce": ms_nosync, "exposed_allreduce_ms": max(0.0, ms - ms_nosync),
            "allreduce_bytes_per_step": grad_bytes,
            "allreduce_ideal_ms_at_measured_busbw": (2.0 * (world - 1) / world * grad_bytes / (busbw * 1e9) * 1e3) if busbw else 0.0,
            "nccl_allreduce_busbw_gbs_1gib": busbw, "nccl_busbw_reference_gbs": 725.0,
            "h2d_bytes_per_step": int(Bp * L * 8 * 3 + Bp * N * 3072 * 2), "d2h_bytes_per_step": 4}


def sft_main(args, rank, world, local):
    import torch.distributed as dist
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        init_nccl(dev)
    sampler = ClockSampler(local)
    sampler.start(); sampler.mark_begin()
    r = sft_section(args, dev, rank, world, local, args.steps, args.warmup)
    clocks = sampler.stop()
    if rank == 0:
        emit(({
            "metric": "sft_tokens_per_s", "value": r["tokens_per_s"], "unit": "tokens/s", "n_gpus": world,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": r["step_ms"], "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "bf16 autocast, fp32 master weights", "data": "synthetic",
            "config": {"workload": r["workload"], "parallelism": r["parallelism"]},
            "sft": r, "loss": r["loss"], "clocks": clocks,
            "e2e": {"value": r["tokens_per_s"], "unit": "tokens/s", "h2d_bytes_per_step": r["h2d_bytes_per_step"],
                    "d2h_bytes_per_step": 4}}))
    if world > 1:
        dist.destroy_process_group()


# ------------------------------------------------------------------------------------------------ config 5
def longctx_main(args, rank, world, local):
    """BASELINE config 5: multi-image long-context prefill + decode of the AKI-4B language model, batch-sharded over
    the GPUs (no data-path collective): 4 x 128 image tokens interleaved in a T = 8192 context, B = 2 per GPU, then
    128 greedy decode steps from one CUDA graph.  One JSON line: prefill tokens/s (value), decode tokens/s, K/V bytes."""
    import torch.distributed as dist
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        init_nccl(dev)
    sampler = ClockSampler(local) if rank == 0 else None
    if sampler:
        sampler.start()
        sampler.mark_begin()
    r = prefill_section(dev, rank, world, args.steps, args.warmup, longctx=(args.batch, args.seq, args.images, 128))
    clocks = sampler.stop() if sampler else None
    if rank == 0:
        emit(({"metric": "prefill_tokens_per_s", "value": r["prefill_tokens_per_s"], "unit": "tokens/s",
                          "n_gpus": world, "steps": args.steps, "warmup": args.warmup, "ms_per_step": r["prefill_ms"],
                          "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "bf16",
                          "data": "synthetic", "config": {"workload": r["workload"],
                                                          "parallelism": f"batch-sharded x{world}, no collective"},
                          "longctx": r, "clocks": clocks,
                          "e2e": {"value": r["prefill_e2e_tokens_per_s"], "unit": "tokens/s",
                                  "h2d_bytes_per_step": r["e2e_h2d_bytes"], "d2h_bytes_per_step": r["e2e_d2h_bytes"]}}))
    if world > 1:
        dist.destroy_process_group()


# ------------------------------------------------------------------------------------------------ main
_REAL_STDOUT_FD = None
_T0 = time.time()


def emit(obj):
    """Print the ONE JSON line of this run on the real stdout (see main())."""
    sys.stdout.flush()
    if _REAL_STDOUT_FD is not None:
        os.dup2(_REAL_STDOUT_FD, 1)
    print(json.dumps(obj), flush=True)


def main():
    # rank 0 prints exactly ONE line on stdout.  Native libraries also write there (NCCL's version banner when the box
    # sets NCCL_DEBUG=VERSION in the environment or /etc/nccl.conf; NCCL_DEBUG_FILE=/dev/stderr did not move it under
    # torchrun), so file descriptor 1 points at stderr for the whole run and is restored only for that line.
    global _REAL_STDOUT_FD
    sys.stdout.flush()
    _REAL_STDOUT_FD = os.dup(1)
    os.dup2(2, 1)
    args = parse()
    rank = int(os.environ.get("RANK", 0)); world = int(os.environ.get("WORLD_SIZE", 1))
    local = int(os.environ.get("LOCAL_RANK", 0))
    T, B, n_img = args.seq, args.batch, args.images
    cfg = {"workload": f"mma_attn_fwd_bwd T={T} B={B}/gpu H={H} D={D} images={n_img}x{N_VIS} q_end=T-64 rope=longrope",
           "l2": "inputs (q,k,v,o,dO: 5 x %.0f MB per GPU) larger than the 126 MB L2" % (B * T * H * D * 2 / 1e6),
           "parallelism": f"batch-sharded x{world}, no collective"}

    if args.workload == "sft" and args.impl != "reference":
        return sft_main(args, rank, world, local)
    if args.workload == "longctx" and args.impl != "reference":
        return longctx_main(args, rank, world, local)
    if args.impl == "reference":
        if rank != 0:
            return
        # The reference's own CPU path on the SAME config as our arm (T, B, images): one step = one forward + backward
        # of the attention core over the batch, fp32, all host threads, row-blocked so the T x T tensors fit host RAM.
        # ~4-10 s per step at T=8192 B=2: every requested step is run unless the whole run would pass ~4 minutes, in
        # which case the steps actually timed are reported in "steps".
        val, ms, threads, nnz, n_timed = cpu_reference_run(T, B, n_img, args.steps, min(args.warmup, 1), budget_s=240.0)
        sample = (f"T={T} B={B} H={H} images={n_img} fwd+bwd fp32 eager with the materialised 4-D mask, row blocks of 1024 "
                  f"queries, {n_timed} timed step(s) of {ms:.0f} ms after {min(args.warmup, 1)} warm-up")
        emit(({"impl": "reference", "metric": "mma_attn_fwd_bwd_tflops", "value": val, "unit": "TFLOP/s",
                          "n_gpus": args.gpus, "steps": n_timed, "warmup": min(args.warmup, 1), "ms_per_step": ms,
                          "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32",
                          "data": "synthetic", "config": cfg,
                          "cpu_baseline": {"value": val, "unit": "TFLOP/s", "cores": threads, "kind": "port",
                                           "sample": sample},
                          "e2e": {"value": val, "unit": "TFLOP/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
                          "gpu_launches": 0}))
        return

    import torch.distributed as dist
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        init_nccl(dev)
    import aki_b200
    from aki_b200 import ops
    from oracle import mma_oracle as O

    lang, am = make_prompt(B, T, n_img, seed=rank)
    segs = ops.build_segments(torch.from_numpy(lang).to(dev), torch.from_numpy(am).to(dev), N_VIS, MEDIA_ID, t_cap=T,
                              exact_shape=False)
    nnz = O.count_allowed(O.segments_ref(lang, am, N_VIS, MEDIA_ID))       # closed form from the oracle's segments ...
    nnz_dev = int(sum(int(ops.rebuild_tile_bounds(ops.MMASegments(
        segs.seq_len[b_:b_ + 1], segs.q_end[b_:b_ + 1], segs.seg[b_:b_ + 1], segs.row_lo[b_:b_ + 1], segs.row_hi[b_:b_ + 1],
        segs.src[b_:b_ + 1], segs.kv_valid_bits[b_:b_ + 1], segs.kv_mutual_bits[b_:b_ + 1], None, None, T)).expand_to_4d().sum())
        for b_ in range(B))) if T <= 16384 else nnz                        # ... and counted on the device from the kernels' own description
    assert nnz_dev == nnz, (nnz_dev, nnz)
    meta = ops.meta_tuple(segs)
    g = torch.Generator(device=dev).manual_seed(rank)
    qkv = torch.randn(B, T, 3 * H * D, generator=g, device=dev, dtype=torch.float32).to(torch.bfloat16)
    d_o = torch.randn(B, T, H, D, generator=g, device=dev, dtype=torch.float32).to(torch.bfloat16)
    rope = aki_b200.LongRope(device=dev)
    cos, sin = rope.tables(torch.arange(T, device=dev)[None], max_position=T - 1)
    scale = D ** -0.5
    q4 = qkv[..., :H * D].unflatten(-1, (H, D)); v4 = qkv[..., 2 * H * D:].unflatten(-1, (H, D))
    k_rot = torch.empty(B, H, T, D, dtype=torch.bfloat16, device=dev)
    d_qkv = torch.empty_like(qkv)
    dviews = [d_qkv[..., i * H * D:(i + 1) * H * D].unflatten(-1, (H, D)) for i in range(3)]

    ev = lambda: torch.cuda.Event(enable_timing=True)
    per_fwd, per_bwd, per_fwd_k, per_bwd_k = [], [], [], []
    from aki_b200._lib import lib as _clib

    def hook():
        """Pair of events the C library records right around its next tcgen05 attention kernel
        (aki_mma_set_timing_events): the kernel-only duration the roofline is computed from."""
        a, b_ = ev(), ev()
        a.record(); b_.record()                       # creates the cudaEvent_t handles
        _clib.aki_mma_set_timing_events(a.cuda_event, b_.cuda_event)
        return a, b_

    def step(timed, keep=None):
        e0, e1, e2 = ev(), ev(), ev()
        e0.record()
        ops.rope_kv_write(qkv, cos, sin, k_rot, None, 0, H)
        kf = hook() if timed else None
        o, lse = ops.attn_fwd_raw(q4, k_rot.transpose(1, 2), v4, cos, sin, meta, scale)
        e1.record()
        kb = hook() if timed else None
        ops.attn_bwd_raw(d_o, q4, k_rot.transpose(1, 2), v4, o, lse, cos, sin, meta, scale, *dviews)
        e2.record()
        if timed:
            per_fwd.append((e0, e1)); per_bwd.append((e1, e2)); per_fwd_k.append(kf); per_bwd_k.append(kb)
        if keep is not None:
            keep.update(o=o, lse=lse)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    sampler = ClockSampler(local)
    sampler.start()
    for _ in range(args.warmup):
        step(False)
    barrier()
    sampler.mark_begin()
    t_start, t_end = ev(), ev()
    launches0 = _clib.aki_mma_launch_count()
    last = {} if args.dump_outputs else None                      # o and lse of the last timed step
    t_start.record()
    for i in range(args.steps):
        step(True, last if i == args.steps - 1 else None)
    t_end.record()
    gpu_launches = int(_clib.aki_mma_launch_count() - launches0)      # kernels of libaki_mma.so enqueued in the timed region
    barrier()
    clocks = sampler.stop()
    ms_total = t_start.elapsed_time(t_end)
    ms_step = ms_total / args.steps
    fwd_ms = statistics.mean(a.elapsed_time(b) for a, b in per_fwd)
    bwd_ms = statistics.mean(a.elapsed_time(b) for a, b in per_bwd)
    fwd_k_ms = statistics.mean(a.elapsed_time(b) for a, b in per_fwd_k)
    bwd_k_ms = statistics.mean(a.elapsed_time(b) for a, b in per_bwd_k)
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, B, T, {"o": last["o"], "lse": last["lse"].transpose(1, 2), "d_q": dviews[0],
                                               "d_k": dviews[1], "d_v": dviews[2], "k_rot": k_rot.transpose(1, 2)})
    del last

    # ---- decode attention kernel alone (HBM-bound): B=8 sequences x 32 heads against an 8K-token cache --------
    Bd, Td = 8, 8192
    kc = torch.randn(Bd, H, Td, D, device=dev, dtype=torch.float32).to(torch.bfloat16)
    vc = torch.randn(Bd, H, Td, D, device=dev, dtype=torch.float32).to(torch.bfloat16)
    qd = torch.randn(Bd, H, D, device=dev, dtype=torch.float32).to(torch.bfloat16)
    kvl = torch.full((Bd,), Td, dtype=torch.int32, device=dev)
    for _ in range(3):
        ops.decode_op(qd, kc, vc, kvl, Td, scale)
    torch.cuda.synchronize()
    d0, d1 = ev(), ev()
    n_dec_rep = 20
    d0.record()
    for _ in range(n_dec_rep):
        ops.decode_op(qd, kc, vc, kvl, Td, scale)
    d1.record()
    torch.cuda.synchronize()
    dec_ms = d0.elapsed_time(d1) / n_dec_rep
    dec_bytes = 2.0 * Bd * H * Td * D * 2
    del kc, vc

    # ---- e2e: public module API with host inputs --------------------------------------------------
    e2e = None
    if not args.no_e2e:
        from transformers import Phi3Config
        pc = Phi3Config(hidden_size=H * D, num_attention_heads=H, num_key_value_heads=H, intermediate_size=8192,
                        vocab_size=32064)
        torch.manual_seed(0)
        mod = aki_b200.AkiMMAAttention(pc, layer_idx=0).to(dev).to(torch.bfloat16)
        host_x = torch.randn(B, T, H * D).to(torch.bfloat16).pin_memory()
        host_loss = torch.empty(1, dtype=torch.float32).pin_memory()

        # Host -> device copies run on their own stream into two device buffers: step i+1's input uploads while step
        # i computes (every step still copies its own input from pinned host memory and reads its loss back).
        copy_stream = torch.cuda.Stream(device=dev)
        xbuf = [torch.empty(B, T, H * D, dtype=torch.bfloat16, device=dev) for _ in range(2)]
        ready = [torch.cuda.Event() for _ in range(2)]
        consumed = [torch.cuda.Event() for _ in range(2)]

        def upload(i):
            with torch.cuda.stream(copy_stream):
                copy_stream.wait_event(consumed[i % 2])
                xbuf[i % 2].copy_(host_x, non_blocking=True)
                ready[i % 2].record(copy_stream)

        def e2e_step(i, last):
            torch.cuda.current_stream().wait_event(ready[i % 2])
            if not last:
                upload(i + 1)
            x = xbuf[i % 2].detach().requires_grad_(True)
            out, _ = mod(x, None, None, mma_segments=segs, mma_rope=(cos, sin))
            loss = out.float().pow(2).mean()
            loss.backward()
            consumed[i % 2].record()
            host_loss.copy_(loss.detach().reshape(1), non_blocking=True)
            torch.cuda.current_stream().synchronize()
            mod.zero_grad(set_to_none=True)

        for ev_ in consumed:
            ev_.record()
        n_warm = max(3, args.warmup // 2)
        upload(0)
        for i in range(n_warm):
            e2e_step(i, False)
        barrier()
        a, b_ = ev(), ev()
        n_e2e = max(3, args.steps // 2)
        a.record()
        for i in range(n_warm, n_warm + n_e2e):
            e2e_step(i, False)      # every timed step also uploads one input (the one the next step would use)
        b_.record()
        barrier()
        e2e_ms = a.elapsed_time(b_) / n_e2e
    flops = 43008.0 * nnz

    # ---- max over ranks, aggregate ----------------------------------------------------------------
    stats = torch.tensor([ms_step, fwd_ms, bwd_ms, e2e_ms if not args.no_e2e else 0.0, float(flops), fwd_k_ms, bwd_k_ms,
                          dec_ms], dtype=torch.float64, device=dev)
    if world > 1:
        mx = stats.clone(); dist.all_reduce(mx, op=dist.ReduceOp.MAX)
        sm = stats.clone(); dist.all_reduce(sm, op=dist.ReduceOp.SUM)
        ms_step, fwd_ms, bwd_ms, e2e_ms_r = (float(x) for x in mx[:4])
        fwd_k_ms, bwd_k_ms, dec_ms = (float(x) for x in mx[5:8])
        total_flops = float(sm[4])
    else:
        e2e_ms_r = float(stats[3]); total_flops = flops
    prefill = longctx = sft = None
    del qkv, d_o, d_qkv, k_rot
    torch.cuda.empty_cache()
    note = lambda m: (sys.stderr.write(f"[bench rank {rank}] {m} t={time.time() - _T0:.1f}s\n"), sys.stderr.flush())
    note("attention + e2e done")
    if not args.no_prefill:
        prefill = prefill_section(dev, rank, world, max(5, args.steps // 5), args.warmup)
    note("prefill section done")
    if not args.no_longctx:
        # BASELINE config 5 at every N of the scaling run: 4 x 128 image tokens in an 8K context, B=2 per GPU, 128 decode steps
        longctx = prefill_section(dev, rank, world, max(5, args.steps // 10), args.warmup, longctx=(2, 8192, 4, 128))
    note("longctx section done")
    if not args.no_sft:
        # BASELINE config 4 at every N of the scaling run: the one workload of the path with a real collective (DDP)
        sft = sft_section(args, dev, rank, world, local, max(4, args.steps // 8), 3)
    note("sft section done")
    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return

    pk, pk_src = peaks()
    value = total_flops / (ms_step * 1e-3) / 1e12
    bwd_tf = 30720.0 * nnz / (bwd_ms * 1e-3) / 1e12
    fwd_tf = 12288.0 * nnz / (fwd_ms * 1e-3) / 1e12
    bwd_k_tf = 30720.0 * nnz / (bwd_k_ms * 1e-3) / 1e12      # attn_bwd_sm100_kernel alone (events from the C library)
    fwd_k_tf = 12288.0 * nnz / (fwd_k_ms * 1e-3) / 1e12
    traffic = None                                           # dram bytes per launch of the dominant kernel (ncu --set full)
    tp = os.path.join(ROOT, "profiles", "ncu_traffic.json")
    if os.path.exists(tp) and T == 8192 and B == 2 and n_img == 4:
        traffic = json.load(open(tp)).get("attn_bwd_sm100_kernel")
    # Peak rule (B200_PROFILING.md): the burst figure for a kernel timed alone / in a short region at full clocks, the
    # sustained one for a kernel inside a seconds-long step under the power cap.  The timed region here is well under a
    # second; if the SM clock sampled during it stayed within 10 % of the maximum the burst peak is the denominator.
    sm_mhz, sm_max = clocks.get("sm_mhz"), clocks.get("sm_max_mhz")
    region_s = ms_total * 1e-3
    use_burst = (region_s < 2.0) and (sm_mhz is None or sm_max is None or sm_mhz >= 0.9 * sm_max)
    peak = pk["bf16_tflops"] if use_burst else pk["bf16_tflops_sustained"]
    roofline = {"bound": "tensor", "kernel": "attn_bwd_sm100_kernel", "achieved": bwd_k_tf, "peak": peak,
                "unit": "TFLOP/s", "frac": bwd_k_tf / peak,
                "peak_source": pk_src + (", burst (timed region %.2f s at %s of %s MHz)" % (region_s, sm_mhz, sm_max) if use_burst
                                         else ", sustained (timed region %.2f s at %s of %s MHz)" % (region_s, sm_mhz, sm_max)),
                "frac_of_burst_peak": bwd_k_tf / pk["bf16_tflops"], "frac_of_sustained_peak": bwd_k_tf / pk["bf16_tflops_sustained"],
                "algorithmic": "30720 * nnz FLOP per launch (SURVEY 8d)", "traffic": traffic,
                "forward_kernel": {"kernel": "attn_fwd_sm100_kernel", "achieved": fwd_k_tf, "frac": fwd_k_tf / peak,
                                   "algorithmic": "12288 * nnz FLOP per launch"}}
    line = {
        "metric": "mma_attn_fwd_bwd_tflops", "value": value, "unit": "TFLOP/s", "n_gpus": world, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": ms_step, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "bf16", "data": "synthetic", "config": cfg,
        "frac_of_bf16_peak": value / (pk["bf16_tflops"] * world),
        "kernels": {"fwd_ms": fwd_ms, "fwd_tflops": fwd_tf, "bwd_ms": bwd_ms, "bwd_tflops": bwd_tf, "nnz_per_gpu": nnz,
                    "attn_fwd_sm100_kernel_ms": fwd_k_ms, "attn_fwd_sm100_kernel_tflops": fwd_k_tf,
                    "attn_bwd_sm100_kernel_ms": bwd_k_ms, "attn_bwd_sm100_kernel_tflops": bwd_k_tf,
                    "note": "fwd/bwd = whole C-ABI calls (rope_kv_write + forward; preprocess + memset + backward + "
                            "finalize); *_kernel = the tcgen05 kernel alone between events recorded by the library"},
        "roofline": roofline,
        "decode_kernel": {"bound": "hbm", "workload": f"aki_mma_decode B={Bd} H={H} T_kv={Td} D={D} (one layer)",
                          "ms": dec_ms, "achieved": dec_bytes / (dec_ms * 1e-3) / 1e9, "peak": pk["hbm_gbs"],
                          "unit": "GB/s", "frac": dec_bytes / (dec_ms * 1e-3) / 1e9 / pk["hbm_gbs"],
                          "algorithmic": "2*B*H*T_kv*D*2 bytes (K and V read once)"},
        "clocks": clocks, "gpu_launches": gpu_launches,
        "gpu_launches_note": "counted by libaki_mma.so (aki_mma_launch_count): per step rope_kv_write, attn_fwd_sm100, "
                             "bwd_preprocess, attn_bwd_sm100, dq_finalize (+ one cudaMemsetAsync, not counted)",
    }
    if not args.no_e2e:
        line["e2e"] = {"value": total_flops / (e2e_ms_r * 1e-3) / 1e12, "unit": "TFLOP/s",
                       "h2d_bytes_per_step": B * T * H * D * 2, "d2h_bytes_per_step": 4, "ms_per_step": e2e_ms_r,
                       "api": "AkiMMAAttention.forward + backward (qkv_proj, o_proj included in time, not in FLOPs); the "
                              "next step's pinned-host input uploads on a copy stream while this step computes"}
    if prefill is not None:
        line["prefill"] = prefill
    if longctx is not None:
        line["longctx"] = longctx
    if sft is not None:
        line["sft"] = sft
    if not args.no_cpu and world == 1:
        # bounded sample of the SAME workload on the host cores (rank 0, N=1 only): same T / images / geometry, half the
        # batch (B=1), one warm-up + two timed steps (~10-25 s); TFLOP/s is normalised by the exact nnz, so it compares
        # directly with `value`.  Plus config 1 (one layer forward on the CPU) in ms.
        val, ms, threads, _, n_timed = cpu_reference_run(T, 1, n_img, 2, 1, budget_s=60.0)
        line["cpu_baseline"] = {"value": val, "unit": "TFLOP/s", "cores": threads, "kind": "port",
                                "sample": f"T={T} B=1 of {B} H={H} images={n_img} fwd+bwd fp32 eager (materialised 4-D mask, "
                                          f"row blocks of 1024 queries), {n_timed} timed step(s) of {ms:.0f} ms",
                                "cfg1_layer_forward_ms": cpu_cfg1_layer_ms(threads),
                                "cfg1_note": "BASELINE config 1: one MMA attention layer forward (qkv_proj, RoPE, 4-D mask, "
                                             "eager softmax, o_proj), batch 1, 128 image + 256 text tokens, fp32, host cores"}
    emit(line)
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
