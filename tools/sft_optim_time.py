"""The SFT step (BASELINE config 4: bench.py's harness, 32 layers, B = 4, T = 656, amp_bf16) on one GPU, two ways:
  torch : clip_grad_norm_(1.0) + torch.optim.AdamW(fused=True), autocast casts every Linear weight in each forward
  fused : AkiAdamW(max_grad_norm=1.0) + use_bf16_weights (the update writes the bf16 copies the Linears read)
Reports, in one run: the step time both ways alternated twice, the two new passes alone against their HBM byte floors
(norm 4 B / param; update 28 B / param + 2 B / Linear-weight element), torch.cuda.max_memory_allocated both ways (the
other way's optimizer state stays resident in both windows), a torch-profiler kernel table of one step each way (after
the timing), and the card's name and power limit.  usage: python tools/sft_optim_time.py [layers] [steps]"""
import os
import subprocess
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import aki_b200                                                        # noqa: E402
from aki_b200 import AkiAdamW, unuse_bf16_weights, use_bf16_weights   # noqa: E402
from aki_b200.model import AkiPhi3SFT, phi35_mini_config              # noqa: E402
from aki_b200.optim import _entries, grad_sq_norm                      # noqa: E402
from aki_b200 import _lib                                              # noqa: E402
from torch.profiler import ProfilerActivity, profile                   # noqa: E402

MEDIA_ID, ASST_ID = 32012, 32001
COPY_GBS = 6548.0          # measured device-to-device copy bandwidth of the B200 (README)


def main():
    layers = int(sys.argv[1]) if len(sys.argv) > 1 else 32
    steps = int(sys.argv[2]) if len(sys.argv) > 2 else 10
    dev = torch.device("cuda", 0)
    smi = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                         capture_output=True, text=True).stdout.strip()
    print(f"card: {smi}")
    Bp, L, N = 4, 513, 144
    model = AkiPhi3SFT(phi35_mini_config(num_layers=layers), device=dev, seed=0)
    params = list(model.parameters())
    n_params = sum(p.numel() for p in params)
    n_lin = sum(m.weight.numel() for m in model.modules() if isinstance(m, torch.nn.Linear))
    print(f"{layers} layers: {n_params / 1e9:.3f} B parameters in {len(params)} tensors, {n_lin / 1e9:.3f} B in Linear "
          f"weights; B = {Bp}, T = {L - 1 + N}")
    opt_t = torch.optim.AdamW(params, lr=2e-5, weight_decay=1e-4, fused=True)
    opt_a = AkiAdamW(params, lr=2e-5, weight_decay=1e-4, max_grad_norm=1.0)
    g = np.random.default_rng(1000)
    me = type("M", (), {})()
    me.lang_model = model.lm; me.media_token_id = MEDIA_ID; me.num_tokens_per_vis = N; me.pad_token_id = 32000
    batches = []
    for _ in range(4):
        lang = g.integers(3, 31000, size=(Bp, L)).astype(np.int64)
        lang[:, 10] = MEDIA_ID; lang[:, 120] = ASST_ID
        labels = lang.copy(); labels[:, :121] = -100
        batches.append((torch.from_numpy(lang).to(dev), torch.ones(Bp, L, dtype=torch.int64, device=dev),
                        torch.from_numpy(labels).to(dev), (torch.randn(Bp, 1, N, 3072) * 0.02).to(torch.bfloat16).to(dev)))

    def fwd_bwd(i):
        ids, am, lab, vis = batches[i % len(batches)]
        pr = aki_b200.prepare_inputs_for_forward(me, vis, ids, am, labels=lab, padding_side="right")
        loss = model(pr["inputs_embeds"].float(), pr["mma_segments"], pr["labels"])
        loss.backward()
        return loss

    def step_torch(i):
        loss = fwd_bwd(i)
        torch.nn.utils.clip_grad_norm_(params, 1.0)
        opt_t.step(); opt_t.zero_grad(set_to_none=True)
        return loss

    def step_fused(i):
        loss = fwd_bwd(i)
        opt_a.step(); opt_a.zero_grad(set_to_none=True)
        return loss

    ways = {"torch": step_torch, "fused": step_fused}

    def window(name, n):
        if name == "fused":
            use_bf16_weights(model, opt_a)
        fn = ways[name]
        for i in range(3):
            fn(i)
        torch.cuda.synchronize()
        torch.cuda.reset_peak_memory_stats(dev)
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        for i in range(n):
            loss = fn(i)
        b.record()
        torch.cuda.synchronize()
        peak = torch.cuda.max_memory_allocated(dev) / 1e9
        if name == "fused":
            unuse_bf16_weights(model)
        return a.elapsed_time(b) / n, peak, float(loss.detach())

    print(f"\nstep time, {steps} timed steps per window after 3 warm-up steps (device events):")
    res = {"torch": [], "fused": []}
    for rep in range(2):
        for name in ("torch", "fused"):
            ms, peak, loss = window(name, steps)
            res[name].append(ms)
            print(f"  {name:5s} rep {rep}: {ms:8.2f} ms/step  peak allocated {peak:6.1f} GB  last loss {loss:.4f}")
    st_a = sum(v.numel() * v.element_size() for s in opt_a.state.values() for k, v in s.items() if k != "step") / 1e9
    st_t = sum(v.numel() * v.element_size() for s in opt_t.state.values() for k, v in s.items() if k != "step") / 1e9
    print(f"  (both optimizers' state stays resident in every window: torch {st_t:.1f} GB, fused {st_a:.1f} GB; the "
          f"fused windows add {n_lin * 2 / 1e9:.1f} GB of bf16 copies)")
    print(f"  torch {min(res['torch']):.2f}-{max(res['torch']):.2f} ms, fused {min(res['fused']):.2f}-"
          f"{max(res['fused']):.2f} ms")

    # the two passes alone, on the model's own gradients
    fwd_bwd(0)
    torch.cuda.synchronize()
    work = [(p, p.grad, opt_a.state[p]["exp_avg"], opt_a.state[p]["exp_avg_sq"], None) for p in params]
    w16 = {m.weight: torch.empty_like(m.weight, dtype=torch.bfloat16) for m in model.modules()
           if isinstance(m, torch.nn.Linear)}
    ent = _entries([(p, gr, m, v, w16.get(p)) for p, gr, m, v, _ in work])
    sq = grad_sq_norm([p.grad for p in params])
    ws = torch.empty(_lib.lib.aki_mma_grad_sq_norm_workspace_bytes(ent.ctypes.data, len(work)), dtype=torch.uint8,
                     device=dev)
    stream = torch.cuda.current_stream(dev).cuda_stream

    def norm_pass():
        _lib.check(_lib.lib.aki_mma_grad_sq_norm(ent.ctypes.data, len(work), ws.data_ptr(), ws.numel(), sq.data_ptr(),
                                                 stream), "norm")

    def update_pass():
        _lib.check(_lib.lib.aki_mma_adamw_step(ent.ctypes.data, len(work), sq.data_ptr(), 1.0, 0.0, 0.9, 0.999, 1e-8,
                                               0.0, 100, stream), "adamw")   # lr = 0: the weights do not drift

    def clip_torch():
        torch.nn.utils.clip_grad_norm_(params, 1e30)

    def adamw_torch():
        lr = opt_t.param_groups[0]["lr"]
        opt_t.param_groups[0]["lr"] = 0.0
        opt_t.step()
        opt_t.param_groups[0]["lr"] = lr

    def timeit(fn, n=20):
        for _ in range(3):
            fn()
        torch.cuda.synchronize()
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        for _ in range(n):
            fn()
        b.record()
        torch.cuda.synchronize()
        return a.elapsed_time(b) / n

    print("\nthe passes alone (device events, 20 calls each; the working set is far above the 126 MB L2):")
    for name, fn, nbytes in (("aki norm pass", norm_pass, 4 * n_params),
                             ("aki update pass (+ bf16 copies)", update_pass, 28 * n_params + 2 * n_lin),
                             ("torch clip_grad_norm_ (norm + scale)", clip_torch, 4 * n_params + 8 * n_params),
                             ("torch AdamW(fused=True).step", adamw_torch, 28 * n_params)):
        ms = timeit(fn)
        floor = nbytes / (COPY_GBS * 1e9) * 1e3
        print(f"  {name:38s} {ms:8.3f} ms  {nbytes / 1e9:6.1f} GB  {nbytes / ms / 1e6:7.0f} GB/s  floor at "
              f"{COPY_GBS:.0f} GB/s {floor:7.3f} ms  ({floor / ms:.2f} of it)")
    for p in params:
        p.grad = None
    del w16, ws

    print("\nkernel table of one step each way (torch.profiler, after the timing):")
    for name in ("torch", "fused"):
        if name == "fused":
            use_bf16_weights(model, opt_a)
        ways[name](0)
        torch.cuda.synchronize()
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            ways[name](1)
            torch.cuda.synchronize()
        if name == "fused":
            unuse_bf16_weights(model)
        rows = [(e.key, getattr(e, "device_time_total", 0), e.count) for e in prof.key_averages()]
        rows = [r for r in rows if r[1] > 0]
        rows.sort(key=lambda r: -r[1])
        tot = sum(r[1] for r in rows)
        print(f"  -- {name}: {tot / 1e3:.2f} ms of kernels")
        for k, t, n in rows[:22]:
            print(f"  {t / 1e3:8.3f} ms {100 * t / tot:5.1f}%  n={n:4d}  {k[:110]}")


if __name__ == "__main__":
    main()
