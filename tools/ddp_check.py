"""DDP check for the SFT step (BASELINE config 4, SURVEY 8e): gradients of a 2-rank DDP step (per-rank batch 2) must
equal the gradients of the same 4 samples run as one batch on a single GPU; a DDP step with AkiAdamW + use_bf16_weights
(bucket views, static graph) must update the parameters like that single-GPU step; batch-sharded prefill must equal the
unsharded prefill.  Launch:  python -m torch.distributed.run --nnodes=1 --nproc-per-node 2 --master-addr 127.0.0.1
--master-port 29511 tools/ddp_check.py      (gpurun --gpus 2)"""
import os
import sys

import numpy as np
import torch
import torch.distributed as dist
from torch.nn.parallel import DistributedDataParallel as DDP

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import aki_b200                                                     # noqa: E402
from aki_b200.dist import gather_batch, shard_batch                # noqa: E402
from aki_b200.model import AkiPhi3Runner, AkiPhi3SFT, phi35_mini_config   # noqa: E402

MEDIA_ID, ASST_ID = 32012, 32001


def main():
    rank, world, local = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"]), int(os.environ["LOCAL_RANK"])
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    dist.init_process_group("nccl", device_id=dev)
    B, L, N = 2 * world, 200, 144
    g = np.random.default_rng(7)
    lang = g.integers(3, 31000, size=(B, L)).astype(np.int64)
    lang[:, 10] = MEDIA_ID; lang[:, 120] = ASST_ID
    labels = lang.copy(); labels[:, :121] = -100
    am = np.ones_like(lang); am[1, 180:] = 0                       # one right-padded sample
    ids, amt, lab = (torch.from_numpy(x).to(dev) for x in (lang, am, labels))
    vis = (torch.randn(B, 1, N, 3072, generator=torch.Generator().manual_seed(3)) * 0.02).to(torch.bfloat16).to(dev)

    cfg = phi35_mini_config(num_layers=2)
    model = AkiPhi3SFT(cfg, device=dev, seed=0)                    # identical init on every rank (same seed)
    me = type("M", (), {})()
    me.lang_model = model.lm; me.media_token_id = MEDIA_ID; me.num_tokens_per_vis = N; me.pad_token_id = 32000

    def loss_of(net, i, a, l, v):
        pr = aki_b200.prepare_inputs_for_forward(me, v, i, a, labels=l, padding_side="right")
        return net(pr["inputs_embeds"].float(), pr["mma_segments"], pr["labels"]), pr

    # single-process reference on the full batch (every rank computes it; only rank 0 reports)
    full_loss, _ = loss_of(model, ids, amt, lab, vis)
    full_loss.backward()
    ref = {n: p.grad.detach().clone() for n, p in model.named_parameters() if p.grad is not None}
    n_tok_full = int((lab[:, 1:] != -100).sum())
    model.zero_grad(set_to_none=True)

    # DDP on the batch shard.  DDP averages per-rank MEAN losses; the full-batch loss is a mean over all target tokens,
    # so each rank's loss is re-weighted by its share of the target tokens (the shards hold the same count here).
    net = DDP(model, device_ids=[local])
    si, sa, sl, sv = shard_batch([ids, amt, lab, vis], rank, world)
    n_tok = int((sl[:, 1:] != -100).sum())
    loss, _ = loss_of(net, si, sa, sl, sv)
    (loss * (n_tok * world / n_tok_full)).backward()
    worst = 0.0
    for n, p in model.named_parameters():
        if p.grad is None:
            continue
        d = float((p.grad - ref[n]).abs().max())
        s = float(ref[n].abs().max()) + 1e-12
        worst = max(worst, d / s)
    t = torch.tensor([worst], device=dev)
    dist.all_reduce(t, op=dist.ReduceOp.MAX)

    # AkiAdamW + the bf16 weight copies under DDP: one clipped step on the shards moves the parameters like the same step
    # on the full batch on one GPU (relative to the size of the update)
    def fused_step(ddp):
        m2 = AkiPhi3SFT(cfg, device=dev, seed=0)
        p0 = [p.detach().clone() for p in m2.parameters()]
        opt = aki_b200.AkiAdamW(m2.parameters(), lr=1e-4, weight_decay=1e-4, max_grad_norm=1.0)
        aki_b200.use_bf16_weights(m2, opt)
        me.lang_model = m2.lm
        if ddp:
            n2 = DDP(m2, device_ids=[local], gradient_as_bucket_view=True, static_graph=True)
            l2, _ = loss_of(n2, si, sa, sl, sv)
            (l2 * (n_tok * world / n_tok_full)).backward()
        else:
            l2, _ = loss_of(m2, ids, amt, lab, vis)
            l2.backward()
        opt.step()
        return [p.detach() - q for p, q in zip(m2.parameters(), p0)]

    d_ref, d_ddp = fused_step(False), fused_step(True)
    num = sum(float((a - b).double().pow(2).sum()) for a, b in zip(d_ddp, d_ref)) ** 0.5
    den = sum(float(b.double().pow(2).sum()) for b in d_ref) ** 0.5
    t_opt = torch.tensor([num / (den + 1e-30)], device=dev)
    dist.all_reduce(t_opt, op=dist.ReduceOp.MAX)

    # batch-sharded prefill == unsharded prefill (no collective on the data path; results gathered afterwards)
    runner = AkiPhi3Runner(cfg, device=dev, seed=0)
    me.lang_model = runner.lm
    with torch.no_grad():
        pr = aki_b200.prepare_inputs_for_forward(me, vis, ids, amt, padding_side="left", exact_shape=False)
        full = runner.prefill(pr["inputs_embeds"], pr["mma_segments"], None)
        prs = aki_b200.prepare_inputs_for_forward(me, sv, si, sa, padding_side="left", exact_shape=False)
        part = runner.prefill(prs["inputs_embeds"], prs["mma_segments"], None)
    gathered = gather_batch(part, B)
    e_pf = float((gathered.float().cpu() - full.float().cpu()).abs().max())
    if rank == 0:
        ok = float(t[0]) < 3e-2 and float(t_opt[0]) < 3e-2 and e_pf < 5e-2
        print(f"ddp_check world={world}: max relative grad error vs single-GPU full batch = {float(t[0]):.3e}; "
              f"AkiAdamW + bf16 weights step, |update - single-GPU update| / |update| = {float(t_opt[0]):.3e}; "
              f"sharded-vs-unsharded prefill logits max abs diff = {e_pf:.3e}  ->  {'PASS' if ok else 'FAIL'}")
    dist.destroy_process_group()


if __name__ == "__main__":
    main()
