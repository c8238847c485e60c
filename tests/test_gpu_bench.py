"""-m gpu: bench.py -- --dump-outputs writes what the last timed step returned (checked against the fp32 oracle on the
same seeded inputs), the inputs are identical from run to run, and --steps sets the number of timed steps."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest
import torch

from conftest import ROOT
from oracle import mma_oracle as O

pytestmark = pytest.mark.gpu
H, D = 32, 96
B, T, N_IMG = 2, 1024, 1      # 2048 token rows: the dump is a sample of them, from both samples of the batch
SMALL = ["--seq", str(T), "--batch", str(B), "--images", str(N_IMG), "--warmup", "1", "--no-e2e", "--no-cpu",
         "--no-prefill", "--no-longctx", "--no-sft"]
NAMES = ("o", "lse", "d_q", "d_k", "d_v", "k_rot")


def _bench(*argv):
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), *argv], capture_output=True, text=True,
                       timeout=400, cwd=ROOT)
    assert r.returncode == 0, r.stderr[-2000:]
    lines = [l for l in r.stdout.splitlines() if l.strip()]
    assert len(lines) == 1, r.stdout
    return json.loads(lines[0])


@pytest.fixture(scope="module")
def attn_runs(tmp_path_factory):
    """The attention workload at --steps 2 and 3, each dumping its outputs: [(steps, json line, dump dir)]."""
    runs = []
    for steps in (2, 3):
        d = tmp_path_factory.mktemp(f"dump_s{steps}")
        runs.append((steps, _bench("--steps", str(steps), "--dump-outputs", str(d), *SMALL), d))
    return runs


def test_dump_outputs_same_inputs_and_steps_honoured(attn_runs):
    # the library counts its own kernel launches inside the timed region: the same number per step at any --steps
    for steps, line, _ in attn_runs:
        assert line["steps"] == steps and line["gpu_launches"] > 0 and line["gpu_launches"] % steps == 0
    assert attn_runs[0][1]["gpu_launches"] // 2 == attn_runs[1][1]["gpu_launches"] // 3
    dirs = [d for _, _, d in attn_runs]
    assert sorted(os.listdir(dirs[0])) == sorted(f"{n}.npy" for n in NAMES)
    assert sum(os.path.getsize(dirs[0] / f"{n}.npy") for n in NAMES) <= 64_000_000
    for name in NAMES:
        a, b = (np.load(d / f"{name}.npy") for d in dirs)
        assert a.dtype == np.float32 and a.shape[0] == min(B * T, 1024), (name, a.dtype, a.shape)
        if name == "d_q":        # accumulated with fp32 atomics: the summation order may differ between runs
            assert np.abs(a - b).max() <= 1e-2 * np.abs(b).max(), name
        else:
            assert np.array_equal(a, b), name


def test_dump_outputs_match_the_oracle(attn_runs):
    """The dumped rows are the attention of bench.py's seeded inputs: o, LSE, the gradients of the pre-RoPE q / k / v
    and the post-RoPE K, each at the rows dump_rows() names, against the fp32 oracle with autograd."""
    sys.path.insert(0, ROOT)
    import aki_b200
    import bench
    dev = torch.device("cuda", 0)
    # bench.py's inputs (rank 0)
    lang, am = bench.make_prompt(B, T, N_IMG, seed=0)
    S = O.segments_ref(lang, am, bench.N_VIS, bench.MEDIA_ID)
    g = torch.Generator(device=dev).manual_seed(0)
    qkv = torch.randn(B, T, 3 * H * D, generator=g, device=dev, dtype=torch.float32).to(torch.bfloat16)
    d_o = torch.randn(B, T, H, D, generator=g, device=dev, dtype=torch.float32).to(torch.bfloat16)
    cos, sin = aki_b200.LongRope(device=dev).tables(torch.arange(T, device=dev)[None], max_position=T - 1)
    # oracle
    xf = qkv.float().cpu().requires_grad_(True)
    q, k, v = (xf[..., i * H * D:(i + 1) * H * D].view(B, T, H, D).transpose(1, 2) for i in range(3))
    c = torch.cat([cos.cpu(), cos.cpu()], -1); s = torch.cat([sin.cpu(), sin.cpu()], -1)
    qr, kr = O.apply_rope(q, c, s), O.apply_rope(k, c, s)
    out = O.eager_attention(qr, kr, v, O.additive_mask_from_segments(S), D ** -0.5)          # (B,T,H,D)
    out.backward(d_o.float().cpu())
    m4 = torch.from_numpy(O.expand_segments_to_4d(S)).bool()
    scores = torch.einsum("bhtd,bhsd->bhts", qr.detach(), kr.detach()) * D ** -0.5
    lse = torch.logsumexp(scores.masked_fill(~m4, float("-inf")), dim=-1)                   # (B,H,T)
    grads = xf.grad.view(B, T, 3, H, D)
    ref = {"o": out.detach(), "lse": lse.transpose(1, 2), "d_q": grads[:, :, 0], "d_k": grads[:, :, 1],
           "d_v": grads[:, :, 2], "k_rot": kr.detach().transpose(1, 2)}
    rows = torch.from_numpy(bench.dump_rows(B, T))
    assert len(rows) == 1024 and (rows < T).any() and (rows >= T).any()
    for name in NAMES:
        want = ref[name][rows // T, rows % T].numpy()
        got = np.load(attn_runs[0][2] / f"{name}.npy")
        assert got.shape == want.shape, (name, got.shape, want.shape)
        err = float(np.abs(got - want).max())
        bound = 3e-2 if name == "lse" else 3e-2 * max(1.0, float(np.abs(want).max()))
        assert err <= bound, (name, err, bound)


def test_longctx_times_exactly_steps_prefills():
    """--workload longctx: the headline prefill loop runs --steps times (the library's launch count in the timed
    region is the same per prefill at any --steps)."""
    lines = {steps: _bench("--workload", "longctx", "--steps", str(steps), "--warmup", "0", "--seq", str(T), "--batch",
                           str(B), "--images", str(N_IMG)) for steps in (2, 3)}
    for steps, line in lines.items():
        assert line["steps"] == steps and line["longctx"]["prefill_steps"] == steps
        assert line["longctx"]["prefill_gpu_launches"] > 0 and line["longctx"]["prefill_gpu_launches"] % steps == 0
    assert lines[2]["longctx"]["prefill_gpu_launches"] // 2 == lines[3]["longctx"]["prefill_gpu_launches"] // 3
