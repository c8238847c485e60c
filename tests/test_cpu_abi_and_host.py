"""CPU-only checks: the C-ABI library loads and exports exactly what include/aki_mma.h declares, argument
validation returns status codes without touching a GPU, and the host-side logic (cache contract, sharding,
longrope factor, bench geometry) behaves like the reference's."""
import ctypes as C
import os
import re
import subprocess
import sys

import numpy as np
import pytest
import torch

from conftest import ROOT


@pytest.fixture(scope="module")
def lib():
    from aki_b200 import _lib
    return _lib


def test_header_symbols_exported(lib):
    hdr = open(os.path.join(ROOT, "include", "aki_mma.h")).read()
    declared = set(re.findall(r"\b(aki_mma_[a-z0-9_]+)\s*\(", hdr))
    assert declared, "no declarations found"
    out = subprocess.run(["nm", "-D", "--defined-only", lib.LIB_PATH], capture_output=True, text=True, check=True).stdout
    exported = set(re.findall(r" T (aki_mma_[a-z0-9_]+)", out))
    assert declared <= exported, f"declared but not exported: {sorted(declared - exported)}"
    assert set(lib.EXPORTED_SYMBOLS) == declared, (sorted(set(lib.EXPORTED_SYMBOLS) ^ declared))


def test_abi_version_and_strerror(lib):
    assert lib.lib.aki_mma_abi_version() == 2
    assert lib.lib.aki_mma_strerror(0) == b"ok"
    for code in range(-6, 0):
        assert len(lib.lib.aki_mma_strerror(code)) > 3
    assert lib.lib.aki_mma_last_cuda_error() is not None


def test_argument_validation_without_gpu(lib):
    """Error behaviour of the ABI: status codes, no exception, no abort (mirrors the reference's asserts)."""
    L = lib.lib
    assert L.aki_mma_segments(None, None, 1, 4, 2, 5, 6, 8, 0, None, None, None, None, None, None, None, None, None, None) == -1
    buf = (C.c_int64 * 8)()
    out = (C.c_int32 * 8)()
    assert L.aki_mma_segments(buf, buf, 0, 4, 2, 5, 6, 8, 0, out, None, None, None, None, None, None, None, None, None) == -2
    p = lib.AttnParams()
    assert L.aki_mma_attn_fwd(None, None) == -1
    p.B, p.H, p.T, p.D = 1, 32, 128, 64          # head_dim 64 is not supported
    assert L.aki_mma_attn_fwd(C.byref(p), None) == -3
    p.D = 96
    assert L.aki_mma_attn_fwd(C.byref(p), None) == -1          # q.ptr NULL
    p.B = 0
    assert L.aki_mma_attn_fwd(C.byref(p), None) == -2
    assert L.aki_mma_attn_bwd_workspace_bytes(2, 32, 1000, 96) >= 2 * 32 * 1000 * 96 * (2 + 4)
    assert L.aki_mma_attn_bwd_workspace_bytes(2, 32, 1000, 64) == 0
    assert L.aki_mma_decode_workspace_bytes(1, 32, 96, 1000) == 1 * 32 * 2 * 98 * 4
    assert L.aki_mma_rope_kv_write(None, 0, 0, None, None, 0, 1, 1, 32, 96, None, None, 0, 0, 0, 1, None, None) == -1


def test_layer_kernel_argument_validation_without_gpu(lib):
    """Status codes of the f-1 / f-2 entry points (no launch happens: every call fails validation first)."""
    L = lib.lib
    assert L.aki_mma_skinny_linear(None, 0, None, None, 1e-5, None, 0, None, 0, 1, 16, 1024, 0, None) == -1
    buf = (C.c_int64 * 64)()
    assert L.aki_mma_skinny_linear(buf, 1024, buf, None, 1e-5, None, 0, buf, 16, 9, 16, 1024, 0, None) == -2      # B > 8
    assert L.aki_mma_skinny_linear(buf, 1024, buf, None, 1e-5, None, 0, buf, 16, 1, 24, 1024, 0, None) == -3      # N % 16
    assert L.aki_mma_skinny_linear(buf, 1024, buf, None, 1e-5, None, 0, buf, 16, 1, 16, 1000, 0, None) == -3      # K % 1024
    assert L.aki_mma_add_rmsnorm(None, 0, None, 0, None, 1e-5, None, 0, None, 0, 1, 1024, None) == -1
    assert L.aki_mma_add_rmsnorm(buf, 1024, None, 0, buf, 1e-5, None, 0, buf, 1024, 0, 1024, None) == -2          # M = 0
    assert L.aki_mma_add_rmsnorm(buf, 1024, None, 0, buf, 1e-5, None, 0, buf, 1024, 1, 8192, None) == -3          # K > 4096
    assert L.aki_mma_add_rmsnorm(buf, 1024, None, 0, buf, 1e-5, buf, 1024, buf, 1024, 1, 1024, None) == -2        # h_out without residual
    assert L.aki_mma_swiglu(None, 0, None, 0, 1, 8, None) == -1
    assert L.aki_mma_swiglu(buf, 16, buf, 8, 1, 12, None) == -3                                                   # N % 8
    assert L.aki_mma_cross_entropy_fwd(None, 0, 0, None, 0, 1, 1, 8, -100, None, None, None) == -1
    assert L.aki_mma_cross_entropy_fwd(buf, 80, 40, buf, 2, 1, 2, 36, -100, buf, buf, None) == -3                 # V % 8
    assert L.aki_mma_cross_entropy_bwd(buf, 80, 40, buf, 2, 1, 2, 40, -100, buf, None, buf, 80, 40, None) == -1   # scale NULL
    assert L.aki_mma_add_rmsnorm_amp_fwd(buf, None, buf, 1e-5, buf, buf, buf, 1, 256, None) == -1                 # h_out without a
    assert L.aki_mma_add_rmsnorm_amp_fwd(buf, None, buf, 1e-5, None, buf, buf, 1, 4096, None) == -3               # K > 3072
    assert L.aki_mma_rmsnorm_amp_bwd_partials(0) == 0 and L.aki_mma_rmsnorm_amp_bwd_partials(9) == 16
    assert L.aki_mma_rmsnorm_amp_bwd_partials(10 ** 6) == 296 * 8
    assert L.aki_mma_rmsnorm_amp_bwd(buf, None, buf, buf, buf, buf, None, 1, 256, None) == -1
    assert L.aki_mma_swiglu_bwd(buf, buf, buf, 1, 12, None) == -3


def test_fuse_phi3_elementwise_is_reversible_and_steps_aside_on_cpu():
    """aki_b200.fuse_phi3_elementwise: per-instance rebinding, idempotent, undone by unfuse; on tensors the fused kernels do
    not serve (CPU, fp32, autograd on) the original forwards run and the outputs are unchanged."""
    import aki_b200
    from transformers import Phi3Config, Phi3ForCausalLM
    cfg = Phi3Config(hidden_size=256, num_attention_heads=4, num_key_value_heads=4, intermediate_size=512, vocab_size=64,
                     num_hidden_layers=2, pad_token_id=0)
    torch.manual_seed(0)
    m = Phi3ForCausalLM(cfg).eval()
    ids = torch.randint(1, 64, (2, 9))
    with torch.no_grad():
        ref = m(input_ids=ids).logits
    assert aki_b200.fuse_phi3_elementwise(m) == 2 * 3 + 1
    assert aki_b200.fuse_phi3_elementwise(m) == 0
    with torch.no_grad():
        got = m(input_ids=ids).logits
    assert torch.equal(ref, got)
    assert aki_b200.unfuse_phi3_elementwise(m) == 7
    assert not any(hasattr(x, "_aki_orig_forward") for x in m.modules())


def test_ops_refuse_cpu_tensors(lib):
    from aki_b200 import ops
    x = torch.zeros(1, 8, dtype=torch.int64)
    with pytest.raises(lib.AkiMmaError):
        ops.build_segments(x, x, 4, 32012)
    q = torch.zeros(1, 128, 32, 96, dtype=torch.bfloat16)
    with pytest.raises(lib.AkiMmaError):
        ops.attn_fwd_raw(q, q, q, None, None, None, 0.1)


def test_kv_cache_contract_cpu():
    """past_key_values[0][0].shape[2] is the past length (vlm.py:463-468, aki_generation.py:80); append along dim 2."""
    from aki_b200 import AkiKVCache
    c = AkiKVCache(num_layers=2, batch=1, num_heads=4, head_dim=96, t_cap=16, device="cpu", dtype=torch.float32)
    assert c[0][0].shape == (1, 4, 0, 96) and c.get_seq_length() == 0 and len(c) == 2
    k = torch.randn(1, 4, 5, 96); v = torch.randn(1, 4, 5, 96)
    for layer in range(2):
        kk, vv = c.update(k, v, layer)
        assert kk.shape == (1, 4, 5, 96) and torch.equal(kk, k) and torch.equal(vv, v)
    assert c[0][0].shape[2] == 5 and int(c.kv_len[0]) == 5
    k2 = torch.randn(1, 4, 1, 96)
    kk, _ = c.update(k2, k2, 0)
    assert kk.shape[2] == 6 and torch.equal(kk[:, :, :5], k) and torch.equal(kk[:, :, 5:], k2)
    legacy = c.to_legacy_cache()
    assert legacy[0][0].shape[2] == 6 and legacy[1][0].shape[2] == 5
    with pytest.raises(ValueError):
        c.update(torch.randn(1, 4, 11, 96), torch.randn(1, 4, 11, 96), 0)


def test_prepare_inputs_passthrough_and_assert_cpu():
    """vision_tokens is None -> ids and the 2-D mask pass through (vlm.py:470-475); the KV-length assert of
    vlm.py:463-468 is kept."""
    from types import SimpleNamespace
    from aki_b200 import prepare_inputs_for_forward
    me = SimpleNamespace(num_tokens_per_vis=4, media_token_id=32012, pad_token_id=32000, lang_model=None)
    ids = torch.tensor([[1, 2, 3]]); am = torch.ones(1, 3, dtype=torch.long)
    out = prepare_inputs_for_forward(me, None, ids, am, labels=ids)
    assert out["input_ids"] is ids and out["attention_mask"] is am and out["labels"] is ids
    past = ((torch.zeros(1, 2, 7, 96), torch.zeros(1, 2, 7, 96)),)
    with pytest.raises(AssertionError):
        prepare_inputs_for_forward(me, None, ids, am, past_key_values=past)
    prepare_inputs_for_forward(me, None, ids, torch.ones(1, 10, dtype=torch.long), past_key_values=past)


def test_longrope_attention_factor():
    from aki_b200 import longrope_attention_factor
    assert abs(longrope_attention_factor(131072, 4096) - 1.1902380714238083) < 1e-12
    assert longrope_attention_factor(4096, 4096) == 1.0


def test_shard_range_partitions():
    from aki_b200.dist import shard_range
    for n in (1, 7, 8, 64):
        for world in (1, 2, 4, 8):
            spans = [shard_range(n, r, world) for r in range(world)]
            assert spans[0][0] == 0 and spans[-1][1] == n
            assert all(spans[r][1] == spans[r + 1][0] for r in range(world - 1))
            sizes = [hi - lo for lo, hi in spans]
            assert max(sizes) - min(sizes) <= 1


def test_bench_prompt_geometry():
    """bench.py's synthetic prompt: spliced length exactly T, image spans of 128, q_end = T - 64 (config 3)."""
    sys.path.insert(0, ROOT)
    import bench
    from oracle import mma_oracle as O
    lang, am = bench.make_prompt(2, 1024, 4)
    S = O.segments_ref(lang, am, 128, 32012)
    assert S.seg.shape == (2, 1024) and (S.seq_len == 1024).all() and (S.q_end == 1024 - 64).all()
    assert int((S.seg[0] > 0).sum()) == 4 * 128 and int(S.seg[0].max()) == 4
    assert O.count_allowed(S) == int(O.expand_segments_to_4d(S).sum())


def test_bench_rejects_arguments_it_cannot_honour(monkeypatch):
    """No timed step to report, or an output dump of a path other than the attention step of this library."""
    sys.path.insert(0, ROOT)
    import bench
    for argv in (["--steps", "0"], ["--warmup", "-1"], ["--impl", "reference", "--dump-outputs", "d"],
                 ["--workload", "sft", "--dump-outputs", "d"]):
        monkeypatch.setattr(sys, "argv", ["bench.py"] + argv)
        with pytest.raises(SystemExit):
            bench.parse()
    monkeypatch.setattr(sys, "argv", ["bench.py", "--steps", "3", "--dump-outputs", "d"])
    args = bench.parse()
    assert args.steps == 3 and args.dump_outputs == "d"


def test_bench_reference_arm_prints_exactly_one_json_line():
    """Driver contract: `bench.py --impl reference` runs on the host cores only and prints ONE JSON line on stdout
    (anything native libraries write to fd 1 is diverted to stderr); other ranks of a torchrun launch print nothing."""
    import json, subprocess
    env = dict(os.environ, NCCL_DEBUG="VERSION")
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "1",
                          "--warmup", "0", "--seq", "512", "--batch", "1", "--images", "1"],
                         capture_output=True, text=True, timeout=600, env=env, cwd=ROOT)
    assert out.returncode == 0, out.stderr[-2000:]
    lines = [l for l in out.stdout.splitlines() if l.strip()]
    assert len(lines) == 1, out.stdout
    d = json.loads(lines[0])
    assert d["impl"] == "reference" and d["metric"] == "mma_attn_fwd_bwd_tflops" and d["unit"] == "TFLOP/s"
    assert d["value"] > 0 and d["cpu_baseline"]["kind"] == "port" and d["cpu_baseline"]["cores"] >= 1
    assert d["e2e"]["h2d_bytes_per_step"] == 0 and d["e2e"]["d2h_bytes_per_step"] == 0
    # the line reports what actually ran: the requested config (not a reduced sample) and the steps really timed
    assert d["steps"] == 1 and d["warmup"] == 0 and "T=512 B=1" in d["config"]["workload"]
    assert "T=512 B=1" in d["cpu_baseline"]["sample"]
    quiet = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "1",
                            "--warmup", "0"], capture_output=True, text=True, timeout=600,
                           env=dict(env, RANK="1", WORLD_SIZE="2", LOCAL_RANK="1"), cwd=ROOT)
    assert quiet.returncode == 0 and quiet.stdout.strip() == ""


def _gloo_worker(rank, world, port, q):
    import torch.distributed as dist
    os.environ["MASTER_ADDR"] = "127.0.0.1"; os.environ["MASTER_PORT"] = str(port)
    dist.init_process_group("gloo", rank=rank, world_size=world)
    from aki_b200.dist import gather_batch, max_over_ranks, shard_batch
    from oracle import mma_oracle as O
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    import helpers as Hp
    lang, am = Hp.make_prompt(5, 40, 4, 1, seed=3)
    my_lang, my_am = shard_batch([torch.from_numpy(lang), torch.from_numpy(am)], rank, world)
    # every rank builds the masks of its own samples only; no data-path collective
    S = O.segments_ref(my_lang.numpy(), my_am.numpy(), 4, Hp.MEDIA_ID, t_cap=43)
    mine = torch.from_numpy(O.expand_segments_to_4d(S))
    full = gather_batch(mine, 5)
    t = max_over_ranks(float(rank + 1), "cpu")
    if rank == 0:
        ref = torch.from_numpy(O.expand_segments_to_4d(O.segments_ref(lang, am, 4, Hp.MEDIA_ID, t_cap=43)))
        q.put((bool(torch.equal(full, ref)), t))
    dist.destroy_process_group()


def test_batch_sharding_world2_gloo():
    import torch.multiprocessing as mp
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    port = 29500 + (os.getpid() % 2000)
    procs = [ctx.Process(target=_gloo_worker, args=(r, 2, port, q)) for r in range(2)]
    for p in procs:
        p.start()
    ok, t = q.get(timeout=120)
    for p in procs:
        p.join(timeout=60)
        assert p.exitcode == 0
    assert ok and t == 2.0
