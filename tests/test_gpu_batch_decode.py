"""-m gpu: aki_mma_batch_linear (batch_linear.cu, 9 - 64 tokens) against fp64 references that round where the kernel
rounds, its determinism, and the fused decode step of AkiPhi3Runner at batches of 9 - 64 sequences.

The references follow tests/test_gpu_layer_numerics.py (skinny-linear section): integer operands make every partial sum
an exact fp32 integer, so modes 0 / 1 must be bit-exact and mode 2 is tie-aware (helpers.accept_branches) with its flip
count bounded.  N is chosen on both sides of every boundary of the dispatch rule, which aki_mma_batch_linear_split reports
(it depends on how many clusters of each size the device holds at once)."""
import ctypes as C
import math

import pytest
import torch

import helpers as Hp

pytestmark = pytest.mark.gpu
dev = "cuda"
U = Hp.U32
BF, F64 = torch.bfloat16, torch.float64
NAN = float("nan")
HIGHER_ORDER = 2.0 ** -30
KS = [1024, 3072, 8192, 12288]
BS = [9, 16, 17, 33, 48, 64]


def _lib():
    from aki_b200._lib import lib
    return lib


def _ops():
    from aki_b200 import ops
    return ops


def _split(B, N, K, mode):
    s = _lib().aki_mma_batch_linear_split(B, N, K, mode)
    assert 1 <= s <= 8, s
    return s


def _boundary_ns(B, K, mode):
    """N on both sides of every change of the split as the row-tile count grows: 128 t (the last tile of t still full)
    and 128 t + 16 (one more, partial tile), up to one tile past the SM count."""
    sms = torch.cuda.get_device_properties(0).multi_processor_count
    splits = [_split(B, 128 * t, K, mode) for t in range(1, sms + 2)]
    ns = {16}
    for t in range(1, sms + 1):
        if splits[t - 1] != splits[t]:
            ns |= {128 * t, 128 * t + 16}
    return sorted(ns), set(splits)


def _weights(N, K, mode, g):
    """Integer weights in [-3, 3]; in the SwiGLU mode the gate rows hold four +-1 entries each (|gate| <= 12)."""
    w = torch.randint(-3, 4, (2 * N if mode == 2 else N, K), generator=g, device=dev, dtype=torch.int32).to(BF)
    if mode == 2:
        gate = torch.zeros(N, K, device=dev)
        idx = torch.randint(0, K, (N, 4), generator=g, device=dev)
        sgn = torch.randint(0, 2, (N, 4), generator=g, device=dev).float() * 2 - 1
        w[:N] = gate.scatter_add_(1, idx, sgn).to(BF)
    return w


def _strided_x(vals):
    B, K = vals.shape
    buf = torch.full((B, K + 64), NAN, dtype=BF, device=dev)
    buf[:, 32:32 + K] = vals
    return buf[:, 32:32 + K]


def _sentinel_intact(buf, inner):
    m = torch.ones_like(buf, dtype=torch.bool)
    m[inner] = False
    return bool(torch.isnan(buf[m].float()).all())


def _run(x, w, mode, N, rms=None, eps=0.0, res=None):
    """One ops.skinny_linear call (B >= 9: aki_mma_batch_linear) into a (B, N) view of stride N + 8 inside a NaN
    sentinel, which must stay intact."""
    B = x.shape[0]
    buf = torch.full((B + 2, N + 8), NAN, dtype=BF, device=dev)
    out = buf[1:B + 1, :N]
    _ops().skinny_linear(x, w, rms, eps, residual=res, swiglu=mode == 2, out=out)
    torch.cuda.synchronize()
    assert _sentinel_intact(buf, (slice(1, B + 1), slice(0, N))), "batch_linear wrote outside its output rows"
    return out


def _run_lib(x, w, mode, N, rms=None, eps=0.0, res=None):
    """Direct aki_mma_batch_linear call (any B in 1..64, also B <= 8)."""
    B, K = x.shape
    out = torch.empty(B, N, dtype=BF, device=dev)
    p = lambda t: None if t is None else C.c_void_p(t.data_ptr())
    rc = _lib().aki_mma_batch_linear(p(x), x.stride(0), p(w), p(rms), C.c_float(eps), p(res),
                                     res.stride(0) if res is not None else 0, p(out), out.stride(0), B, N, K, mode,
                                     C.c_void_p(torch.cuda.current_stream().cuda_stream))
    assert rc == 0, rc
    torch.cuda.synchronize()
    return out


def _check_flips(what, flips, v64, eps_rel):
    n, bound = int(flips.sum()), Hp.flip_bound(v64, eps_rel)
    print(f"{what}: {n} accepted flips of {flips.numel()} (bound {bound})")
    assert n <= bound, (what, n, bound)


def _exact_check(out, x64, w, mode, N, res64=None, what=""):
    """s = x @ w.T is an integer below 2^17, exact in fp32 in any order (assumes the tensor core's fp32 accumulation is
    exact on integer partial sums below 2^24).  mode 0: bf16(s); mode 1: bf16(fp32(bf16(s) + res)); mode 2:
    bf16(bf16(up) * bf16(gq / (1 + __expf(-gq)))) with __expf 2 + floor(|1.16 x|) ulp, 1 + e and the division u each."""
    s = x64 @ w.to(F64).t()
    if mode == 2:
        gq, uq = Hp.bf16_rne(s[:, :N]), Hp.bf16_rne(s[:, N:])
        assert float(gq.abs().max()) <= 12
        v = gq / (1 + torch.exp(-gq))
        eps = (2 + torch.floor(1.16 * gq.abs())) * 2 * U + 2 * U + HIGHER_ORDER
        a_ref, a_alt, band = Hp.bf16_branches(v, eps)
        flips = Hp.accept_branches(out, Hp.bf16_rne(uq * a_ref), Hp.bf16_rne(uq * a_alt), band, what)
        _check_flips(what, flips, v, eps)
        return
    ref = Hp.bf16_rne(s) if mode == 0 else Hp.bf16_rne(Hp.f32(Hp.bf16_rne(s) + res64))
    assert torch.equal(out.to(F64), ref), (what, int((out.to(F64) != ref).sum()))


# ------------------------------------------------------------------------------------------------ exact integers
@pytest.mark.parametrize("mode", [0, 1, 2])
@pytest.mark.parametrize("K", KS)
def test_batch_linear_exact_integers(K, mode):
    """Integer x, w in [-3, 3]: bit-exact (tie-aware in mode 2) against the fp64 GEMM at N on both sides of every
    split boundary (of every token padding) and N = 32064 (a partial last tile), B cycling through 9, 16, 17, 33, 48,
    64; strided x, residual of odd row stride N + 3, output view inside a NaN sentinel.  Every split the rule can pick
    for this K and mode runs at least once."""
    g = torch.Generator(device=dev).manual_seed(K * 7 + mode)
    ns, picks = set(), set()
    for pad_b in (16, 32, 48, 64):
        n_, p_ = _boundary_ns(pad_b, K, mode)
        ns |= set(n_)
        picks |= p_
    seen = set()
    for i, N in enumerate(sorted(ns) + [32064]):
        B = BS[i % len(BS)]
        s = _split(B, N, K, mode)
        seen.add(s)
        what = f"batch mode={mode} N={N} K={K} B={B} split={s}"
        print(what)
        w = _weights(N, K, mode, g)
        xv = torch.randint(-3, 4, (B, K), generator=g, device=dev, dtype=torch.int32).to(BF)
        res = (torch.randn(B, N + 3, generator=g, device=dev) * 64).to(BF)[:, :N] if mode == 1 else None
        out = _run(_strided_x(xv), w, mode, N, res=res)
        _exact_check(out, xv.to(F64), w, mode, N, res.to(F64) if mode == 1 else None, what)
        del w
    print(f"splits picked {sorted(picks)}, run {sorted(seen)}")
    assert seen >= picks, (picks, seen)


# ------------------------------------------------------------------------------------------------ RMSNorm prologue
@pytest.mark.parametrize("mode", [0, 1, 2])
@pytest.mark.parametrize("B,N,K", [(9, 9216, 3072), (33, 3072, 8192), (64, 1024, 3072), (48, 32064, 3072)])
def test_batch_linear_norm_prologue_exact(B, N, K, mode):
    """x in {-1, +1}, integer gamma, eps = 0: mean square 1, rsqrtf(1) = 1, every normalised element is +-gamma, so the
    output is bit-exact to the integer GEMM on gamma * x."""
    g = torch.Generator(device=dev).manual_seed(N + K * 3 + mode + B)
    w = _weights(N, K, mode, g)
    xv = (torch.randint(0, 2, (B, K), generator=g, device=dev) * 2 - 1).to(BF)
    gamma = torch.randint(-3, 4, (K,), generator=g, device=dev, dtype=torch.int32).to(BF)
    if mode == 2:
        gamma = gamma.clamp(-1, 1)
    res = (torch.randn(B, N + 3, generator=g, device=dev) * 64).to(BF)[:, :N] if mode == 1 else None
    what = f"batch prologue-exact mode={mode} N={N} K={K} B={B} split={_split(B, N, K, mode)}"
    print(what)
    out = _run(_strided_x(xv), w, mode, N, rms=gamma, eps=0.0, res=res)
    _exact_check(out, xv.to(F64) * gamma.to(F64), w, mode, N, res.to(F64) if mode == 1 else None, what)


def _depth(B, N, K, mode):
    """Roundings a square passes through in the kernel's sum: each of the 4 threads of a token adds 8 squares per
    16-byte piece by FMA over at most ceil(ceil(nch / S) * 8 / 4) pieces, 2 xor-shuffle adds, then S rank partials."""
    S = _split(B, N, K, mode)
    pieces = math.ceil(math.ceil(K // 64 / S) * 8 / 4)
    return 8 * pieces + 2 + S


@pytest.mark.parametrize("B,N,K", [(9, 9216, 3072), (40, 3072, 8192), (64, 3072, 3072), (17, 32064, 3072),
                                   (64, 2048, 12288)])
def test_batch_linear_norm_prologue_bound(B, N, K):
    """Gaussian x through the RMSNorm prologue against an fp64 GEMM of the reference's normalised operand, within
        ulp_bf16(|ref| + E) + E,   E = sum_k |w_k| |xg_alt_k - xg_ref_k| [k in band] + K u sum_k |w_k xg_k|
    with the prologue's branches from the reasoning of test_gpu_layer_numerics._norm_prologue_ref at this kernel's
    summation depth (_depth)."""
    g = torch.Generator(device=dev).manual_seed(N + K + B)
    w = (torch.randn(N, K, generator=g, device=dev) * K ** -0.5).to(BF)
    xv = torch.randn(B, K, generator=g, device=dev).to(BF)
    gamma = (1 + 0.1 * torch.randn(K, generator=g, device=dev)).to(BF)
    depth = _depth(B, N, K, 0)
    x64 = xv.to(F64)
    r = 1 / torch.sqrt((x64 * x64).sum(-1, keepdim=True) / K + Hp.f32(torch.tensor(1e-5, dtype=F64)))
    eps_xn = (depth + 2) * U / 2 + 4 * U + U + HIGHER_ORDER
    v = x64 * r
    xn_ref, xn_alt, band = Hp.bf16_branches(v, eps_xn)
    g64 = gamma.to(F64)
    xg_ref, xg_alt = Hp.bf16_rne(g64 * xn_ref), Hp.bf16_rne(g64 * xn_alt)
    what = f"batch prologue-bound N={N} K={K} B={B} depth={depth}"
    out = _run(_strided_x(xv), w, 0, N, rms=gamma, eps=1e-5).to(F64)
    w64 = w.to(F64)
    ref = xg_ref @ w64.t()
    E = ((xg_alt - xg_ref).abs() * band) @ w64.abs().t() + K * U * (xg_ref.abs() @ w64.abs().t())
    err = (out - ref).abs()
    lim = Hp.ulp_bf16(ref.abs() + E) + E
    print(f"{what}: prologue in-band {int(band.sum())} (flip bound {Hp.flip_bound(v, eps_xn)}), "
          f"max err / bound {float((err / lim).max()):.3f}")
    assert bool((err <= lim).all()), (what, float((err / lim).max()))
    assert int(band.sum()) <= Hp.flip_bound(v, eps_xn)


# ------------------------------------------------------------------------------------------------ determinism
@pytest.mark.parametrize("mode", [0, 1, 2])
def test_batch_linear_determinism(mode):
    """Two calls are bit-identical; for each token padding, rows of a B-token call equal the same rows of a call with a
    different B of the same padding.  Whether rows also match across paddings (and against skinny_linear at B <= 8) is
    reported, not asserted."""
    N, K = 3072, 8192
    g = torch.Generator(device=dev).manual_seed(11 + mode)
    w = (torch.randn(2 * N if mode == 2 else N, K, generator=g, device=dev) * K ** -0.5).to(BF)
    xv = torch.randn(64, K, generator=g, device=dev).to(BF)
    gamma = (1 + 0.1 * torch.randn(K, generator=g, device=dev)).to(BF)
    res = (torch.randn(64, N, generator=g, device=dev) * 4).to(BF) if mode == 1 else None
    rms = None if mode == 1 else gamma

    def call(B):
        return _run_lib(xv[:B], w, mode, N, rms=rms, eps=1e-5, res=res[:B] if res is not None else None)

    full = {}
    for lo, hi in [(9, 16), (17, 32), (33, 48), (49, 64)]:
        a, b = call(hi), call(hi)
        assert torch.equal(a, b), (mode, hi)
        c = call(lo)
        assert torch.equal(c, a[:lo]), (mode, lo, hi)
        full[hi] = a
    cross = {hi: torch.equal(full[hi][:9], full[16][:9]) for hi in (32, 48, 64)}
    sk = _ops().skinny_linear(xv[:8], w, rms, 1e-5, residual=res[:8] if res is not None else None, swiglu=mode == 2)
    bl8 = call(8)
    print(f"mode={mode}: rows 0-8 equal across paddings 16 / 32 / 48 / 64: {cross}; batch_linear B=8 == "
          f"skinny_linear B=8: {torch.equal(sk, bl8)} (max |diff| {float((sk.float() - bl8.float()).abs().max()):.3e})")


# ------------------------------------------------------------------------------------------------ model level
@pytest.fixture(scope="module")
def runner():
    from aki_b200.model import AkiPhi3Runner, phi35_mini_config
    return AkiPhi3Runner(phi35_mini_config(num_layers=2), device=torch.device("cuda", 0), seed=0)


@pytest.mark.parametrize("B", [9, 32, 64])
def test_fused_decode_step_at_batch(runner, B):
    """2-layer runner at B sequences: decode_step_fused (aki_mma_batch_linear for every projection and the lm_head)
    against decode_step through HF's layers for 5 steps, within the tolerance of test_fused_decode_step_matches_the_
    hf_layer_path; decode_step_graphed(fused=True) gives the eager fused tokens and bit-identical K/V cache rows."""
    T, n_new = 50, 5
    emb = (torch.randn(B, T, 3072, generator=torch.Generator().manual_seed(B)) * 0.05).to(BF).to(dev)
    caches = [runner.new_cache(B, T + n_new + 3) for _ in range(3)]
    toks = [runner.prefill(emb, None, c)[:, -1].argmax(-1, keepdim=True) for c in caches]
    tok = toks[0]
    for step in range(n_new):
        ref = runner.decode_step(tok, caches[0]).float()
        got = runner.decode_step_fused(tok, caches[1]).float()
        scale = float(ref.abs().max())
        assert float((got - ref).abs().max()) < 3e-2 * max(scale, 1.0), (B, step, float((got - ref).abs().max()), scale)
        nxt_graph = runner.decode_step_graphed(tok, caches[2], fused=True)
        assert torch.equal(nxt_graph, got[:, -1].argmax(-1, keepdim=True)), (B, step)
        tok = got[:, -1].argmax(-1, keepdim=True)
    n = T + n_new
    for l in range(2):
        assert torch.equal(caches[1].k[l][:, :, :n], caches[2].k[l][:, :, :n]), (B, l)
        assert torch.equal(caches[1].v[l][:, :, :n], caches[2].v[l][:, :, :n]), (B, l)
        a_, b_ = caches[0].k[l][:, :, :n].float(), caches[1].k[l][:, :, :n].float()
        assert float((a_ - b_).abs().max()) < 3e-2 * max(1.0, float(a_.abs().max()))


def test_graphed_step_above_64_keeps_the_hf_layers(runner):
    """B = 65 is past the fused kernels' range: decode_step_graphed(fused=True) runs HF's layers, the same tokens as
    fused=False, and skinny_linear refuses 65 tokens."""
    B, T, n_new = 65, 20, 3
    emb = (torch.randn(B, T, 3072, generator=torch.Generator().manual_seed(65)) * 0.05).to(BF).to(dev)
    ca, cb = runner.new_cache(B, T + n_new + 3), runner.new_cache(B, T + n_new + 3)
    ta = runner.prefill(emb, None, ca)[:, -1].argmax(-1, keepdim=True)
    tb = runner.prefill(emb, None, cb)[:, -1].argmax(-1, keepdim=True)
    for _ in range(n_new):
        ta = runner.decode_step_graphed(ta, ca, fused=True)
        tb = runner.decode_step_graphed(tb, cb, fused=False)
        assert torch.equal(ta, tb)
    with pytest.raises(ValueError):
        _ops().skinny_linear(torch.zeros(65, 1024, dtype=BF, device=dev), torch.zeros(16, 1024, dtype=BF, device=dev))
