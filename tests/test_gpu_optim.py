"""-m gpu: the fused optimizer step (optim.cu, aki_b200.optim): the squared gradient norm and the AdamW update against
fp64 references and against clip_grad_norm_ + torch.optim.AdamW(fused=True), the bf16 weight copy against autocast's
cast, and AkiAdamW / use_bf16_weights in the SFT step.

u = 2^-24 is the fp32 unit roundoff; gamma(k) = k u / (1 - k u) bounds k roundings of non-negative quantities."""
import copy
import math

import numpy as np
import pytest
import torch

import helpers as Hp

pytestmark = pytest.mark.gpu
dev = "cuda"
F32, F64, BF = torch.float32, torch.float64, torch.bfloat16
U = 2.0 ** -24
TINY = 2.0 ** -149          # absolute error of one rounding into the fp32 subnormal range (<= half of it)
CHUNK = 16384               # elements per fp32 partial of the norm (optim.cu OPT_CHUNK)


def gamma(k):
    return k * U / (1 - k * U)


def _norm(grads):
    from aki_b200.optim import grad_sq_norm
    return grad_sq_norm(grads)


def _ulps(a, b):
    """Distance in fp32 ulps (ordered-integer view; NaN positions must agree)."""
    ia = a.contiguous().view(torch.int32).to(torch.int64)
    ib = b.contiguous().view(torch.int32).to(torch.int64)
    ia = torch.where(ia < 0, -(ia & 0x7FFFFFFF), ia)
    ib = torch.where(ib < 0, -(ib & 0x7FFFFFFF), ib)
    assert torch.equal(torch.isnan(a), torch.isnan(b))
    d = (ia - ib).abs()[~torch.isnan(a)]
    return int(d.max()) if d.numel() else 0


# ---- squared norm -------------------------------------------------------------------------------------------------
def _int_grads(sizes, seed):
    g = torch.Generator(device=dev).manual_seed(seed)
    return [torch.randint(-31, 32, (n,), generator=g, device=dev).to(F32) for n in sizes]


@pytest.mark.parametrize("sizes", [[1], [3], [7], [4096 + 5], [1, 3, 7, 4096 + 5, CHUNK, CHUNK + 1, 1_000_003],
                                   [0, 5, 0, 9]])
def test_norm_exact_for_integer_gradients(sizes):
    """|g| <= 31: a 16384-element partial is at most 16384 * 961 < 2^24, an exact fp32 integer; the fp64 sum of the
    partials is exact, so the single rounding to fp32 must equal the rounding of the exact integer sum."""
    gs = _int_grads(sizes, 1)
    want = sum(int((g.to(torch.int64) ** 2).sum()) for g in gs)
    got = _norm(gs)
    assert got.item() == float(np.float32(want)), (got.item(), want)


def test_norm_list_longer_than_one_launch_is_exact_and_deterministic():
    """600 entries (a launch takes 256): the partials of all launches are added in one fixed order."""
    sizes = [(i * 37) % 5000 + 1 for i in range(600)]
    gs = _int_grads(sizes, 2)
    want = sum(int((g.to(torch.int64) ** 2).sum()) for g in gs)
    a = _norm(gs)
    b = _norm(gs)
    assert a.item() == float(np.float32(want))
    assert torch.equal(a.view(torch.int32), b.view(torch.int32))


def test_norm_above_2_31_elements():
    """Five read-only entries alias one 2^29 + 3 element gradient (2.7e9 elements in all, chunk indices and offsets past
    2^31); integer values at both ends of the buffer and at scattered places keep every partial exact."""
    n = (1 << 29) + 3
    g = torch.zeros(n, dtype=F32, device=dev)
    idx = torch.tensor([0, 1, 2, CHUNK - 1, CHUNK, 123_456_789, n - 4, n - 3, n - 2, n - 1], device=dev)
    g[idx] = torch.tensor([3., -5., 7., 31., -31., 2., -9., 11., 13., -17.], device=dev)
    tail = g[4:]                                          # 16-byte aligned view: numel % 4 == 3 exercises the tail
    entries = [g, g, g, g, tail]
    want = 4 * int((g.to(torch.int64) ** 2).sum()) + int((tail.to(torch.int64) ** 2).sum())
    assert sum(e.numel() for e in entries) > 2 ** 31
    assert _norm(entries).item() == float(np.float32(want))


def test_norm_gaussian_within_summation_depth_and_repeatable():
    """Each partial passes every g^2 through at most 64 sequential FMAs of one thread, 5 warp-shuffle adds and 7 adds of
    the warp sums: 76 roundings; the fp64 sum of the partials adds < 2^-40 relative and the final fp32 rounding one
    more u.  So |got - ref| <= (gamma(76) + U + 2^-40) * sum g^2 (all terms non-negative)."""
    g = torch.Generator(device=dev).manual_seed(3)
    gs = [torch.randn(n, generator=g, device=dev) * s for n, s in
          ((1, 1.0), (3, 1e-3), (4101, 10.0), (CHUNK * 3 + 7, 1.0), (5_000_000, 0.01), (98_765, 1e3))]
    ref = sum(float((x.to(F64) ** 2).sum()) for x in gs)
    runs = [_norm(gs) for _ in range(4)]
    assert abs(runs[0].item() - ref) <= (gamma(76) + U + 2 ** -40) * ref, (runs[0].item(), ref)
    for r in runs[1:]:
        assert torch.equal(r.view(torch.int32), runs[0].view(torch.int32))


# ---- update against fp64 -----------------------------------------------------------------------------------------
def _adamw(rows, sq=None, max_norm=1.0, lr=1e-3, b1=0.9, b2=0.999, eps=1e-8, wd=0.0, step=1):
    from aki_b200 import _lib
    from aki_b200.optim import _entries
    ent = _entries(rows)
    _lib.check(_lib.lib.aki_mma_adamw_step(ent.ctypes.data, len(rows), sq.data_ptr() if sq is not None else None,
                                           max_norm, lr, b1, b2, eps, wd, step,
                                           torch.cuda.current_stream().cuda_stream), "aki_mma_adamw_step")


def _f(x):
    return float(np.float32(x))


def _ref64(p, g, m, v, c, lr, b1, b2, eps, wd, step):
    """torch.optim.AdamW's formula in fp64 on the fp32 hyperparameters, rounding only the stored m, v, p to fp32 (the
    update reads the stored m and v, as the fp32 code does).  c: the clip factor (fp64)."""
    lr, b1, b2, eps, wd = (_f(x) for x in (lr, b1, b2, eps, wd))
    g = g.to(F64) * c
    p1 = p.to(F64) * (1 - lr * wd)
    m1 = Hp.f32(b1 * m.to(F64) + (1 - b1) * g)
    v1 = Hp.f32(b2 * v.to(F64) + (1 - b2) * g * g)
    bc1, bc2 = 1 - b1 ** step, 1 - b2 ** step
    p2 = Hp.f32(p1 - lr / bc1 * m1 / (torch.sqrt(v1) / math.sqrt(bc2) + eps))
    return p2, m1, v1, (p1, g, bc1, bc2)


def _bounds(p, m, v, m1, v1, aux, c_rel, lr, b1, b2, eps, wd, step):
    """First-order bounds of the kernel's fp32 evaluation against _ref64 (+ TINY per rounding for subnormal results):
      g' = g * c: 1 rounding, plus c_rel from the clip factor's own roundings (sqrt, add, reciprocal, multiply: 4u)
      m  = fma(b1, m, fma(-b1, g', g')): 2 roundings       -> dm <= gamma(2 + 1 + c_rel/u)(|b1 m| + |(1-b1) g'|)
      v  = fma(b2, v, fma(-b2, g'g', g'g')): 3 roundings, g' error twice -> dv <= gamma(3 + 2(1 + c_rel/u))(b2 v + (1-b2) g'^2)
      p1 = p - (lr wd) p: 2 roundings                      -> dp1 <= gamma(2) |p|
      bc = 1 - powf(b, t): powf <= 4 ulp (8u relative) of b^t, 1 rounding; sqrt of bc2 halves its error, 1 rounding
      step_size = lr / bc1: 1 rounding; denom = sqrt(v)/bc2s + eps: 3 roundings + dv/2v + e(bc2s)
      upd = step_size * m / denom: 2 roundings; p = p1 - upd: 1 rounding (0.5 ulp: u |p|)
    Stored m, v of the kernel may differ from the reference's by dm, dv: the update is bounded with them."""
    lr, b1, b2, eps, wd = (_f(x) for x in (lr, b1, b2, eps, wd))
    p1, g, bc1, bc2 = aux
    k = 1 + c_rel / U
    dm = gamma(2 + k) * ((b1 * m.to(F64)).abs() + ((1 - b1) * g).abs()) + 2 * TINY
    dv = gamma(3 + 2 * k) * (b2 * v.to(F64) + (1 - b2) * g * g) + 3 * TINY
    dp1 = gamma(2) * p.to(F64).abs() + 2 * TINY
    e_bc1 = 8 * U * b1 ** step / bc1 + U
    e_bc2s = (8 * U * b2 ** step / bc2 + U) / 2 + U
    e_ss = e_bc1 + U
    den = torch.sqrt(v1) / math.sqrt(bc2) + eps
    sv = torch.sqrt(v1)
    d_sqrt = torch.where(sv > 0, torch.minimum(dv / (2 * sv), torch.sqrt(dv)), torch.sqrt(dv))   # |sqrt a - sqrt b|
    e_den = d_sqrt / math.sqrt(bc2) / den + e_bc2s + 3 * U
    upd = lr / bc1 * m1.abs() / den
    dupd = lr / bc1 * dm / den + upd * (e_ss + e_den + 2 * U) + 2 * TINY
    dp = dp1 + dupd + U * (p1.abs() + upd) + TINY
    return dp * (1 + 1e-6), dm * (1 + 1e-6), dv * (1 + 1e-6)


def _state(n, step, seed, gscale):
    g_ = torch.Generator(device=dev).manual_seed(seed)
    p = torch.randn(n, generator=g_, device=dev)
    g = torch.randn(n, generator=g_, device=dev) * gscale
    if step == 1:
        m = torch.zeros(n, device=dev)
        v = torch.zeros(n, device=dev)
    else:
        m = torch.randn(n, generator=g_, device=dev) * 1e-3
        v = torch.rand(n, generator=g_, device=dev) * 1e-6
    return p, g, m, v


def _check_vs_fp64(n, step, wd, clip, gscale, lr=1e-3, max_norm=1.0, seed=0):
    p0, g, m0, v0 = _state(n, step, seed, gscale)
    p, m, v = p0.clone(), m0.clone(), v0.clone()
    sq = None
    c, c_rel = 1.0, 0.0
    if clip is not None:
        sq = torch.tensor([clip], dtype=F32, device=dev)
        cc = max_norm / (math.sqrt(float(sq)) + _f(1e-6))
        c, c_rel = min(1.0, cc), (0.0 if cc >= 1.0 * (1 + 8 * U) else 4 * U)
    _adamw([(p, g, m, v, None)], sq=sq, max_norm=max_norm, lr=lr, wd=wd, step=step)
    p2, m1, v1, aux = _ref64(p0, g, m0, v0, c, lr, 0.9, 0.999, 1e-8, wd, step)
    dp, dm, dv = _bounds(p0, m0, v0, m1, v1, aux, c_rel, lr, 0.9, 0.999, 1e-8, wd, step)
    for name, got, ref, b in (("m", m, m1, dm), ("v", v, v1, dv), ("p", p, p2, dp)):
        fin = torch.isfinite(ref)
        assert torch.equal(got[~fin].to(F64), ref[~fin]), name           # overflow: the same inf
        err = (got.to(F64) - ref)[fin].abs()
        assert bool((err <= b[fin]).all()), (name, float((err / b[fin]).max()))
    return p, m, v


@pytest.mark.parametrize("step", [1, 10000])
@pytest.mark.parametrize("wd", [0.0, 1e-4])
@pytest.mark.parametrize("clip", [None, 0.25, 400.0, 0.0], ids=["noclip", "inactive", "active", "zero_norm"])
def test_update_against_fp64(step, wd, clip):
    """n = 4096 * 3 + 3 elements (vector path and scalar tail); clip: the squared norm handed to the kernel (0.25: factor
    1/(0.5 + 1e-6) > 1, clamped; 400: factor 0.05; 0: a zero-norm step, factor clamped to 1)."""
    _check_vs_fp64(4096 * 3 + 3, step, wd, clip, 1.0)


def test_update_zero_gradients():
    """All-zero gradients with a zero norm: m and v only decay, p moves by weight decay and the decaying moments."""
    n = 1027
    p0, _, m0, v0 = _state(n, 10000, 5, 1.0)
    g = torch.zeros(n, device=dev)
    p, m, v = p0.clone(), m0.clone(), v0.clone()
    sq = _norm([g])
    assert sq.item() == 0.0
    _adamw([(p, g, m, v, None)], sq=sq, wd=1e-4, step=10000)
    p2, m1, v1, aux = _ref64(p0, g, m0, v0, 1.0, 1e-3, 0.9, 0.999, 1e-8, 1e-4, 10000)
    dp, dm, dv = _bounds(p0, m0, v0, m1, v1, aux, 0.0, 1e-3, 0.9, 0.999, 1e-8, 1e-4, 10000)
    assert bool(((m.to(F64) - m1).abs() <= dm).all() and ((v.to(F64) - v1).abs() <= dv).all())
    assert bool(((p.to(F64) - p2).abs() <= dp).all())


@pytest.mark.parametrize("gscale", [1e-30, 1e18, 1e30])
@pytest.mark.parametrize("step", [1, 10000])
def test_update_extreme_gradients(gscale, step):
    """|g| ~ 1e-30: g^2 underflows to 0 in fp32 (the reference's stored v rounds to 0 too).  |g| ~ 1e18: g^2 near the
    top of the fp32 range.  |g| ~ 1e30: g^2 overflows, and torch's fma(-b2, g*g, g*g) is inf - inf = NaN, so v and p
    become NaN while m stays finite -- torch.optim.AdamW(fused=True) gives the same.  With clipping, the device norm
    of such gradients is 0 (factor clamped to 1) or inf (factor 0: every gradient becomes 0)."""
    n = 4099
    g_ = _state(n, step, 11, gscale)[1]
    sq = _norm([g_])
    if gscale < 1e20:
        _check_vs_fp64(n, step, 1e-4, None, gscale, seed=11)
    else:
        p0, g, m0, v0 = _state(n, step, 11, gscale)
        p, m, v = p0.clone(), m0.clone(), v0.clone()
        _adamw([(p, g, m, v, None)], wd=1e-4, step=step)
        _, m1, _, aux = _ref64(p0, g, m0, v0, 1.0, 1e-3, 0.9, 0.999, 1e-8, 1e-4, step)
        dm = gamma(3) * ((0.9 * m0.to(F64)).abs() + (_f(0.1) * aux[1]).abs())
        assert bool(((m.to(F64) - m1).abs() <= dm).all())
        assert bool(torch.isnan(v).all() and torch.isnan(p).all())
        if step == 1:
            q = torch.nn.Parameter(p0.clone())
            q.grad = g.clone()
            torch.optim.AdamW([q], lr=1e-3, weight_decay=1e-4, fused=True).step()
            assert bool(torch.isnan(q).all())
    _check_vs_fp64(n, step, 1e-4, float(sq), gscale, seed=11)


# ---- against torch -----------------------------------------------------------------------------------------------
SIZES = [1, 3, 7, 4096 + 5, 100_003]


def _pair(seed, gscale=1.0):
    g_ = torch.Generator(device=dev).manual_seed(seed)
    ps = [torch.nn.Parameter(torch.randn(n, generator=g_, device=dev)) for n in SIZES]
    qs = [torch.nn.Parameter(p.detach().clone()) for p in ps]
    return ps, qs, g_


def _set_grads(ps, qs, g_, gscale=1.0):
    for p, q in zip(ps, qs):
        p.grad = torch.randn(p.shape, generator=g_, device=dev) * gscale
        q.grad = p.grad.clone()


@pytest.mark.parametrize("max_norm", [None, 1.0, 1e6], ids=["noclip", "active", "inactive"])
def test_update_against_torch_fused_adamw(max_norm):
    """Three steps against clip_grad_norm_ + torch.optim.AdamW(fused=True) on the same inputs: m and v within 1 ulp,
    p within 2 ulp.  The only difference is the norm's summation order (a last-bit difference of the clip factor)."""
    from aki_b200 import AkiAdamW
    ps, qs, g_ = _pair(0)
    a = AkiAdamW(ps, lr=1e-3, weight_decay=1e-4, max_grad_norm=max_norm)
    t = torch.optim.AdamW(qs, lr=1e-3, weight_decay=1e-4, fused=True)
    for _ in range(3):
        _set_grads(ps, qs, g_)
        a.step()
        if max_norm is not None:
            tn = torch.nn.utils.clip_grad_norm_(qs, max_norm)
            assert abs(a.last_grad_norm.item() - tn.item()) <= 4 * U * tn.item()
        t.step()
        for p, q in zip(ps, qs):
            sa, st = a.state[p], t.state[q]
            assert _ulps(sa["exp_avg"], st["exp_avg"]) <= 1
            assert _ulps(sa["exp_avg_sq"], st["exp_avg_sq"]) <= 1
            assert _ulps(p.detach(), q.detach()) <= 2


@pytest.mark.parametrize("bad", [float("nan"), float("inf")])
def test_non_finite_gradients_as_torch(bad):
    """A NaN gradient makes the norm NaN and every parameter NaN; an inf gradient makes the norm inf, the clip factor 0,
    that element NaN (inf * 0) and the others zero gradients -- as clip_grad_norm_ + AdamW produce them."""
    from aki_b200 import AkiAdamW
    ps, qs, g_ = _pair(1)
    a = AkiAdamW(ps, lr=1e-3, weight_decay=1e-4, max_grad_norm=1.0)
    t = torch.optim.AdamW(qs, lr=1e-3, weight_decay=1e-4, fused=True)
    _set_grads(ps, qs, g_)
    ps[3].grad[17] = bad
    qs[3].grad[17] = bad
    a.step()
    torch.nn.utils.clip_grad_norm_(qs, 1.0)
    t.step()
    if bad != bad:
        assert all(bool(torch.isnan(p).all()) for p in ps)
    for p, q in zip(ps, qs):
        assert _ulps(p.detach(), q.detach()) <= 2


# ---- the bf16 copy ----------------------------------------------------------------------------------------------
def test_bf16_copy_bits_for_every_value_class():
    """lr = 0 leaves p unchanged (p - 0 * m / denom; a NaN comes out as the canonical NaN), so the copy must be bf16(p)
    for crafted p: rounding ties to even and odd, values next to ties, values that round to +-inf, the largest finite bf16, subnormals, zeros, inf, NaN."""
    bits = [0x3F808000, 0x3F818000, 0x3F808001, 0x3F807FFF, 0xBF808000, 0xBF818000,       # ties, near ties
            0x7F7F8000, 0x7F7FFFFF, 0xFF7F8000, 0x7F7F7FFF, 0x7F7F0000,                     # -> inf, largest finite
            0x00000001, 0x00008000, 0x00018000, 0x007FFFFF, 0x80008000, 0x00800000,         # subnormals, min normal
            0x00000000, 0x80000000, 0x7F800000, 0xFF800000, 0x7FC00000, 0x7F800001, 0xFFC12345]
    n = len(bits) * 11 + 3
    x = torch.tensor((bits * 12)[:n], dtype=torch.int64).to(torch.int32).view(F32).to(dev)
    p = x.clone()
    g = torch.zeros_like(p)
    m, v = torch.zeros_like(p), torch.zeros_like(p)
    w16 = torch.full((n,), 7.0, dtype=BF, device=dev)
    _adamw([(p, g, m, v, w16)], lr=0.0, step=1)
    nan = torch.isnan(x)
    assert torch.equal(torch.isnan(p), nan)            # arithmetic on a NaN gives the canonical NaN, as in torch
    assert torch.equal(p[~nan].view(torch.int32), x[~nan].view(torch.int32))
    assert torch.equal(w16.view(torch.int16), p.to(BF).view(torch.int16))
    assert torch.equal(w16[~nan].view(torch.int16), x[~nan].to(BF).view(torch.int16))


def test_bf16_copy_after_each_step():
    from aki_b200 import AkiAdamW
    ps, _, g_ = _pair(4)
    a = AkiAdamW(ps, lr=1e-2, weight_decay=1e-4, max_grad_norm=1.0)
    copies = {p: torch.zeros(p.shape, dtype=BF, device=dev) for p in ps}
    a._bf16.update(copies)
    for _ in range(3):
        for p in ps:
            p.grad = torch.randn(p.shape, generator=g_, device=dev)
        a.step()
        for p in ps:
            assert torch.equal(copies[p].view(torch.int16), p.detach().to(BF).view(torch.int16))


# ---- optimizer behaviour ----------------------------------------------------------------------------------------
def test_lr_scheduler_is_followed():
    """LambdaLR changes lr every step (0 on the second): AkiAdamW follows it step by step as torch's AdamW does."""
    from aki_b200 import AkiAdamW
    ps, qs, g_ = _pair(5)
    a = AkiAdamW(ps, lr=1e-2, weight_decay=1e-4)
    t = torch.optim.AdamW(qs, lr=1e-2, weight_decay=1e-4, fused=True)
    f = [1.0, 0.0, 0.3, 0.05].__getitem__
    sa, st = torch.optim.lr_scheduler.LambdaLR(a, f), torch.optim.lr_scheduler.LambdaLR(t, f)
    for i in range(3):
        _set_grads(ps, qs, g_)
        before = [p.detach().clone() for p in ps]
        a.step(); t.step()
        if i == 1:
            assert all(torch.equal(p, b) for p, b in zip(ps, before))
        for p, q in zip(ps, qs):
            assert _ulps(p.detach(), q.detach()) <= 2
        sa.step(); st.step()
        assert a.param_groups[0]["lr"] == t.param_groups[0]["lr"]


@pytest.mark.parametrize("direction", ["aki_to_torch", "torch_to_aki"])
def test_state_dict_round_trips_with_torch_adamw(direction):
    from aki_b200 import AkiAdamW
    ps, qs, g_ = _pair(6)
    first = AkiAdamW(ps, lr=1e-3, weight_decay=1e-4) if direction == "aki_to_torch" else \
        torch.optim.AdamW(ps, lr=1e-3, weight_decay=1e-4, fused=True)
    for _ in range(2):
        for p in ps:
            p.grad = torch.randn(p.shape, generator=g_, device=dev)
        first.step()
    for p, q in zip(ps, qs):
        q.data.copy_(p.data)
    second = torch.optim.AdamW(qs, lr=1e-3, weight_decay=1e-4, fused=True) if direction == "aki_to_torch" else \
        AkiAdamW(qs, lr=1e-3, weight_decay=1e-4)
    second.load_state_dict(copy.deepcopy(first.state_dict()))   # a checkpoint: no tensor shared with `first`
    assert set(second.state_dict()["state"][0]) == {"step", "exp_avg", "exp_avg_sq"}
    assert float(second.state_dict()["state"][0]["step"]) == 2.0
    _set_grads(ps, qs, g_)
    first.step(); second.step()
    for p, q in zip(ps, qs):
        assert _ulps(p.detach(), q.detach()) <= 2
        assert _ulps(first.state[p]["exp_avg"], second.state[q]["exp_avg"]) <= 1
        assert float(second.state[q]["step"]) == 3.0


def test_step_does_not_synchronise():
    from aki_b200 import AkiAdamW
    ps, _, g_ = _pair(7)
    a = AkiAdamW(ps, lr=1e-3, max_grad_norm=1.0)
    a._bf16.update({p: torch.empty(p.shape, dtype=BF, device=dev) for p in ps})
    for _ in range(2):
        for p in ps:
            p.grad = torch.randn(p.shape, generator=g_, device=dev)
        torch.cuda.synchronize()
        torch.cuda.set_sync_debug_mode("error")
        try:
            a.step()
        finally:
            torch.cuda.set_sync_debug_mode("default")
    assert math.isfinite(a.last_grad_norm.item())


# ---- the SFT step ------------------------------------------------------------------------------------------------
@pytest.fixture
def det_attention_bwd(monkeypatch):
    """The tcgen05 attention backward adds dQ partials in L2 in a varying order (last-bit differences from run to run);
    the SIMT verification backward is deterministic, so bit-identity of two SFT steps tests the weight path alone."""
    from aki_b200 import ops
    orig = ops.attn_bwd_raw
    monkeypatch.setattr(ops, "attn_bwd_raw", lambda *a, **k: orig(*a, **{**k, "simt": True}))


def _sft_model(seed=1):
    from aki_b200 import ops
    from aki_b200.model import AkiPhi3SFT, phi35_mini_config
    model = AkiPhi3SFT(phi35_mini_config(num_layers=2), device=dev, seed=seed)
    B, L, N = 2, 120, 48
    lang, am = Hp.make_prompt(B, L, N, 1, pad_right=17)
    segs = ops.build_segments(torch.from_numpy(lang).to(dev), torch.from_numpy(am).to(dev), N, Hp.MEDIA_ID)
    torch.manual_seed(2)
    emb = torch.randn(B, segs.T, 3072, device=dev) * 0.05
    labels = torch.randint(0, 32000, (B, segs.T), device=dev)
    labels[:, :40] = -100
    return model, (emb, segs, labels)


def _loss_grads(model, batch):
    model.zero_grad(set_to_none=True)
    loss = model(*batch)
    loss.backward()
    return loss.detach().clone(), {n: p.grad.clone() for n, p in model.named_parameters() if p.grad is not None}


def _assert_bits(a, b):
    (la, ga), (lb, gb) = a, b
    assert torch.equal(la.view(torch.int32), lb.view(torch.int32)), (la, lb)
    assert ga.keys() == gb.keys() and len(ga) > 10
    for n in ga:
        assert torch.equal(ga[n].view(torch.int32), gb[n].view(torch.int32)), n


def test_sft_step1_bit_identical_to_autocast(det_attention_bwd):
    """Fused layers (as test_sft_step_with_fused_layer_kernels_matches_the_hf_layer_objects builds them): loss and every
    parameter gradient with the bf16 copies equal plain autocast bit for bit, and exactly the five Linears of each layer
    plus lm_head read a copy."""
    from aki_b200 import AkiAdamW, use_bf16_weights
    model, batch = _sft_model()
    ref = _loss_grads(model, batch)
    keys = set(model.state_dict())
    opt = AkiAdamW(model.parameters(), lr=1e-4, weight_decay=1e-4, max_grad_norm=1.0)
    assert use_bf16_weights(model, opt) == 2 * 4 + 1
    names = {n for n, m in model.named_modules() if hasattr(m, "_aki_weight_bf16")}
    assert names == {f"lm.model.layers.{i}.{s}" for i in range(2) for s in
                     ("self_attn.qkv_proj", "self_attn.o_proj", "mlp.gate_up_proj", "mlp.down_proj")} | {"lm.lm_head"}
    assert set(model.state_dict()) == keys
    _assert_bits(_loss_grads(model, batch), ref)


def test_sft_later_steps_and_trajectory(det_attention_bwd):
    """After 3 AkiAdamW steps the copies the kernel wrote give bit-identical outputs to plain autocast on the same
    masters.  Then a 5-step trajectory with AkiAdamW(max_grad_norm=1.0) + copies against clip_grad_norm_ +
    AdamW(fused=True) under plain autocast.  The optimizers differ only in last bits per step (the norm's summation
    order), but a last-bit change of a master can flip the rounding of its bf16 copy (a 2^-8 relative change of that
    weight in the next forward), and a random-init model fitting one batch at lr 1e-4 (loss 11 -> 1e-4 in 5 steps)
    amplifies that.  Stated tolerance: losses within 1e-2 relative; per element |dp| <= 5 * 2 * 3.2 lr (twice the
    largest Adam step lr (1 - b1) / sqrt(1 - b2) < 3.2 lr, per step); the parameter difference within 5 % of the
    distance travelled, per tensor."""
    from aki_b200 import AkiAdamW, unuse_bf16_weights, use_bf16_weights
    model, batch = _sft_model()
    twin, _ = _sft_model()
    p0 = {n: p.detach().clone() for n, p in model.named_parameters()}
    lr = 1e-4
    opt = AkiAdamW(model.parameters(), lr=lr, weight_decay=1e-4, max_grad_norm=1.0)
    topt = torch.optim.AdamW(twin.parameters(), lr=lr, weight_decay=1e-4, fused=True)
    use_bf16_weights(model, opt)
    la, lt = [], []
    for i in range(5):
        la.append(_loss_grads(model, batch)[0].item())
        opt.step()
        lt.append(_loss_grads(twin, batch)[0].item())
        torch.nn.utils.clip_grad_norm_(twin.parameters(), 1.0)
        topt.step()
        if i == 2:
            with_copies = _loss_grads(model, batch)
            unuse_bf16_weights(model)
            plain = _loss_grads(model, batch)
            _assert_bits(with_copies, plain)
            use_bf16_weights(model, opt)
    for a, b in zip(la, lt):
        assert abs(a - b) <= 1e-2 * abs(b), (la, lt)
    tw = dict(twin.named_parameters())
    for n, p in model.named_parameters():
        d = (p.detach() - tw[n].detach()).abs()
        assert float(d.max()) <= 5 * 2 * 3.2 * lr, (n, float(d.max()))
        moved = (tw[n].detach() - p0[n]).norm()
        assert float(d.norm()) <= 0.05 * float(moved) + 1e-12, (n, float(d.norm()), float(moved))


def test_model_load_state_dict_refreshes_the_copy(det_attention_bwd):
    from aki_b200 import AkiAdamW, unuse_bf16_weights, use_bf16_weights
    model, batch = _sft_model()
    other, _ = _sft_model(seed=5)
    opt = AkiAdamW(model.parameters(), lr=1e-4)
    use_bf16_weights(model, opt)
    _loss_grads(model, batch)                                   # copies written from the seed-1 masters
    model.load_state_dict(other.state_dict())
    with_copies = _loss_grads(model, batch)
    unuse_bf16_weights(model)
    _assert_bits(with_copies, _loss_grads(model, batch))


def test_unuse_restores_the_original_forwards():
    from aki_b200 import AkiAdamW, unuse_bf16_weights, use_bf16_weights
    model, _ = _sft_model()
    before = {n: m.forward for n, m in model.named_modules() if isinstance(m, torch.nn.Linear)}
    opt = AkiAdamW(model.parameters(), lr=1e-4)
    n = use_bf16_weights(model, opt)
    assert use_bf16_weights(model, opt) == 0                    # idempotent
    assert len(opt._bf16) == n
    assert unuse_bf16_weights(model) == n
    assert len(opt._bf16) == 0
    for name, m in model.named_modules():
        assert not any(a.startswith("_aki_bf16") or a == "_aki_weight_bf16" for a in vars(m))
        if name in before:
            assert m.forward == before[name]
