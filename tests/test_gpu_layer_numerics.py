"""-m gpu: the decoder-layer kernels around attention (skinny_linear.cu, layer_elementwise.cu, rope.cu) element by
element against fp64 references that round where the kernels round.

Where a kernel's value is exact before its last rounding (integer GEMMs, bf16 x bf16 products, fp32 adds of bf16 values)
the output must be bit-exact.  Where it is not (rsqrtf, expf, __expf, sincosf, reassociated fp32 sums), the comparison
is tie-aware (helpers.accept_bf16): bit-exact to the correctly rounded fp64 value except within eps_rel |v| (+ eps_abs)
of a bf16 rounding midpoint, where either neighbour is accepted (and where a cancellation makes eps_abs span several
bf16 ulps, every value of the rounded interval [bf16(v - tol), bf16(v + tol)]); eps comes from the CUDA math accuracy table
(rsqrtf, expf: 2 ulp; __expf: 2 + floor(|1.16 x|) ulp; sincosf: 2 ulp; logf: 1 ulp) plus first-order rounding terms
derived next to each kernel line they model.  Where an accepted flip feeds a later rounding, both branches are
carried.  Every such check prints its flip count and asserts it below helpers.flip_bound.

u = 2^-24 below is the fp32 unit roundoff; an fp32 ulp is at most 2u relative."""
import ctypes as C
import math

import pytest
import torch

import helpers as Hp

pytestmark = pytest.mark.gpu
dev = "cuda"
U = Hp.U32
BF, F32, F64 = torch.bfloat16, torch.float32, torch.float64
NAN = float("nan")
ERR_UNSUPPORTED = -3
HIGHER_ORDER = 2.0 ** -30         # covers the second-order products of the first-order bounds below


def _lib():
    from aki_b200._lib import lib
    return lib


def _ops():
    from aki_b200 import ops
    return ops


def _p(t):
    return None if t is None else C.c_void_p(t.data_ptr())


def _check_flips(what, flips, v64, eps_rel, eps_abs=0.0):
    n, bound = int(flips.sum()), Hp.flip_bound(v64, eps_rel, eps_abs)
    print(f"{what}: {n} accepted flips of {flips.numel()} (bound {bound})")
    assert n <= bound, (what, n, bound)


def _sentinel_intact(buf, inner):
    """Every element of buf outside the view `inner` (a (rows, cols) slice of it) is still NaN."""
    m = torch.ones_like(buf, dtype=torch.bool)
    m[inner] = False
    return bool(torch.isnan(buf[m].float()).all())


# ------------------------------------------------------------------------------------------------ skinny linear
def _per(N, sms):
    """Row tiles per CTA, the dispatch rule of aki_mma_skinny_linear (skinny_linear.cu)."""
    tiles = N // 16
    return 1 if tiles <= sms else 2 if tiles <= 2 * sms else 4 if tiles <= 4 * sms else 16


N_TAGS = {"16": lambda s: 16, "16sms": lambda s: 16 * s, "16sms+16": lambda s: 16 * s + 16, "32sms": lambda s: 32 * s,
          "32sms+16": lambda s: 32 * s + 16, "64sms": lambda s: 64 * s, "64sms+16": lambda s: 64 * s + 16,
          "32064": lambda s: 32064}
# each dispatch width twice, at both sides of its boundaries, and at two K values; K = 1024 with per = 1 is one
# 64-element K slice per warp (a single ring entry), 12288 is the largest K whose x fits the shared-memory limit
SK_SHAPES = [("16", 1, 12288), ("16sms", 1, 1024), ("16sms+16", 2, 3072), ("32sms", 2, 8192), ("32sms+16", 4, 1024),
             ("64sms", 4, 3072), ("64sms+16", 16, 8192), ("32064", 16, 3072)]


def _n_of(tag, per):
    sms = torch.cuda.get_device_properties(0).multi_processor_count
    N = N_TAGS[tag](sms)
    assert _per(N, sms) == per, (tag, N, sms)
    return N


def _skinny_weights(N, K, mode, g):
    """Integer weights in [-3, 3] (exact in bf16).  In the SwiGLU mode the gate rows hold four +-1 entries each, so
    with |x| <= 3 every gate sum lies in [-12, 12], where silu is not trivial; the up rows stay dense."""
    w = torch.randint(-3, 4, (2 * N if mode == 2 else N, K), generator=g, device=dev, dtype=torch.int32).to(BF)
    if mode == 2:
        gate = torch.zeros(N, K, device=dev)
        idx = torch.randint(0, K, (N, 4), generator=g, device=dev)
        sgn = torch.randint(0, 2, (N, 4), generator=g, device=dev).float() * 2 - 1
        w[:N] = gate.scatter_add_(1, idx, sgn).to(BF)
    return w


def _strided_x(vals):
    """vals (B, K) placed as a column slice of a NaN-filled (B, K + 64) buffer: x_stride = K + 64."""
    B, K = vals.shape
    buf = torch.full((B, K + 64), NAN, dtype=BF, device=dev)
    buf[:, 32:32 + K] = vals
    return buf[:, 32:32 + K]


def _run_skinny(x, w, mode, N, rms=None, eps=0.0, res=None):
    """One ops.skinny_linear call writing into a (B, N) view of stride N + 8 inside a NaN-filled buffer; asserts that the
    pad columns and the neighbour rows keep the sentinel."""
    B = x.shape[0]
    buf = torch.full((B + 2, N + 8), NAN, dtype=BF, device=dev)
    out = buf[1:B + 1, :N]
    _ops().skinny_linear(x, w, rms, eps, residual=res, swiglu=mode == 2, out=out)
    torch.cuda.synchronize()
    assert _sentinel_intact(buf, (slice(1, B + 1), slice(0, N))), "skinny_linear wrote outside its output rows"
    return out


def _silu_branches(gq):
    """silu of the (integer, bf16-exact) gate as skinny_linear_kernel<*, 2> computes it:
        act = bf16(gq / (1 + __expf(-gq)))
    __expf: 2 + floor(|1.16 x|) ulp (<= 2u each, relative) on e = exp(-gq); 1 + e and the IEEE division add u each."""
    v = gq / (1 + torch.exp(-gq))
    eps = (2 + torch.floor(1.16 * gq.abs())) * 2 * U + 2 * U + HIGHER_ORDER
    return (*Hp.bf16_branches(v, eps), v, eps)


def _skinny_exact_check(out, x64, w, mode, N, res64=None, what=""):
    """Modes 0 / 1 / 2 with integer operands: s = x @ w.T is an integer below 2^17 (K <= 12288, |x w| <= 9), exact in
    fp32 in any summation order, so the fragment order, the K-slice reduction and the MMA's accumulation cannot change
    it (assumes mma.sync's fp32 accumulation is exact on integer partial sums below 2^24).
        mode 0: y = bf16(s);  mode 1: y = bf16(fp32(bf16(s) + res));  mode 2: y = bf16(bf16(up) * act(bf16(gate)))
    bf16(up) * act is a product of two 8-bit significands, exact in fp32 before its rounding."""
    s = x64 @ w.to(F64).t()
    if mode == 0:
        ref = Hp.bf16_rne(s)
    elif mode == 1:
        ref = Hp.bf16_rne(Hp.f32(Hp.bf16_rne(s) + res64))
    else:
        gq, uq = Hp.bf16_rne(s[:, :N]), Hp.bf16_rne(s[:, N:])
        assert float(gq.abs().max()) <= 12
        a_ref, a_alt, band, v, eps = _silu_branches(gq)
        flips = Hp.accept_branches(out, Hp.bf16_rne(uq * a_ref), Hp.bf16_rne(uq * a_alt), band, what)
        _check_flips(what, flips, v, eps)
        return
    assert torch.equal(out.to(F64), ref), (what, int((out.to(F64) != ref).sum()))


@pytest.mark.parametrize("mode", [0, 1, 2])
@pytest.mark.parametrize("tag,per,K", SK_SHAPES)
def test_skinny_linear_exact_integers(tag, per, K, mode):
    """aki_mma_skinny_linear with integer x, w in [-3, 3]: bit-exact against the fp64 GEMM (see _skinny_exact_check), at
    N on both sides of every dispatch boundary, B = 1, 5, 8, strided x, residual of odd row stride N + 3, output view of
    stride N + 8 inside a NaN sentinel."""
    N = _n_of(tag, per)
    g = torch.Generator(device=dev).manual_seed(N * 31 + K + mode)
    w = _skinny_weights(N, K, mode, g)
    xv = torch.randint(-3, 4, (8, K), generator=g, device=dev, dtype=torch.int32).to(BF)
    res_buf = (torch.randn(8, N + 3, generator=g, device=dev) * 64).to(BF) if mode == 1 else None
    for B in (1, 5, 8):
        what = f"skinny mode={mode} N={N} K={K} B={B} per={per}"
        print(what)
        res = res_buf[:B, :N] if mode == 1 else None
        out = _run_skinny(_strided_x(xv[:B]), w, mode, N, res=res)
        _skinny_exact_check(out, xv[:B].to(F64), w, mode, N, res.to(F64) if mode == 1 else None, what)


@pytest.mark.parametrize("mode", [0, 1, 2])
@pytest.mark.parametrize("tag,per,K", [("16", 1, 3072), ("16sms+16", 2, 1024), ("64sms", 4, 8192), ("64sms+16", 16, 1024)])
def test_skinny_linear_norm_prologue_exact(tag, per, K, mode):
    """RMSNorm prologue with x in {-1, +1}, integer gamma and eps = 0: the mean square is exactly 1, rsqrtf(1) = 1
    (assumed: the test reports otherwise), every normalised element is +-gamma, far from any tie, and the output must
    be bit-exact to the integer GEMM on gamma * x."""
    N = _n_of(tag, per)
    g = torch.Generator(device=dev).manual_seed(N + K * 3 + mode)
    w = _skinny_weights(N, K, mode, g)
    xv = (torch.randint(0, 2, (8, K), generator=g, device=dev) * 2 - 1).to(BF)
    gamma = torch.randint(-3, 4, (K,), generator=g, device=dev, dtype=torch.int32).to(BF)
    if mode == 2:
        gamma = gamma.clamp(-1, 1)        # |gate| = |sum of four +-1 weights times +-gamma| <= 4
    res = (torch.randn(8, N + 3, generator=g, device=dev) * 64).to(BF)[:, :N] if mode == 1 else None
    what = f"skinny prologue-exact mode={mode} N={N} K={K} B=8 per={per}"
    print(what)
    out = _run_skinny(_strided_x(xv), w, mode, N, rms=gamma, eps=0.0, res=res)
    _skinny_exact_check(out, xv.to(F64) * gamma.to(F64), w, mode, N, res.to(F64) if mode == 1 else None, what)


def _norm_prologue_ref(xv, gamma, eps, K, depth):
    """Branches of the prologue's two roundings, Phi3RMSNorm's: xn = bf16(x * r), xg = bf16(gamma * xn) (exact bf16
    product, one rounding).  r = rsqrtf(ss / K + eps) with ss an fp32 sum of x^2 whose terms pass through at most
    `depth` roundings: rel(ss / K + eps) <= (depth + 2) u, rsqrtf 2 ulp <= 4u, so rel(r) <= (depth + 2) u / 2 + 4u,
    and x * r adds u."""
    x64 = xv.to(F64)
    r = 1 / torch.sqrt((x64 * x64).sum(-1, keepdim=True) / K + Hp.f32(torch.tensor(eps, dtype=F64)))
    eps_xn = (depth + 2) * U / 2 + 4 * U + U + HIGHER_ORDER
    v = x64 * r
    xn_ref, xn_alt, band = Hp.bf16_branches(v, eps_xn)
    g64 = gamma.to(F64)
    return Hp.bf16_rne(g64 * xn_ref), Hp.bf16_rne(g64 * xn_alt), band, v, eps_xn


@pytest.mark.parametrize("tag,per,K", [("16sms", 1, 3072), ("32sms", 2, 12288), ("32sms+16", 4, 3072),
                                       ("32064", 16, 3072)])
def test_skinny_linear_norm_prologue_bound(tag, per, K):
    """RMSNorm prologue on Gaussian x: against an fp64 GEMM of the reference's normalised operand, within
        ulp_bf16(|ref| + E) + E,   E = sum_k |w_k| |xg_alt_k - xg_ref_k| [k in band] + K u sum_k |w_k xg_k|
    (the bf16 rounding of the fp32 sum, the accepted flips of the prologue, the fp32 accumulation).  The prologue's
    sum of squares: every thread adds the squares of its 8-element chunks (3 roundings on entry, 4 updates per chunk,
    ceil(K / 4096) chunks), then 5 shuffle levels and the 16 warp partials."""
    N = _n_of(tag, per)
    g = torch.Generator(device=dev).manual_seed(N + K)
    w = (torch.randn(N, K, generator=g, device=dev) * K ** -0.5).to(BF)
    xv = torch.randn(8, K, generator=g, device=dev).to(BF)
    gamma = (1 + 0.1 * torch.randn(K, generator=g, device=dev)).to(BF)
    depth = 3 + 4 * math.ceil(K / 4096) + 5 + 16
    xg_ref, xg_alt, band, v, eps_xn = _norm_prologue_ref(xv, gamma, 1e-5, K, depth)
    what = f"skinny prologue-bound mode=0 N={N} K={K} B=8 per={per}"
    print(what)
    out = _run_skinny(_strided_x(xv), w, 0, N, rms=gamma, eps=1e-5).to(F64)
    w64 = w.to(F64)
    ref = xg_ref @ w64.t()
    E = ((xg_alt - xg_ref).abs() * band) @ w64.abs().t() + K * U * (xg_ref.abs() @ w64.abs().t())
    err = (out - ref).abs()
    lim = Hp.ulp_bf16(ref.abs() + E) + E
    assert bool((err <= lim).all()), (what, float((err / lim).max()))
    print(f"{what}: prologue in-band elements {int(band.sum())} of {band.numel()} (flip bound "
          f"{Hp.flip_bound(v, eps_xn)}), max err / bound {float((err / lim).max()):.3f}")
    assert int(band.sum()) <= Hp.flip_bound(v, eps_xn)


def test_skinny_linear_token_independence_and_unsupported_k():
    """B = 1 ... 8 with the (inexact) norm prologue and a residual: row b of every call is bit-identical to a B = 1 call
    on that row alone -- the per-token accumulation order does not depend on B.  K = 13312 needs more shared memory than
    the kernel allows and is refused with AKI_ERR_UNSUPPORTED."""
    sms = torch.cuda.get_device_properties(0).multi_processor_count
    N, K = 16 * sms + 16, 3072
    g = torch.Generator(device=dev).manual_seed(5)
    w = (torch.randn(N, K, generator=g, device=dev) * K ** -0.5).to(BF)
    xv = torch.randn(8, K, generator=g, device=dev).to(BF)
    gamma = (1 + 0.1 * torch.randn(K, generator=g, device=dev)).to(BF)
    res = (torch.randn(8, N + 3, generator=g, device=dev) * 4).to(BF)[:, :N]
    single = [_run_skinny(_strided_x(xv[b:b + 1]), w, 1, N, rms=gamma, eps=1e-5, res=res[b:b + 1]) for b in range(8)]
    for B in range(1, 9):
        print(f"skinny token-independence mode=1 N={N} K={K} B={B} per={_per(N, sms)}")
        out = _run_skinny(_strided_x(xv[:B]), w, 1, N, rms=gamma, eps=1e-5, res=res[:B])
        for b in range(B):
            assert torch.equal(out[b], single[b][0]), (B, b)
    big = torch.zeros(8 * 13312 * 2, dtype=BF, device=dev)
    rc = _lib().aki_mma_skinny_linear(_p(big), 13312, _p(big), None, C.c_float(1e-5), None, 0, _p(big), 16, 1, 16, 13312,
                                      0, None)
    assert rc == ERR_UNSUPPORTED


# ------------------------------------------------------------------------------------------------ add_rmsnorm / swiglu
def _norm_depth(K):
    """Roundings a square passes through in add_rmsnorm_kernel's sum: product, FMA, add on entry, then the lane's later
    updates (4 per 256-element chunk), then 5 shuffle levels."""
    return 3 + 4 * (K // 256) + 5


@pytest.mark.parametrize("M,K", [(1, 256), (7, 1024), (8, 4096), (9, 256), (9, 3072), (5240, 3072), (5240, 4096)])
@pytest.mark.parametrize("layout", ["inplace", "separate", "no-residual"])
def test_add_rmsnorm_rounding_points(M, K, layout):
    """aki_mma_add_rmsnorm through the C API with strided x (K + 16), residual (K + 32), h (K + 24) and y (K + 8) rows,
    each inside a NaN-filled buffer with a guard row on either side.
      h = bf16(fp32(res + x)): bit-exact.
      y = bf16(w * bf16(h * r)), r = rsqrtf(ss / K + eps): tie-aware at bf16(h * r) (eps from _norm_prologue_ref with
          _norm_depth), both branches through the exact bf16 multiply by w.
    With the residual updated in place, nothing outside its own rows and columns changes.  K above 4096 is refused."""
    lib, ops = _lib(), _ops()
    g = torch.Generator(device=dev).manual_seed(M * 13 + K)
    xb = torch.full((M, K + 16), NAN, dtype=BF, device=dev)
    xb[:, :K] = torch.randn(M, K, generator=g, device=dev).to(BF)
    rb = torch.full((M + 2, K + 32), NAN, dtype=BF, device=dev)
    rb[1:M + 1, :K] = (torch.randn(M, K, generator=g, device=dev) * 3).to(BF)
    w = (1 + 0.1 * torch.randn(K, generator=g, device=dev)).to(BF)
    x, res = xb[:, :K], rb[1:M + 1, :K]
    x64, res64 = x.to(F64), res.to(F64)
    yb = torch.full((M + 2, K + 8), NAN, dtype=BF, device=dev)
    y = yb[1:M + 1, :K]
    hb = torch.full((M + 2, K + 24), NAN, dtype=BF, device=dev)
    if layout == "inplace":
        h, hs = res, rb.stride(0)
    elif layout == "separate":
        h, hs = hb[1:M + 1, :K], hb.stride(0)
    else:
        h, hs = None, 0
    r_arg = None if layout == "no-residual" else res
    rc = lib.aki_mma_add_rmsnorm(_p(x), xb.stride(0), _p(r_arg), rb.stride(0) if r_arg is not None else 0, _p(w),
                                 C.c_float(1e-5), _p(h), hs, _p(y), yb.stride(0), M, K, ops._stream())
    assert rc == 0
    torch.cuda.synchronize()
    hv = x64 if layout == "no-residual" else Hp.bf16_rne(Hp.f32(res64 + x64))
    if h is not None:
        assert torch.equal(h.to(F64), hv)
        buf = rb if layout == "inplace" else hb
        assert _sentinel_intact(buf, (slice(1, M + 1), slice(0, K)))
    else:
        assert torch.equal(res.to(F64), res64) and _sentinel_intact(rb, (slice(1, M + 1), slice(0, K)))
    assert _sentinel_intact(yb, (slice(1, M + 1), slice(0, K)))
    y_ref, y_alt, band, v, eps = _norm_prologue_ref(hv, w, 1e-5, K, _norm_depth(K))
    flips = Hp.accept_branches(y, y_ref, y_alt, band, f"add_rmsnorm y M={M} K={K}")
    _check_flips(f"add_rmsnorm y M={M} K={K} {layout}", flips, v, eps)
    assert lib.aki_mma_add_rmsnorm(_p(x), xb.stride(0), None, 0, _p(w), C.c_float(1e-5), None, 0, _p(y), yb.stride(0), M,
                                   4352, ops._stream()) == ERR_UNSUPPORTED


def _silu_expf(g64):
    """v = g / (1 + expf(-g)) as swiglu_kernel evaluates it: expf 2 ulp (<= 4u relative on e, and on 1 + e), the add and
    the IEEE division u each.  Where expf(-g) overflows fp32 (g <= -89 in bf16) the kernel divides by inf: -0."""
    e = torch.exp(-g64)
    over = torch.isinf(Hp.f32(e))
    v = torch.where(over, torch.zeros_like(g64), g64 / (1 + e))
    return v, 4 * U + 2 * U + HIGHER_ORDER


@pytest.mark.parametrize("M,N,dist", [(5, 8, "wide"), (37, 3072, "wide"), (1300, 8192, "normal")])
def test_swiglu_rounding_points(M, N, dist):
    """aki_mma_swiglu: y = bf16(up * bf16(silu(gate))).  Tie-aware at the silu (_silu_expf), both branches through the
    exact bf16 product with up.  gate_up rows of stride 2N + 16, y rows of stride N + 8 in a NaN sentinel.  'wide' draws
    gates uniformly from [-90, 90] (the expf overflow side included) with |up| in [1, 2), so no product leaves the
    normal range; M = 1300, N = 8192 is more than 148 x 32 CTAs of 256 threads: the grid-stride loop runs twice."""
    lib, ops = _lib(), _ops()
    g = torch.Generator(device=dev).manual_seed(M + N)
    gb = torch.full((M, 2 * N + 16), NAN, dtype=BF, device=dev)
    if dist == "wide":
        gate = (torch.rand(M, N, generator=g, device=dev) * 180 - 90)
        up = (1 + torch.rand(M, N, generator=g, device=dev)) * (torch.randint(0, 2, (M, N), generator=g, device=dev) * 2 - 1)
        gate[0, :4] = torch.tensor([-90.0, -89.0, -88.5, 90.0])      # overflow of expf(-g) starts between -88.5 and -89
    else:
        gate = torch.randn(M, N, generator=g, device=dev) * 3
        up = torch.randn(M, N, generator=g, device=dev)
    gb[:, :N], gb[:, N:2 * N] = gate.to(BF), up.to(BF)
    yb = torch.full((M + 2, N + 8), NAN, dtype=BF, device=dev)
    y = yb[1:M + 1, :N]
    assert lib.aki_mma_swiglu(_p(gb), gb.stride(0), _p(y), yb.stride(0), M, N, ops._stream()) == 0
    torch.cuda.synchronize()
    assert _sentinel_intact(yb, (slice(1, M + 1), slice(0, N)))
    g64, u64 = gb[:, :N].to(F64), gb[:, N:2 * N].to(F64)
    v, eps = _silu_expf(g64)
    a_ref, a_alt, band = Hp.bf16_branches(v, eps)
    flips = Hp.accept_branches(y, Hp.bf16_rne(u64 * a_ref), Hp.bf16_rne(u64 * a_alt), band, f"swiglu M={M} N={N}")
    _check_flips(f"swiglu M={M} N={N} {dist}", flips, v, eps)
    if dist == "wide":
        assert int((g64 <= -89).sum()) > 0 and bool((y[g64 <= -89].float() == 0).all())


# ------------------------------------------------------------------------------------------------ SFT (amp) kernels
@pytest.mark.parametrize("M,K,with_a", [(1, 256, True), (9, 3072, True), (2369, 1024, False), (2369, 3072, True)])
def test_add_rmsnorm_amp_fwd_rounding_points(M, K, with_a):
    """aki_mma_add_rmsnorm_amp_fwd.  h' = fp32(h + a): bit-exact.  r = rsqrtf(ss / K + eps) against fp64 within
    (depth + 2) u / 2 + 4u relative (ss: one FMA per square, 8 per 256-element chunk, then 5 shuffle levels).
    x = bf16(w * (h' * r)) with the kernel's own r: two fp32 roundings, tie-aware with eps = 2u."""
    g = torch.Generator(device=dev).manual_seed(M + K)
    h = torch.randn(M, K, generator=g, device=dev) * 2
    a = torch.randn(M, K, generator=g, device=dev).to(BF) if with_a else None
    w = 1 + 0.1 * torch.randn(K, generator=g, device=dev)
    hn = torch.full((M, K), NAN, device=dev) if with_a else None
    x = torch.full((M, K), NAN, dtype=BF, device=dev)
    r = torch.full((M,), NAN, device=dev)
    assert _lib().aki_mma_add_rmsnorm_amp_fwd(_p(h), _p(a), _p(w), C.c_float(1e-5), _p(hn), _p(x), _p(r), M, K,
                                              _ops()._stream()) == 0
    torch.cuda.synchronize()
    h64 = Hp.f32(h.to(F64) + a.to(F64)) if with_a else h.to(F64)
    if with_a:
        assert torch.equal(hn.to(F64), h64)
    r64 = 1 / torch.sqrt((h64 * h64).mean(-1) + Hp.f32(torch.tensor(1e-5, dtype=F64)))
    depth = 2 + 8 * (K // 256) + 5
    rel = ((r.to(F64) - r64).abs() / r64).max()
    print(f"amp fwd M={M} K={K}: max rel err of r {float(rel):.3e} (bound {(depth + 2) * U / 2 + 4 * U:.3e})")
    assert float(rel) <= (depth + 2) * U / 2 + 4 * U + HIGHER_ORDER
    v = w.to(F64) * (h64 * r.to(F64)[:, None])
    flips = Hp.accept_bf16(x, v, 2 * U + HIGHER_ORDER, what=f"amp fwd x M={M} K={K}")
    _check_flips(f"amp fwd x M={M} K={K}", flips, v, 2 * U)


@pytest.mark.parametrize("M,K,with_dh", [(1, 256, False), (2369, 256, True), (2369, 3072, False), (40, 1024, True)])
def test_rmsnorm_amp_bwd_against_fp64(M, K, with_dh):
    """aki_mma_rmsnorm_amp_bwd: dh = dh_out + r g w - h coef, coef = r^3 dot / K, dot = sum_k g w h, and the per-warp dw
    partials sum_{rows of warp p} g h r, against fp64 per element.  Bounds (first order, S = sum_k |g w h| of the row):
      dot: g*w, *h and the add into the lane's sum (K / 32 terms), 5 shuffle levels: (K / 32 + 7) u S;
      coef: 3 multiplies and a division add 4u |coef|: |d coef| <= r^3 / K (K / 32 + 11) u S;
      dh: r*g, *w, the add of dh_out, the FMA with h*coef: <= 4u (|dh_out| + |r g w| + |h coef|) + |h| |d coef|;
      dw partial: g*h, *r and the add on entry, one more add per later row walked: (3 + rows per warp) u sum |g h r|.
    M = 2369 is one row past 296 x 8 warps: warp 0 walks two rows."""
    lib = _lib()
    g_ = torch.Generator(device=dev).manual_seed(M * 3 + K)
    dx = torch.randn(M, K, generator=g_, device=dev).to(BF)
    h = torch.randn(M, K, generator=g_, device=dev) * 2
    w = 1 + 0.1 * torch.randn(K, generator=g_, device=dev)
    r = Hp.f32(1 / torch.sqrt((h.to(F64) ** 2).mean(-1) + 1e-5)).to(F32)
    dh_out = torch.randn(M, K, generator=g_, device=dev) * 0.1 if with_dh else None
    n_part = lib.aki_mma_rmsnorm_amp_bwd_partials(M)
    dh = torch.full((M, K), NAN, device=dev)
    dwp = torch.full((n_part, K), NAN, device=dev)
    assert lib.aki_mma_rmsnorm_amp_bwd(_p(dx), _p(dh_out), _p(h), _p(r), _p(w), _p(dh), _p(dwp), M, K,
                                       _ops()._stream()) == 0
    torch.cuda.synchronize()
    g64, h64, w64, r64 = dx.to(F64), h.to(F64), w.to(F64), r.to(F64)[:, None]
    A = dh_out.to(F64) if with_dh else torch.zeros_like(h64)
    gwh = g64 * w64 * h64
    dot, S = gwh.sum(-1, keepdim=True), gwh.abs().sum(-1, keepdim=True)
    coef = r64 ** 3 * dot / K
    Bt, Ct = r64 * g64 * w64, h64 * coef
    ref = A + Bt - Ct
    bound = 4 * U * (A.abs() + Bt.abs() + Ct.abs()) + h64.abs() * r64 ** 3 / K * (K / 32 + 11) * U * S
    err = (dh.to(F64) - ref).abs()
    print(f"amp bwd M={M} K={K}: dh max err / bound {float((err / bound).max()):.3f}")
    assert bool((err <= bound * (1 + HIGHER_ORDER) + 2.0 ** -140).all()), float((err / bound).max())
    ghr = g64 * h64 * r64
    part = torch.zeros(n_part, K, dtype=F64, device=dev).index_add_(0, torch.arange(M, device=dev) % n_part, ghr)
    part_abs = torch.zeros(n_part, K, dtype=F64, device=dev).index_add_(0, torch.arange(M, device=dev) % n_part, ghr.abs())
    rows_per_warp = math.ceil(M / n_part)
    pb = (3 + rows_per_warp) * U * part_abs
    perr = (dwp.to(F64) - part).abs()
    print(f"amp bwd M={M} K={K}: dw partial max err / bound {float((perr / pb.clamp(min=1e-300)).max()):.3f}")
    assert bool((perr <= pb * (1 + HIGHER_ORDER)).all())
    assert bool(((dwp.to(F64).sum(0) - ghr.sum(0)).abs() <= pb.sum(0) * (1 + HIGHER_ORDER) + 2.0 ** -100).all())


@pytest.mark.parametrize("M,N", [(3, 8), (77, 8192), (1300, 8192)])
def test_swiglu_bwd_rounding_points(M, N):
    """aki_mma_swiglu_bwd, per element with s = 1 / (1 + expf(-g)) (expf 4u, the add and the division u each:
    eps_s = 6u):
      d_up  = bf16(d * bf16(g * s)): tie-aware at bf16(g * s) (eps_s + u), both branches through the exact product;
      d_act = bf16(d * up): exact product, bit-exact;
      d_gate = bf16(d_act * (s * (1 + g * (1 - s)))) against fp64 silu'(g) times the bf16 d_act, with the absolute
          error of the fp32 chain propagated from eps_s through 1 - s, g *, 1 +, s * (u each) and the last multiply."""
    g_ = torch.Generator(device=dev).manual_seed(M + N * 7)
    gu = torch.cat([torch.randn(M, N, generator=g_, device=dev) * 4, torch.randn(M, N, generator=g_, device=dev)], 1).to(BF)
    d = torch.randn(M, N, generator=g_, device=dev).to(BF)
    out = torch.full((M, 2 * N), NAN, dtype=BF, device=dev)
    assert _lib().aki_mma_swiglu_bwd(_p(d), _p(gu), _p(out), M, N, _ops()._stream()) == 0
    torch.cuda.synchronize()
    g64, u64, d64 = gu[:, :N].to(F64), gu[:, N:].to(F64), d.to(F64)
    s = 1 / (1 + torch.exp(-g64))
    eps_s = 6 * U
    a_ref, a_alt, band = Hp.bf16_branches(g64 * s, eps_s + U + HIGHER_ORDER)
    flips = Hp.accept_branches(out[:, N:], Hp.bf16_rne(d64 * a_ref), Hp.bf16_rne(d64 * a_alt), band, "swiglu_bwd d_up")
    _check_flips(f"swiglu_bwd d_up M={M} N={N}", flips, g64 * s, eps_s + U)
    d_act = Hp.bf16_rne(d64 * u64)
    inner = 1 + g64 * (1 - s)
    e_in = g64.abs() * (s * eps_s + U * (1 - s)) + U * (g64 * (1 - s)).abs() + U * (1 + (g64 * (1 - s)).abs())
    e_sd = inner.abs() * s * eps_s + s * e_in + U * s * inner.abs()
    v = d_act * s * inner
    eps_abs = d_act.abs() * e_sd * (1 + HIGHER_ORDER)
    flips = Hp.accept_bf16(out[:, :N], v, U + HIGHER_ORDER, eps_abs, "swiglu_bwd d_gate")
    _check_flips(f"swiglu_bwd d_gate M={M} N={N}", flips, v, U, eps_abs)


# ------------------------------------------------------------------------------------------------ cross-entropy
def _ce_kernels(logits, labels, ignore_index, scale):
    """row_loss, row_lse and dlogits (NaN-prefilled, contiguous) from the two C entry points."""
    lib, ops = _lib(), _ops()
    B, T, V = logits.shape
    loss = torch.full((B, T), NAN, device=dev)
    lse = torch.full((B, T), NAN, device=dev)
    assert lib.aki_mma_cross_entropy_fwd(_p(logits), logits.stride(0), logits.stride(1), _p(labels), labels.stride(0), B,
                                         T, V, ignore_index, _p(loss), _p(lse), ops._stream()) == 0
    d = torch.full((B, T, V), NAN, dtype=BF, device=dev)
    sc = torch.tensor([scale], dtype=F32, device=dev)
    assert lib.aki_mma_cross_entropy_bwd(_p(logits), logits.stride(0), logits.stride(1), _p(labels), labels.stride(0), B,
                                         T, V, ignore_index, _p(lse), _p(sc), _p(d), d.stride(0), d.stride(1),
                                         ops._stream()) == 0
    torch.cuda.synchronize()
    return loss, lse, d


def _ce_case(name):
    """(logits (B, T, V) bf16 view, labels (B, T) int64, ignore_index) for the named edge case."""
    g = torch.Generator(device=dev).manual_seed(sum(map(ord, name)))
    shapes = {"v8": (2, 6, 8), "v1000": (3, 17, 1000), "v32064": (2, 9, 32064), "wide": (2, 9, 32064),
              "neg-inf-chunk": (2, 4, 32064), "neg-inf-chunk-short": (2, 4, 3000), "strided": (2, 11, 1000),
              "t1": (3, 1, 1000), "all-ignored": (2, 7, 1000)}
    B, T, V = shapes[name]
    ignore = -1 if name == "v1000" else -100
    pad = 64 if name == "strided" else 0
    buf = torch.full((B, T, V + pad), NAN, dtype=BF, device=dev)
    x = torch.randn(B, T, V, generator=g, device=dev) * 3
    if name == "wide":
        x = torch.rand(B, T, V, generator=g, device=dev) * 6000 - 3000
    buf[..., :V] = x.to(BF)
    logits = buf[..., :V]
    labels = torch.randint(0, V, (B, T), generator=g, device=dev)
    if T > 1:
        labels[0, 1], labels[-1, -1] = 0, V - 1                 # the first and the last class
    if T > 3:
        labels[0, 2], labels[-1, 2] = V, -5                    # out of range, not ignore_index: ignored
        labels[0, 3] = ignore
    if name == "v1000":
        labels[1, 4] = -100                                    # not this call's ignore_index, negative: ignored
    if name.startswith("neg-inf-chunk"):
        # the first 8-element chunk of every thread (elements [0, 8 x 256)) is -inf: that chunk's exp sum is NaN and only
        # the m == -inf guards drop it; with V = 3000 threads >= 119 have no second chunk, so the NaN reaches ce_combine
        logits[:, :, :2048] = -math.inf
        labels[:, 1:] = torch.randint(2048, V, (B, T - 1), generator=g, device=dev)
    if name == "all-ignored":
        labels[:] = -100
    return logits, labels, ignore


CE_CASES = ["v8", "v1000", "v32064", "wide", "neg-inf-chunk", "neg-inf-chunk-short", "strided", "t1", "all-ignored"]


@pytest.mark.parametrize("name", CE_CASES)
def test_cross_entropy_edges_against_fp64(name):
    """aki_mma_cross_entropy_{fwd,bwd} against the fp64 logsumexp of the bf16 logits.
    Forward, per row: s = sum expf(x - m) in the online form, so a term passes through expf (4u), the 7 adds of its
    chunk, one rescale (expf 4u + multiply u) and add per later chunk of its thread (nc = ceil(V / 2048)), and 5 shuffle
    + 7 warp combines (6u each): rel(s) <= (12 + 6 (nc + 11)) u.  The rounding of x - m costs sum_i p_i |x_i - m| u <=
    u log V (the entropy), logf 1 ulp <= 2u log V, m + log s and lse - x_t u each:
        |loss - ref| <= (12 + 6 (nc + 11)) u + 3u log V + u |lse| + u |loss|      (a c 2^-23 (|lse| + log V) bound).
    Backward, per element: v = (exp(x - lse) - [target]) scale with the kernel's lse and scale; x - lse (u |x - lse|),
    expf (4u), the subtraction of 1 and the scale (u each), and 2^-148 absolute where expf's result is subnormal.
    A target outside [0, V) that is not ignore_index is ignored (torch would raise); ignored rows, the last position and
    every row of an all-ignored batch give loss 0, lse 0 and an all-zero gradient row."""
    logits, labels, ignore = _ce_case(name)
    B, T, V = logits.shape
    scale = 1.7 / 13
    loss, lse, d = _ce_kernels(logits, labels, ignore, scale)
    tgt = torch.full((B, T), ignore, dtype=torch.int64, device=dev)
    tgt[:, :-1] = labels[:, 1:]
    live = (tgt != ignore) & (tgt >= 0) & (tgt < V)
    print(f"cross-entropy {name}: B={B} T={T} V={V}, {int(live.sum())} live rows")
    assert torch.equal(loss[~live], torch.zeros_like(loss[~live])) and torch.equal(lse[~live], torch.zeros_like(lse[~live]))
    assert torch.equal(d[~live].float(), torch.zeros_like(d[~live].float()))
    if name in ("t1", "all-ignored"):
        assert int(live.sum()) == 0
        return
    x64 = logits.to(F64)[live]                                 # (R, V)
    t = tgt[live]
    lse64 = torch.logsumexp(x64, -1)
    loss64 = lse64 - x64.gather(1, t[:, None])[:, 0]
    nc = math.ceil(V / 2048)
    lb = (12 + 6 * (nc + 11)) * U + 3 * U * math.log(V) + U * lse64.abs()
    e_lse = (lse[live].to(F64) - lse64).abs()
    e_loss = (loss[live].to(F64) - loss64).abs()
    print(f"cross-entropy {name}: max |lse err| / bound {float((e_lse / lb).max()):.3f}, "
          f"max |loss err| / bound {float((e_loss / (lb + U * loss64.abs())).max()):.3f}")
    assert bool((e_lse <= lb).all()) and bool((e_loss <= lb + U * loss64.abs()).all())
    lse_k = lse[live].to(F64)[:, None]
    arg = torch.where(torch.isfinite(x64), x64 - lse_k, torch.zeros_like(x64))
    p = torch.exp(x64 - lse_k)
    onehot = torch.zeros_like(p).scatter_(1, t[:, None], 1.0)
    sc = float(torch.tensor(scale, dtype=F32))
    v = (p - onehot) * sc
    eps_abs = sc * (p * (U * arg.abs() + 4 * U) + 2.0 ** -148) + 2.0 ** -149
    flips = Hp.accept_bf16(d[live], v, 2 * U + HIGHER_ORDER, eps_abs, f"cross-entropy bwd {name}")
    _check_flips(f"cross-entropy bwd {name}", flips, v, 2 * U, eps_abs)


def test_cross_entropy_op_ignores_out_of_range_labels_and_empty_batches():
    """ops.cross_entropy_shifted: labels outside [0, V) are ignored, not an error, and do not count in the mean; a batch
    with no valid target returns loss 0 and an all-zero gradient (torch's mean over no element is NaN)."""
    ops = _ops()
    g = torch.Generator(device=dev).manual_seed(9)
    B, T, V = 2, 9, 1000
    logits = (torch.randn(B, T, V, generator=g, device=dev) * 3).to(BF)
    labels = torch.randint(0, V, (B, T), generator=g, device=dev)
    labels[0, 3], labels[1, 5], labels[1, 6] = V, -7, -100
    a = logits.clone().requires_grad_(True)
    got = ops.cross_entropy_shifted(a, labels)
    keep = labels.clone()
    keep[(keep < 0) | (keep >= V)] = -100
    ref = torch.nn.functional.cross_entropy(logits[:, :-1].double().reshape(-1, V), keep[:, 1:].reshape(-1), ignore_index=-100)
    assert abs(float(got) - float(ref)) <= 1e-5 * abs(float(ref))
    got.backward()
    assert torch.equal(a.grad[0, 2].float(), torch.zeros(V, device=dev))             # row 2 pairs with labels[0, 3] = V
    labels[:] = -100
    b = logits.clone().requires_grad_(True)
    got = ops.cross_entropy_shifted(b, labels)
    assert float(got) == 0.0
    assert math.isnan(float(torch.nn.functional.cross_entropy(logits[:, :-1].float().reshape(-1, V),
                                                              labels[:, 1:].reshape(-1), ignore_index=-100)))
    got.backward()
    assert torch.equal(b.grad.float(), torch.zeros(B, T, V, device=dev))


# ------------------------------------------------------------------------------------------------ RoPE
LONG_EXT = [2.0 + 3.0 * i / 48 for i in range(48)]


def _long_rope():
    import aki_b200
    return aki_b200.LongRope(long_factor=LONG_EXT, device=dev)


def test_rope_table_against_fp64_near_128k():
    """aki_mma_rope_table with the long factors at positions up to 131071: cos / sin against fp64 cos / sin of the fp32
    product f = fp32(pos * inv_freq) (the rounding point the kernel and HF share), times the fp32 attention factor.
    Bound: sincosf 2 ulp of the fp32 result (scaled by the factor) + half an ulp of the final multiply."""
    rope = _long_rope()
    g = torch.Generator(device=dev).manual_seed(1)
    pos = torch.stack([131071 - torch.arange(512, device=dev), torch.randint(0, 131072, (512,), generator=g, device=dev)])
    pos[1, 0] = 0
    cos, sin = rope.tables(pos, max_position=131071)
    inv64 = rope.inv_freq_long.to(F64)
    f = Hp.f32(pos.to(F64)[..., None] * inv64)
    af = float(torch.tensor(rope.attention_factor, dtype=F32))
    for got, ref in ((cos, torch.cos(f)), (sin, torch.sin(f))):
        lim = 2 * Hp.ulp32(ref) * af + 0.5 * Hp.ulp32(ref.abs() * af * (1 + 2 ** -20))
        err = (got.to(F64) - ref * af).abs()
        print(f"rope_table: max err / bound {float((err / lim).max()):.3f}")
        assert bool((err <= lim).all()), float((err / lim).max())


def _rot_branches(lo, hi, c, s):
    """lo' = lo c - hi s, hi' = hi c + lo s (fp64, exact from bf16 x fp32).  rope_kv_write_kernel compiles each to one
    FMA over one rounded product (SASS: 32 FFMA + 32 FMUL), in either order, e.g. fma(lo, c, -fp32(hi s)): the fp32
    value is within u max(|lo c|, |hi s|) + u |v| of v."""
    v_lo, v_hi = lo * c - hi * s, hi * c + lo * s
    a_lo = U * torch.maximum((lo * c).abs(), (hi * s).abs()) * (1 + 2 * U)
    a_hi = U * torch.maximum((hi * c).abs(), (lo * s).abs()) * (1 + 2 * U)
    return torch.cat([v_lo, v_hi], -1), torch.cat([a_lo, a_hi], -1)


def _rope_check(got, x, cos, sin, what):
    """got (B, H, T, 96) bf16 against the rotation of x (B, T, H, 96) bf16 by the kernel's tables (B, T, 48)."""
    x64 = x.to(F64).transpose(1, 2)
    c, s = cos.to(F64)[:, None], sin.to(F64)[:, None]
    v, ea = _rot_branches(x64[..., :48], x64[..., 48:], c, s)
    flips = Hp.accept_bf16(got, v, U + HIGHER_ORDER, ea, what)
    _check_flips(what, flips, v, U, ea)


@pytest.mark.parametrize("H,with_v", [(32, True), (5, False), (40, True)])
def test_rope_kv_write_rotation_and_rows(H, with_v):
    """aki_mma_rope_kv_write at positions near 128K: K rows [past, past + T) rotated (tie-aware, _rot_branches), V an
    exact copy, Q rotated into q_rot; every other cache element keeps its NaN sentinel.  H = 40 makes the 192 threads
    of a CTA loop; H = 5 runs without a V cache."""
    ops = _ops()
    B, T, D, past, t_cap = 2, 33, 96, 10, 43                  # past + T == t_cap: the last row of the cache
    g = torch.Generator(device=dev).manual_seed(H)
    qkv = (torch.randn(B, T, 3 * H * D, generator=g, device=dev) * 2).to(BF)
    pos = 131071 - T + torch.arange(T, device=dev)[None].repeat(B, 1)
    pos[1] -= 5000
    cos, sin = _long_rope().tables(pos, max_position=131071)
    kc = torch.full((B, H, t_cap, D), NAN, dtype=BF, device=dev)
    vc = torch.full_like(kc, NAN) if with_v else None
    qr = torch.full((B, H, T, D), NAN, dtype=BF, device=dev)
    ops.rope_kv_write(qkv, cos, sin, kc, vc, past, H, q_rot=qr)
    torch.cuda.synchronize()
    q, k, v = (qkv[..., i * H * D:(i + 1) * H * D].view(B, T, H, D) for i in range(3))
    _rope_check(kc[:, :, past:], k, cos, sin, f"rope_kv_write K H={H}")
    _rope_check(qr, q, cos, sin, f"rope_kv_write Q H={H}")
    assert bool(torch.isnan(kc[:, :, :past].float()).all())
    if with_v:
        assert torch.equal(vc[:, :, past:], v.transpose(1, 2)) and bool(torch.isnan(vc[:, :, :past].float()).all())


@pytest.mark.parametrize("H", [32, 7])
def test_rope_kv_write_dev_drops_rows_past_capacity(H):
    """aki_mma_rope_kv_write_dev with per-sequence device lengths: sequence b writes rows [past_b, min(past_b + T, t_cap));
    rows at or past t_cap are dropped.  Every other element of both caches keeps its sentinel -- in particular row 0 of
    the next head (and of the next sequence), where row t_cap of a contiguous (B, H, t_cap, D) cache would land, and the
    guard rows after the last head.  Q is rotated for every token regardless."""
    ops = _ops()
    B, T, D, t_cap = 6, 9, 96, 20
    past = torch.tensor([0, 5, 11, 12, 19, 20], dtype=torch.int32, device=dev)
    g = torch.Generator(device=dev).manual_seed(100 + H)
    qkv = (torch.randn(B, T, 3 * H * D, generator=g, device=dev) * 2).to(BF)
    pos = past[:, None].long() + torch.arange(T, device=dev)[None] + 120000
    cos, sin = _long_rope().tables(pos, max_position=131071)
    n_el = B * H * t_cap * D
    kbuf = torch.full((n_el + 2 * D,), NAN, dtype=BF, device=dev)     # two guard rows after the last head's last row
    vbuf = torch.full_like(kbuf, NAN)
    kc, vc = kbuf[:n_el].view(B, H, t_cap, D), vbuf[:n_el].view(B, H, t_cap, D)
    qr = torch.full((B, H, T, D), NAN, dtype=BF, device=dev)
    ops.rope_kv_write(qkv, cos, sin, kc, vc, 0, H, q_rot=qr, past_len_dev=past)
    torch.cuda.synchronize()
    assert bool(torch.isnan(kbuf[n_el:].float()).all()) and bool(torch.isnan(vbuf[n_el:].float()).all())
    q, k, v = (qkv[..., i * H * D:(i + 1) * H * D].view(B, T, H, D) for i in range(3))
    _rope_check(qr, q, cos, sin, f"rope_kv_write_dev Q H={H}")
    written = torch.zeros(B, t_cap, dtype=torch.bool, device=dev)
    for b, p0 in enumerate(past.tolist()):
        n = max(0, min(T, t_cap - p0))
        if n:
            written[b, p0:p0 + n] = True
            _rope_check(kc[b:b + 1, :, p0:p0 + n], k[b:b + 1, :n], cos[b:b + 1, :n], sin[b:b + 1, :n],
                        f"rope_kv_write_dev K b={b} H={H}")
            assert torch.equal(vc[b, :, p0:p0 + n], v[b, :n].transpose(0, 1))
    keep = ~written[:, None, :, None].expand_as(kc)
    assert bool(torch.isnan(kc[keep].float()).all()) and bool(torch.isnan(vc[keep].float()).all())
