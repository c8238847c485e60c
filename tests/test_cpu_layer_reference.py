"""CPU checks of the rounding-point reference helpers that test_gpu_layer_numerics.py compares the decoder-layer kernels
with: bf16_rne against torch's fp32 -> bf16 cast (a single round-to-nearest-even), the neighbour and ulp helpers, and the
tie-aware comparison accept_bf16 on constructed cases."""
import math

import pytest
import torch

import helpers as Hp

F32 = torch.float32


def _f32_bits(bits):
    return torch.tensor(bits, dtype=torch.int64).to(torch.int32).view(F32)


def test_bf16_rne_matches_torch_on_ties_subnormals_and_overflow():
    g = torch.Generator().manual_seed(0)
    special = [
        0.0, -0.0, 1.0, -1.0, math.inf, -math.inf,
        1.0 + 2 ** -8, 1.0 + 3 * 2 ** -8, -(1.0 + 2 ** -8), -(1.0 + 3 * 2 ** -8),        # ties: to even down / up
        1.0 + 2 ** -8 + 2 ** -23, 1.0 + 2 ** -8 - 2 ** -23,                              # one fp32 ulp off a tie
        Hp.BF16_MAX, -Hp.BF16_MAX,                                                       # largest finite
        (2 - 2 ** -8) * 2.0 ** 127, -(2 - 2 ** -8) * 2.0 ** 127,                         # the tie above it -> inf
        (2 - 2 ** -8 - 2 ** -20) * 2.0 ** 127,                                           # just below that tie
        2.0 ** -126, 2.0 ** -133, 2.0 ** -134, 3 * 2.0 ** -134, 2.0 ** -135, 5 * 2.0 ** -136, 2.0 ** -149,
        -3 * 2.0 ** -134, (2 - 2 ** -7) * 2.0 ** -127, (2 - 2 ** -8) * 2.0 ** -127,      # bf16 subnormal range
        float.fromhex("0x1.fffffep+127"), float.fromhex("0x1.fe0000p+127"),
    ]
    x = torch.cat([torch.tensor(special, dtype=F32),
                   torch.randn(20000, generator=g) * torch.exp2(torch.randint(-140, 128, (20000,), generator=g).float()),
                   _f32_bits(torch.randint(-2 ** 31, 2 ** 31, (20000,), generator=g).tolist())])
    x = x[~torch.isnan(x)]
    want = x.to(torch.bfloat16)
    got = Hp.bf16_rne(x.double())
    assert torch.equal(got.to(torch.bfloat16).view(torch.int16), want.view(torch.int16))
    assert torch.equal(got, want.double())                     # the fp64 result is exactly the bf16 value
    assert torch.isnan(Hp.bf16_rne(torch.tensor([math.nan], dtype=torch.float64))).all()


def test_bf16_rne_rounds_once_from_fp64():
    """A value just above a bf16 tie that fp32 would round onto the tie: one rounding from fp64 goes up, the double
    rounding through fp32 goes to even (down)."""
    v = torch.tensor([1.0 + 2 ** -8 + 2 ** -40], dtype=torch.float64)
    assert float(Hp.bf16_rne(v)) == 1.0 + 2 ** -7
    assert float(v.float().to(torch.bfloat16)) == 1.0


def test_neighbours_and_ulps():
    v = torch.tensor([1.0, -1.0, 0.0, Hp.BF16_MAX, 2.0 ** -133, 3.0], dtype=torch.float64)
    assert Hp.bf16_step(v, True).tolist() == [1 + 2 ** -7, -(1 - 2 ** -8), 2.0 ** -133, math.inf, 2.0 ** -132, 3 + 2 ** -6]
    assert Hp.bf16_step(v, False).tolist() == [1 - 2 ** -8, -(1 + 2 ** -7), -2.0 ** -133, (2 - 2 ** -6) * 2.0 ** 127,
                                               0.0, 3 - 2 ** -6]
    assert Hp.ulp32(torch.tensor([1.0, 1.5, 2.0 ** -140, 3e38], dtype=torch.float64)).tolist() == \
        [2.0 ** -23, 2.0 ** -23, 2.0 ** -149, 2.0 ** 104]
    assert Hp.ulp_bf16(torch.tensor([1.0, -3.0, 2.0 ** -130], dtype=torch.float64)).tolist() == \
        [2.0 ** -7, 2.0 ** -6, 2.0 ** -133]
    assert Hp.f32(torch.tensor([1.0 + 2 ** -30], dtype=torch.float64)).item() == 1.0


def test_accept_bf16_on_constructed_cases():
    tie = 1.0 + 2 ** -8                                   # midpoint of 1 and 1 + 2^-7; RNE -> 1.0
    eps = 2 ** -20
    bf = lambda *v: torch.tensor(v, dtype=torch.float64).to(torch.bfloat16)
    v = torch.tensor([tie, tie + 2 ** -23, tie - 2 ** -23], dtype=torch.float64)
    # both neighbours of the tie are accepted for an exact tie and one fp32 ulp either side of it
    flips = Hp.accept_bf16(bf(1.0, 1.0, 1.0), v, eps)
    assert flips.tolist() == [False, True, False]         # tie + 1 ulp rounds up: 1.0 is the accepted flip
    flips = Hp.accept_bf16(bf(1.0 + 2 ** -7, 1.0 + 2 ** -7, 1.0 + 2 ** -7), v, eps)
    assert flips.tolist() == [True, False, True]
    # with no uncertainty only the correct rounding passes
    Hp.accept_bf16(bf(1.0, 1.0 + 2 ** -7, 1.0), v, 0.0)
    with pytest.raises(AssertionError):
        Hp.accept_bf16(bf(1.0 + 2 ** -7, 1.0 + 2 ** -7, 1.0), v, 0.0)
    # far from any tie (a quarter ulp from it) the wrong neighbour is rejected
    far = torch.tensor([1.0 + 2 ** -9, -(3.0 + 2 ** -8)], dtype=torch.float64)
    Hp.accept_bf16(bf(1.0, -3.0), far, eps)
    with pytest.raises(AssertionError):
        Hp.accept_bf16(bf(1.0 + 2 ** -7, -3.0), far, eps)
    with pytest.raises(AssertionError):
        Hp.accept_bf16(bf(1.0, -(3.0 + 2 ** -6)), far, eps)
    # a value two ulps away is never accepted, even inside the band
    with pytest.raises(AssertionError):
        Hp.accept_bf16(bf(1.0 + 2 ** -6), torch.tensor([tie], dtype=torch.float64), eps)
    # the absolute term widens the band near zero (a rotation that cancels), and NaN only matches NaN
    Hp.accept_bf16(bf(2.0 ** -20), torch.tensor([2.0 ** -20 + 2.0 ** -28 + 2.0 ** -40], dtype=torch.float64), 0.0, 2.0 ** -35)
    with pytest.raises(AssertionError):
        Hp.accept_bf16(bf(2.0 ** -20), torch.tensor([2.0 ** -20 + 2.0 ** -28 + 2.0 ** -33], dtype=torch.float64), 0.0, 2.0 ** -35)
    Hp.accept_bf16(bf(math.nan, math.inf), torch.tensor([math.nan, math.inf], dtype=torch.float64), eps)
    # a cancellation whose absolute term spans several bf16 ulps (2^-24 around 2^-20, ulp 2^-27): every bf16 value of
    # the rounded interval is accepted, nothing beyond it; the two-branch model refuses such a band
    v = torch.tensor([2.0 ** -20], dtype=torch.float64)
    flips = Hp.accept_bf16(bf(2.0 ** -20 + 7 * 2.0 ** -27, 2.0 ** -20 - 7 * 2.0 ** -28), v.expand(2), 0.0, 2.0 ** -24)
    assert flips.tolist() == [True, True]
    with pytest.raises(AssertionError):
        Hp.accept_bf16(bf(2.0 ** -20 + 9 * 2.0 ** -27), v, 0.0, 2.0 ** -24)
    with pytest.raises(AssertionError):
        Hp.bf16_branches(v, 0.0, 2.0 ** -24)


def test_flip_bound_scales_with_eps():
    v = torch.linspace(1, 2, 10000, dtype=torch.float64)
    assert Hp.flip_bound(v, 0.0) == 8
    assert Hp.flip_bound(v, 2 ** -20) == int(2 * 10000 * 2 ** -11) + 8
