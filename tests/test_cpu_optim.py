"""CPU-only: status codes of the optimizer entry points (aki_mma_grad_sq_norm, aki_mma_adamw_step), returned before any
launch or device query, and the parameter checks of AkiAdamW."""
import ctypes as C

import pytest
import torch

ERR_NULL, ERR_BAD_SHAPE, ERR_MISALIGNED = -1, -2, -4


@pytest.fixture(scope="module")
def lib():
    from aki_b200 import _lib
    return _lib


def _list(lib, n=2, buf=None, **over):
    """n entries pointing into `buf` (host memory: nothing is launched when validation fails)."""
    base = C.addressof(buf)
    arr = (lib.AdamWTensor * n)()
    for i in range(n):
        arr[i].param, arr[i].grad, arr[i].exp_avg, arr[i].exp_avg_sq = base, base + 16, base + 32, base + 48
        arr[i].param_bf16 = base + 64
        arr[i].numel = 4
    for k, v in over.items():
        setattr(arr[n - 1], k, v)
    return arr


def _adamw(lib, arr, n=None, sq=None, max_norm=1.0, lr=1e-3, b1=0.9, b2=0.999, eps=1e-8, wd=0.0, step=1):
    return lib.lib.aki_mma_adamw_step(arr, len(arr) if n is None else n, sq, max_norm, lr, b1, b2, eps, wd, step, None)


def _norm(lib, arr, n=None, ws=True, ws_bytes=4096, sq=True, buf=None):
    p = C.addressof(buf)
    return lib.lib.aki_mma_grad_sq_norm(arr, len(arr) if n is None else n, p if ws else None, ws_bytes, p if sq else None,
                                        None)


def test_adamw_status_codes(lib):
    buf = (C.c_int64 * 64)()
    ok = _list(lib, buf=buf)
    assert _adamw(lib, None, n=1) == ERR_NULL
    for field in ("param", "grad", "exp_avg", "exp_avg_sq"):
        assert _adamw(lib, _list(lib, buf=buf, **{field: None})) == ERR_NULL, field
    assert _adamw(lib, ok, n=0) == ERR_BAD_SHAPE
    assert _adamw(lib, ok, n=-3) == ERR_BAD_SHAPE
    assert _adamw(lib, _list(lib, buf=buf, numel=-1)) == ERR_BAD_SHAPE
    for field in ("param", "grad", "exp_avg", "exp_avg_sq", "param_bf16"):
        bad = _list(lib, buf=buf)
        setattr(bad[1], field, getattr(bad[1], field) + 4)
        assert _adamw(lib, bad) == ERR_MISALIGNED, field
    nan, inf = float("nan"), float("inf")
    for kw in (dict(b1=1.0), dict(b1=-0.1), dict(b1=nan), dict(b2=1.0), dict(b2=nan), dict(eps=-1e-8), dict(eps=inf),
               dict(eps=nan), dict(lr=-1e-3), dict(lr=inf), dict(lr=nan), dict(wd=-0.1), dict(wd=nan), dict(step=0),
               dict(step=-5)):
        assert _adamw(lib, ok, **kw) == ERR_BAD_SHAPE, kw
    sq = C.addressof(buf)
    for mn in (0.0, -1.0, inf, nan):
        assert _adamw(lib, ok, sq=sq, max_norm=mn) == ERR_BAD_SHAPE, mn


def test_grad_sq_norm_status_codes(lib):
    buf = (C.c_int64 * 64)()
    ok = _list(lib, buf=buf)
    assert lib.lib.aki_mma_grad_sq_norm(None, 1, C.addressof(buf), 4096, C.addressof(buf), None) == ERR_NULL
    assert _norm(lib, _list(lib, buf=buf, grad=None), buf=buf) == ERR_NULL
    assert _norm(lib, ok, ws=False, buf=buf) == ERR_NULL
    assert _norm(lib, ok, sq=False, buf=buf) == ERR_NULL
    assert _norm(lib, ok, n=0, buf=buf) == ERR_BAD_SHAPE
    assert _norm(lib, _list(lib, buf=buf, numel=-2), buf=buf) == ERR_BAD_SHAPE
    assert _norm(lib, ok, ws_bytes=0, buf=buf) == ERR_BAD_SHAPE
    bad = _list(lib, buf=buf)
    bad[0].grad += 8
    assert _norm(lib, bad, buf=buf) == ERR_MISALIGNED
    # the norm reads grad and numel only: NULL or misaligned optimizer-state pointers are not its business
    nostate = _list(lib, buf=buf, param=None, exp_avg=None, exp_avg_sq=None, param_bf16=None, numel=-1)
    assert _norm(lib, nostate, buf=buf) == ERR_BAD_SHAPE


def test_grad_sq_norm_workspace_bytes(lib):
    buf = (C.c_int64 * 64)()
    f = lib.lib.aki_mma_grad_sq_norm_workspace_bytes
    assert f(None, 1) == 0 and f(_list(lib, buf=buf), 0) == 0 and f(_list(lib, buf=buf, numel=-1), 2) == 0
    small = f(_list(lib, n=2, buf=buf), 2)                        # two chunks
    big = f(_list(lib, n=2, buf=buf, numel=3_000_000_000), 2)      # 64-bit element counts
    assert small >= 2 * 4 and small % 16 == 0
    assert big >= (1 + (3_000_000_000 + 16383) // 16384) * 4 and big % 16 == 0


def test_akiadamw_refuses_what_it_does_not_implement():
    from aki_b200 import AkiAdamW
    w = torch.nn.Parameter(torch.zeros(4))
    with pytest.raises(ValueError, match="CPU"):
        AkiAdamW([w])
    with pytest.raises(ValueError, match="fp32"):
        AkiAdamW([torch.nn.Parameter(torch.zeros(4, dtype=torch.bfloat16))])
    with pytest.raises(ValueError, match="sparse"):
        AkiAdamW([torch.nn.Parameter(torch.zeros(4, 4).to_sparse())])
    with pytest.raises(ValueError, match="non-leaf"):
        AkiAdamW([torch.zeros(4, requires_grad=True) * 2])
    with pytest.raises(ValueError, match="amsgrad"):
        AkiAdamW([w], amsgrad=True)
    with pytest.raises(ValueError, match="maximize"):
        AkiAdamW([w], maximize=True)
    for kw in (dict(lr=-1.0), dict(eps=-1.0), dict(betas=(1.0, 0.999)), dict(betas=(0.9, -0.1)), dict(weight_decay=-1.0),
               dict(max_grad_norm=0.0)):
        with pytest.raises(ValueError):
            AkiAdamW([w], **kw)


def test_use_bf16_weights_needs_the_fused_optimizer():
    from aki_b200 import use_bf16_weights
    lin = torch.nn.Linear(8, 8, bias=False)
    with pytest.raises(TypeError):
        use_bf16_weights(lin, torch.optim.AdamW(lin.parameters()))


def test_exports():
    import aki_b200
    for name in ("AkiAdamW", "use_bf16_weights", "unuse_bf16_weights"):
        assert name in aki_b200.__all__ and hasattr(aki_b200, name)
