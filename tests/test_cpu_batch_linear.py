"""CPU-only: argument validation of aki_mma_batch_linear (the 9 - 64 token decode linear) returns the status codes of
aki_mma_skinny_linear for the same faults, before any launch or device query."""
import ctypes as C

import pytest

ERR_NULL, ERR_BAD_SHAPE, ERR_UNSUPPORTED, ERR_MISALIGNED = -1, -2, -3, -4


@pytest.fixture(scope="module")
def L():
    from aki_b200 import _lib
    return _lib.lib


def _call(L, x=True, xs=1024, w=True, rms=None, res=None, rs=0, y=True, ys=16, B=16, N=16, K=1024, mode=0, buf=None):
    p = C.cast(buf, C.c_void_p) if buf is not None else None
    return L.aki_mma_batch_linear(p if x else None, xs, p if w else None, rms, 1e-5, res, rs, p if y else None, ys, B, N,
                                  K, mode, None)


def test_batch_linear_status_codes(L):
    buf = (C.c_int64 * 64)()
    ok = C.cast(buf, C.c_void_p)
    assert _call(L, x=False, buf=buf) == ERR_NULL
    assert _call(L, w=False, buf=buf) == ERR_NULL
    assert _call(L, y=False, buf=buf) == ERR_NULL
    assert _call(L, B=0, buf=buf) == ERR_BAD_SHAPE
    assert _call(L, B=65, buf=buf) == ERR_BAD_SHAPE
    assert _call(L, N=0, buf=buf) == ERR_BAD_SHAPE
    assert _call(L, mode=3, buf=buf) == ERR_BAD_SHAPE
    assert _call(L, N=24, buf=buf) == ERR_UNSUPPORTED                 # N % 16
    assert _call(L, K=1000, xs=1000, buf=buf) == ERR_UNSUPPORTED      # K % 64
    assert _call(L, mode=1, buf=buf) == ERR_NULL                      # residual epilogue without a residual
    assert _call(L, mode=0, res=ok, rs=16, buf=buf) == ERR_NULL        # a residual outside the residual epilogue
    assert _call(L, mode=2, res=ok, rs=16, buf=buf) == ERR_NULL
    assert _call(L, xs=1028, buf=buf) == ERR_UNSUPPORTED              # x row stride not a multiple of 8
    assert _call(L, xs=512, buf=buf) == ERR_UNSUPPORTED               # rows overlap (x_stride < K)
    odd = C.c_void_p(ok.value + 2)
    assert _call(L, rms=odd, buf=buf) == ERR_MISALIGNED


def test_batch_linear_split_status_codes(L):
    assert L.aki_mma_batch_linear_split(0, 16, 1024, 0) == ERR_BAD_SHAPE
    assert L.aki_mma_batch_linear_split(65, 16, 1024, 0) == ERR_BAD_SHAPE
    assert L.aki_mma_batch_linear_split(16, 24, 1024, 0) == ERR_UNSUPPORTED
    assert L.aki_mma_batch_linear_split(16, 16, 1000, 0) == ERR_UNSUPPORTED
