"""ctypes binding of libaki_mma.so (C ABI: include/aki_mma.h).

The library is the product: there is no CPU or PyTorch fallback.  If the shared object is missing the import
fails loudly with the command that builds it.
"""
from __future__ import annotations

import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("AKI_MMA_LIB") or os.path.join(_HERE, "libaki_mma.so")   # AKI_MMA_LIB: A/B builds (tools only)

AKI_OK = 0
ABI_VERSION = 2
HEAD_DIM = 96
TILE = 128


class AkiMmaError(RuntimeError):
    pass


class Tensor4(C.Structure):
    _fields_ = [("ptr", C.c_void_p), ("stride_b", C.c_int64), ("stride_t", C.c_int64), ("stride_h", C.c_int64)]


class AttnParams(C.Structure):
    _fields_ = [
        ("B", C.c_int32), ("H", C.c_int32), ("T", C.c_int32), ("D", C.c_int32),
        ("scale", C.c_float),
        ("q", Tensor4), ("k", Tensor4), ("v", Tensor4), ("o", Tensor4),
        ("lse", C.c_void_p),
        ("rope_cos", C.c_void_p), ("rope_sin", C.c_void_p), ("rope_stride_b", C.c_int64),
        ("seq_len", C.c_void_p), ("row_lo", C.c_void_p), ("row_hi", C.c_void_p),
        ("kv_valid_bits", C.c_void_p), ("kv_mutual_bits", C.c_void_p),
        ("q_tile_kv_end", C.c_void_p), ("kv_tile_q_mask", C.c_void_p),
        ("meta_pitch", C.c_int32), ("bits_pitch", C.c_int32),
        ("fwd_plan", C.c_void_p), ("plan_pairs", C.c_int32), ("q_offset", C.c_int32),
    ]


class AttnBwdParams(C.Structure):
    _fields_ = [
        ("fwd", AttnParams),
        ("d_o", Tensor4), ("d_q", Tensor4), ("d_k", Tensor4), ("d_v", Tensor4),
        ("workspace", C.c_void_p), ("workspace_bytes", C.c_size_t),
        ("deterministic", C.c_int32),
    ]


class AdamWTensor(C.Structure):
    _fields_ = [("param", C.c_void_p), ("grad", C.c_void_p), ("exp_avg", C.c_void_p), ("exp_avg_sq", C.c_void_p),
                ("param_bf16", C.c_void_p), ("numel", C.c_int64)]


_SIGNATURES = {
    "aki_mma_abi_version": (C.c_int, []),
    "aki_mma_strerror": (C.c_char_p, [C.c_int]),
    "aki_mma_last_cuda_error": (C.c_char_p, []),
    "aki_mma_segments": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_int64, C.c_int64, C.c_int,
                                   C.c_int, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p,
                                   C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]),
    "aki_mma_tile_bounds": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_void_p,
                                      C.c_void_p, C.c_void_p]),
    "aki_mma_tile_bounds_at": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_int,
                                         C.c_void_p, C.c_void_p, C.c_void_p]),
    "aki_mma_fwd_plan": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_int,
                                   C.c_int, C.c_int, C.c_void_p, C.c_void_p]),
    "aki_mma_fwd_plan_at": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_int,
                                      C.c_int, C.c_int, C.c_int, C.c_void_p, C.c_void_p]),
    "aki_mma_expand_mask": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_int,
                                      C.c_int, C.c_void_p, C.c_void_p]),
    "aki_mma_splice": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_int,
                                 C.c_int, C.c_int, C.c_int, C.c_int, C.c_float, C.c_int, C.c_void_p, C.c_void_p,
                                 C.c_void_p]),
    "aki_mma_rope_table": (C.c_int, [C.c_void_p, C.c_void_p, C.c_float, C.c_int, C.c_int, C.c_int, C.c_void_p,
                                     C.c_void_p, C.c_void_p]),
    "aki_mma_rope_kv_write": (C.c_int, [C.c_void_p, C.c_int64, C.c_int64, C.c_void_p, C.c_void_p, C.c_int64, C.c_int,
                                        C.c_int, C.c_int, C.c_int, C.c_void_p, C.c_void_p, C.c_int64, C.c_int64,
                                        C.c_int, C.c_int, C.c_void_p, C.c_void_p]),
    "aki_mma_rope_kv_write_dev": (C.c_int, [C.c_void_p, C.c_int64, C.c_int64, C.c_void_p, C.c_void_p, C.c_int64, C.c_int,
                                            C.c_int, C.c_int, C.c_int, C.c_void_p, C.c_void_p, C.c_int64, C.c_int64,
                                            C.c_void_p, C.c_int, C.c_void_p, C.c_void_p]),
    "aki_mma_attn_fwd": (C.c_int, [C.POINTER(AttnParams), C.c_void_p]),
    "aki_mma_attn_bwd": (C.c_int, [C.POINTER(AttnBwdParams), C.c_void_p]),
    "aki_mma_attn_bwd_workspace_bytes": (C.c_size_t, [C.c_int, C.c_int, C.c_int, C.c_int]),
    "aki_mma_decode_workspace_bytes": (C.c_size_t, [C.c_int, C.c_int, C.c_int, C.c_int]),
    "aki_mma_decode": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int64, C.c_int64, C.c_void_p, C.c_void_p,
                                 C.c_int, C.c_int, C.c_int, C.c_int, C.c_float, C.c_void_p, C.c_void_p, C.c_size_t,
                                 C.c_void_p]),
    "aki_mma_decode_masked": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int64, C.c_int64, C.c_void_p, C.c_void_p,
                                        C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.c_float, C.c_void_p,
                                        C.c_void_p, C.c_size_t, C.c_void_p]),
    "aki_mma_skinny_linear": (C.c_int, [C.c_void_p, C.c_int64, C.c_void_p, C.c_void_p, C.c_float, C.c_void_p, C.c_int64,
                                        C.c_void_p, C.c_int64, C.c_int, C.c_int, C.c_int, C.c_int, C.c_void_p]),
    "aki_mma_batch_linear": (C.c_int, [C.c_void_p, C.c_int64, C.c_void_p, C.c_void_p, C.c_float, C.c_void_p, C.c_int64,
                                       C.c_void_p, C.c_int64, C.c_int, C.c_int, C.c_int, C.c_int, C.c_void_p]),
    "aki_mma_batch_linear_split": (C.c_int, [C.c_int, C.c_int, C.c_int, C.c_int]),
    "aki_mma_add_rmsnorm": (C.c_int, [C.c_void_p, C.c_int64, C.c_void_p, C.c_int64, C.c_void_p, C.c_float, C.c_void_p,
                                      C.c_int64, C.c_void_p, C.c_int64, C.c_int, C.c_int, C.c_void_p]),
    "aki_mma_swiglu": (C.c_int, [C.c_void_p, C.c_int64, C.c_void_p, C.c_int64, C.c_int, C.c_int, C.c_void_p]),
    "aki_mma_cross_entropy_fwd": (C.c_int, [C.c_void_p, C.c_int64, C.c_int64, C.c_void_p, C.c_int64, C.c_int, C.c_int, C.c_int,
                                            C.c_longlong, C.c_void_p, C.c_void_p, C.c_void_p]),
    "aki_mma_cross_entropy_bwd": (C.c_int, [C.c_void_p, C.c_int64, C.c_int64, C.c_void_p, C.c_int64, C.c_int, C.c_int, C.c_int,
                                            C.c_longlong, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int64, C.c_int64,
                                            C.c_void_p]),
    "aki_mma_add_rmsnorm_amp_fwd": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_float, C.c_void_p, C.c_void_p,
                                              C.c_void_p, C.c_int, C.c_int, C.c_void_p]),
    "aki_mma_rmsnorm_amp_bwd_partials": (C.c_int, [C.c_int]),
    "aki_mma_rmsnorm_amp_bwd": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p,
                                          C.c_void_p, C.c_int, C.c_int, C.c_void_p]),
    "aki_mma_swiglu_bwd": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_void_p]),
    "aki_mma_grad_sq_norm_workspace_bytes": (C.c_size_t, [C.c_void_p, C.c_int]),
    "aki_mma_grad_sq_norm": (C.c_int, [C.c_void_p, C.c_int, C.c_void_p, C.c_size_t, C.c_void_p, C.c_void_p]),
    "aki_mma_adamw_step": (C.c_int, [C.c_void_p, C.c_int, C.c_void_p, C.c_float, C.c_float, C.c_float, C.c_float, C.c_float,
                                     C.c_float, C.c_int64, C.c_void_p]),
    "aki_mma_set_timing_events": (C.c_int, [C.c_void_p, C.c_void_p]),
    "aki_mma_launch_count": (C.c_ulonglong, []),
    "aki_mma_attn_fwd_simt": (C.c_int, [C.POINTER(AttnParams), C.c_void_p]),
    "aki_mma_attn_bwd_simt": (C.c_int, [C.POINTER(AttnBwdParams), C.c_void_p]),
}

EXPORTED_SYMBOLS = tuple(_SIGNATURES)


def _load():
    if not os.path.exists(LIB_PATH):
        raise ImportError(
            f"{LIB_PATH} is missing: the CUDA library is the product and there is no fallback. Build it with "
            f"`python -c 'import __graft_entry__ as g; g.build()'` or `make -C aki_b200/csrc`.")
    lib = C.CDLL(LIB_PATH)
    for name, (res, args) in _SIGNATURES.items():
        fn = getattr(lib, name)          # AttributeError if the ABI is incomplete
        fn.restype = res
        fn.argtypes = args
    if lib.aki_mma_abi_version() != ABI_VERSION:
        raise ImportError(f"{LIB_PATH}: ABI version {lib.aki_mma_abi_version()} != {ABI_VERSION}; rebuild")
    return lib


lib = _load()


def check(status: int, what: str) -> None:
    if status != AKI_OK:
        msg = lib.aki_mma_strerror(status).decode()
        if status == -5:
            msg += ": " + lib.aki_mma_last_cuda_error().decode()
        raise AkiMmaError(f"{what} failed: {msg} (status {status})")
