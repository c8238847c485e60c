"""aki_b200 -- B200-native modality-mutual attention (MMA) for AKI's Phi-3.5-mini decoder layers.

Importing the package loads aki_b200/libaki_mma.so (C ABI: include/aki_mma.h); there is no fallback."""
from . import ops                                                    # noqa: F401  (loads the library)
from .attention import (AkiMMAAttention, aki_mma_attention, mma_context, register_attention_interface,   # noqa: F401
                        replace_phi3_attention)
from .cache import AkiKVCache                                        # noqa: F401
from .inputs import prepare_inputs_for_forward                       # noqa: F401
from .layers import fuse_phi3_elementwise, unfuse_phi3_elementwise   # noqa: F401
from .optim import AkiAdamW, unuse_bf16_weights, use_bf16_weights   # noqa: F401
from .ops import MMASegments, build_segments                         # noqa: F401
from .rope import LongRope, longrope_attention_factor               # noqa: F401

__all__ = ["AkiMMAAttention", "aki_mma_attention", "mma_context", "register_attention_interface", "replace_phi3_attention", "fuse_phi3_elementwise", "unfuse_phi3_elementwise",
           "AkiAdamW", "use_bf16_weights", "unuse_bf16_weights",
           "AkiKVCache", "prepare_inputs_for_forward", "MMASegments", "build_segments", "LongRope",
           "longrope_attention_factor", "ops"]
