"""Model-level input preparation: the drop-in for VLMWithLanguageStream._prepare_inputs_for_forward
(codes/open_flamingo/src/vlm.py:445-603) with identical arguments and return keys.  `attention_mask` stays the 2-D
spliced mask (B,T) and the extra key `mma_segments` carries the compact MMA description; `expand_to_4d()` on it
reproduces the reference's (B,1,T,T) int64 tensor bit-for-bit.  No Python loop over samples, no T^2 object."""
from __future__ import annotations

from typing import Optional

import torch

from . import ops

ASSISTANT_TOKEN_ID = 32001   # hard-coded in the reference (vlm.py:492)


def prepare_inputs_for_forward(self, vision_tokens: Optional[torch.Tensor], lang_x: torch.Tensor,
                               attention_mask: torch.Tensor, labels: Optional[torch.Tensor] = None,
                               past_key_values=None, vision_attention_mask: Optional[torch.Tensor] = None,
                               past_media_locations: Optional[torch.Tensor] = None,
                               past_vision_tokens: Optional[torch.Tensor] = None, padding_side: str = "left",
                               num_beams: int = 1, assistant_token_id: int = ASSISTANT_TOKEN_ID,
                               text_only: bool = False, exact_shape: bool = True):
    """`self` needs the attributes the reference method reads: lang_model (get_input_embeddings), media_token_id,
    num_tokens_per_vis, pad_token_id.  Call it unbound or bind it over the reference class."""
    if past_key_values is not None:                                                        # vlm.py:463-468
        pkv0 = past_key_values[0][0]
        past_len = pkv0.shape[2]
        assert attention_mask.shape[1] == past_len + lang_x.shape[1], (
            "Attention_mask must be as long as the entire past len (including image tokens) and current input IDs. "
            "Check that you've expanded the attention mask to account for past image tokens.")
    if vision_tokens is None:                                                              # vlm.py:470-475
        return {"input_ids": lang_x, "attention_mask": attention_mask, "labels": labels}
    N = int(self.num_tokens_per_vis)
    assert vision_tokens.shape[2] == N, (
        f"vision token number mismatch: image embedding ({vision_tokens.shape[2]}) vs. "
        f"model.num_tokens_per_vis ({N})")                                                 # vlm.py:525-528
    lang_embeds = self.lang_model.get_input_embeddings()(lang_x)                           # vlm.py:478
    B, L = lang_x.shape
    t_cap = L + vision_tokens.shape[1] * (N - 1)
    # a continuation (follow-up turn) describes its own tokens: the mask's last L columns; the cached rows keep theirs
    past_mask = attention_mask[:, :attention_mask.shape[1] - L] if past_key_values is not None else None
    segs = ops.build_segments(lang_x, attention_mask[:, -L:] if past_mask is not None else attention_mask, N,
                              int(self.media_token_id), assistant_token_id, t_cap=t_cap, text_only=text_only,
                              exact_shape=exact_shape)
    embeds, new_labels = ops.splice(lang_embeds.to(torch.bfloat16), vision_tokens, labels, segs,
                                    pad_value=float(self.pad_token_id), padding_side=padding_side)
    if torch.is_grad_enabled() and padding_side == "right" and (
            lang_embeds.requires_grad or (vision_tokens is not None and vision_tokens.requires_grad)):
        # training: same values, but with the scatter-add backward so that the embedding table / vision side train
        embeds = ops.splice_trainable(lang_embeds.to(torch.bfloat16), vision_tokens, segs, float(self.pad_token_id))
    mask = segs.spliced_mask_2d()
    if past_mask is not None:                 # HF's contract: the 2-D mask covers past + new tokens
        mask = torch.cat([past_mask.to(mask.dtype), mask], 1)
    return {"inputs_embeds": embeds.to(lang_embeds.dtype), "attention_mask": mask,
            "labels": new_labels, "mma_segments": segs}
