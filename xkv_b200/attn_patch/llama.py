"""Llama attention forward for the xKV cache (reference: xKV/attn_patch/llama.py:19-88).

Semantics kept from the reference:
* RoPE is applied to Q only before the cache is touched (llama.py:39-40);
* prefill hands the PRE-RoPE keys plus cos/sin to ``cache.update(..., mode='prefill')`` and then
  attends on the ORIGINAL keys/values (llama.py:45-50) — compression only affects later decode steps;
* decode appends the post-RoPE keys (llama.py:51-53) and attends over the cache;
* only the sdpa attention implementation is accepted (llama.py:55-56);
* a sliding-window layer whose context exceeds the window attends through SDPA with transformers' mask
  (mistral.py:69): the fused kernel has no window, so it is bypassed there.
What differs: the reference calls every q_len > 1 forward a prefill; here only the first forward of a layer is
(``is_prefill_step``: several tokens, empty layer).  A later multi-token forward (assisted decoding verifying a
draft, a second chunk of a prompt) is a decode step of q_len tokens, causal among themselves: the fused kernel takes
it within its bounds, past them ``cache.attend`` declines and the dense path runs with transformers' causal mask.
Also: the decode step calls ``cache.attend`` — the fused reconstruct + RoPE + GQA-softmax kernel over
the stored factors — instead of SDPA over dense reconstructed tensors.  Written against the installed
transformers (``past_key_values`` kwarg; the reference's ``past_key_value`` spelling is accepted too).
"""
from __future__ import annotations

import types
from typing import Optional, Tuple

import torch
from transformers.cache_utils import Cache
from transformers.modeling_utils import ALL_ATTENTION_FUNCTIONS
from transformers.models.llama.modeling_llama import LlamaAttention, apply_rotary_pos_emb

from ..customized_cache.fake_layer_merge_dynamic_cache import FakeLayerMergingCache, is_prefill_step


def _heads(proj, hidden_states: torch.Tensor, head_dim: int) -> torch.Tensor:
    """(bs, q_len, hidden) -> (bs, heads, q_len, head_dim) view of a projection's output."""
    bs, q_len = hidden_states.shape[:2]
    return proj(hidden_states).view(bs, q_len, -1, head_dim).transpose(1, 2)


def _rope(x: torch.Tensor, cos: torch.Tensor, sin: torch.Tensor) -> torch.Tensor:
    return apply_rotary_pos_emb(x, x, cos, sin)[0]


def _dense_attention(module, q, k, v, attention_mask, **kwargs):
    if module.config._attn_implementation != "sdpa":
        raise ValueError("Only sdpa is supported for now")
    return ALL_ATTENTION_FUNCTIONS["sdpa"](module, q, k, v, attention_mask, scaling=module.scaling,
                                           dropout=module.attention_dropout if module.training else 0.0, **kwargs)


def xKV_llama_forward(  # noqa: N802
    self,
    hidden_states: torch.Tensor,
    position_embeddings: Tuple[torch.Tensor, torch.Tensor] = None,
    attention_mask: Optional[torch.Tensor] = None,
    past_key_values: Optional[Cache] = None,
    past_key_value: Optional[Cache] = None,
    cache_position: Optional[torch.LongTensor] = None,
    **kwargs,
):
    cache = past_key_value if past_key_values is None else past_key_values
    out_shape = (*hidden_states.shape[:-1], -1)
    cos, sin = position_embeddings
    q = _rope(_heads(self.q_proj, hidden_states, self.head_dim), cos, sin)
    k_pre = _heads(self.k_proj, hidden_states, self.head_dim)       # PRE-RoPE: what the cache compresses
    v = _heads(self.v_proj, hidden_states, self.head_dim)
    k = _rope(k_pre, cos, sin)

    if cache is not None and is_prefill_step(cache, self.layer_idx, hidden_states.shape[1]):
        # prefill: the cache gets the pre-RoPE keys and the tables; attention below runs on the ORIGINAL K / V
        assert isinstance(cache, FakeLayerMergingCache)
        cache.update(k_pre, v, self.layer_idx, mode="prefill", cos=cos, sin=sin, return_dense=False)
    elif cache is not None:
        # decode: fused attention over the factored cache when the layer's group is factored, else the dense path.
        # The fused kernel attends over EVERY cached token; a sliding-window layer (Mistral / Qwen2 checkpoints with
        # config.sliding_window, reference mistral.py:69) whose context has outgrown its window must honour the mask
        # transformers built, so it takes the dense path (materialised K^ / V^ + SDPA with that mask).
        window = kwargs.get("sliding_window")
        windowed = window is not None and cache.get_seq_length(self.layer_idx) + hidden_states.shape[1] > window
        if isinstance(cache, FakeLayerMergingCache) and getattr(self, "xkv_fused_decode", True) and not windowed:
            fused = cache.attend(q, k, v, self.layer_idx, self.scaling, key_pre_rope=k_pre, cos=cos, sin=sin)
            if fused is not None:
                return self.o_proj(fused.transpose(1, 2).reshape(out_shape).contiguous()), None
        k, v = cache.update(k, v, self.layer_idx, mode="decode")

    attn_output, attn_weights = _dense_attention(self, q, k, v, attention_mask, **kwargs)
    return self.o_proj(attn_output.reshape(out_shape).contiguous()), attn_weights


def _bind(model, expected_cls, forward, what: str):
    for layer in model.model.layers:
        module = layer.self_attn
        if not isinstance(module, expected_cls):
            raise ValueError(f"Only {what} is supported for now")
        module.forward = types.MethodType(forward, module)


def enable_llama_xKV_eval(model):  # noqa: N802
    """Rebind every layer's ``self_attn.forward`` (reference llama.py:77-88)."""
    _bind(model, LlamaAttention, xKV_llama_forward, "LlamaAttention")
