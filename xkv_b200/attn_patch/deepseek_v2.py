"""DeepSeek-V2 (MLA) attention forward for the xKV cache (reference: xKV/attn_patch/deepseek_v2.py:160-302).

Semantics kept from the reference:
* the cache holds the LATENT ``compressed_kv`` (b, 1, l, kv_lora_rank) in the key slot and the RoPE'd ``k_pe``
  (b, 1, l, qk_rope_head_dim) in the value slot (:217-232);
* latents carry no RoPE, so ``re_apply_rope=False`` and ``cos = sin = None`` (:226, :231);
* only the latents are compressed: ``merge_value`` must be off (:222-223);
* the cache's return IS used, in prefill too (:224): the last layer of a group already attends on the
  compressed latents, earlier layers of the group on their exact ones (SURVEY.md §3 D);
* every step the (reconstructed) latents go through ``kv_a_layernorm`` + ``kv_b_proj`` (:235).
What differs: written against transformers' native ``DeepseekV2Attention`` (the reference patches the Hub's
remote-code ``DeepseekV2FlashAttention2``, which is not vendored), attention through the installed sdpa
interface instead of flash-attn 2.  Prefill gets the reconstructed latents from the factors through the tcgen05 GEMM
(``FakeLayerMergingCache.materialize``), as the reference's cache return requires.

Decode never rebuilds them.  The reference re-expands the WHOLE cache through ``kv_a_layernorm`` + ``kv_b_proj`` on
every step (:235); here the step runs in the factors' rank space (``_absorbed_decode``).  With the stored latent
``c_t = V_l a_t`` (``a_t``: row t of the group's token factor, ``V_l``: this layer's 512 rows of the right factor),
``kv_a_layernorm(c_t) = gamma o c_t / rms_t`` and ``kv_b_proj = [W_UK; W_UV]`` per head:

    q_nope[h] . k_nope[t,h] = (1 / rms_t) (V_l^T (gamma o W_UK[h]^T q_nope[h])) . a_t  =  (1 / rms_t) q_hat[h] . a_t
    sum_t p[h,t] v[t,h]     = W_UV[h] (gamma o V_l sum_t (p[h,t] / rms_t) a_t)

so one pass over ``A`` for the scores and one for the values replace the S x 512 reconstruction, the RMSNorm and the
S x 512 x (heads x 256) projection; ``1 / rms_t`` is computed once per layer (first decode step) and kept.  Decode tokens
stay dense and exact (cache:131) and join through a log-sum-exp merge.
"""
from __future__ import annotations

import types
from typing import Optional

import torch
from transformers.cache_utils import Cache
from transformers.modeling_utils import ALL_ATTENTION_FUNCTIONS
from transformers.models.deepseek_v2.modeling_deepseek_v2 import DeepseekV2Attention, apply_rotary_emb

from ..customized_cache.fake_layer_merge_dynamic_cache import FakeLayerMergingCache, is_prefill_step


def xKV_mla_forward(  # noqa: N802
    self,
    hidden_states: torch.Tensor,
    attention_mask: Optional[torch.Tensor] = None,
    past_key_values: Optional[Cache] = None,
    position_embeddings: Optional[torch.Tensor] = None,
    past_key_value: Optional[Cache] = None,
    **kwargs,
):
    cache = past_key_values if past_key_values is not None else past_key_value
    bsz, q_len = hidden_states.shape[:-1]
    # the first forward of a layer; later multi-token forwards are decode steps and take the dense path below
    # (latent_slot declines q_len > 1)
    is_prefill = is_prefill_step(cache, self.layer_idx, q_len)

    if self.q_lora_rank is None:
        q = self.q_proj(hidden_states)
    else:
        q = self.q_b_proj(self.q_a_layernorm(self.q_a_proj(hidden_states)))
    q = q.view(bsz, q_len, -1, self.qk_head_dim).transpose(1, 2)
    q_nope, q_pe = torch.split(q, [self.qk_nope_head_dim, self.qk_rope_head_dim], dim=-1)

    compressed_kv = self.kv_a_proj_with_mqa(hidden_states)
    compressed_kv, k_pe = torch.split(compressed_kv, [self.kv_lora_rank, self.qk_rope_head_dim], dim=-1)
    k_pe = k_pe.view(bsz, 1, q_len, self.qk_rope_head_dim)
    q_pe, k_pe = apply_rotary_emb(q_pe, k_pe, position_embeddings.to(q_pe.device))

    latent = compressed_kv.view(bsz, q_len, 1, self.kv_lora_rank).transpose(1, 2)   # (b, 1, l, kv_lora_rank)
    if (cache is not None and not is_prefill and isinstance(cache, FakeLayerMergingCache)
            and getattr(self, "xkv_fused_decode", True)):
        fused = _absorbed_decode(self, cache, q_nope, q_pe, latent, k_pe.contiguous())
        if fused is not None:
            return self.o_proj(fused.reshape(bsz, q_len, -1).contiguous()), None
    if cache is not None:
        if is_prefill:
            assert isinstance(cache, FakeLayerMergingCache)
            if cache.is_value_merged():
                raise ValueError("DeepseekV2Attention does not support --merge_v")
            latent, k_pe = cache.update(latent, k_pe.contiguous(), self.layer_idx, mode="prefill", cos=None, sin=None,
                                        re_apply_rope=False)
        else:
            latent, k_pe = cache.update(latent, k_pe.contiguous(), self.layer_idx, mode="decode", cos=None, sin=None,
                                        re_apply_rope=False)
    kv_len = latent.shape[-2]
    kv = self.kv_b_proj(self.kv_a_layernorm(latent.squeeze(1)))
    kv = kv.view(bsz, kv_len, -1, self.qk_nope_head_dim + self.v_head_dim).transpose(1, 2)
    k_nope, value_states = torch.split(kv, [self.qk_nope_head_dim, self.v_head_dim], dim=-1)

    query_states = torch.cat((q_nope, q_pe), dim=-1)
    key_states = torch.cat((k_nope, k_pe.expand(*k_nope.shape[:-1], -1)), dim=-1)

    if self.config._attn_implementation != "sdpa":
        raise ValueError("Only sdpa is supported for now")
    attention_interface = ALL_ATTENTION_FUNCTIONS["sdpa"]
    attn_output, attn_weights = attention_interface(
        self,
        query_states,
        key_states,
        value_states,
        attention_mask,
        dropout=0.0 if not self.training else self.attention_dropout,
        scaling=self.scaling,
        **kwargs,
    )
    attn_output = attn_output.reshape(bsz, q_len, -1).contiguous()
    return self.o_proj(attn_output), attn_weights


@torch.no_grad()
def _absorbed_decode(self, cache: FakeLayerMergingCache, q_nope, q_pe, latent, k_pe) -> Optional[torch.Tensor]:
    """One decode step of an MLA layer over the factored latent cache, in the rank space (see the module docstring).
    q_nope (1, Hq, 1, dn), q_pe (1, Hq, 1, dr), latent (1, 1, 1, C), k_pe (1, 1, 1, dr) -> (1, 1, Hq, dv) or None."""
    from .. import ops

    slot = cache.latent_slot(latent, k_pe, self.layer_idx)
    if slot is None:
        return None
    a, v_l, extras = slot["A"], slot["V"], slot["extras"]
    hq, dn, dv, c = q_nope.shape[1], self.qk_nope_head_dim, self.v_head_dim, self.kv_lora_rank
    gamma = self.kv_a_layernorm.weight.float()
    w = self.kv_b_proj.weight.view(hq, dn + dv, c).float()
    w_uk, w_uv = w[:, :dn], w[:, dn:]
    if "inv_rms" not in extras:
        # once per layer: 1 / rms of the reconstructed (bf16, as the reference stores them) latents
        s_tok = a.shape[0]
        lat = torch.empty(s_tok, c, dtype=torch.bfloat16, device=a.device)
        ops.gemm_grouped([ops.make_problem([a], [v_l], lat, M=s_tok, N=c, K=a.shape[1])])
        extras["inv_rms"] = torch.rsqrt(lat.float().pow(2).mean(-1) + self.kv_a_layernorm.variance_epsilon).contiguous()
        del lat
    qn, qp = q_nope[0, :, 0].float(), q_pe[0, :, 0]
    q_hat = ((torch.einsum("hd,hdc->hc", qn, w_uk) * gamma) @ v_l.float()).to(torch.bfloat16).contiguous()
    u, lse_p = ops.decode_absorbed(q_hat, a, self.scaling, row_scale=extras["inv_rms"], bias_q=qp.contiguous(),
                                   bias_k=slot["v_prefix"])
    out_p = torch.einsum("hc,hvc->hv", (u @ v_l.float().t()) * gamma, w_uv)
    # decode tokens (the new one included): dense, exact latents through the module's own layernorm + projection
    kv_t = self.kv_b_proj(self.kv_a_layernorm(slot["k_tail"])).view(-1, hq, dn + dv).float()
    s_t = (torch.einsum("hd,thd->ht", qn, kv_t[:, :, :dn]) + qp.float() @ slot["v_tail"].float().t()) * self.scaling
    lse_t = torch.logsumexp(s_t, dim=-1)
    out_t = torch.einsum("ht,thv->hv", torch.softmax(s_t, dim=-1), kv_t[:, :, dn:])
    lse = torch.logaddexp(lse_p, lse_t)
    out = torch.exp(lse_p - lse)[:, None] * out_p + torch.exp(lse_t - lse)[:, None] * out_t
    return out.to(q_nope.dtype)[None, None]


def enable_deepseek_v2_xKV_eval(model):  # noqa: N802
    """Rebind every MLA layer's forward (reference deepseek_v2.py:290-302)."""
    for layer in model.model.layers:
        module = layer.self_attn
        if not isinstance(module, DeepseekV2Attention):
            raise ValueError("Only DeepseekV2Attention is supported for now")
        module.forward = types.MethodType(xKV_mla_forward, module)
