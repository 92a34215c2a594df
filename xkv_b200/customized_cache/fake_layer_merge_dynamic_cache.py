"""``FakeLayerMergingCache`` on the B200 kernels.

Same public surface as the reference class (fake_layer_merge_dynamic_cache.py:103-213) —
``FakeLayerMergingCache(merge_setup)``, ``update(key, value, layer_idx, mode='prefill', cos=None, sin=None,
re_apply_rope=True)``, ``is_key_merged``/``is_value_merged``, ``grouped_layer_merging``, ``update_cache`` —
written against the installed transformers (layer-object caches).  What differs is what it *stores*:

* the reference multiplies the truncated SVD back and keeps dense K^/V^ for every layer;
* this cache keeps, per layer group, the factors ``A (S x r)`` and ``V (n x r)`` produced by
  :func:`xkv_b200.compress.compress_groups`, plus a dense tail of the tokens appended during decode
  (the reference never compresses those either: ``mode != 'prefill'`` skips merging, cache:131).

Dense per-layer tensors are only produced on request (``update`` must return them for API parity, and the
MLA caller uses the return value): ``K^_l = rope(bf16(A_k V_k[l]^T))`` through the tcgen05 GEMM engine and
the bf16 RoPE kernel.  The decode hot path does not go through that: the patched attention forward calls
:meth:`FakeLayerMergingCache.attend`, which runs the fused reconstruct+attention kernel.

``layer_merge_impl='slerp'`` (the MiniCache baseline, reference cache:183-197) runs the row-wise SLERP kernel and
keeps the merged layers dense, as the reference does.  Batch size 1 (every configuration of BASELINE.json); larger
batches raise ``XkvError``: the reference's batched SVD is one SVD per sample, and padded batches would need an
attention mask in the fused decode kernel.
"""
from __future__ import annotations

from typing import Dict, List, Optional, Tuple

import torch
from transformers.cache_utils import DynamicCache, DynamicLayer

from .. import compress, factorize, ops
from .._lib import XkvError
from ..configurations import LayerGroup, xKVConfig


def is_prefill_step(cache, layer_idx: int, q_len: int) -> bool:
    """The routing rule of the patched attention forwards: a forward is the prefill only when it brings several tokens
    to a layer that holds none yet.  Every later forward is a decode step of q_len tokens (one token, a speculative
    draft being verified, or a continuation chunk), appended exact to the dense tail."""
    return q_len > 1 and (cache is None or cache.get_seq_length(layer_idx) == 0)


class _XkvLayer(DynamicLayer):
    """One layer's slot: dense prefill K/V until its group is compressed, then (group factors, dense tail)."""

    def __init__(self):
        super().__init__()
        self.group: Optional["_GroupState"] = None   # set once the layer's group has been compressed
        self.index_in_group = 0
        self.prefill_len = 0
        self.tail_k: Optional[torch.Tensor] = None   # (1, H, T, D) post-RoPE keys appended during decode
        self.tail_v: Optional[torch.Tensor] = None
        self.tail_kpre: Optional[torch.Tensor] = None  # pre-RoPE copies, kept only when decode tokens get folded
        self.kpre_from = 0                           # first tail row whose pre-RoPE copy is valid (0 = all of them)
        self.tail_len = 0
        self.dense_k: Optional[torch.Tensor] = None  # a slot of a compressed group that stayed dense (merge flag off)
        self.dense_v: Optional[torch.Tensor] = None
        self.extras: Dict[str, torch.Tensor] = {}    # per-layer quantities callers derive once from the factors (MLA: 1 / rms)

    # --- sequence bookkeeping used by transformers' mask / position logic ---
    def get_seq_length(self) -> int:
        if self.group is None:
            return super().get_seq_length()
        return self.prefill_len + self.tail_len

    def append_tail(self, k: torch.Tensor, v: torch.Tensor, k_pre: Optional[torch.Tensor] = None) -> None:
        t = k.shape[-2]
        need = self.tail_len + t
        if self.tail_k is None or self.tail_k.shape[-2] < need:
            cap = max(64, 2 * need)
            new_k = torch.empty(k.shape[0], k.shape[1], cap, k.shape[3], dtype=k.dtype, device=k.device)
            new_v = torch.empty(v.shape[0], v.shape[1], cap, v.shape[3], dtype=v.dtype, device=v.device)  # MLA: other width
            new_p = torch.empty_like(new_k) if (k_pre is not None or self.tail_kpre is not None) else None
            if new_p is not None and self.tail_kpre is None:
                self.kpre_from = self.tail_len       # rows appended before pre-RoPE copies were kept cannot be folded
            if self.tail_len:
                new_k[:, :, : self.tail_len] = self.tail_k[:, :, : self.tail_len]
                new_v[:, :, : self.tail_len] = self.tail_v[:, :, : self.tail_len]
                if new_p is not None and self.tail_kpre is not None:
                    new_p[:, :, : self.tail_len] = self.tail_kpre[:, :, : self.tail_len]
            self.tail_k, self.tail_v, self.tail_kpre = new_k, new_v, new_p
        if k_pre is not None and self.tail_kpre is None:   # the buffer predates the first pre-RoPE copy
            self.tail_kpre = torch.empty_like(self.tail_k)
            self.kpre_from = self.tail_len
        self.tail_k[:, :, self.tail_len:need] = k
        self.tail_v[:, :, self.tail_len:need] = v
        if k_pre is not None:
            self.tail_kpre[:, :, self.tail_len:need] = k_pre
        elif self.tail_kpre is not None:
            self.kpre_from = need                    # a token without a pre-RoPE copy: nothing up to here can be folded
        self.tail_len = need

    def check_crop(self, max_length: int) -> int:
        """Tokens a compressed layer keeps after crop(max_length); XkvError when that cuts into the compressed prefix.
        One exception: right after the prefill (no decode token yet, nothing folded), the prefill's own last tokens
        may be dropped -- assisted decoding verifies its first drafts in the prefill forward.  Their token-factor rows
        are cut; the group's basis, fitted with them, stays."""
        current = self.get_seq_length()
        keep = current - abs(max_length) if max_length < 0 else max_length
        fresh = self.tail_len == 0 and self.group.length == self.group.prefill_tokens
        if keep < current and keep < self.prefill_len and not (fresh and keep >= 1):
            raise XkvError(f"FakeLayerMergingCache.crop: cannot crop to {keep} tokens, below the {self.prefill_len} "
                           "tokens already compressed into the layer group's factors")
        return keep

    def crop(self, max_length: int) -> None:
        """Keep the first ``max_length`` tokens (negative: drop ``-max_length``), as ``DynamicLayer.crop``.  A compressed
        layer loses tokens of its dense tail; its compressed prefix is cut only in the case check_crop allows."""
        if self.group is None:
            return super().crop(max_length)
        keep = self.check_crop(max_length)
        if keep >= self.get_seq_length():
            return
        if keep < self.prefill_len:                  # the prefill's last tokens (check_crop allowed it)
            self.prefill_len = self.group.length = keep
            self.group.prefill_tokens = keep
            for name in ("dense_k", "dense_v"):
                if getattr(self, name) is not None:
                    setattr(self, name, getattr(self, name)[..., :keep, :])
        self.tail_len = keep - self.prefill_len
        # RoPE rows waiting for the fold belong to the tail tokens: the rejected ones leave with them
        del self.group.tail_rope[self.tail_len:]


class _GroupState:
    """Factors of one compressed group and the RoPE tables of its prefill positions."""

    def __init__(self, info: LayerGroup, factors: compress.GroupFactors, heads: int, head_dim: int,
                 cos: Optional[torch.Tensor], sin: Optional[torch.Tensor], re_apply_rope: bool):
        self.info = info
        self.factors = factors
        self.heads = heads
        self.head_dim = head_dim
        self.cos = cos      # (S, D) bf16 or None
        self.sin = sin
        self.re_apply_rope = re_apply_rope
        self.length = 0            # tokens in the factors (prefill, then folded decode tokens)
        self.prefill_tokens = 0    # of which the prefill compressed
        # RoPE rows (cos, sin) of the decode tokens waiting in the dense tails, one per token (recorded when the group's
        # first layer sees the token); consumed when the tokens are folded into the factors, trimmed by crop()
        self.tail_rope: List[Tuple[torch.Tensor, torch.Tensor]] = []


class FakeLayerMergingCache(DynamicCache):
    def __init__(self, merge_setup: xKVConfig, compress_decode_tokens: bool = False, decode_capacity: int = 4096):
        """``compress_decode_tokens`` (extension, off by default: the reference keeps decode tokens exact,
        cache:131): once every layer of a group has seen a decode token, its pre-RoPE key / value rows are
        projected onto the group's right factors (xkv_append_project) and leave the dense tail.  Up to
        ``decode_capacity`` tokens can be folded per group."""
        super().__init__()
        self.compress_decode_tokens = compress_decode_tokens
        self.decode_capacity = decode_capacity if compress_decode_tokens else 0
        self.layer_class_to_replicate = _XkvLayer
        self.num_layers = merge_setup.num_layers
        self.merge_setup = merge_setup
        self._groups: Dict[int, _GroupState] = {}
        self._workspace: Optional[torch.Tensor] = None
        self._merge_cos_sin = (None, None, True)     # (cos, sin, re_apply_rope) of the prefill call being merged
        self.num_heads: Optional[int] = None
        self.head_dim: Optional[int] = None

    # ------------------------------------------------------------------ reference surface
    def _should_merge(self, layer_idx: int) -> bool:
        """True when ``layer_idx`` is the last layer of its group (reference cache:113-119)."""
        info = self.merge_setup.get_group_for_layer(layer_idx)
        return info is not None and layer_idx == info.layers[-1]

    def is_value_merged(self) -> bool:
        return self.merge_setup.merge_value

    def is_key_merged(self) -> bool:
        return self.merge_setup.merge_key

    def _layer(self, layer_idx: int) -> _XkvLayer:
        while len(self.layers) <= layer_idx:
            self.layers.append(_XkvLayer())
        return self.layers[layer_idx]

    def update(self, key, value, layer_idx, mode="prefill", cos=None, sin=None, re_apply_rope=True,
               return_dense=True):
        """Reference cache:127-153.  Prefill happens once, on an empty layer; every later forward is a decode step
        whatever its token count (speculative verification, a continuation chunk): the tokens are appended to the dense
        tail, exact, and nothing is re-compressed (the reference assumes a single prefill, SURVEY 9.7; this extends it).
        Prefill: stash the layer's (pre-RoPE) K and V; when the last layer of a group arrives, compress the group; keys of un-grouped layers get RoPE immediately.  Decode: append
        the (post-RoPE) token to the dense tail.  Returns dense (K_l, V_l) as the reference does;
        ``return_dense=False`` (an extension used by callers that ignore the return, llama.py:46-49) skips
        the materialisation."""
        layer = self._layer(layer_idx)
        if mode != "prefill":
            if layer.group is None:
                return DynamicLayer.update(layer, key, value)
            layer.append_tail(key, value)
            return self.materialize(layer_idx) if return_dense else (None, None)
        if key.shape[0] != 1:
            raise XkvError("FakeLayerMergingCache: batch size 1 only on the B200 path")
        if layer.group is not None:
            # The reference would re-run its SVD on a cache whose keys already carry RoPE (SURVEY.md section 9.7: a
            # single prefill call is assumed); here the dense prefill tensors are gone, so say so instead of failing
            # inside torch.cat.
            raise XkvError(f"FakeLayerMergingCache: layer {layer_idx} is already compressed; a second prefill-mode update "
                           "(chunked prefill, multi-turn reuse of one cache object) is not supported -- use a fresh cache")
        self.num_heads = key.shape[1]
        self.head_dim = key.shape[3]
        info = self.merge_setup.get_group_for_layer(layer_idx)
        if info is None:
            # un-grouped layer: exact cache, RoPE applied now (reference cache:149-152)
            if re_apply_rope:
                key = self._rope_dense(key, cos, sin)
            return DynamicLayer.update(layer, key, value)
        # Stash the layer's prefill tensors AS THEY ARE (views of the projections' token-major output): the reference's
        # cat-append (cache:129) would copy them into head-major tensors, and the factorisation reads token-major layer
        # tensors in place (no gather, no packed copy).  A grouped layer sees exactly one prefill call (checked above).
        if not layer.is_initialized:
            layer.lazy_initialization(key, value)
        elif layer.keys is not None and layer.keys.numel() > 0:
            raise XkvError(f"FakeLayerMergingCache: layer {layer_idx} already holds prefill tokens; chunked prefill of a "
                           "grouped layer is not supported (the reference assumes a single prefill call, SURVEY.md 9.7)")
        layer.keys, layer.values = key, value
        if self._should_merge(layer_idx):
            self._merge_cos_sin = (cos, sin, re_apply_rope)
            self.grouped_layer_merging(layer_idx)
        if not return_dense:
            return None, None
        return self.materialize(layer_idx) if layer.group is not None else (layer.keys, layer.values)

    @torch.no_grad()
    def grouped_layer_merging(self, last_layer_idx: int) -> None:
        """Reference cache:155-208 (svd branch): gather the group's layers, factorise K and V, drop the dense
        copies.  Stream-ordered; no host synchronisation (the reference's cuda.synchronize/gc at :205-208 is
        not a contract)."""
        info = self.merge_setup.get_group_for_layer(last_layer_idx)
        if info is None:
            return
        first, last = info.layers[0], info.layers[-1]
        ids = list(range(first, last + 1))            # the reference assumes contiguous groups (cache:165)
        layers = [self._layer(i) for i in ids]
        keys = [l.keys for l in layers]
        values = [l.values for l in layers]
        seq = keys[0].shape[-2]
        if self.merge_setup.layer_merge_impl == "slerp":
            self._slerp_merge(info, layers, keys, values)
            return
        if self.merge_setup.layer_merge_impl != "svd":
            raise NotImplementedError(f"Unknown implementation: {self.merge_setup.layer_merge_impl}")
        merge_k = self.merge_setup.merge_key and self._rank_fits(info.rank_k, seq, len(ids))
        merge_v = self.merge_setup.merge_value and self._rank_fits(info.rank_v, seq, len(ids))
        if not (merge_k or merge_v):
            cos, sin, re_rope = self._merge_cos_sin
            if re_rope:       # nothing to compress (rank >= min(m, n) is a no-op in the reference, §9.6)
                for l in layers:
                    l.keys = self._rope_dense(l.keys, cos, sin)
            return
        (gf,) = compress.compress_groups([keys], [values], info.rank_k, info.rank_v, merge_key=merge_k,
                                         merge_value=merge_v, layer_ids=[ids],
                                         extra_rows=self.decode_capacity)
        cos, sin, re_rope = self._merge_cos_sin
        cs = sn = None
        if re_rope and cos is not None:
            cs = torch.empty(seq + self.decode_capacity, cos.shape[-1], dtype=torch.bfloat16, device=cos.device)
            sn = torch.empty_like(cs)
            cs[:seq] = cos[0]
            sn[:seq] = sin[0]
        state = _GroupState(info, gf, self.num_heads, self.head_dim, cs, sn, bool(re_rope))
        state.length = seq
        state.prefill_tokens = seq                   # compressed by the prefill itself (crop may still cut those)
        state.layer_ids = ids
        self._groups[first] = state
        for pos, l in enumerate(layers):
            l.group = state
            l.index_in_group = pos
            l.prefill_len = seq
            # dense copies of whatever was factorised are released; a slot that stayed dense keeps its tensor
            if gf.key is None:
                l.dense_k = self._rope_dense(keys[pos], cos, sin) if re_rope else keys[pos]
            l.dense_v = values[pos] if gf.value is None else None
            l.keys = l.values = None

    def _slerp_merge(self, info: LayerGroup, layers, keys, values) -> None:
        """MiniCache baseline (reference cache:183-197, fake_minicache_merge :93-100): row-wise SLERP of the two
        layers of a group. The result is dense (nothing is compressed in storage), so these layers stay on the
        dense cache path; keys get RoPE afterwards like every merged group (cache:142-148)."""
        assert len(keys) == 2 and len(values) == 2, "SLERP only supports group size 2"
        cos, sin, re_rope = self._merge_cos_sin

        def merge(pair):
            bs, h, s, d = pair[0].shape
            rows = [t.transpose(1, 2).reshape(bs * s * h, d) for t in pair]     # token-major rows (view when possible)
            rows = [r if r.stride(1) == 1 and r.stride(0) == d else r.contiguous() for r in rows]
            e1, e2 = ops.slerp_merge(rows[0], rows[1], float(info.slerp_t), float(info.slerp_gamma))
            return [e.view(bs, s, h, d).transpose(1, 2) for e in (e1, e2)]

        new_k = merge(keys) if self.merge_setup.merge_key else list(keys)
        new_v = merge(values) if self.merge_setup.merge_value else list(values)
        for l, k, v in zip(layers, new_k, new_v):
            l.keys = self._rope_dense(k, cos, sin) if re_rope else k
            l.values = v

    def _rank_fits(self, rank: Optional[int], seq: int, nlayers: int) -> bool:
        if rank is None:
            return False
        n = nlayers * self.num_heads * self.head_dim
        # rank >= min(m, n) is a no-op in the reference (slicing past the end, cache:21-23): the slot stays dense
        return 0 < rank < min(seq, n) and factorize.sketch_width(rank) <= n

    def update_cache(self, layer_idx, key_approx, value_approx):
        """Reference cache:210-213: overwrite a layer's dense tensors (kept for API parity; a layer whose
        group has been factorised becomes dense again)."""
        layer = self._layer(layer_idx)
        layer.group = None
        layer.keys, layer.values = key_approx, value_approx
        layer.is_initialized = True

    # ------------------------------------------------------------------ dense views (API parity path)
    def _rope_dense(self, k: torch.Tensor, cos: torch.Tensor, sin: torch.Tensor) -> torch.Tensor:
        """HF apply_rotary_pos_emb on (1, H, S, D) keys via the bf16 RoPE kernel."""
        bs, h, s, d = k.shape
        # token-major COPY: the caller's tensor must stay pre-RoPE (llama.py:50 rotates it again for prefill attention)
        x = torch.empty(s, h, d, dtype=k.dtype, device=k.device)
        x.copy_(k[0].transpose(0, 1))
        ops.rope_bf16_(x, cos[0].to(torch.bfloat16).contiguous(), sin[0].to(torch.bfloat16).contiguous())
        return x.view(1, s, h, d).transpose(1, 2)

    @torch.no_grad()
    def materialize(self, layer_idx: int) -> Tuple[torch.Tensor, torch.Tensor]:
        """Dense (K_l, V_l) of a compressed layer: rope(bf16(A_k V_k[l]^T)) || tail — what the reference keeps
        in ``key_cache[l]`` / ``value_cache[l]`` after prefill."""
        layer = self._layer(layer_idx)
        st = layer.group
        if st is None:
            return layer.keys, layer.values
        h, d, s = st.heads, st.head_dim, layer.prefill_len
        rows = slice(layer.index_in_group * h * d, (layer.index_in_group + 1) * h * d)

        def dense(f: Optional[factorize.Factors], kept: Optional[torch.Tensor], rope: bool) -> torch.Tensor:
            if f is None:
                return kept
            x = torch.empty(s, h * d, dtype=torch.bfloat16, device=f.A.device)
            ops.gemm_grouped([ops.make_problem([f.A_storage[:s]], [f.V[rows]], x, M=s, N=h * d, K=f.rank)])
            if rope and st.cos is not None:
                ops.rope_bf16_(x.view(s, h, d), st.cos[:s], st.sin[:s])
            return x.view(1, s, h, d).transpose(1, 2)

        k = dense(st.factors.key, layer.dense_k, st.re_apply_rope)
        v = dense(st.factors.value, layer.dense_v, False)
        if layer.tail_len:
            k = torch.cat([k, layer.tail_k[:, :, : layer.tail_len]], dim=-2)
            v = torch.cat([v, layer.tail_v[:, :, : layer.tail_len]], dim=-2)
        return k, v

    # ------------------------------------------------------------------ decode hot path
    @torch.no_grad()
    def attend(self, query: torch.Tensor, key: torch.Tensor, value: torch.Tensor, layer_idx: int,
               scaling: float, key_pre_rope: Optional[torch.Tensor] = None, cos: Optional[torch.Tensor] = None,
               sin: Optional[torch.Tensor] = None) -> Optional[torch.Tensor]:
        """Decode step of one layer: append the Tq new (post-RoPE) tokens and attend over the factored cache with
        the fused kernel, causally among the new tokens.  query (1, Hq, Tq, D) -> (1, Hq, Tq, D).  Returns None, having
        appended nothing, when the layer is not factored on both sides or the step is past the fused kernel's bounds
        ((Hq / H) * Tq > 64 or Hq * Tq > 512); the caller then uses the dense path.  key_pre_rope / cos / sin of the new
        positions are only needed when decode tokens are folded into the factors (compress_decode_tokens); the fold
        runs at single-token steps only, since the tokens of a multi-token step may still be rejected (crop)."""
        layer = self._layer(layer_idx)
        st = layer.group
        if st is None or st.factors.key is None or st.factors.value is None:
            return None
        hq, tq = query.shape[1], query.shape[2]
        h, d = st.heads, st.head_dim
        if (hq // h) * tq > 64 or hq * tq > 512:
            return None
        fold = self.compress_decode_tokens and key_pre_rope is not None
        layer.append_tail(key, value, key_pre_rope if fold else None)
        if fold and layer_idx == st.layer_ids[0] and st.re_apply_rope and cos is not None:
            cs = cos.reshape(-1, cos.shape[-1])[-tq:].to(torch.bfloat16)
            sn = sin.reshape(-1, sin.shape[-1])[-tq:].to(torch.bfloat16)
            st.tail_rope.extend(zip(cs, sn))
        rows = slice(layer.index_in_group * h * d, (layer.index_in_group + 1) * h * d)
        fk, fv = st.factors.key, st.factors.value
        need = ops.decode_workspace_bytes(hq * tq, layer.prefill_len, layer.tail_len, fv.rank)
        if self._workspace is None or self._workspace.numel() < need:
            self._workspace = torch.empty(int(need * 1.25) + 4096, dtype=torch.uint8, device=query.device)
        n_tok = layer.prefill_len
        out = ops.decode_attention(
            query[0, :, 0, :] if tq == 1 else query[0], fk.A_storage[:n_tok], fk.V[rows], fv.A_storage[:n_tok], fv.V[rows],
            h, st.cos[:n_tok] if st.re_apply_rope else None, st.sin[:n_tok] if st.re_apply_rope else None,
            layer.tail_k[0, :, : layer.tail_len], layer.tail_v[0, :, : layer.tail_len], scaling,
            workspace=self._workspace)
        if fold and tq == 1 and layer_idx == st.layer_ids[-1]:
            self._fold_tail(st)
        return out[None, :, None, :] if tq == 1 else out[None]

    @torch.no_grad()
    def latent_slot(self, key: torch.Tensor, value: torch.Tensor, layer_idx: int) -> Optional[dict]:
        """Decode step of a layer whose KEY slot is factored and whose VALUE slot stayed dense and needs no RoPE — the MLA
        layout (reference deepseek_v2.py:217-232: latents in the key slot, rotated k_pe in the value slot,
        re_apply_rope=False, merge_value off).  Appends the new token to the dense tails and hands the caller the pieces
        of the layer's cache WITHOUT materialising the latents:
          A (S, r) token factor of the group, V (D, r) this layer's rows of the right factor (latent_t = V a_t),
          v_prefix (S, Dv) the dense value slot of the prefill tokens, k_tail (T, D) / v_tail (T, Dv) the decode tokens,
          extras: a dict that lives as long as the layer's cache entry (callers memoise derived quantities in it).
        Returns None when the layer is not in that state (the caller then uses update(mode='decode'))."""
        layer = self._layer(layer_idx)
        st = layer.group
        if (st is None or st.factors.key is None or st.factors.value is not None or st.re_apply_rope or st.heads != 1
                or layer.dense_v is None or key.shape[2] != 1):
            return None
        layer.append_tail(key, value)
        d = st.head_dim
        rows = slice(layer.index_in_group * d, (layer.index_in_group + 1) * d)
        fk = st.factors.key
        n_tok, t = layer.prefill_len, layer.tail_len
        return {"A": fk.A_storage[:n_tok], "V": fk.V[rows], "v_prefix": layer.dense_v[0, 0, :n_tok],
                "k_tail": layer.tail_k[0, 0, :t], "v_tail": layer.tail_v[0, 0, :t], "extras": layer.extras}

    @torch.no_grad()
    def _fold_tail(self, st: "_GroupState") -> None:
        """North-star step 4: every layer of the group has now seen the same T tail tokens; gather their
        pre-RoPE keys / values into the group's token-major rows, project them onto the right factors and
        append the result to A_k / A_v.  The tokens leave the dense tails.  Each token's RoPE row was recorded when
        it was appended (``st.tail_rope``); if the tails are not uniform (a layer took the dense path for a step, a
        pre-RoPE copy is missing, a RoPE row is missing) nothing is folded and the tokens simply stay dense (exact)."""
        layers = [self._layer(i) for i in st.layer_ids]
        t = layers[0].tail_len
        if t == 0 or any(l.tail_len != t or l.tail_kpre is None or l.kpre_from > 0 for l in layers):
            return
        if st.re_apply_rope and st.cos is not None and len(st.tail_rope) != t:
            return
        fk, fv = st.factors.key, st.factors.value
        if st.length + t > fk.A_storage.shape[0]:
            return   # capacity exhausted: keep the tokens dense (still exact)
        xk = ops.pack_group([l.tail_kpre[:, :, :t] for l in layers])[0]
        xv = ops.pack_group([l.tail_v[:, :, :t] for l in layers])[0]
        ops.append_project_many([xk, xv], [fk.V, fv.V], [fk.A_storage[st.length: st.length + t],
                                                         fv.A_storage[st.length: st.length + t]])
        if st.re_apply_rope and st.cos is not None:
            st.cos[st.length: st.length + t] = torch.stack([c for c, _ in st.tail_rope])
            st.sin[st.length: st.length + t] = torch.stack([x for _, x in st.tail_rope])
        st.tail_rope.clear()
        st.length += t
        for l in layers:
            l.prefill_len = st.length
            l.tail_len = 0
            l.kpre_from = 0

    # ------------------------------------------------------------------ cache surgery
    def crop(self, max_length: int):
        """Drop tokens from the end (assisted / speculative decoding rejects drafted tokens this way).  Compressed layers
        lose tokens of their dense tail; cropping into a group's compressed tokens raises ``XkvError`` and leaves the
        cache as it was, except right after the prefill (``_XkvLayer.check_crop``).  Un-grouped layers crop as
        ``DynamicLayer`` does."""
        for l in self.layers:
            if getattr(l, "group", None) is not None:
                l.check_crop(max_length)
        return super().crop(max_length)

    def _refuse_if_compressed(self, what: str) -> None:
        if any(getattr(l, "group", None) is not None for l in self.layers):
            raise XkvError(f"FakeLayerMergingCache.{what}: not supported once layer groups are factorised (beam search "
                           "and batch > 1 need per-sample caches)")

    def batch_repeat_interleave(self, repeats: int):
        self._refuse_if_compressed("batch_repeat_interleave")
        return super().batch_repeat_interleave(repeats)

    def batch_select_indices(self, indices: torch.Tensor):
        self._refuse_if_compressed("batch_select_indices")
        return super().batch_select_indices(indices)

    def reorder_cache(self, beam_idx: torch.LongTensor):
        self._refuse_if_compressed("reorder_cache")
        return super().reorder_cache(beam_idx)
