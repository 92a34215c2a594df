"""CPU: which decode path ``FakeLayerMergingCache.attend`` takes for each state of a layer group (both sides factored, one
side factored with the other kept dense, nothing factored, past the bounds), with stub layer states and the ops replaced
by recorders; and that decode tokens are never folded into a one-sided group."""
from types import SimpleNamespace

import pytest
import torch

from xkv_b200 import ops
from xkv_b200.configurations import generate_consecutive_xKV_config
from xkv_b200.customized_cache.fake_layer_merge_dynamic_cache import FakeLayerMergingCache, _GroupState, _XkvLayer

HQ, H, D, S = 8, 2, 4, 10


def _factors(rank):
    return SimpleNamespace(A_storage=torch.zeros(S + 4, rank), V=torch.zeros(2 * H * D, rank), rank=rank)


def _cache(key, value, compress_decode_tokens=False):
    """Two layers of one group; `key` / `value`: True = factored, False = kept dense (the merge's dense slot)."""
    cfg = generate_consecutive_xKV_config(num_layers=2, end_layer=-1, group_size=2, rank_k=8, rank_v=8)
    cache = FakeLayerMergingCache(cfg, compress_decode_tokens=compress_decode_tokens)
    factors = SimpleNamespace(key=_factors(6) if key else None, value=_factors(8) if value else None)
    st = _GroupState(None, factors, H, D, torch.ones(S, D), torch.zeros(S, D), True)
    st.layer_ids = [0, 1]
    st.length = st.prefill_tokens = S
    for i in range(2):
        layer = _XkvLayer()
        layer.group, layer.index_in_group, layer.prefill_len = st, i, S
        dense = torch.randn(1, S, H, D).transpose(1, 2)           # (1, H, S, D) view of token-major storage
        layer.dense_k = None if key else dense
        layer.dense_v = None if value else dense.clone()
        cache.layers.append(layer)
    return cache


@pytest.fixture
def recorded(monkeypatch):
    calls = []

    def both(q, a_k, vk, a_v, vv, h, cos, sin, k_tail, v_tail, scale, **kw):
        calls.append(("both", dict(a_k=a_k, a_v=a_v, cos=cos)))
        return torch.zeros_like(q)

    def half(q, h, **kw):
        calls.append(("half", kw))
        return torch.zeros_like(q)

    monkeypatch.setattr(ops, "decode_attention", both)
    monkeypatch.setattr(ops, "decode_attention_half", half)
    monkeypatch.setattr(ops, "decode_workspace_bytes", lambda *a: 64)
    monkeypatch.setattr(ops, "decode_half_workspace_bytes", lambda *a: 64)
    monkeypatch.setattr(ops, "pack_group", lambda *a, **k: pytest.fail("a one-sided group must not fold"))
    return calls


def _step(cache, layer_idx, tq=1, **kw):
    q = torch.randn(1, HQ, tq, D)
    k, v = torch.randn(1, H, tq, D), torch.randn(1, H, tq, D)
    return cache.attend(q, k, v, layer_idx, 0.5, **kw)


def test_both_factored_runs_the_fused_kernel(recorded):
    out = _step(_cache(True, True), 0)
    assert out.shape == (1, HQ, 1, D) and [c[0] for c in recorded] == ["both"]


@pytest.mark.parametrize("key,value", [(True, False), (False, True)])
def test_one_sided_groups_run_the_half_kernel(recorded, key, value):
    cache = _cache(key, value)
    out = _step(cache, 1, tq=3)
    assert out.shape == (1, HQ, 3, D)
    (name, kw), = recorded
    assert name == "half"
    factored, dense = ("a_k", "v_dense") if key else ("a_v", "k_dense")
    assert kw[factored] is not None and kw[factored].shape[0] == S
    slot = kw[dense]
    assert slot.shape == (S, H, D) and slot.stride(-1) == 1                       # token-major view, read in place
    src = cache.layers[1].dense_v if key else cache.layers[1].dense_k
    assert slot.data_ptr() == src.data_ptr() and torch.equal(slot, src[0].transpose(0, 1))
    assert kw["k_dense" if key else "a_k"] is None and kw["a_v" if key else "v_dense"] is None
    assert (kw["cos"] is not None) == key                                         # RoPE only for a factored key side
    assert cache.layers[1].tail_len == 3


def test_a_cropped_dense_slot_is_passed_at_its_length(recorded):
    cache = _cache(True, False)
    for layer in cache.layers:
        layer.crop(7)                                                              # right after the prefill
    _step(cache, 0)
    assert recorded[0][1]["v_dense"].shape == (7, H, D) and recorded[0][1]["a_k"].shape[0] == 7


def test_nothing_factored_or_past_the_bounds_declines(recorded):
    cache = _cache(False, False)
    assert _step(cache, 0) is None
    cache = _cache(True, False)
    cache.layers[0].dense_v = None                                                 # no dense slot to read
    assert _step(cache, 0) is None
    cache = _cache(False, True)
    assert _step(cache, 0, tq=17) is None                                          # 4 q heads per kv head x 17 tokens
    assert cache.layers[0].tail_len == 0 and recorded == []


@pytest.mark.parametrize("key,value", [(True, False), (False, True)])
def test_one_sided_groups_fold_nothing(recorded, key, value):
    cache = _cache(key, value, compress_decode_tokens=True)
    st = cache.layers[0].group
    for li in (0, 1):
        _step(cache, li, key_pre_rope=torch.randn(1, H, 1, D), cos=torch.ones(1, 1, D), sin=torch.zeros(1, 1, D))
    assert all(l.tail_len == 1 and l.tail_kpre is None for l in cache.layers)     # decode tokens stay dense and exact
    assert st.length == S and st.tail_rope == []
    cache._fold_tail(st)                                                           # a direct call does nothing either
    assert all(l.tail_len == 1 and l.prefill_len == S for l in cache.layers)
