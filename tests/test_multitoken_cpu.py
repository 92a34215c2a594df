"""CPU: host-side bookkeeping of multi-token steps -- the prefill / decode routing rule of the attention patches and
``crop`` on compressed layers (dense tail and RoPE rows trimmed, the compressed prefix refused)."""
import pytest
import torch
from transformers.cache_utils import DynamicLayer

from xkv_b200._lib import XkvError
from xkv_b200.configurations import generate_consecutive_xKV_config
from xkv_b200.customized_cache.fake_layer_merge_dynamic_cache import (FakeLayerMergingCache, _GroupState, _XkvLayer,
                                                                      is_prefill_step)

H, D = 2, 4


def _kv(t, seed=0):
    g = torch.Generator().manual_seed(seed)
    return torch.randn(1, H, t, D, generator=g), torch.randn(1, H, t, D, generator=g)


def _compressed_layer(prefill=10, tail=5, group=None):
    """A layer as grouped_layer_merging leaves it (factors are not touched by crop), plus `tail` decode tokens."""
    layer = _XkvLayer()
    layer.group = group or _GroupState(None, None, H, D, None, None, True)
    layer.prefill_len = prefill
    layer.append_tail(*_kv(tail))
    layer.group.tail_rope = [(torch.full((D,), float(i)), torch.zeros(D)) for i in range(tail)]
    return layer


def test_crop_trims_the_tail_and_its_rope_rows():
    layer = _compressed_layer()
    k_before = layer.tail_k[:, :, :5].clone()
    layer.crop(12)
    assert layer.get_seq_length() == 12 and layer.tail_len == 2
    assert [c[0].item() for c, _ in layer.group.tail_rope] == [0.0, 1.0]
    assert torch.equal(layer.tail_k[:, :, :2], k_before[:, :, :2])
    layer.crop(-1)                                     # negative: drop that many tokens, as in DynamicLayer.crop
    assert layer.tail_len == 1 and len(layer.group.tail_rope) == 1
    layer.crop(50)                                     # longer than the cache: nothing happens
    assert layer.tail_len == 1
    layer.append_tail(*_kv(3, seed=1))                 # appending after a crop overwrites the rejected rows
    assert layer.get_seq_length() == 14


def test_crop_below_the_compressed_length_raises():
    layer = _compressed_layer()
    with pytest.raises(XkvError, match="compressed"):
        layer.crop(9)
    with pytest.raises(XkvError):
        layer.crop(-6)
    assert layer.tail_len == 5
    layer.crop(10)                                     # exactly the compressed prefix: allowed
    assert layer.tail_len == 0 and layer.group.tail_rope == []
    layer.prefill_len = 14                             # after a fold the compressed length includes folded tokens
    layer.append_tail(*_kv(2))
    with pytest.raises(XkvError):
        layer.crop(13)


def test_cache_crop_is_all_or_nothing():
    cfg = generate_consecutive_xKV_config(num_layers=3, end_layer=-1, group_size=2, rank_k=8, rank_v=8)
    cache = FakeLayerMergingCache(cfg)
    st = _GroupState(None, None, H, D, None, None, True)
    cache.layers.extend([_compressed_layer(group=st), _compressed_layer(group=st), _XkvLayer()])
    DynamicLayer.update(cache.layers[2], *_kv(15))    # un-grouped layer: plain dense cache
    cache.crop(-3)
    assert [l.get_seq_length() for l in cache.layers] == [12, 12, 12]
    assert cache.layers[2].keys.shape[-2] == 12
    with pytest.raises(XkvError):
        cache.crop(8)
    assert [l.get_seq_length() for l in cache.layers] == [12, 12, 12]
    for what, arg in (("reorder_cache", torch.tensor([0])), ("batch_select_indices", torch.tensor([0])),
                      ("batch_repeat_interleave", 2)):
        with pytest.raises(XkvError):
            getattr(cache, what)(arg)


def test_routing_rule():
    cfg = generate_consecutive_xKV_config(num_layers=2, end_layer=-1, group_size=2, rank_k=8, rank_v=8)
    cache = FakeLayerMergingCache(cfg)
    assert is_prefill_step(cache, 0, 7)                # several tokens, empty layer: the prefill
    assert not is_prefill_step(cache, 0, 1)            # one token is always a decode step
    assert is_prefill_step(None, 0, 7)
    cache.layers.append(_compressed_layer())
    assert not is_prefill_step(cache, 0, 7)            # a later multi-token forward is a decode step
    assert is_prefill_step(cache, 1, 7)                # layer 1 holds nothing yet


def test_crop_may_cut_the_prefill_before_any_decode_step():
    """Assisted decoding verifies its first drafts in the prefill forward: right after the prefill, crop drops the
    prefill's last tokens (their token-factor rows); once a decode token arrived, the compressed prefix is fixed."""
    st = _GroupState(None, None, H, D, None, None, True)
    st.length = st.prefill_tokens = 10
    layers = [_compressed_layer(tail=0, group=st), _compressed_layer(tail=0, group=st)]
    layers[0].dense_v = torch.zeros(1, 1, 10, D)            # a slot that stayed dense is cut with the factors
    for l in layers:
        l.check_crop(7)
    for l in layers:
        l.crop(7)
    assert [l.get_seq_length() for l in layers] == [7, 7] and st.length == 7 and layers[0].dense_v.shape[-2] == 7
    layers[0].append_tail(*_kv(1))
    with pytest.raises(XkvError):
        layers[0].crop(6)
