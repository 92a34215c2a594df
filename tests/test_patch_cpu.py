"""CPU: the patch entry point mirrors the reference's (xKV/patch.py:32-73): constructor contract, dispatch on
model_type, forward rebinding, fresh cache per generate() call.  No kernels run here."""
import types

import pytest
import torch

from xkv_b200.configurations import generate_consecutive_xKV_config
from xkv_b200.patch import KVCompress, prepare_cache


def _tiny_llama():
    from transformers import LlamaConfig, LlamaForCausalLM

    cfg = LlamaConfig(hidden_size=64, intermediate_size=128, num_hidden_layers=2, num_attention_heads=4,
                      num_key_value_heads=2, head_dim=16, vocab_size=128, max_position_embeddings=256)
    cfg._attn_implementation = "sdpa"
    torch.manual_seed(0)
    return LlamaForCausalLM(cfg)


def test_constructor_contract(tmp_path):
    with pytest.raises(ValueError, match="Must provide either xKV_config or yaml_path"):
        KVCompress()
    cfg = generate_consecutive_xKV_config(num_layers=2, end_layer=-1, group_size=2, rank_k=8, rank_v=8)
    assert KVCompress(xKV_config=cfg).config is cfg
    path = tmp_path / "c.yaml"
    cfg.to_yaml(str(path))
    assert KVCompress(yaml_path=str(path)).config.layer_groups[0].layers == [0, 1]


def test_patch_rebinds_forwards_and_cache_factory():
    from xkv_b200.attn_patch.llama import xKV_llama_forward
    from xkv_b200.customized_cache import FakeLayerMergingCache

    model = _tiny_llama()
    cfg = generate_consecutive_xKV_config(num_layers=2, end_layer=-1, group_size=2, rank_k=8, rank_v=8)
    out = KVCompress(xKV_config=cfg)(model)
    assert out is model and model.kv_compress_config is cfg
    for layer in model.model.layers:
        assert isinstance(layer.self_attn.forward, types.MethodType)
        assert layer.self_attn.forward.__func__ is xKV_llama_forward
    kw1, kw2 = {}, {}
    model._prepare_cache_for_generation(None, kw1, None, 1, 16)
    model._prepare_cache_for_generation(None, kw2, None, 1, 16)
    assert isinstance(kw1["past_key_values"], FakeLayerMergingCache)
    assert kw1["past_key_values"] is not kw2["past_key_values"]        # a fresh cache per generate() call


def test_unknown_method_and_model_type():
    from transformers.cache_utils import DynamicCache

    fn = prepare_cache("not-a-method", None)
    kw = {}
    fn(None, None, kw)
    assert type(kw["past_key_values"]) is DynamicCache
    model = _tiny_llama()
    model.config.model_type = "gpt_neox"
    with pytest.raises(ValueError, match="Model type not supported"):
        KVCompress(xKV_config=generate_consecutive_xKV_config(num_layers=2, end_layer=1))(model)
    model.config.model_type = "deepseek_v2"      # dispatches to the MLA patch, which rejects Llama attention modules
    with pytest.raises(ValueError, match="DeepseekV2Attention"):
        KVCompress(xKV_config=generate_consecutive_xKV_config(num_layers=2, end_layer=1))(model)


def test_reference_import_paths_resolve():
    import xKV.attn_patch.llama as a
    import xKV.configurations as c
    import xKV.customized_cache as cc
    import xKV.patch as p

    assert p.KVCompress is KVCompress and "xKV" in cc.method_to_cache_obj
    assert c.xKVConfig.__name__ == "xKVConfig" and hasattr(a, "enable_llama_xKV_eval")


def test_ops_fail_loudly_without_a_gpu():
    from xkv_b200 import _lib, ops

    with pytest.raises(_lib.XkvError):
        ops.pack_group([torch.zeros(1, 1, 8, 8, dtype=torch.bfloat16)])
