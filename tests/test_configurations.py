"""CPU: the configuration surface mirrors the reference's (xKV/configurations.py) — names, defaults,
per-group override rules, YAML schema and the errors it raises."""
import glob
import os

import pytest

from xkv_b200.configurations import (
    LayerGroup,
    generate_consecutive_layer_groups,
    generate_consecutive_xKV_config,
    xKVConfig,
)

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
# a checkout of the original xKV repository, when one is at hand: the reference-parity tests below read it
REFERENCE = os.environ.get("XKV_REFERENCE_ROOT", "")


def test_defaults_match_reference():
    cfg = xKVConfig()
    assert (cfg.num_layers, cfg.layer_merge_impl, cfg.rank_k, cfg.rank_v) == (None, "svd", None, None)
    assert (cfg.slerp_t, cfg.slerp_gamma, cfg.merge_key, cfg.merge_value) == (0.5, 1.0, True, True)
    assert cfg.layer_groups == [] and cfg.extra_kwargs == {}
    gen = generate_consecutive_xKV_config()
    assert (gen.rank_k, gen.rank_v, len(gen.layer_groups)) == (256, 768, 16)  # layers 0..31 in pairs


def test_group_parameters_are_finalised_per_impl():
    cfg = xKVConfig(rank_k=128, rank_v=32, slerp_t=0.9, layer_groups=[
        LayerGroup(layers=[0, 1], rank_k=256, rank_v=64, slerp_t=0.1),
        LayerGroup(layers=[2, 3]),
        LayerGroup(layers=[4, 5], rank_k=64),
    ])
    g = cfg.layer_groups
    assert (g[0].rank_k, g[0].rank_v) == (256, 64) and (g[1].rank_k, g[1].rank_v) == (128, 32)
    assert (g[2].rank_k, g[2].rank_v) == (64, 32)
    assert all(x.slerp_t is None and x.slerp_gamma is None for x in g)
    cfg = xKVConfig(layer_merge_impl="slerp", rank_k=9, slerp_t=0.75, slerp_gamma=0.05,
                    layer_groups=[LayerGroup(layers=[0, 1], slerp_t=0.95), LayerGroup(layers=[2, 3], slerp_gamma=0.2)])
    g = cfg.layer_groups
    assert (g[0].slerp_t, g[0].slerp_gamma) == (0.95, 0.05) and (g[1].slerp_t, g[1].slerp_gamma) == (0.75, 0.2)
    assert all(x.rank_k is None and x.rank_v is None for x in g)


def test_errors():
    with pytest.raises(ValueError, match="at least one layer"):
        LayerGroup(layers=[])
    with pytest.raises(ValueError, match="Invalid layer_merge_impl"):
        xKVConfig(layer_merge_impl="pca")
    with pytest.raises(ValueError, match="appears in multiple groups"):
        xKVConfig(layer_groups=[LayerGroup(layers=[0, 1]), LayerGroup(layers=[1, 2])])
    with pytest.raises(ValueError, match="exceeds"):
        xKVConfig(num_layers=4, layer_groups=[LayerGroup(layers=[3, 4])])
    with pytest.raises(AssertionError):
        generate_consecutive_xKV_config(end_layer=-1)


def test_layer_lookup_and_consecutive_groups():
    groups = generate_consecutive_layer_groups(0, 5, 2)
    assert [g.layers for g in groups] == [[0, 1], [2, 3], [4, 5]]
    groups = generate_consecutive_layer_groups(2, 8, 4)   # last group is short
    assert [g.layers for g in groups] == [[2, 3, 4, 5], [6, 7, 8]]
    cfg = generate_consecutive_xKV_config(num_layers=32, start_layer=4, end_layer=-1, group_size=4, rank_k=512, rank_v=768)
    assert cfg.get_group_for_layer(3) is None
    assert cfg.get_group_for_layer(4).layers == [4, 5, 6, 7]
    assert cfg.get_group_for_layer(31).layers[-1] == 31 and cfg.get_group_for_layer(31).rank_k == 512
    # 27 layers in groups of 4: the last group has 3 layers (DeepSeek-V2-Lite, config 5)
    cfg = generate_consecutive_xKV_config(num_layers=27, end_layer=-1, group_size=4)
    assert cfg.layer_groups[-1].layers == [24, 25, 26]


def test_yaml_round_trip(tmp_path):
    cfg = xKVConfig(num_layers=12, rank_k=128, rank_v=64, merge_value=False, extra_kwargs={"note": "x"},
                    layer_groups=[LayerGroup(layers=[0, 1], rank_k=256), LayerGroup(layers=[2, 3])])
    path = tmp_path / "cfg.yaml"
    cfg.to_yaml(str(path))
    text = path.read_text()
    assert text.startswith("xKV_config:")
    with pytest.raises(TypeError):
        xKVConfig.from_yaml(str(path))  # reference behaviour: extra_kwargs are flattened and do not round-trip
    cfg.extra_kwargs = {}
    cfg.to_yaml(str(path))
    back = xKVConfig.from_yaml(str(path))
    assert back.num_layers == 12 and back.merge_value is False
    assert [(g.layers, g.rank_k, g.rank_v) for g in back.layer_groups] == [([0, 1], 256, 64), ([2, 3], 128, 64)]
    assert "2 groups" in str(back)


@pytest.mark.parametrize("path", sorted(glob.glob(os.path.join(ROOT, "configs", "*.yaml"))))
def test_shipped_configs_load(path):
    cfg = xKVConfig.from_yaml(path)
    assert cfg.layer_groups and cfg.num_layers is not None
    for g in cfg.layer_groups:
        assert cfg.get_group_for_layer(g.layers[0]) is g


@pytest.mark.skipif(not (REFERENCE and os.path.isdir(os.path.join(REFERENCE, "configs"))),
                    reason="needs XKV_REFERENCE_ROOT, a checkout of the original xKV repository")
@pytest.mark.parametrize("name", ["example.yaml", "example_xkv_config.yaml", "grouped_layers.yaml"])
def test_reference_yaml_files_load_unchanged(name):
    import importlib.util

    cfg = xKVConfig.from_yaml(os.path.join(REFERENCE, "configs", name))
    # the reference class, executed as the checker (loaded by path so it does not shadow the repo's xKV shim)
    spec = importlib.util.spec_from_file_location("_ref_xkv_configurations", os.path.join(REFERENCE, "xKV", "configurations.py"))
    mod = importlib.util.module_from_spec(spec)
    import sys

    sys.modules[spec.name] = mod      # dataclasses resolves string annotations through sys.modules
    spec.loader.exec_module(mod)
    RefConfig = mod.xKVConfig
    ref = RefConfig.from_yaml(os.path.join(REFERENCE, "configs", name))
    assert cfg.to_dict() == ref.to_dict()
    assert [(g.layers, g.rank_k, g.rank_v, g.slerp_t, g.slerp_gamma) for g in cfg.layer_groups] == \
           [(g.layers, g.rank_k, g.rank_v, g.slerp_t, g.slerp_gamma) for g in ref.layer_groups]
    assert str(cfg) == str(ref)
