"""CLI glue (reference utils.py:68-137): flag names, defaults and the configuration they produce."""
import argparse
import os
import re
import sys
import types

import pytest

from xkv_b200 import cli
from xkv_b200.configurations import xKVConfig

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
# a checkout of the original xKV repository, when one is at hand: the reference-parity test below reads it
REFERENCE = os.environ.get("XKV_REFERENCE_ROOT", "")


def _parse(argv):
    return cli.add_common_args(argparse.ArgumentParser()).parse_args(argv)


def test_reference_defaults():
    a = _parse([])
    assert (a.rank_k, a.rank_v, a.layer_group_size) == (256, 768, 1)
    assert (a.layer_merge_impl, a.slerp_t, a.slerp_gamma) == ("svd", 0.5, 0.05)
    assert a.merge_key is False and a.merge_value is False and a.xKV is False and a.flash2 is False
    assert (a.start_layer_idx, a.end_layer_idx, a.customized_merge_config) == (0, -1, None)


def test_readme_abbreviations_work():
    # README.md:88 spells the flags --merge_k / --merge_v: argparse prefix matching resolves them
    a = _parse(["--xKV", "--merge_k", "--merge_v", "--rank_k", "512", "--rank_v", "768", "--layer_group_size", "4"])
    assert a.merge_key and a.merge_value and a.xKV and a.rank_k == 512 and a.layer_group_size == 4


def test_config_from_flags_matches_consecutive_groups():
    a = _parse(["--merge_key", "--merge_value", "--rank_k", "512", "--layer_group_size", "4"])
    cfg = cli.config_from_args(a, 32)
    assert cfg.num_layers == 32 and cfg.rank_k == 512 and cfg.rank_v == 768
    assert [g.layers for g in cfg.layer_groups] == [list(range(i, i + 4)) for i in range(0, 32, 4)]
    # end_layer_idx = -1 means the last layer; a window of layers leaves the others un-grouped
    b = _parse(["--start_layer_idx", "4", "--end_layer_idx", "13", "--layer_group_size", "4"])
    cfg = cli.config_from_args(b, 32)
    assert [g.layers for g in cfg.layer_groups] == [[4, 5, 6, 7], [8, 9, 10, 11], [12, 13]]
    assert cfg.merge_key is False and cfg.get_group_for_layer(0) is None


def test_customized_merge_config_wins():
    path = os.path.join(ROOT, "configs", sorted(os.listdir(os.path.join(ROOT, "configs")))[0])
    a = _parse(["--customized_merge_config", path, "--rank_k", "17", "--layer_group_size", "9"])
    cfg = cli.config_from_args(a, 32)
    assert cfg.to_dict() == xKVConfig.from_yaml(path).to_dict()


def test_apply_patch_installs_config_and_cache_factory():
    transformers = pytest.importorskip("transformers")
    import torch
    from transformers import LlamaConfig, LlamaForCausalLM

    from xkv_b200.customized_cache import FakeLayerMergingCache

    torch.manual_seed(0)
    model = LlamaForCausalLM(LlamaConfig(hidden_size=64, intermediate_size=128, num_hidden_layers=4,
                                         num_attention_heads=4, num_key_value_heads=2, vocab_size=128))
    a = _parse(["--merge_key", "--merge_value", "--rank_k", "8", "--rank_v", "8", "--layer_group_size", "2"])
    out = cli.apply_kv_compress_patch(model, a)
    assert out is model and model.kv_compress_config.num_layers == 4
    kwargs = {}
    model._prepare_cache_for_generation(None, kwargs)
    assert isinstance(kwargs["past_key_values"], FakeLayerMergingCache)


def test_root_utils_module_reexports():
    sys.path.insert(0, ROOT)
    import utils as root_utils

    assert root_utils.add_common_args is cli.add_common_args
    assert root_utils.apply_kv_compress_patch is cli.apply_kv_compress_patch


@pytest.mark.skipif(not (REFERENCE and os.path.isfile(os.path.join(REFERENCE, "utils.py"))),
                    reason="needs XKV_REFERENCE_ROOT, a checkout of the original xKV repository")
def test_flags_equal_the_reference_parser():
    """Every add_argument call of the reference's add_common_args (utils.py:96-137), read from its source text (the
    module itself imports loguru / the HF hub stack), against the parser built here: same flags, defaults, actions."""
    src = open(os.path.join(REFERENCE, "utils.py")).read()
    body = src[src.index("def add_common_args"):]
    calls = re.findall(r"add_argument\(\s*(['\"])(--[\w]+)\1(.*?)\)\s*\n", body, flags=re.S)
    ours = {a.option_strings[0]: a for a in cli.add_common_args(argparse.ArgumentParser())._actions if a.option_strings
            and a.option_strings[0] != "-h"}
    assert {c[1] for c in calls} == set(ours)
    for _, flag, rest in calls:
        act = ours[flag]
        if "store_true" in rest:
            assert isinstance(act, argparse._StoreTrueAction) and act.default is False
        m = re.search(r"default\s*=\s*([^,\s)]+)", rest)
        if m:
            assert act.default == eval(m.group(1))   # noqa: S307 - literals from the reference source
