"""GPU, model level: forwards of several tokens after the prefill (a continuation chunk, assisted decoding's draft
verification) and ``crop`` on a compressed cache, through the patched models of test_generate_gpu against the oracle's
dense cache."""
import pytest
import torch

from tests.test_generate_gpu import _mla_model, _model, _windowed_model

pytestmark = pytest.mark.gpu


def _gqa128_model():
    """GQA 4 at head_dim 128: the decode runs the CTA-pair score kernel."""
    from transformers import LlamaConfig, LlamaForCausalLM

    cfg = LlamaConfig(hidden_size=1024, intermediate_size=512, num_hidden_layers=4, num_attention_heads=8,
                      num_key_value_heads=2, head_dim=128, vocab_size=512, max_position_embeddings=4096,
                      rope_theta=500000.0)
    cfg._attn_implementation = "sdpa"
    torch.manual_seed(0)
    return LlamaForCausalLM(cfg).to(device="cuda", dtype=torch.bfloat16).eval()


MODELS = {"toy64": _model, "gqa128": _gqa128_model}


def _setup(name, rank_k=64, rank_v=128):
    from xkv_b200.configurations import generate_consecutive_xKV_config
    from xkv_b200.patch import KVCompress

    model = MODELS[name]()
    cfg = generate_consecutive_xKV_config(num_layers=4, end_layer=-1, group_size=2, rank_k=rank_k, rank_v=rank_v)
    KVCompress(xKV_config=cfg)(model)
    return model, cfg


def _fused(model, on):
    for layer in model.model.layers:
        layer.self_attn.xkv_fused_decode = on


def _ids(n, seed=1, vocab=512):
    return torch.randint(0, vocab, (1, n), device="cuda", generator=torch.Generator(device="cuda").manual_seed(seed))


class _Spy:
    """Counts calls of a module attribute; records the q rank of ops.decode_attention calls."""

    def __init__(self, owner, name):
        self.owner, self.name, self.calls = owner, name, []
        self.orig = getattr(owner, name)

    def __enter__(self):
        def wrapped(*a, **k):
            self.calls.append(a[0].dim() if self.name == "decode_attention" else 1)
            return self.orig(*a, **k)

        setattr(self.owner, self.name, wrapped)
        return self

    def __exit__(self, *exc):
        setattr(self.owner, self.name, self.orig)


@torch.no_grad()
@pytest.mark.parametrize("name", list(MODELS))
def test_continuation_matches_oracle_and_single_steps(name):
    from tests.oracle_cache import OracleCache
    from xkv_b200 import ops
    from xkv_b200.customized_cache import FakeLayerMergingCache

    model, cfg = _setup(name)
    prompt, chunk = _ids(700), _ids(5, seed=2)
    cache = FakeLayerMergingCache(cfg)
    model(input_ids=prompt, past_key_values=cache, use_cache=True)
    with _Spy(ops, "decode_attention") as spy:
        ours = model(input_ids=chunk, past_key_values=cache, use_cache=True).logits[0].float()
    assert spy.calls == [3] * 4                          # every layer took the fused multi-token kernel
    assert all(l.tail_len == 5 for l in cache.layers)
    one = FakeLayerMergingCache(cfg)
    model(input_ids=prompt, past_key_values=one, use_cache=True)
    single = torch.cat([model(input_ids=chunk[:, i:i + 1], past_key_values=one, use_cache=True).logits[0].float()
                        for i in range(5)])
    _fused(model, False)
    oracle = OracleCache(cfg)
    model(input_ids=prompt, past_key_values=oracle, use_cache=True)
    ref = model(input_ids=chunk, past_key_values=oracle, use_cache=True).logits[0].float()
    _fused(model, True)
    torch.cuda.synchronize()
    scale = ref.abs().max().item()
    dev, dev1 = (ours - ref).abs().max().item(), (ours - single).abs().max().item()
    print(f"{name}: 5-token step vs oracle {dev:.4f}, vs five single steps {dev1:.4f} (logit scale {scale:.3f})")
    assert dev <= 5e-2 * scale
    assert dev1 <= 1e-2 * scale


@torch.no_grad()
@pytest.mark.parametrize("name", list(MODELS))
def test_crop_rejected_tokens(name):
    from xkv_b200._lib import XkvError
    from xkv_b200.customized_cache import FakeLayerMergingCache

    model, cfg = _setup(name)
    prompt, draft, nxt = _ids(600), _ids(6, seed=3), _ids(1, seed=4)
    cache = FakeLayerMergingCache(cfg)
    model(input_ids=prompt, past_key_values=cache, use_cache=True)
    model(input_ids=draft, past_key_values=cache, use_cache=True)
    cache.crop(-4)                                        # 2 of the 6 drafted tokens accepted
    assert cache.get_seq_length() == 602 and all(l.tail_len == 2 for l in cache.layers)
    ours = model(input_ids=nxt, past_key_values=cache, use_cache=True).logits[0, -1].float()
    clean = FakeLayerMergingCache(cfg)
    model(input_ids=prompt, past_key_values=clean, use_cache=True)
    model(input_ids=draft[:, :2], past_key_values=clean, use_cache=True)
    ref = model(input_ids=nxt, past_key_values=clean, use_cache=True).logits[0, -1].float()
    torch.cuda.synchronize()
    assert (ours - ref).abs().max().item() <= 1e-3 * ref.abs().max().item()
    with pytest.raises(XkvError, match="compressed"):
        cache.crop(599)
    assert cache.get_seq_length() == 603                  # the refused crop left the cache as it was
    cache.crop(600)
    assert all(l.tail_len == 0 for l in cache.layers)


@torch.no_grad()
def test_assisted_decoding_matches_greedy():
    """generate(prompt_lookup_num_tokens=4) verifies drafts with multi-token forwards and crops the rejected tokens;
    on a repetitive prompt (48-token vocabulary) drafts are proposed and partly rejected."""
    from xkv_b200 import ops
    from xkv_b200.customized_cache import FakeLayerMergingCache

    model, _ = _setup("gqa128")
    ids = _ids(800, seed=5, vocab=48)
    greedy = model.generate(ids, max_new_tokens=32, do_sample=False, return_dict_in_generate=True, output_logits=True)
    with _Spy(ops, "decode_attention") as spy, _Spy(FakeLayerMergingCache, "crop") as crops:
        assisted = model.generate(ids, max_new_tokens=32, do_sample=False, prompt_lookup_num_tokens=4)
    torch.cuda.synchronize()
    assert 3 in spy.calls, "no fused multi-token step ran"
    assert crops.calls, "crop never ran"
    a, g = assisted[0, ids.shape[1]:], greedy.sequences[0, ids.shape[1]:]
    assert a.shape == g.shape
    diff = (a != g).nonzero()
    if len(diff):
        i = diff[0].item()
        top2 = greedy.logits[i][0].float().topk(2).values
        scale = torch.stack(greedy.logits).float().abs().max().item()
        assert (top2[0] - top2[1]).item() < 5e-2 * scale, f"first difference at step {i} is not a near tie"


@torch.no_grad()
def test_sliding_window_multi_token_step_takes_the_dense_path():
    from tests.oracle_cache import OracleCache
    from xkv_b200 import ops
    from xkv_b200.configurations import generate_consecutive_xKV_config
    from xkv_b200.customized_cache import FakeLayerMergingCache
    from xkv_b200.patch import KVCompress

    model = _windowed_model("mistral", 256)
    cfg = generate_consecutive_xKV_config(num_layers=4, end_layer=-1, group_size=2, rank_k=64, rank_v=128)
    KVCompress(xKV_config=cfg)(model)
    prompt, chunk = _ids(700), _ids(4, seed=2)
    cache = FakeLayerMergingCache(cfg)
    model(input_ids=prompt, past_key_values=cache, use_cache=True)
    with _Spy(ops, "decode_attention") as spy:
        ours = model(input_ids=chunk, past_key_values=cache, use_cache=True).logits[0].float()
    assert spy.calls == []
    _fused(model, False)
    oracle = OracleCache(cfg)
    model(input_ids=prompt, past_key_values=oracle, use_cache=True)
    ref = model(input_ids=chunk, past_key_values=oracle, use_cache=True).logits[0].float()
    torch.cuda.synchronize()
    assert (ours - ref).abs().max().item() <= 5e-2 * ref.abs().max().item()


@torch.no_grad()
def test_mla_multi_token_step_matches_oracle():
    from tests.oracle_cache import OracleCache
    from xkv_b200.configurations import generate_consecutive_xKV_config
    from xkv_b200.customized_cache import FakeLayerMergingCache
    from xkv_b200.patch import KVCompress

    model = _mla_model()
    cfg = generate_consecutive_xKV_config(num_layers=3, end_layer=-1, group_size=3, rank_k=256, rank_v=None,
                                          merge_value=False)
    KVCompress(xKV_config=cfg)(model)
    prompt, chunk = _ids(600, seed=2), _ids(4, seed=3)
    cache = FakeLayerMergingCache(cfg)
    model(input_ids=prompt, past_key_values=cache, use_cache=True)
    ours = model(input_ids=chunk, past_key_values=cache, use_cache=True).logits[0].float()
    oracle = OracleCache(cfg)
    model(input_ids=prompt, past_key_values=oracle, use_cache=True)
    ref = model(input_ids=chunk, past_key_values=oracle, use_cache=True).logits[0].float()
    torch.cuda.synchronize()
    assert cache.get_seq_length() == 604
    assert (ours - ref).abs().max().item() <= 5e-2 * ref.abs().max().item()


@torch.no_grad()
def test_fold_waits_for_a_single_token_step():
    from xkv_b200.customized_cache import FakeLayerMergingCache

    model, cfg = _setup("toy64")
    cache = FakeLayerMergingCache(cfg, compress_decode_tokens=True, decode_capacity=64)
    model(input_ids=_ids(500), past_key_values=cache, use_cache=True)
    model(input_ids=_ids(3, seed=2), past_key_values=cache, use_cache=True)
    assert all(l.prefill_len == 500 and l.tail_len == 3 for l in cache.layers)       # nothing folded at Tq = 3
    assert all(len(cache.layers[i].group.tail_rope) == 3 for i in (0, 2))
    model(input_ids=_ids(1, seed=3), past_key_values=cache, use_cache=True)
    assert all(l.prefill_len == 504 and l.tail_len == 0 for l in cache.layers)       # folded at the next single step
