"""GPU parity of the fused decode over one-sided groups (ops.decode_attention_half): one slot of the layer is factored, the
other is a dense prefix slot read in place.  Reference: the oracle's formula on the device -- the factored side rebuilt as
in test_decode_multi_gpu._oracle (bf16(A V_l^T), HF RoPE in bf16 for keys), the dense side used as given, the tail
concatenated, SDPA with the causal mask over the last Tq tail tokens.  Tolerance: bf16 (2e-2 of the output scale),
log-sum-exp as in test_decode_multi_gpu.  Then the model level: a patched random-init Llama with key-only, value-only and
rank-limited groups against the oracle cache, counting the fused one-sided calls."""
import math

import pytest
import torch

from tests.test_decode_gpu import VARIANTS, _set_variant
from tests.test_decode_multi_gpu import _inputs

pytestmark = pytest.mark.gpu

STATES = ("key_only", "value_only")   # which side is factored


def _half_inputs(S, H, D, qpk, Tq, T0, rk=256, rv=256, seed=0, shape="flat"):
    x = _inputs(S, H, D, qpk, Tq, T0, rk, rv, seed=seed, shape=shape)
    g = torch.Generator().manual_seed(seed + 100)
    x["k_dense"] = torch.randn(S, H, D, generator=g).bfloat16().cuda()   # rotated keys, token-major
    x["v_dense"] = torch.randn(S, H, D, generator=g).bfloat16().cuda()
    return x


def _layout(t, layout):
    """A token-major (S, H, D) slot as the view the call receives."""
    if layout == "token":
        return t
    if layout == "head":
        return t.transpose(0, 1).contiguous()                               # (H, S, D)
    # a view cropped to fewer tokens than its storage holds (a crop right after the prefill)
    big = torch.randn(t.shape[0] + 37, *t.shape[1:], device=t.device).bfloat16()
    big[: t.shape[0]] = t
    return big[: t.shape[0]]


def _oracle(x, H, Tq, state):
    from oracle import xkv_oracle as O

    S, D = x["a_k"].shape[0], x["q"].shape[-1]
    qpk = x["q"].shape[0] // H
    if state == "key_only":
        k_hat = (x["a_k"].float() @ x["v_k"].float().t()).bfloat16().view(S, H, D).permute(1, 0, 2)[None]
        k_hat = O.apply_rope(k_hat, x["cos"][None], x["sin"][None])[0]
        v_hat = x["v_dense"].permute(1, 0, 2)
    else:
        k_hat = x["k_dense"].permute(1, 0, 2)
        v_hat = (x["a_v"].float() @ x["v_v"].float().t()).bfloat16().view(S, H, D).permute(1, 0, 2)
    k = torch.cat([k_hat.float(), x["k_tail"].float()], 1).repeat_interleave(qpk, 0)
    v = torch.cat([v_hat.float(), x["v_tail"].float()], 1).repeat_interleave(qpk, 0)
    L = k.shape[1]
    sc = torch.einsum("htd,hld->htl", x["q"].float(), k) / math.sqrt(D)
    pos = torch.arange(L, device=sc.device)
    mask = pos[None, :] <= (L - Tq + torch.arange(Tq, device=sc.device))[:, None]
    sc = sc.masked_fill(~mask[None], float("-inf"))
    return torch.softmax(sc, -1) @ v, torch.logsumexp(sc, -1)


def _run(x, H, state, layout="token", **kw):
    from xkv_b200 import ops

    D = x["q"].shape[-1]
    if state == "key_only":
        sides = dict(a_k=x["a_k"], vk_layer=x["v_k"], v_dense=_layout(x["v_dense"], layout), cos=x["cos"], sin=x["sin"])
    else:
        sides = dict(a_v=x["a_v"], vv_layer=x["v_v"], k_dense=_layout(x["k_dense"], layout))
    return ops.decode_attention_half(x["q"], H, k_tail=x["k_tail"], v_tail=x["v_tail"], scale=1.0 / math.sqrt(D),
                                     **sides, **kw)


def _check(S, H, D, qpk, Tq, T0, state, rk=256, rv=256, shape="flat", layout="token", variant="auto", seed=0):
    x = _half_inputs(S, H, D, qpk, Tq, T0, rk, rv, seed=seed, shape=shape)
    _set_variant(variant)
    try:
        lse = torch.empty(H * qpk, Tq, dtype=torch.float32, device="cuda")
        out = _run(x, H, state, layout, lse_out=lse)
    finally:
        _set_variant("auto")
    ref, lse_ref = _oracle(x, H, Tq, state)
    torch.cuda.synchronize()
    assert out.shape == (H * qpk, Tq, D)
    err = (out.float() - ref).abs().max().item()
    scale = ref.abs().max().item()
    assert err <= 2e-2 * max(scale, 1e-3), f"max err {err} at output scale {scale}"
    lerr = ((lse - lse_ref).abs() - 1e-2 * lse_ref.abs()).max().item()
    assert lerr <= 2e-2, f"lse err {lerr}"


_TQ_QPK = [(tq, qpk) for tq in (1, 4, 16) for qpk in (1, 4, 8) if qpk * tq <= 64]


@pytest.mark.parametrize("state", STATES)
@pytest.mark.parametrize("D", [64, 128])
@pytest.mark.parametrize("Tq,qpk", _TQ_QPK)
@pytest.mark.parametrize("S,T0", [(100, 5), (4133, 0)])
def test_half_parity(S, T0, Tq, qpk, D, state):
    _check(S, 2, D, qpk, Tq, T0, state)


@pytest.mark.parametrize("state", STATES)
@pytest.mark.parametrize("D,shape", [(128, "sharp"), (64, "later"), (128, "later")])
def test_half_softmax_shapes(shape, D, state):
    """sharp: peaked softmax over the prefix; later: one later tail token dominates (the causal mask).  (sharp at head_dim
    64 is left out for the same reason as in test_decode_multi_gpu: the factored head_dim 64 FFMA scores path.)"""
    _check(4133, 2, D, 4, 4, 5, state, shape=shape, seed=1)


@pytest.mark.parametrize("variant", list(VARIANTS))
@pytest.mark.parametrize("D", [64, 128])
def test_key_only_every_scores_variant(D, variant):
    _check(4133, 2, D, 4, 4, 5, "key_only", variant=variant)


@pytest.mark.parametrize("state", STATES)
@pytest.mark.parametrize("layout", ["token", "head", "crop"])
@pytest.mark.parametrize("D", [64, 128])
def test_dense_slot_layouts(D, layout, state):
    _check(1000, 2, D, 4, 4, 5, state, layout=layout)


@pytest.mark.parametrize("state", STATES)
@pytest.mark.parametrize("Tq", [1, 8])
def test_half_config2_64k(Tq, state):
    """Config 2's layer shape: 32 q / 8 kv heads x 128, rank 512 / 768, a 64K prefix."""
    _check(65536, 8, 128, 4, Tq, 16, state, rk=512, rv=768)


@pytest.mark.parametrize("state", STATES)
def test_half_row_bounds(state):
    """64 rows per kv head (qpk 4 x Tq 16) and 512 rows in all (8 kv heads)."""
    _check(4133, 8, 128, 4, 16, 5, state)


@pytest.mark.parametrize("state", STATES)
@pytest.mark.parametrize("D", [64, 128])
def test_half_multi_token_equals_single_token_calls(D, state):
    H, qpk, Tq, T0 = 2, 4, 5, 7
    x = _half_inputs(1000, H, D, qpk, Tq, T0, seed=2)
    multi = _run(x, H, state)
    singles = [_run(dict(x, q=x["q"][:, t].contiguous(), k_tail=x["k_tail"][:, :T0 + t + 1],
                         v_tail=x["v_tail"][:, :T0 + t + 1]), H, state) for t in range(Tq)]
    torch.cuda.synchronize()
    single = torch.stack(singles, 1).float()
    assert (multi.float() - single).abs().max().item() <= 4e-3 * single.abs().max().item()


@pytest.mark.parametrize("state", STATES)
@pytest.mark.parametrize("D", [64, 128])
def test_exact_reconstruction_as_dense_slot_matches_both_factored(D, state):
    """A dense slot holding exactly the bf16 reconstruction (rotated, for keys) of a factor pair gives the fused
    both-factored result."""
    from oracle import xkv_oracle as O
    from xkv_b200 import ops

    S, H, qpk, Tq = 2000, 2, 4, 4
    x = _half_inputs(S, H, D, qpk, Tq, 5, seed=3)
    k_hat = (x["a_k"].float() @ x["v_k"].float().t()).bfloat16().view(S, H, D).permute(1, 0, 2)[None]
    x["k_dense"] = O.apply_rope(k_hat, x["cos"][None], x["sin"][None])[0].transpose(0, 1).contiguous()
    x["v_dense"] = (x["a_v"].float() @ x["v_v"].float().t()).bfloat16().view(S, H, D).contiguous()
    both = ops.decode_attention(x["q"], x["a_k"], x["v_k"], x["a_v"], x["v_v"], H, x["cos"], x["sin"], x["k_tail"],
                                x["v_tail"], 1.0 / math.sqrt(D))
    half = _run(x, H, state)
    torch.cuda.synchronize()
    assert (half.float() - both.float()).abs().max().item() <= 2e-2 * both.float().abs().max().item()


def test_half_errors():
    from xkv_b200 import ops
    from xkv_b200._lib import XkvError

    H, D = 2, 128
    x = _half_inputs(512, H, D, 4, 2, 3)
    kw = dict(k_tail=x["k_tail"], v_tail=x["v_tail"], scale=0.1)
    with pytest.raises(XkvError, match="exactly one side"):       # both factored
        ops.decode_attention_half(x["q"], H, a_k=x["a_k"], vk_layer=x["v_k"], a_v=x["a_v"], vv_layer=x["v_v"], **kw)
    with pytest.raises(XkvError, match="exactly one side"):       # both dense
        ops.decode_attention_half(x["q"], H, k_dense=x["k_dense"], v_dense=x["v_dense"], **kw)
    lib = ops._lib.load()
    with pytest.raises(XkvError, match="exactly one side"):       # the C ABI says the same, naming the alternatives
        ops.check(lib.xkv_decode_attention_half(
            ops._ptr(x["q"]), 8, 2, H, D, ops._ptr(x["a_k"]), 256, 256, ops._ptr(x["v_k"]), 256, None, 0, 0,
            ops._ptr(x["a_v"]), 256, 256, ops._ptr(x["v_v"]), 256, None, 0, 0, 512, None, None, 0, None, None, 0, 0, 0,
            ops.C.c_float(0.1), ops._ptr(x["q"]), ops._ptr(x["q"]), 0, None, None))
    with pytest.raises(XkvError, match="head_dim 96"):
        y = _half_inputs(512, H, 96, 4, 2, 3)
        ops.decode_attention_half(y["q"], H, a_v=y["a_v"], vv_layer=y["v_v"], k_dense=y["k_dense"], k_tail=y["k_tail"],
                                  v_tail=y["v_tail"], scale=0.1)
    with pytest.raises(XkvError, match="multiples of 8"):           # token stride H*D + 4 elements
        padded = torch.zeros(512, H * D + 4, device="cuda").bfloat16()
        padded[:, : H * D] = x["v_dense"].reshape(512, H * D)
        ops.decode_attention_half(x["q"], H, a_k=x["a_k"], vk_layer=x["v_k"], cos=x["cos"], sin=x["sin"],
                                  v_dense=padded[:, : H * D].view(512, H, D), **kw)
    with pytest.raises(XkvError, match="bounds"):                   # 4 q heads per kv head x 17 tokens: 68 rows
        y = _half_inputs(512, H, D, 4, 17, 0)
        ops.decode_attention_half(y["q"], H, a_k=y["a_k"], vk_layer=y["v_k"], v_dense=y["v_dense"], cos=y["cos"],
                                  sin=y["sin"], k_tail=y["k_tail"], v_tail=y["v_tail"], scale=0.1)
    with pytest.raises(XkvError, match="bounds"):                   # 64 kv heads x 9 tokens: 576 rows
        y = _half_inputs(256, 64, 64, 1, 9, 0)
        ops.decode_attention_half(y["q"], 64, a_v=y["a_v"], vv_layer=y["v_v"], k_dense=y["k_dense"],
                                  k_tail=y["k_tail"], v_tail=y["v_tail"], scale=0.1)
    small = torch.empty(1024, dtype=torch.uint8, device="cuda")
    with pytest.raises(XkvError, match="workspace too small"):
        ops.check(lib.xkv_decode_attention_half(
            ops._ptr(x["q"]), 8, 2, H, D, ops._ptr(x["a_k"]), 256, 256, ops._ptr(x["v_k"]), 256, None, 0, 0, None, 0, 0,
            None, 0, ops._ptr(x["v_dense"]), D, H * D, 512, ops._ptr(x["cos"]), ops._ptr(x["sin"]), D,
            ops._ptr(x["k_tail"]), ops._ptr(x["v_tail"]), 5, x["k_tail"].stride(0), x["k_tail"].stride(1),
            ops.C.c_float(0.1), ops._ptr(x["q"]), ops.C.c_void_p(small.data_ptr()), small.numel(), ops._stream(), None))


# ------------------------------------------------------------------------------------------------ model level
def _counting(fn_owner, name):
    calls = []
    orig = getattr(fn_owner, name)

    def wrapped(*a, **k):
        calls.append(1)
        return orig(*a, **k)

    setattr(fn_owner, name, wrapped)
    return calls, orig


MODEL_SETUPS = {
    # name -> (config kwargs, prompt length, expected factored sides)
    "key_only": (dict(rank_k=64, rank_v=128, merge_value=False), 700, (True, False)),
    "value_only": (dict(rank_k=64, rank_v=128, merge_key=False), 700, (False, True)),
    "rank_v_too_large": (dict(rank_k=64, rank_v=128), 120, (True, False)),   # rank_v >= the 120-token prompt: V dense
}


@pytest.mark.parametrize("setup", list(MODEL_SETUPS))
def test_patched_llama_one_sided_groups_match_oracle_cache(setup):
    from tests.oracle_cache import OracleCache
    from tests.test_generate_gpu import _decode_logits, _model
    from xkv_b200 import ops
    from xkv_b200.configurations import generate_consecutive_xKV_config
    from xkv_b200.customized_cache import FakeLayerMergingCache
    from xkv_b200.patch import KVCompress

    kwargs, n, sides = MODEL_SETUPS[setup]
    model = _model()
    cfg = generate_consecutive_xKV_config(num_layers=4, end_layer=-1, group_size=2, **kwargs)
    KVCompress(xKV_config=cfg)(model)
    ids = torch.randint(0, 512, (1, n), device="cuda", generator=torch.Generator(device="cuda").manual_seed(1))
    cache = FakeLayerMergingCache(cfg)
    calls, orig = _counting(ops, "decode_attention_half")
    try:
        lg_ours, _ = _decode_logits(model, cache, ids, steps=6)
    finally:
        ops.decode_attention_half = orig
    for l in cache.layers:
        assert (l.group.factors.key is not None, l.group.factors.value is not None) == sides
    assert len(calls) == 4 * 6, f"{len(calls)} fused one-sided calls, expected 24"
    for layer in model.model.layers:
        layer.self_attn.xkv_fused_decode = False
    lg_ref, _ = _decode_logits(model, OracleCache(cfg), ids, steps=6)
    torch.cuda.synchronize()
    assert torch.allclose(lg_ours[0], lg_ref[0], atol=1e-3)
    dev = (lg_ours[1:] - lg_ref[1:]).abs().max().item()
    scale = lg_ref[1:].abs().max().item()
    print(f"{setup}: decode logits max |ours - oracle| = {dev:.4f} (logit scale {scale:.3f})")
    assert dev <= 5e-2 * scale


@torch.no_grad()
def test_assisted_decoding_on_a_key_only_cache_matches_greedy():
    from tests.test_multitoken_gpu import _gqa128_model, _ids
    from xkv_b200 import ops
    from xkv_b200.configurations import generate_consecutive_xKV_config
    from xkv_b200.patch import KVCompress

    model = _gqa128_model()
    cfg = generate_consecutive_xKV_config(num_layers=4, end_layer=-1, group_size=2, rank_k=64, rank_v=128,
                                          merge_value=False)
    KVCompress(xKV_config=cfg)(model)
    ids = _ids(800, seed=5, vocab=48)
    greedy = model.generate(ids, max_new_tokens=24, do_sample=False, return_dict_in_generate=True, output_logits=True)
    dims = []
    orig = ops.decode_attention_half
    ops.decode_attention_half = lambda q, *a, **k: (dims.append(q.dim()), orig(q, *a, **k))[1]
    try:
        assisted = model.generate(ids, max_new_tokens=24, do_sample=False, prompt_lookup_num_tokens=3)
    finally:
        ops.decode_attention_half = orig
    torch.cuda.synchronize()
    assert 3 in dims, "no fused multi-token one-sided step ran"
    a, g = assisted[0, ids.shape[1]:], greedy.sequences[0, ids.shape[1]:]
    assert a.shape == g.shape
    diff = (a != g).nonzero()
    if len(diff):
        i = diff[0].item()
        top2 = greedy.logits[i][0].float().topk(2).values
        scale = torch.stack(greedy.logits).float().abs().max().item()
        assert (top2[0] - top2[1]).item() < 5e-2 * scale, f"first difference at step {i} is not a near tie"


@torch.no_grad()
def test_compress_decode_tokens_on_a_key_only_cache_folds_nothing():
    from tests.oracle_cache import OracleCache
    from tests.test_generate_gpu import _decode_logits, _model
    from xkv_b200.configurations import generate_consecutive_xKV_config
    from xkv_b200.customized_cache import FakeLayerMergingCache
    from xkv_b200.patch import KVCompress

    model = _model()
    cfg = generate_consecutive_xKV_config(num_layers=4, end_layer=-1, group_size=2, rank_k=64, rank_v=128,
                                          merge_value=False)
    KVCompress(xKV_config=cfg)(model)
    ids = torch.randint(0, 512, (1, 700), device="cuda", generator=torch.Generator(device="cuda").manual_seed(1))
    cache = FakeLayerMergingCache(cfg, compress_decode_tokens=True, decode_capacity=64)
    lg_ours, _ = _decode_logits(model, cache, ids, steps=6)
    assert all(l.prefill_len == 700 and l.tail_len == 6 for l in cache.layers)   # the decode tokens stayed dense
    assert all(l.group.length == 700 for l in cache.layers)
    for layer in model.model.layers:
        layer.self_attn.xkv_fused_decode = False
    lg_ref, _ = _decode_logits(model, OracleCache(cfg), ids, steps=6)
    torch.cuda.synchronize()
    assert (lg_ours[1:] - lg_ref[1:]).abs().max().item() <= 5e-2 * lg_ref[1:].abs().max().item()
