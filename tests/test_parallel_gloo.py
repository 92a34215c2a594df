"""CPU, world_size 2 over gloo: the host logic of the multi-GPU paths — group ownership, token shards, the
max-over-ranks timing rule, and the Gram all-reduce plumbing of the token-sharded factorisation (the local
Gram is a torch matmul here: this test covers the collective, the kernels are covered on the GPU)."""
import os
import socket

import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

from xkv_b200 import parallel


def test_assign_groups_partitions_exactly():
    for groups, world in [(8, 1), (8, 2), (8, 8), (10, 8), (7, 4), (3, 8)]:
        owned = [parallel.assign_groups(groups, world, r) for r in range(world)]
        flat = [g for o in owned for g in o]
        assert flat == list(range(groups))
        assert max(len(o) for o in owned) - min(len(o) for o in owned) <= 1
    assert [len(parallel.assign_groups(10, 8, r)) for r in range(8)] == [2, 2, 1, 1, 1, 1, 1, 1]
    with pytest.raises(ValueError):
        parallel.assign_groups(8, 2, 2)


def test_token_shards_cover_the_sequence():
    for tokens, world in [(131072, 8), (65536, 2), (1000, 4), (100, 8)]:
        spans = [parallel.token_shard(tokens, world, r) for r in range(world)]
        assert spans[0][0] == 0 and spans[-1][1] == tokens
        for (b0, e0), (b1, e1) in zip(spans[:-1], spans[1:]):
            assert e0 == b1 and b0 <= e0
        assert all(b % 128 == 0 or b == tokens for b, _ in spans)


def _packed_offsets(n):
    """Row offsets of the packed upper triangle (row r keeps columns [32 * (r // 32), n)): the layout of
    xkv_gram_pack_upper, restated in numpy-style Python."""
    off, offs = 0, []
    for r in range(n):
        offs.append(off)
        off += n - (r // 32) * 32
    return offs, off


def _pack_upper(g):
    n = g.shape[0]
    return torch.cat([g[r, (r // 32) * 32:] for r in range(n)])


def _unpack_upper(packed, n):
    offs, _ = _packed_offsets(n)
    full = torch.zeros(n, n, dtype=packed.dtype)
    for r in range(n):
        c0 = (r // 32) * 32
        full[r, c0:] = packed[offs[r]: offs[r] + n - c0]
    upper = torch.triu(full)
    return upper + torch.triu(full, 1).t()


def test_packed_upper_triangle_size_matches_the_library():
    """xkv_gram_packed_elems is host code: callable without a GPU."""
    from xkv_b200 import _lib

    lib = _lib.load()
    for n in (32, 64, 100, 1024, 4096, 8192):
        assert int(lib.xkv_gram_packed_elems(n)) == _packed_offsets(n)[1]
    assert int(lib.xkv_gram_packed_elems(8192)) * 4 < 0.51 * 8192 * 8192 * 4      # half the all-reduce payload


def _free_port():
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        return s.getsockname()[1]


def _worker(rank, world, port, ret):
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    dist.init_process_group("gloo", rank=rank, world_size=world)
    try:
        torch.manual_seed(0)
        x = torch.randn(512, 64).bfloat16().float()        # the full matrix, identical on every rank
        b, e = parallel.token_shard(512, world, rank)
        g_local = x[b:e].t() @ x[b:e]                        # stand-in for the Gram kernel on the local rows
        # as factorize_token_sharded does: only the packed upper triangle is reduced, then mirrored back
        packed = _pack_upper(g_local)
        dist.all_reduce(packed, op=dist.ReduceOp.SUM)
        g_local = _unpack_upper(packed, 64)
        ok_gram = torch.allclose(g_local, x.t() @ x, rtol=1e-5, atol=1e-4) and torch.equal(g_local, g_local.t())
        # every rank derives the same right factor from the reduced Gram and projects its own rows
        evals, evecs = torch.linalg.eigh(g_local.double())
        v = evecs[:, -16:].float()
        a_local = x[b:e] @ v
        gathered = [torch.empty_like(a_local) for _ in range(world)]
        dist.all_gather(gathered, a_local)
        ok_proj = torch.allclose(torch.cat(gathered), x @ v, atol=1e-4)
        slow = parallel.max_over_ranks(10.0 + rank)
        groups = parallel.assign_groups(8, world, rank)
        counts = torch.tensor([len(groups)])
        dist.all_reduce(counts)
        ret[rank] = (ok_gram, ok_proj, slow, int(counts.item()))
    finally:
        dist.destroy_process_group()


def test_world_size_two_gram_allreduce_and_timing():
    world = 2
    mgr = mp.Manager()
    ret = mgr.dict()
    mp.spawn(_worker, args=(world, _free_port(), ret), nprocs=world, join=True)
    for rank in range(world):
        ok_gram, ok_proj, slow, total = ret[rank]
        assert ok_gram and ok_proj
        assert slow == 11.0          # max over ranks, on both ranks
        assert total == 8


def test_merge_partial_attention_equals_softmax_over_the_union():
    torch.manual_seed(1)
    hq, d, s = 8, 16, 300
    scores = torch.randn(hq, s) * 3
    v = torch.randn(s, d)
    ref = torch.softmax(scores, dim=1) @ v
    cuts = [0, 128, 128, 300]             # three shards, the middle one empty
    outs, lses = [], []
    for b, e in zip(cuts[:-1], cuts[1:]):
        if e > b:
            outs.append(torch.softmax(scores[:, b:e], dim=1) @ v[b:e])
            lses.append(torch.logsumexp(scores[:, b:e], dim=1))
        else:
            outs.append(torch.zeros(hq, d))
            lses.append(torch.full((hq,), float("-inf")))
    out, lse = parallel.merge_partial_attention(torch.stack(outs), torch.stack(lses))
    assert torch.allclose(out, ref, atol=1e-5)
    assert torch.allclose(lse, torch.logsumexp(scores, dim=1), atol=1e-5)


def _decode_worker(rank, world, port, ret):
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    dist.init_process_group("gloo", rank=rank, world_size=world)
    try:
        torch.manual_seed(0)
        hq, d, s = 8, 32, 1000
        scores = torch.randn(hq, s) * 2                      # identical on every rank
        v = torch.randn(s, d)
        b, e = parallel.token_shard(s, world, rank)
        out_local = (torch.softmax(scores[:, b:e], dim=1) @ v[b:e]).bfloat16()   # stand-in for the decode kernel
        lse_local = torch.logsumexp(scores[:, b:e], dim=1)
        merged = parallel.merge_token_shards(out_local, lse_local)
        ref = torch.softmax(scores, dim=1) @ v
        ret[rank] = (merged.dtype == torch.bfloat16, float((merged.float() - ref).abs().max()))
    finally:
        dist.destroy_process_group()


def test_world_size_two_token_sharded_decode_merge():
    world = 2
    mgr = mp.Manager()
    ret = mgr.dict()
    mp.spawn(_decode_worker, args=(world, _free_port(), ret), nprocs=world, join=True)
    for rank in range(world):
        same_dtype, err = ret[rank]
        assert same_dtype and err < 2e-2
