"""Multi-GPU partitioning of the xKV path (one process per GPU, torch.distributed).

Two natural shards (DESIGN.md §6):

* layer groups are independent (reference cache:161-165 touches only the group's layers) — ranks own
  disjoint sets of groups and never exchange data on the hot path;
* long contexts can be split by token rows (``factorize.factorize_token_sharded``) — each matrix's n x n fp32
  Gram is summed over the ranks (one all-reduce of its packed upper triangle), the matrix's owner derives the right
  factor and broadcasts it, and every rank projects its own rows.
"""
from __future__ import annotations

from typing import List, Sequence, Tuple

import torch


def assign_groups(num_groups: int, world_size: int, rank: int) -> List[int]:
    """Contiguous, balanced ownership of layer groups: the first ``num_groups % world_size`` ranks get one
    extra group (e.g. 10 groups on 8 GPUs -> 2,2,1,1,1,1,1,1). Every group is owned by exactly one rank."""
    if world_size < 1 or not (0 <= rank < world_size):
        raise ValueError(f"bad rank {rank} / world size {world_size}")
    base, extra = divmod(num_groups, world_size)
    start = rank * base + min(rank, extra)
    count = base + (1 if rank < extra else 0)
    return list(range(start, start + count))


def token_shard(num_tokens: int, world_size: int, rank: int, multiple: int = 128) -> Tuple[int, int]:
    """[begin, end) token rows of ``rank``: contiguous, balanced in units of ``multiple`` tokens (tile height)."""
    units = (num_tokens + multiple - 1) // multiple
    base, extra = divmod(units, world_size)
    b = (rank * base + min(rank, extra)) * multiple
    e = b + (base + (1 if rank < extra else 0)) * multiple
    return min(b, num_tokens), min(e, num_tokens)


def max_over_ranks(value: float, device=None, group=None) -> float:
    """Device-side timing convention: a multi-GPU step takes as long as its slowest rank."""
    import torch.distributed as dist

    if not (dist.is_available() and dist.is_initialized()) or dist.get_world_size(group) == 1:
        return float(value)
    t = torch.tensor([float(value)], dtype=torch.float64, device=device or "cpu")
    dist.all_reduce(t, op=dist.ReduceOp.MAX, group=group)
    return float(t.item())


def allreduce_gram(local_grams: Sequence[torch.Tensor], group=None) -> None:
    """Sum the per-rank Gram matrices in place (the only data-path collective of the token-sharded path)."""
    import torch.distributed as dist

    for g in local_grams:
        dist.all_reduce(g, op=dist.ReduceOp.SUM, group=group)


def merge_partial_attention(outs: torch.Tensor, lses: torch.Tensor) -> Tuple[torch.Tensor, torch.Tensor]:
    """Flash-decoding merge of P partial attentions over disjoint token sets.

    outs: (P, Hq, D) normalised partial outputs (softmax over each shard's own tokens), lses: (P, Hq) log-sum-exp of each
    shard's scaled scores.  Returns (out (Hq, D) fp32, lse (Hq,)) of the softmax over the union of the tokens:
        lse = log sum_p exp(lse_p),   out = sum_p exp(lse_p - lse) out_p.
    A shard without tokens contributes lse_p = -inf (weight 0)."""
    lses = lses.float()
    lse = torch.logsumexp(lses, dim=0)
    w = torch.exp(lses - lse[None]).nan_to_num(0.0)
    return (w[:, :, None] * outs.float()).sum(0), lse


def merge_token_shards(out_local: torch.Tensor, lse_local: torch.Tensor, group=None) -> torch.Tensor:
    """Decode over a token-sharded factored cache (SURVEY §8e): every rank has run
    ``ops.decode_attention(..., lse_out=lse_local)`` over ITS token rows of A_k / A_v (the decode tail lives on one rank,
    the others pass none); one all-gather of (Hq x (D + 1)) floats per layer and a local merge give every rank the
    attention output over the whole context.  Returns (Hq, D) in out_local's dtype.  The merge is per row, so a
    multi-token step (q (Hq, Tq, D)) merges unchanged: pass its output and log-sum-exp as (Hq * Tq, D) and (Hq * Tq,)."""
    import torch.distributed as dist

    world = dist.get_world_size(group)
    packed = torch.cat([out_local.float(), lse_local.float()[:, None]], dim=1).contiguous()   # (Hq, D + 1)
    gathered = [torch.empty_like(packed) for _ in range(world)]
    dist.all_gather(gathered, packed, group=group)
    allp = torch.stack(gathered)
    out, _ = merge_partial_attention(allp[:, :, :-1], allp[:, :, -1])
    return out.to(out_local.dtype)
