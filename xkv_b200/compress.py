"""Prefill compression of whole layer groups: gather (pack) + factorise, K and V on separate streams.

This is the device-side body of ``FakeLayerMergingCache.grouped_layer_merging``
(reference fake_layer_merge_dynamic_cache.py:155-208) for many groups at once: where the reference
loops ``cat -> fake_svd(K) -> fake_svd(V) -> split`` per group with host synchronisation after each
(:205-208), all groups' K matrices form one batch and all V matrices another, the two batches run
concurrently on two CUDA streams, and nothing synchronises with the host.
"""
from __future__ import annotations

from dataclasses import dataclass
from typing import List, Optional, Sequence

import torch

from . import factorize, ops
from ._lib import XkvError


@dataclass
class GroupFactors:
    """Compressed form of one layer group (either slot may stay dense when its merge flag is off)."""

    layers: List[int]
    key: Optional[factorize.Factors]
    value: Optional[factorize.Factors]


_side_streams = {}


def _side_stream(device: torch.device, index: int = 0, priority: int = 0) -> torch.cuda.Stream:
    key = (device.type, device.index, index, priority)
    if key not in _side_streams:
        _side_streams[key] = torch.cuda.Stream(device=device, priority=priority)
    return _side_streams[key]


def pack_groups(groups: Sequence[Sequence[torch.Tensor]], out: Optional[Sequence[torch.Tensor]] = None) -> List[torch.Tensor]:
    """One token-major matrix (S, G*H*D) per group (batch size 1)."""
    xs = []
    for i, layers in enumerate(groups):
        if layers[0].shape[0] != 1:
            raise XkvError("compress: batch size 1 per call (the reference's batched SVD is one SVD per sample)")
        x = ops.pack_group(layers, out=None if out is None else out[i][None])
        xs.append(x[0])
    return xs


def compress_groups(
    keys: Sequence[Sequence[torch.Tensor]],
    values: Sequence[Sequence[torch.Tensor]],
    rank_k: Optional[int],
    rank_v: Optional[int],
    merge_key: bool = True,
    merge_value: bool = True,
    opts: Optional[factorize.FactorizeOptions] = None,
    layer_ids: Optional[Sequence[Sequence[int]]] = None,
    num_streams: int = 4,
    extra_rows: int = 0,
    in_place: bool = True,
    job_events: Optional[list] = None,
) -> List[GroupFactors]:
    """Compress equally-shaped layer groups. keys[g][i] / values[g][i]: (1, H, S, D) bf16 of layer i of
    group g (keys PRE-RoPE, as the reference hands them over, llama.py:49).

    The K matrices and the V matrices are independent factorisations; they are cut into up to
    `num_streams` batches that run on separate CUDA streams, so that the latency-bound stages of one batch
    (Cholesky panels, Jacobi) overlap the tensor-core GEMMs of another.  `in_place=False` forces the gather kernel +
    packed-matrix path (the two give bit-identical factors; tests compare them)."""
    ng = len(keys)
    if ng == 0:
        return []
    dev = keys[0][0].device
    main = torch.cuda.current_stream(dev)
    kf: List[Optional[factorize.Factors]] = [None] * ng
    vf: List[Optional[factorize.Factors]] = [None] * ng
    if keys[0][0].shape[0] != 1:
        raise XkvError("compress: batch size 1 per call (the reference's batched SVD is one SVD per sample)")
    sides = (["k"] if merge_key else []) + (["v"] if merge_value else [])
    jobs = []   # (target list, first group, groups, rank)
    per_side = max(1, num_streams // max(len(sides), 1))
    for side in sides:
        src, dst, rank = (keys, kf, rank_k) if side == "k" else (values, vf, rank_v)
        nchunk = min(per_side, ng)
        size = (ng + nchunk - 1) // nchunk
        for lo in range(0, ng, size):
            jobs.append((dst, lo, src[lo:lo + size], rank))
    used = []
    # Every chain on its own side stream with a CTA-level priority (0, the lowest, is what the projection GEMMs are
    # launched with: xkv_host.h gemm_low_priority): when SMs free up, the pending CTAs of a higher-priority chain go first, so
    # one chain's latency-bound kernels (Cholesky clusters, Jacobi windows) are not queued behind the hundreds of GEMM CTAs
    # of another.  Measured (bench step, 10 steps, two runs): no priorities, last job on the caller's stream 44.3 / 43.1 ms;
    # all side streams 41.9; priorities -1 / -2 / -3 dealt round-robin 39.2 - 39.8 (8 jobs).  With both sides compressed the
    # chains of the larger rank (the longer ones: wider sketch, more Cholesky block steps) get the top priority -3 and the
    # others -1, so that all chains end together: 37.9 / 38.1 -> 37.1 / 37.2 ms same box (profiles/r02_priorities_ab.jsonl;
    # the device has four levels, 0 .. -3; the reverse order costs 0.6 ms, distinct levels per chain gain nothing).
    for j, (dst, lo, groups, rank) in enumerate(jobs):
        if len(sides) == 2 and rank_k != rank_v:
            prio = -3 if rank == max(rank_k, rank_v) else -1   # the longer chains (wider sketch) first
        else:
            prio = -1 - (j % 3)
        stream = main if num_streams <= 1 else _side_stream(dev, 200 + j, priority=prio)
        if stream is not main:
            stream.wait_stream(main)
            used.append(stream)
        with torch.cuda.stream(stream):
            if job_events is not None:
                ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                job_events.append((j, rank, len(groups), ev0, ev1))
                ev0.record()
            # token-major layer tensors (what HF hands over) are read in place through per-layer tensor maps; any other
            # layout goes through the gather kernel first (reference cache:170-171 + :13-14)
            rows = [[factorize.layer_rows(t) for t in grp] for grp in groups] if in_place else None
            if rows is not None and all(r is not None for grp in rows for r in grp) and len(groups[0]) <= 16:
                fs = factorize.factorize_groups(rows, rank, opts, extra_rows=extra_rows)
            else:
                xs = pack_groups(groups)
                fs = factorize.factorize_batch(xs, rank, opts, extra_rows=extra_rows)
                if stream is not main:
                    for x in xs:
                        x.record_stream(stream)
        if job_events is not None:
            with torch.cuda.stream(stream):
                job_events[-1][4].record()
        for i, f in enumerate(fs):
            dst[lo + i] = f
            if stream is not main:
                for t in (f.A_storage, f.Vt, f.V, f.sigma_lead):
                    if t is not None:
                        t.record_stream(main)
    for stream in used:
        main.wait_stream(stream)
    ids = layer_ids if layer_ids is not None else [list(range(len(g))) for g in keys]
    return [GroupFactors(layers=list(ids[g]), key=kf[g], value=vf[g]) for g in range(ng)]


def compress_groups_from_host(
    h_keys: Sequence[Sequence[torch.Tensor]],
    h_values: Sequence[Sequence[torch.Tensor]],
    rank_k: Optional[int],
    rank_v: Optional[int],
    device: torch.device,
    chunk_groups: int = 1,
    opts: Optional[factorize.FactorizeOptions] = None,
    host_out: Optional[List[torch.Tensor]] = None,
    num_streams: int = 2,
    staging=None,
):
    """Compress a KV cache that lives in (pinned) HOST memory, pipelined by chunks of `chunk_groups` layer groups:
    the host->device copy of chunk c+1 runs on a copy stream while chunk c is factorised, and the factors of chunk
    c-1 go back to the host on a third stream, so that the step costs about one pass of the KV over PCIe plus the
    factorisation of the last chunk instead of copy + compute + copy in sequence.

    h_keys[g][i] / h_values[g][i]: pinned (1, S, H, D) bf16 tensors (token-major, as HF produces K/V before the
    (bs, H, S, D) view).  `staging`: device buffers from :func:`host_staging` (a serving loop allocates them once;
    without them they are allocated here, on every call).  Returns (factors per group, host tensors [A_k, Vt_k,
    A_v, Vt_v per group] or None)."""
    ng = len(h_keys)
    main = torch.cuda.current_stream(device)
    copy_s = _side_stream(device, 101)
    back_s = _side_stream(device, 102)
    # The K side and the V side of a chunk are independent factorisations: each starts as soon as ITS tensors have landed
    # (V is sent first: its chain is the longer one and runs under the K copy; what remains after the last byte arrives
    # is one K chain + the copy-back of its factors), on its own stream.
    side_s = {"v": _side_stream(device, 103), "k": _side_stream(device, 104, priority=-1)}
    # device staging for every group, allocated on the main stream (the copy stream only writes into it)
    dk, dv = staging if staging is not None else host_staging(h_keys, h_values, device)
    copy_s.wait_stream(main)
    for st in side_s.values():
        st.wait_stream(main)
    sides = (["v"] if rank_v is not None else []) + (["k"] if rank_k is not None else [])
    ready = {"k": [], "v": []}
    with torch.cuda.stream(copy_s):
        for lo in range(0, ng, chunk_groups):
            for side in ("v", "k"):
                dst, src = (dv, h_values) if side == "v" else (dk, h_keys)
                for g in range(lo, min(lo + chunk_groups, ng)):
                    for d, h in zip(dst[g], src[g]):
                        d.copy_(h, non_blocking=True)
                ev = torch.cuda.Event()
                ev.record(copy_s)
                ready[side].append(ev)
    kf: List[Optional[factorize.Factors]] = [None] * ng
    vf: List[Optional[factorize.Factors]] = [None] * ng
    slot = {side: i for i, side in enumerate(x for x in ("k", "v") if x in sides)}   # host_out: [A, Vt] per compressed side, K first
    host_tensors: Optional[List[Optional[torch.Tensor]]] = [None] * (2 * len(sides) * ng) if host_out is not None else None
    for c, lo in enumerate(range(0, ng, chunk_groups)):
        hi = min(lo + chunk_groups, ng)
        keys = [[t.transpose(1, 2) for t in dk[g]] for g in range(lo, hi)]
        vals = [[t.transpose(1, 2) for t in dv[g]] for g in range(lo, hi)]
        for side in sides:
            st = side_s[side]
            st.wait_event(ready[side][c])
            with torch.cuda.stream(st):
                res = compress_groups(keys, vals, rank_k, rank_v, merge_key=side == "k", merge_value=side == "v", opts=opts,
                                      num_streams=max(1, num_streams // 2))
                done = torch.cuda.Event()
                done.record(st)
            for g, gf in zip(range(lo, hi), res):
                f = gf.key if side == "k" else gf.value
                (kf if side == "k" else vf)[g] = f
                for t in (f.A_storage, f.Vt, f.V, f.sigma_lead):
                    if t is not None:
                        t.record_stream(main)
            if host_out is not None:
                back_s.wait_event(done)
                with torch.cuda.stream(back_s):
                    for g in range(lo, hi):
                        f = kf[g] if side == "k" else vf[g]
                        for j, t in enumerate((f.A, f.Vt)):
                            k = 2 * len(sides) * g + 2 * slot[side] + j
                            host_out[k].copy_(t, non_blocking=True)
                            t.record_stream(back_s)
                            host_tensors[k] = host_out[k]
    for st in side_s.values():
        main.wait_stream(st)
    main.wait_stream(back_s)
    main.wait_stream(copy_s)
    out = [GroupFactors(layers=list(range(len(h_keys[g]))), key=kf[g], value=vf[g]) for g in range(ng)]
    return out, host_tensors


def host_staging(h_keys, h_values, device: torch.device):
    """Device staging buffers for :func:`compress_groups_from_host` (same shapes as the host tensors)."""
    dk = [[torch.empty(h.shape, dtype=h.dtype, device=device) for h in grp] for grp in h_keys]
    dv = [[torch.empty(h.shape, dtype=h.dtype, device=device) for h in grp] for grp in h_values]
    return dk, dv


class GraphedCompressor:
    """compress_groups captured once into a CUDA graph and replayed (static input buffers).

    The factorisation enqueues a few thousand small kernels per step; replaying a captured graph removes the
    per-launch host cost, which otherwise leaves the GPU waiting during the latency-bound stages.  Inputs must
    keep their addresses between replays (a serving loop that reuses its KV buffers, or bench.py)."""

    def __init__(self, keys, values, rank_k, rank_v, merge_key=True, merge_value=True, opts=None, num_streams=4):
        self._args = (keys, values, rank_k, rank_v, merge_key, merge_value, opts)
        self._num_streams = num_streams
        dev = keys[0][0].device
        # warm-up outside capture: first-use attribute setting, allocator pools of the side streams
        compress_groups(*self._args, num_streams=num_streams)
        torch.cuda.synchronize(dev)
        self.graph = torch.cuda.CUDAGraph()
        with torch.cuda.graph(self.graph):
            self.result = compress_groups(*self._args, num_streams=num_streams)

    def replay(self) -> List[GroupFactors]:
        self.graph.replay()
        return self.result
