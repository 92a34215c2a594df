"""Low-rank factorisation of a layer group's token-major KV matrix on the B200 kernels.

Replaces the reference's ``fake_svd`` (fake_layer_merge_dynamic_cache.py:11-29: exact
``torch.linalg.svd`` -> truncate -> multiply back) by a factorisation that is *stored*:

    X (m x n, bf16)  ~=  A (m x r, bf16) @ Vt (r x n, bf16),    A = X V,  V orthonormal columns

so that ``A @ Vt`` is the orthogonal projection of X onto (an accurate approximation of) its dominant
rank-r right singular subspace, i.e. the same matrix ``U_r S_r V_r^T`` the reference multiplies back.

Algorithm (every product is a tcgen05 GEMM of xkv_gemm.cu, everything stays on the device and on the
caller's stream; nothing synchronises):

  1. Gram            G = X^T X            one pass over X, symmetric tile set, fp32 accumulation in TMEM
  2. range finder    Y = G Omega           Omega Gaussian n x l, l = round_up(r + 64, 64)
  3. CholeskyQR      Q = orth(Y)           row-normalise, S = Y^T Y (6-term bf16-limb product ~ fp32),
                                           blocked Cholesky + explicit inverse, Q = Y L^-T; repeated
  4. power steps     Y = (G - c I) Q; CholeskyQR   4 times (3-term limb product; two CholeskyQR passes
                     after the first step, ONE accurate pass after the others); from the second
                     step on c ~ lambda_l / 2 (lambda_l read off the diagonal of the previous step's
                     triangular factor), which does the work of ~6 plain steps in 4
  5. Rayleigh-Ritz   shared-memory Jacobi on the window of T = Q^T G Q that straddles column r: the
                     triangular (Cholesky) orthogonalisation keeps the columns ordered by dominance,
                     so only the boundary window needs rotating (DESIGN.md, "windowed Rayleigh-Ritz")
  6. right factor    V = first r columns;  Vt / V in bf16
  7. projection      A = X V               second and last pass over X

The Gram route is exact up to fp32 rounding of G, needs exactly two reads of X, and was chosen over
sketching X directly because r is a sizeable fraction of n here (512..768 of 4096).
"""
from __future__ import annotations

from dataclasses import dataclass, field
from typing import Dict, List, Optional, Sequence

import ctypes as C

import torch

from . import _lib, ops
from ._lib import XkvError


@dataclass
class FactorizeOptions:
    """The factorisation's schedule is fixed in the library (DESIGN.md section 2); what a caller chooses is here."""

    profile: bool = False   # record the driver's 7 stage events and report the stage times in Factors.timings


@dataclass
class Factors:
    """Stored form of one compressed (group, K-or-V) matrix."""

    A: torch.Tensor                     # (m, r)  bf16  token-side factor  (= U_r S_r up to rotation)
    Vt: torch.Tensor                    # (r, n)  bf16  right factor, rows = basis vectors
    V: torch.Tensor                     # (n, r)  bf16  same, transposed (layout the decode kernel reads)
    rank: int
    sigma_lead: Optional[torch.Tensor] = None   # leading singular values (Ritz estimates), fp32
    A_storage: Optional[torch.Tensor] = None    # A plus spare rows for appended tokens (A is a view of it)
    timings: Dict[str, float] = field(default_factory=dict)

    def reconstruct(self) -> torch.Tensor:
        """Dense bf16 reconstruction (test/debug helper; the product path never materialises it)."""
        return (self.A.float() @ self.Vt.float()).to(torch.bfloat16)


def _round_up(x: int, k: int) -> int:
    return (x + k - 1) // k * k


def sketch_width(rank: int) -> int:
    """Columns of the driver's sketch of a rank-`rank` factorisation; the matrix must have at least as many."""
    return _round_up(rank + 64, 64)


_STAGES = ("gram_gemm", "gram_reduce_split", "range_finder", "power_iters", "rayleigh_ritz", "project")


def workspace_bytes(batch: int, m: int, n: int, rank: int, opts: Optional[FactorizeOptions] = None) -> int:
    """Workspace of one driver call (0 for a problem the driver rejects); `opts` does not change it."""
    return int(_lib.load().xkv_factorize_workspace_bytes(batch, m, n, rank))


def layer_rows(t: torch.Tensor) -> Optional[torch.Tensor]:
    """(S, H*D) row-major view of a (1, H, S, D) layer tensor whose memory is token-major (what HF produces:
    ``proj(x).view(b, s, H, D).transpose(1, 2)``), or None when the layout is different (then the gather kernel runs)."""
    if t.dim() != 4 or t.shape[0] != 1 or t.dtype != torch.bfloat16:
        return None
    _, h, s, d = t.shape
    sb, sh, ss, sd = t.stride()
    if sd != 1 or (h > 1 and sh != d) or ss < h * d or ss % 8 or (t.data_ptr() & 15) or (h * d) % 64:
        return None
    return t.as_strided((s, h * d), (ss, 1))


def _factorize_chunks(items: Sequence, chunk: int, m: int, n: int, rank: int, opts: FactorizeOptions,
                      workspace: Optional[torch.Tensor], extra_rows: int, dev, run) -> List[Factors]:
    """What factorize_groups and factorize_batch share: sizes (and if needed allocates) the workspace for `chunk` matrices,
    then per chunk of `items` allocates A (with `extra_rows` spare token rows behind it, for tokens appended later by
    xkv_append_project), Vt, V and sigma, and makes the driver call ``run(part, outs, tail)`` — outs: the A / Vt / V /
    sigma pointer arrays, tail: the workspace, its size, the stage events and the stream, in the C argument order.  With
    `opts.profile` the 7 stage events of every call are recorded and their intervals summed into each Factors.timings."""
    lib = _lib.load()
    need = int(lib.xkv_factorize_workspace_bytes(chunk, m, n, rank))
    if need == 0:
        raise XkvError(lib.xkv_last_error().decode() or "factorize: invalid problem")
    if workspace is None or workspace.numel() * workspace.element_size() < need:
        workspace = torch.empty(need, dtype=torch.uint8, device=dev)
    stream = C.c_void_p(torch.cuda.current_stream().cuda_stream)
    out: List[Factors] = []
    all_events = []
    for lo in range(0, len(items), chunk):
        part = items[lo:lo + chunk]
        nb = len(part)
        a_store = [torch.empty(m + extra_rows, rank, dtype=torch.bfloat16, device=dev) for _ in range(nb)]
        a = [t[:m] for t in a_store]
        vt = [torch.empty(rank, n, dtype=torch.bfloat16, device=dev) for _ in range(nb)]
        v = [torch.empty(n, rank, dtype=torch.bfloat16, device=dev) for _ in range(nb)]
        sig = [torch.empty(_lib.FACTORIZE_SIGMA_COUNT, dtype=torch.float32, device=dev) for _ in range(nb)]
        ev_arr = None
        if opts.profile:
            events = [torch.cuda.Event(enable_timing=True) for _ in range(7)]
            for e in events:
                e.record()  # torch creates the cudaEvent lazily; recording materialises the handle
            ev_arr = (C.c_void_p * 7)(*[e.cuda_event for e in events])
            all_events.append(events)
        outs = (ops._ptr_array(a), ops._ptr_array(vt), ops._ptr_array(v), ops._ptr_array(sig))
        tail = (C.c_void_p(workspace.data_ptr()), workspace.numel() * workspace.element_size(), ev_arr, stream)
        run(part, outs, tail)
        for b in range(nb):
            out.append(Factors(A=a[b], Vt=vt[b], V=v[b], rank=rank, sigma_lead=sig[b], A_storage=a_store[b]))
    if opts.profile:
        torch.cuda.synchronize()
        timings: Dict[str, float] = {}
        for events in all_events:
            for i, name in enumerate(_STAGES):
                timings[name] = timings.get(name, 0.0) + events[i].elapsed_time(events[i + 1])
        for f in out:
            f.timings = timings
    return out


def factorize_groups(groups: Sequence[Sequence[torch.Tensor]], rank: int, opts: Optional[FactorizeOptions] = None,
                     workspace: Optional[torch.Tensor] = None, extra_rows: int = 0) -> List[Factors]:
    """Factorise layer groups IN PLACE at rank `rank`: groups[g][i] is the (S, H*D) row-major matrix of layer i of group g
    (:func:`layer_rows`); the group matrix is their column-wise concatenation — the reference's ``torch.cat(dim=1)`` +
    ``transpose(1, 2).reshape`` (cache:170-171, :13-14) — and is never materialised: the Gram pass and the projection pass
    read the layer tensors through per-layer tensor maps (xkv_factorize_groups)."""
    opts = opts or FactorizeOptions()
    if len(groups) == 0:
        return []
    lib = _lib.load()
    nl = len(groups[0])
    m, lc = groups[0][0].shape
    ld = groups[0][0].stride(0)
    for grp in groups:
        if len(grp) != nl:
            raise XkvError("factorize_groups: equally sized groups required")
        for t in grp:
            if (not t.is_cuda or t.dtype != torch.bfloat16 or tuple(t.shape) != (m, lc) or t.stride() != (ld, 1)
                    or t.data_ptr() & 15):
                raise XkvError("factorize_groups: layers must be equally shaped row-major bf16 CUDA matrices, 16-byte aligned")
    r = int(rank)
    per_call = max(1, min(_lib.MAX_BATCH, 64 // nl))     # XKV_MAX_LAYER_MAPS layer matrices per launch

    def run(part, outs, tail):
        flat = [t for grp in part for t in grp]
        _lib.check(lib.xkv_factorize_groups(ops._ptr_array(flat), len(part), nl, lc, m, ld, r, *outs, *tail))

    return _factorize_chunks(groups, min(len(groups), per_call), m, nl * lc, r, opts, workspace, extra_rows,
                             groups[0][0].device, run)


def factorize_batch(xs: Sequence[torch.Tensor], rank: int, opts: Optional[FactorizeOptions] = None,
                    workspace: Optional[torch.Tensor] = None, extra_rows: int = 0) -> List[Factors]:
    """Factorise a batch of equally-shaped token-major matrices (m x n bf16) at rank `rank`.

    One call into the library's stream-ordered driver (xkv_factorize_batch); batches larger than the
    C-ABI's per-call limit are processed in chunks that reuse one workspace.  Matrices whose rows are split over
    several GPUs go through :func:`factorize_token_sharded`."""
    opts = opts or FactorizeOptions()
    if len(xs) == 0:
        return []
    lib = _lib.load()
    m, n = xs[0].shape
    for x in xs:
        if not x.is_cuda:
            raise XkvError("factorize: CUDA tensors required (no CPU path)")
        if x.dtype != torch.bfloat16 or tuple(x.shape) != (m, n) or x.stride(1) != 1 or x.stride(0) != xs[0].stride(0):
            raise XkvError("factorize: inputs must be equally-shaped row-major bf16 matrices")
    r = int(rank)

    def run(part, outs, tail):
        _lib.check(lib.xkv_factorize_batch(ops._ptr_array(part), len(part), m, n, part[0].stride(0), r, *outs, None, 0,
                                           *tail))

    return _factorize_chunks(xs, min(len(xs), _lib.MAX_BATCH), m, n, r, opts, workspace, extra_rows, xs[0].device, run)


_chain_streams = {}


def _chain_stream(device, index: int):
    """Prioritised side stream for one of several concurrent factorisation chains (see compress.compress_groups)."""
    key = (device.index, index)
    if key not in _chain_streams:
        _chain_streams[key] = torch.cuda.Stream(device=device, priority=-1 - (index % 3))
    return _chain_streams[key]


def factorize_token_sharded(jobs: Sequence, process_group, opts: Optional[FactorizeOptions] = None,
                            comm_events: Optional[list] = None) -> List[Factors]:
    """Token-sharded factorisation of several matrices with the small-matrix stages DISTRIBUTED over the ranks.

    jobs: [(x_local, rank), ...] — x_local is this rank's (m_local, n) bf16 row shard of matrix i (same i on every rank).
    1. every rank runs the Gram of its rows of every matrix (phase 1);
    2. the packed upper triangle of every Gram (half the bytes of the full matrix) is summed over the ranks (NCCL
       all-reduce, overlapping the next matrix's Gram); matrix i has an owner, rank i mod P;
    3. the owner alone runs the range finder / CholeskyQR / power steps / Rayleigh-Ritz of its matrices (phase 3) — the part
       that does not shrink with the number of token shards — and broadcasts the right factor Vt (r x n bf16);
    4. every rank projects its own rows, A_p = X_p V (phase 4).
    With one matrix per rank or more the whole factorisation scales.  Returns Factors with the LOCAL rows of A.
    `opts.profile` does not apply here.  `comm_events`: optional [start, end] CUDA events (enable_timing) recorded around
    the exchanges; the payload bytes are appended."""
    import torch.distributed as dist

    lib = _lib.load()
    world = dist.get_world_size(process_group)
    me = dist.get_rank(process_group)
    stream = C.c_void_p(torch.cuda.current_stream().cuda_stream)
    dev = jobs[0][0].device
    n = jobs[0][0].shape[1]
    per = ops.gram_packed_elems(n)
    nj = len(jobs)

    def call(phase, xs, r, a_s, vts_, vs, grams, ws, on=None):
        """One driver call for a batch of matrices of equal shape and rank (xs / a_s / vs / grams may be None per phase)."""
        nb = len(vts_)
        m = xs[0].shape[0] if xs is not None else n
        _lib.check(lib.xkv_factorize_batch(
            ops._ptr_array(xs) if xs is not None else None, nb, m, n, xs[0].stride(0) if xs is not None else n, r,
            ops._ptr_array(a_s) if a_s is not None else None, ops._ptr_array(vts_), ops._ptr_array(vs) if vs is not None else None,
            None, ops._ptr_array(grams) if grams is not None else None, phase, C.c_void_p(ws.data_ptr()),
            ws.numel(), None, stream if on is None else C.c_void_p(on.cuda_stream)))

    m_loc = jobs[0][0].shape[0]
    for x, r in jobs:
        if x.dtype != torch.bfloat16 or tuple(x.shape) != (m_loc, n) or x.stride(1) != 1 or not x.is_cuda:
            raise XkvError("factorize_token_sharded: equally shaped row-major bf16 CUDA shards required")
    # the matrices this rank owns, by rank value: their small-matrix stages run as ONE batch per rank value
    owned = {}
    for i, (_, r) in enumerate(jobs):
        if i % world == me:
            owned.setdefault(r, []).append(i)
    need = max(int(lib.xkv_factorize_workspace_bytes(1, max(m_loc, r), n, r)) for _, r in jobs)
    for r, idx in owned.items():
        for lo in range(0, len(idx), _lib.MAX_BATCH):
            need = max(need, int(lib.xkv_factorize_workspace_bytes(len(idx[lo:lo + _lib.MAX_BATCH]), n, n, r)))
    ws = torch.empty(need, dtype=torch.uint8, device=dev)
    gram = torch.empty(n, n, dtype=torch.float32, device=dev)
    packed = [torch.empty(per, dtype=torch.float32, device=dev) for _ in range(nj)]
    vts = [torch.empty(r, n, dtype=torch.bfloat16, device=dev) for _, r in jobs]
    # 1 + 2. local Grams; the packed upper triangle of every matrix is summed as soon as it exists (NCCL runs on its own
    # stream: the sum of matrix i overlaps the Gram of matrix i + 1).  all-reduce rather than reduce-to-owner: with
    # NVSwitch the in-switch reduction makes it the fastest collective for this size (measured 317 GB/s at 2 ranks)
    if comm_events is not None:
        comm_events[0].record()
    sums = []
    for i, (x, r) in enumerate(jobs):
        if m_loc > 0:
            call(1, [x], r, None, [vts[i]], None, [gram], ws)
            ops.gram_pack_upper(gram, packed[i])
        else:
            packed[i].zero_()
        sums.append(dist.all_reduce(packed[i], op=dist.ReduceOp.SUM, group=process_group, async_op=True))
    # 3. the owner of matrix i (rank i mod P) derives its right factor: all the matrices a rank owns at one rank value in
    # ONE batched call (the latency-bound stages carry several matrices per launch); the owners work side by side
    # Each rank value's batch is a latency-bound chain of ~160 launches (Cholesky clusters at l = 1088 / 1600 are most of it):
    # the chains of different rank values run on their own prioritised side streams, each with its own workspace, so that
    # the K chain fills the SMs the V chain leaves idle (one stream: the chains ran back to back).
    main_stream = torch.cuda.current_stream(dev)
    chain_streams = []
    for gi, (r, idx) in enumerate(owned.items()):
        st = _chain_stream(dev, gi) if len(owned) > 1 else main_stream
        if st is not main_stream:
            st.wait_stream(main_stream)
            chain_streams.append(st)
        with torch.cuda.stream(st):
            ws_r = ws if st is main_stream else torch.empty(
                max(int(lib.xkv_factorize_workspace_bytes(len(idx[lo:lo + _lib.MAX_BATCH]), n, n, r))
                    for lo in range(0, len(idx), _lib.MAX_BATCH)), dtype=torch.uint8, device=dev)
            for lo in range(0, len(idx), _lib.MAX_BATCH):
                part = idx[lo:lo + _lib.MAX_BATCH]
                grams = torch.empty(len(part), n, n, dtype=torch.float32, device=dev)
                for k, i in enumerate(part):
                    sums[i].wait()
                    ops.gram_unpack_upper(packed[i], grams[k])
                v_tmp = [torch.empty(n, r, dtype=torch.bfloat16, device=dev) for _ in part]
                call(3, None, r, None, [vts[i] for i in part], v_tmp, list(grams), ws_r, on=st)
                del v_tmp, grams
            del ws_r
    for st in chain_streams:
        main_stream.wait_stream(st)
    # ... and broadcasts it; everybody issues the broadcasts in the same order
    casts = []
    for i in range(nj):
        owner = i % world
        src = dist.get_global_rank(process_group, owner) if process_group is not None else owner
        casts.append(dist.broadcast(vts[i], src=src, group=process_group, async_op=True))
    for w in sums + casts:
        w.wait()
    if comm_events is not None:
        comm_events[1].record()
        comm_events.append(sum(p.numel() * 4 for p in packed) + sum(v.numel() * 2 for v in vts))
    # 4. local projection (one call per matrix: a 64K x 8192 projection fills the GPU on its own)
    out: List[Factors] = []
    for i, (x, r) in enumerate(jobs):
        a = torch.empty(m_loc, r, dtype=torch.bfloat16, device=dev)
        if m_loc > 0:
            call(4, [x], r, [a], [vts[i]], None, None, ws)
        out.append(Factors(A=a, Vt=vts[i], V=vts[i].t().contiguous(), rank=r, A_storage=a))
    return out
