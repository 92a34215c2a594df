"""Tensor-level wrappers over the C-ABI (``include/xkv_b200.h``).

PyTorch is used only for device memory and streams: every function takes CUDA tensors, passes raw
``data_ptr()``s and the current stream to the library, and returns without synchronising.
"""
from __future__ import annotations

import ctypes as C
from typing import List, Optional, Sequence, Tuple

import torch

from . import _lib
from ._lib import GemmProblem, check

# term lists (indices into the limb arrays: 0 = hi, 1 = mid, 2 = lo)
TERMS_1 = ((0, 0),)
TERMS_3 = ((0, 0), (0, 1), (1, 0))
TERMS_6 = ((0, 0), (0, 1), (1, 0), (1, 1), (0, 2), (2, 0))


def _stream() -> C.c_void_p:
    return C.c_void_p(torch.cuda.current_stream().cuda_stream)


def _require_cuda(*tensors: torch.Tensor) -> None:
    """Every operand must live on the CURRENT CUDA device: the library launches on the current device's current
    stream (kernels, tensor maps and per-device attributes all belong to it).  A process that shards a model over
    several GPUs (device_map) wraps the call in ``torch.cuda.device(tensor.device)``."""
    cur = None
    for t in tensors:
        if t is None:
            continue
        if not t.is_cuda:
            raise _lib.XkvError("xkv_b200 ops need CUDA tensors: there is no CPU path")
        if cur is None:
            cur = torch.cuda.current_device()
        if t.device.index != cur:
            raise _lib.XkvError(f"xkv_b200 op called with a tensor on cuda:{t.device.index} while cuda:{cur} is the current "
                                "device: wrap the call in torch.cuda.device(tensor.device)")


def launch_count() -> int:
    return int(_lib.load().xkv_launch_count())


# ---------------------------------------------------------------------------------------------
# (1) gather
# ---------------------------------------------------------------------------------------------
def pack_group(layers: Sequence[torch.Tensor], out: Optional[torch.Tensor] = None) -> torch.Tensor:
    """Gather G tensors (bs, H, S, D) bf16 into X (bs, S, G*H*D) bf16, columns ordered (layer, head, dim).

    Same result as ``torch.cat(layers, dim=1).transpose(1, 2).reshape(bs, S, G*H*D)``
    (reference: fake_layer_merge_dynamic_cache.py:170-171 and :13-14)."""
    lib = _lib.load()
    _require_cuda(*layers)
    g = len(layers)
    bs, h, s, d = layers[0].shape
    sb, sh, ss, sd = layers[0].stride()
    for t in layers:
        if t.dtype != torch.bfloat16:
            raise _lib.XkvError("pack_group: bf16 tensors required")
        if tuple(t.shape) != (bs, h, s, d) or t.stride() != (sb, sh, ss, sd):
            raise _lib.XkvError("pack_group: all layers of a group must share shape and strides")
    if s > 0 and sd != 1:
        raise _lib.XkvError("pack_group: head_dim must be contiguous")
    if out is None:
        out = torch.empty((bs, s, g * h * d), dtype=torch.bfloat16, device=layers[0].device)
    ptrs = (C.c_void_p * g)(*[t.data_ptr() for t in layers])
    check(lib.xkv_pack_group(ptrs, g, bs, h, s, d, sb, sh, ss, C.c_void_p(out.data_ptr()), _stream()))
    return out


def unpack_group(x: torch.Tensor, layers: Sequence[torch.Tensor]) -> None:
    """Inverse of :func:`pack_group`: scatter X (bs, S, G*H*D) back into the per-layer tensors."""
    lib = _lib.load()
    _require_cuda(x, *layers)
    g = len(layers)
    bs, h, s, d = layers[0].shape
    sb, sh, ss, sd = layers[0].stride()
    ptrs = (C.c_void_p * g)(*[t.data_ptr() for t in layers])
    check(lib.xkv_unpack_group(C.c_void_p(x.data_ptr()), g, bs, h, s, d, sb, sh, ss, ptrs, _stream()))


# ---------------------------------------------------------------------------------------------
# (2) GEMM engine
# ---------------------------------------------------------------------------------------------
def make_problem(
    a_limbs: Sequence[torch.Tensor],
    b_limbs: Sequence[torch.Tensor],
    out: torch.Tensor,
    *,
    M: int,
    N: int,
    K: int,
    a_mn_major: bool = False,
    b_mn_major: bool = False,
    terms: Sequence[Tuple[int, int]] = TERMS_1,
    out_transposed: bool = False,
    sym_upper: bool = False,
    split_k: int = 1,
    split_stride: int = 0,
    accum_phases: int = 1,
    a_layers: Optional[Sequence[torch.Tensor]] = None,
    b_layers: Optional[Sequence[torch.Tensor]] = None,
) -> GemmProblem:
    """Describe D = sum_t A[ta] @ B[tb]^T.  A limbs: (M, K) row-major, or (K, M) if a_mn_major;
    B limbs: (N, K) row-major, or (K, N) if b_mn_major. `out`: fp32/bf16, (M, N) or (N, M) if transposed;
    with split_k > 1 `out` is the first of split_k slabs `split_stride` elements apart.  accum_phases > 1: every
    CTA accumulates its k range in that many pieces on the tensor core and sums the pieces in fp32 (fp32 output).
    a_layers / b_layers: the operand is the column-wise concatenation of these equally shaped row-major matrices, read in
    place (a layer group's K / V without the gather); `a_limbs` / `b_limbs` are then ignored (pass [])."""
    p = GemmProblem()
    p.M, p.N, p.K = M, N, K
    p.num_terms = len(terms)
    p.a_mn_major, p.b_mn_major = int(a_mn_major), int(b_mn_major)
    for i in range(3):
        a = a_limbs[i] if i < len(a_limbs) else None
        b = b_limbs[i] if i < len(b_limbs) else None
        p.A[i] = a.data_ptr() if a is not None else None
        p.B[i] = b.data_ptr() if b is not None else None
    for t in list(a_limbs) + list(b_limbs) + list(a_layers or []) + list(b_layers or []):
        if t is not None and (t.dtype != torch.bfloat16 or t.stride(-1) != 1):
            raise _lib.XkvError("gemm operands must be bf16 with unit inner stride")
    for side, layers in (("a", a_layers), ("b", b_layers)):
        if not layers:
            continue
        if len(layers) > _lib.MAX_GROUP_LAYERS or any(t.shape != layers[0].shape or t.stride() != layers[0].stride() for t in layers):
            raise _lib.XkvError("gemm: layered operands must be equally shaped and strided (at most 16 layers)")
        setattr(p, side + "_layers", len(layers))
        p.layer_cols = layers[0].shape[1]
        arr = p.A_layer if side == "a" else p.B_layer
        for i, t in enumerate(layers):
            arr[i] = t.data_ptr()
    p.lda = (a_layers[0] if a_layers else a_limbs[0]).stride(0)
    p.ldb = (b_layers[0] if b_layers else b_limbs[0]).stride(0)
    for t, (ta, tb) in enumerate(terms):
        p.term_a[t], p.term_b[t] = ta, tb
    if out.dtype not in (torch.float32, torch.bfloat16) or out.stride(-1) != 1:
        raise _lib.XkvError("gemm output must be fp32 or bf16 with unit inner stride")
    p.D = out.data_ptr()
    p.ldd = out.stride(-2)
    p.out_bf16 = int(out.dtype == torch.bfloat16)
    p.out_transposed = int(out_transposed)
    p.sym_upper = int(sym_upper)
    p.split_k = split_k
    p.split_stride = split_stride
    p.accum_phases = accum_phases
    return p


def gemm_grouped(problems: Sequence[GemmProblem]) -> None:
    lib = _lib.load()
    arr = (GemmProblem * len(problems))(*problems)
    check(lib.xkv_gemm_grouped(arr, len(problems), _stream()))


# ---------------------------------------------------------------------------------------------
# small fp32 helpers of the factorisation
# ---------------------------------------------------------------------------------------------
def _ptr(t: Optional[torch.Tensor]) -> C.c_void_p:
    return C.c_void_p(t.data_ptr() if t is not None else None)


def _ptr_array(ts: Optional[Sequence[Optional[torch.Tensor]]]):
    if ts is None:
        return None
    return (C.c_void_p * len(ts))(*[(t.data_ptr() if t is not None else None) for t in ts])


def reduce_slabs(slabs: torch.Tensor, out: torch.Tensor, symmetrize: bool = False) -> None:
    """out = slabs.sum(0); with symmetrize the strictly-lower triangle mirrors the upper one.
    `slabs` is (S, rows, cols) fp32 (only upper-triangle tiles need be valid when symmetrize)."""
    _require_cuda(slabs, out)
    s, rows, cols = slabs.shape
    check(_lib.load().xkv_reduce_slabs(_ptr(slabs), s, slabs.stride(0), rows, cols, slabs.stride(1), int(symmetrize),
                                       _ptr(out), out.stride(0), _stream()))


def split_bf16(x: torch.Tensor, hi: torch.Tensor, mid: Optional[torch.Tensor] = None,
               lo: Optional[torch.Tensor] = None) -> None:
    """hi = bf16(x), mid = bf16(x - hi), lo = bf16(x - hi - mid) for a 2-D fp32 matrix."""
    _require_cuda(x, hi)
    rows, cols = x.shape
    check(_lib.load().xkv_split_bf16(_ptr(x), rows, cols, x.stride(0), _ptr(hi), _ptr(mid), _ptr(lo), hi.stride(0),
                                     _stream()))


def symmetrize_split_bf16(slabs: Sequence[torch.Tensor], hi: Sequence[torch.Tensor], mid: Sequence[torch.Tensor],
                          lo: Sequence[torch.Tensor]) -> None:
    """For each (S, n, n) fp32 slab stack (upper-triangle tiles valid): bf16 limbs of the full symmetric sum, one pass."""
    _require_cuda(*slabs, *hi)
    s, n, _ = slabs[0].shape
    check(_lib.load().xkv_symmetrize_split_bf16(_ptr_array(slabs), len(slabs), s, slabs[0].stride(0), n,
                                                slabs[0].stride(1), _ptr_array(hi), _ptr_array(mid), _ptr_array(lo),
                                                hi[0].stride(0), _stream()))


def gram_packed_elems(n: int) -> int:
    """Floats of the packed upper triangle of an n x n symmetric matrix (row r keeps its columns from 32 * (r // 32))."""
    return int(_lib.load().xkv_gram_packed_elems(n))


def gram_pack_upper(full: torch.Tensor, packed: Optional[torch.Tensor] = None) -> torch.Tensor:
    """Upper triangle of a symmetric (n, n) fp32 matrix, packed: the payload of the token-sharded Gram all-reduce."""
    _require_cuda(full, packed)
    n = full.shape[0]
    if full.dtype != torch.float32 or full.shape != (n, n) or full.stride(1) != 1:
        raise _lib.XkvError("gram_pack_upper: square fp32 matrix with unit inner stride required")
    if packed is None:
        packed = torch.empty(gram_packed_elems(n), dtype=torch.float32, device=full.device)
    check(_lib.load().xkv_gram_pack_upper(_ptr(full), n, full.stride(0), _ptr(packed), _stream()))
    return packed


def gram_unpack_upper(packed: torch.Tensor, full: torch.Tensor) -> torch.Tensor:
    """Inverse of gram_pack_upper: fills `full` (n, n) symmetrically (lower triangle = mirrored upper)."""
    _require_cuda(full, packed)
    n = full.shape[0]
    if packed.dtype != torch.float32 or packed.numel() < gram_packed_elems(n) or not packed.is_contiguous():
        raise _lib.XkvError("gram_unpack_upper: contiguous fp32 buffer of gram_packed_elems(n) floats required")
    check(_lib.load().xkv_gram_unpack_upper(_ptr(packed), n, _ptr(full), full.stride(0), _stream()))
    return full


def fill_gaussian_bf16(out: torch.Tensor, seed: int) -> None:
    _require_cuda(out)
    rows, cols = out.shape
    check(_lib.load().xkv_fill_gaussian_bf16(_ptr(out), rows, cols, out.stride(0), C.c_uint64(seed), _stream()))


def normalize_rows(ys: Sequence[torch.Tensor], hi=None, mid=None, lo=None) -> None:
    """Scale every row of each fp32 matrix to unit norm in place, optionally emitting bf16 limbs."""
    _require_cuda(*ys)
    rows, cols = ys[0].shape
    ldo = hi[0].stride(0) if hi is not None else cols
    check(_lib.load().xkv_normalize_rows(_ptr_array(ys), _ptr_array(hi), _ptr_array(mid), _ptr_array(lo), len(ys),
                                         rows, cols, ys[0].stride(0), ldo, _stream()))


def shift_normalize_rows(ys: Sequence[torch.Tensor], qs: Optional[Sequence[torch.Tensor]] = None,
                         shifts: Optional[torch.Tensor] = None, rdiag: Optional[Sequence[torch.Tensor]] = None,
                         rdiag_first: bool = True, hi=None, mid=None, lo=None) -> None:
    """Y <- Y - shifts[b] * Q (when `qs` is given), then row-normalise like normalize_rows; the row norms are
    recorded in (rdiag_first) or multiplied into `rdiag` (running diagonal of the triangular factor)."""
    _require_cuda(*ys)
    rows, cols = ys[0].shape
    ldo = hi[0].stride(0) if hi is not None else cols
    check(_lib.load().xkv_shift_normalize_rows(_ptr_array(ys), _ptr_array(qs), _ptr(shifts) if shifts is not None else None,
                                               _ptr_array(rdiag), int(rdiag_first), _ptr_array(hi), _ptr_array(mid),
                                               _ptr_array(lo), len(ys), rows, cols, ys[0].stride(0), ldo, _stream()))


def ritz_shift_update(rdiag: Sequence[torch.Tensor], shifts: torch.Tensor, tail_rows: int = 8, shift_scale: float = 0.5) -> None:
    """shifts[b] <- shift_scale * (mean of the last tail_rows entries of rdiag[b] + shifts[b])."""
    check(_lib.load().xkv_ritz_shift_update(_ptr_array(rdiag), len(rdiag), rdiag[0].numel(), tail_rows,
                                            C.c_float(shift_scale), _ptr(shifts), _stream()))


def rdiag_update(rdiag: Sequence[torch.Tensor], linvs: Sequence[torch.Tensor]) -> None:
    """rdiag[b][j] /= Linv[b][j][j]."""
    check(_lib.load().xkv_rdiag_update(_ptr_array(rdiag), _ptr_array(linvs), len(rdiag), rdiag[0].numel(),
                                       linvs[0].stride(0), _stream()))


def pass_flags(linvs: Sequence[torch.Tensor], min_pivot: float, flags: torch.Tensor) -> None:
    """flags[b] = 1 when the Cholesky pass that produced linvs[b] met a pivot L_jj^2 < min_pivot (or a NaN), else 0.
    `flags`: int32 CUDA tensor with one entry per matrix."""
    _require_cuda(*linvs, flags)
    l = linvs[0].shape[0]
    check(_lib.load().xkv_pass_flags(_ptr_array(linvs), len(linvs), l, linvs[0].stride(0), C.c_float(min_pivot),
                                     _ptr(flags), _stream()))


class launch_predicate:
    """Context manager: while active, this thread's batched launches of shift_normalize_rows, the batched slab reduction,
    cholesky_inverse and rdiag_update skip matrix b when flags[b] == 0 ON THE DEVICE (no host synchronisation)."""

    def __init__(self, flags: torch.Tensor):
        _require_cuda(flags)
        if flags.dtype != torch.int32:
            raise _lib.XkvError("launch_predicate: int32 flags required")
        self.flags = flags

    def __enter__(self):
        _lib.load().xkv_set_launch_predicate(_ptr(self.flags))
        return self

    def __exit__(self, *exc):
        _lib.load().xkv_set_launch_predicate(None)
        return False


def cholesky_inverse(ss: Sequence[torch.Tensor], linvs: Sequence[torch.Tensor], shift: float = 0.0,
                     pivot_floor: float = 1e-12, limbs=None) -> None:
    """Batched (S + shift*I) = L L^T and Linv = L^{-1} in one cluster launch (S is destroyed); `limbs` =
    (hi, mid, lo) lists of bf16 matrices that receive the limb split of Linv (mid / lo may be None).
    The library takes one row stride for every S and Linv and one for every limb matrix: a batch whose matrices do
    not share them would be read and written at the wrong addresses, so it is rejected."""
    _require_cuda(*ss, *linvs)
    l = ss[0].shape[0]
    ld = ss[0].stride(0)
    if len(linvs) != len(ss):
        raise _lib.XkvError("cholesky_inverse: one Linv per S required")
    for t in list(ss) + list(linvs):
        if t.dtype != torch.float32 or tuple(t.shape) != (l, l) or t.stride() != (ld, 1):
            raise _lib.XkvError(f"cholesky_inverse: every S and Linv must be a ({l}, {l}) fp32 matrix with the row stride "
                                f"of ss[0] ({ld}) and unit inner stride")
    if limbs is None:
        check(_lib.load().xkv_cholesky_inverse(_ptr_array(ss), _ptr_array(linvs), len(ss), l, ld, C.c_float(shift),
                                               C.c_float(pivot_floor), _stream()))
        return
    hi, mid, lo = limbs
    _require_cuda(*hi, *(mid or []), *(lo or []))
    ld_limb = hi[0].stride(0)
    for side in (hi, mid, lo):
        if side is None:
            continue
        if len(side) != len(ss):
            raise _lib.XkvError("cholesky_inverse: one limb matrix per S required")
        for t in side:
            if t is not None and (t.dtype != torch.bfloat16 or tuple(t.shape) != (l, l) or t.stride() != (ld_limb, 1)):
                raise _lib.XkvError(f"cholesky_inverse: every limb must be a ({l}, {l}) bf16 matrix with the row stride of "
                                    f"hi[0] ({ld_limb}) and unit inner stride")
    check(_lib.load().xkv_cholesky_inverse_limbs(_ptr_array(ss), _ptr_array(linvs), _ptr_array(hi), _ptr_array(mid),
                                                 _ptr_array(lo), len(ss), l, ld, ld_limb, C.c_float(shift),
                                                 C.c_float(pivot_floor), _stream()))


def jacobi_eigh(ts: Sequence[torch.Tensor], evals: Sequence[torch.Tensor],
                wts: Optional[Sequence[Optional[torch.Tensor]]] = None, sweeps: int = 8) -> None:
    """Eigen-decomposition of small symmetric windows (W <= 160): evals descending, eigenvectors as rows."""
    _require_cuda(*ts, *evals)
    w = ts[0].shape[0]
    ldw = w
    if wts is not None:
        for t in wts:
            if t is not None:
                ldw = t.stride(0)
    check(_lib.load().xkv_jacobi_eigh(_ptr_array(ts), _ptr_array(evals), _ptr_array(wts), len(ts), w, ts[0].stride(0),
                                      ldw, sweeps, _stream()))


def convert_bf16(src: torch.Tensor, dst: Optional[torch.Tensor] = None, dst_t: Optional[torch.Tensor] = None) -> None:
    """fp32 (rows, cols) -> bf16 copy and/or transposed bf16 copy (cols, rows)."""
    _require_cuda(src)
    rows, cols = src.shape
    check(_lib.load().xkv_convert_bf16(_ptr(src), rows, cols, src.stride(0), _ptr(dst),
                                       dst.stride(0) if dst is not None else 0, _ptr(dst_t),
                                       dst_t.stride(0) if dst_t is not None else 0, _stream()))


# ---------------------------------------------------------------------------------------------
# (3) decode-time attention over the factored cache
# ---------------------------------------------------------------------------------------------
def decode_workspace_bytes(hq: int, s: int, t: int, rv: int) -> int:
    return int(_lib.load().xkv_decode_workspace_bytes(hq, s, t, rv))


def decode_attention(q: torch.Tensor, a_k: torch.Tensor, vk_layer: torch.Tensor, a_v: torch.Tensor,
                     vv_layer: torch.Tensor, num_kv_heads: int, cos: Optional[torch.Tensor],
                     sin: Optional[torch.Tensor], k_tail: Optional[torch.Tensor], v_tail: Optional[torch.Tensor],
                     scale: float, out: Optional[torch.Tensor] = None,
                     workspace: Optional[torch.Tensor] = None,
                     lse_out: Optional[torch.Tensor] = None) -> torch.Tensor:
    """softmax(scale * q [K^; K_tail]^T) [V^; V_tail] for one layer, batch 1, with K^ = rope(bf16(A_k Vk_l^T)) and
    V^ = A_v Vv_l^T never materialised.  q (Hq, D); a_k (S, rk); vk_layer (H*D, rk); a_v (S, rv);
    vv_layer (H*D, rv); cos/sin (S, D) or None; k_tail/v_tail (H, T, D) or None.  Returns (Hq, D) bf16.
    lse_out: optional (Hq,) fp32 tensor that receives log sum exp of the scaled scores over THIS call's tokens
    (token-sharded contexts: see parallel.merge_token_shards).

    Multi-token step: q (Hq, Tq, D) returns (Hq, Tq, D) and lse_out is (Hq, Tq).  The last Tq tail tokens are the
    queries' own (T >= Tq) and query token t sees the prefix and tail tokens [0, T - Tq + t].  Bounds:
    (Hq / H) * Tq <= 64 and Hq * Tq <= 512 (XkvError past them)."""
    _require_cuda(q, a_k, vk_layer, a_v, vv_layer, cos, sin, k_tail, v_tail, out, workspace)
    if q.dim() not in (2, 3):
        raise _lib.XkvError("decode_attention: q must be (Hq, D) or (Hq, Tq, D)")
    multi = q.dim() == 3
    hq, d = q.shape[0], q.shape[-1]
    tq = q.shape[1] if multi else 1
    if lse_out is not None and (not lse_out.is_cuda or lse_out.dtype != torch.float32 or lse_out.numel() < hq * tq
                                or not lse_out.is_contiguous()):
        raise _lib.XkvError("decode_attention: lse_out must be a contiguous CUDA fp32 tensor of Hq * Tq elements")
    s, rk = a_k.shape
    rv = a_v.shape[1]
    t = 0 if k_tail is None else k_tail.shape[1]
    need = decode_workspace_bytes(hq * tq, s, t, rv)
    if workspace is None or workspace.numel() < need:
        workspace = torch.empty(need, dtype=torch.uint8, device=q.device)
    if out is None:
        out = torch.empty(*q.shape, dtype=torch.bfloat16, device=q.device)
    for name, x in (("q", q), ("a_k", a_k), ("vk_layer", vk_layer), ("a_v", a_v), ("vv_layer", vv_layer)):
        if x.dtype != torch.bfloat16 or x.stride(-1) != 1:
            raise _lib.XkvError(f"decode_attention: {name} must be bf16 with unit inner stride")
    if not q.is_contiguous():
        q = q.contiguous()
    if cos is not None and (cos.dtype != torch.bfloat16 or cos.stride(-1) != 1 or cos.shape[0] < s):
        raise _lib.XkvError("decode_attention: cos/sin must be bf16 (S, D) tables")
    sh = st = 0
    if t > 0:
        if k_tail.stride() != v_tail.stride() or k_tail.stride(-1) != 1:
            raise _lib.XkvError("decode_attention: k_tail / v_tail must share strides, unit inner stride")
        sh, st = k_tail.stride(0), k_tail.stride(1)
    lib = _lib.load()
    args = (_ptr(a_k), a_k.stride(0), rk, _ptr(vk_layer), vk_layer.stride(0), _ptr(a_v), a_v.stride(0), rv,
            _ptr(vv_layer), vv_layer.stride(0), s, _ptr(cos), _ptr(sin), cos.stride(0) if cos is not None else 0,
            _ptr(k_tail if t else None), _ptr(v_tail if t else None), t, sh, st, C.c_float(scale), _ptr(out),
            C.c_void_p(workspace.data_ptr()), workspace.numel(), _stream(), _ptr(lse_out))
    if multi:
        check(lib.xkv_decode_attention_multi(_ptr(q), hq, tq, num_kv_heads, d, *args))
    else:
        check(lib.xkv_decode_attention_lse(_ptr(q), hq, num_kv_heads, d, *args))
    return out


def decode_half_workspace_bytes(rows: int, s: int, t: int, value_width: int) -> int:
    return int(_lib.load().xkv_decode_half_workspace_bytes(rows, s, t, value_width))


def _dense_slot(x: torch.Tensor, s: int, h: int, d: int, name: str) -> Tuple[int, int]:
    """(head stride, token stride) of a dense prefix slot given as an (S, H, D) or (H, S, D) view."""
    if x.dim() != 3 or x.dtype != torch.bfloat16 or x.stride(-1) != 1:
        raise _lib.XkvError(f"decode_attention_half: {name} must be a bf16 (S, H, D) or (H, S, D) view with unit inner stride")
    if tuple(x.shape) == (s, h, d):
        return x.stride(1), x.stride(0)
    if tuple(x.shape) == (h, s, d):
        return x.stride(0), x.stride(1)
    raise _lib.XkvError(f"decode_attention_half: {name} has shape {tuple(x.shape)}, expected ({s}, {h}, {d}) or ({h}, {s}, {d})")


def decode_attention_half(q: torch.Tensor, num_kv_heads: int, *, a_k: Optional[torch.Tensor] = None,
                          vk_layer: Optional[torch.Tensor] = None, k_dense: Optional[torch.Tensor] = None,
                          a_v: Optional[torch.Tensor] = None, vv_layer: Optional[torch.Tensor] = None,
                          v_dense: Optional[torch.Tensor] = None, cos: Optional[torch.Tensor] = None,
                          sin: Optional[torch.Tensor] = None, k_tail: Optional[torch.Tensor] = None,
                          v_tail: Optional[torch.Tensor] = None, scale: float, out: Optional[torch.Tensor] = None,
                          workspace: Optional[torch.Tensor] = None, lse_out: Optional[torch.Tensor] = None) -> torch.Tensor:
    """:func:`decode_attention` for a one-sided group: exactly one side is factored (a_k / vk_layer, or a_v / vv_layer),
    the other is the dense prefix slot (k_dense: rotated keys, or v_dense), an (S, H, D) or (H, S, D) view with unit inner
    stride read in place (strides multiples of 8 elements, else XkvError; it is never copied).  cos / sin rotate a
    factored key side only.  q, the tail, lse_out, the multi-token form and the bounds are those of decode_attention."""
    _require_cuda(q, a_k, vk_layer, k_dense, a_v, vv_layer, v_dense, cos, sin, k_tail, v_tail, out, workspace, lse_out)
    if (a_k is None) == (k_dense is None) or (a_v is None) == (v_dense is None):
        raise _lib.XkvError("decode_attention_half: give each side either as factors or as a dense slot")
    if (a_k is None) == (a_v is None):
        raise _lib.XkvError("decode_attention_half: exactly one side must be factored (both factored: decode_attention; "
                            "both dense: SDPA)")
    if q.dim() not in (2, 3):
        raise _lib.XkvError("decode_attention_half: q must be (Hq, D) or (Hq, Tq, D)")
    hq, d = q.shape[0], q.shape[-1]
    tq = q.shape[1] if q.dim() == 3 else 1
    if lse_out is not None and (lse_out.dtype != torch.float32 or lse_out.numel() < hq * tq or not lse_out.is_contiguous()):
        raise _lib.XkvError("decode_attention_half: lse_out must be a contiguous CUDA fp32 tensor of Hq * Tq elements")
    s = (a_k if a_k is not None else a_v).shape[0]
    h = num_kv_heads
    for name, x in (("q", q), ("a_k", a_k), ("vk_layer", vk_layer), ("a_v", a_v), ("vv_layer", vv_layer)):
        if x is not None and (x.dtype != torch.bfloat16 or x.stride(-1) != 1):
            raise _lib.XkvError(f"decode_attention_half: {name} must be bf16 with unit inner stride")
    if (a_k is not None and vk_layer is None) or (a_v is not None and vv_layer is None):
        raise _lib.XkvError("decode_attention_half: a factored side needs its right factor rows (vk_layer / vv_layer)")
    ksh, kst = _dense_slot(k_dense, s, h, d, "k_dense") if k_dense is not None else (0, 0)
    vsh, vst = _dense_slot(v_dense, s, h, d, "v_dense") if v_dense is not None else (0, 0)
    if not q.is_contiguous():
        q = q.contiguous()
    if cos is not None and (cos.dtype != torch.bfloat16 or cos.stride(-1) != 1 or cos.shape[0] < s):
        raise _lib.XkvError("decode_attention_half: cos/sin must be bf16 (S, D) tables")
    t = 0 if k_tail is None else k_tail.shape[1]
    sh = st = 0
    if t > 0:
        if k_tail.stride() != v_tail.stride() or k_tail.stride(-1) != 1:
            raise _lib.XkvError("decode_attention_half: k_tail / v_tail must share strides, unit inner stride")
        sh, st = k_tail.stride(0), k_tail.stride(1)
    rk = a_k.shape[1] if a_k is not None else 0
    rv = a_v.shape[1] if a_v is not None else 0
    need = decode_half_workspace_bytes(hq * tq, s, t, rv if a_v is not None else d)
    if workspace is None or workspace.numel() < need:
        workspace = torch.empty(need, dtype=torch.uint8, device=q.device)
    if out is None:
        out = torch.empty(*q.shape, dtype=torch.bfloat16, device=q.device)
    check(_lib.load().xkv_decode_attention_half(
        _ptr(q), hq, tq, h, d, _ptr(a_k), a_k.stride(0) if a_k is not None else 0, rk, _ptr(vk_layer),
        vk_layer.stride(0) if vk_layer is not None else 0, _ptr(k_dense), ksh, kst, _ptr(a_v),
        a_v.stride(0) if a_v is not None else 0, rv, _ptr(vv_layer), vv_layer.stride(0) if vv_layer is not None else 0,
        _ptr(v_dense), vsh, vst, s, _ptr(cos), _ptr(sin), cos.stride(0) if cos is not None else 0,
        _ptr(k_tail if t else None), _ptr(v_tail if t else None), t, sh, st, C.c_float(scale), _ptr(out),
        C.c_void_p(workspace.data_ptr()), workspace.numel(), _stream(), _ptr(lse_out)))
    return out


def decode_absorbed(q_hat: torch.Tensor, a: torch.Tensor, scale: float, row_scale: Optional[torch.Tensor] = None,
                    bias_q: Optional[torch.Tensor] = None, bias_k: Optional[torch.Tensor] = None,
                    workspace: Optional[torch.Tensor] = None) -> Tuple[torch.Tensor, torch.Tensor]:
    """Absorbed attention over a token factor (MLA latents).  q_hat (Hq, r) bf16: the query folded into the rank space;
    a (S, r) bf16; row_scale (S,) fp32 or None; bias_q (Hq, d) / bias_k (S, d) bf16 or None (the RoPE part).
    Returns (u (Hq, r) fp32 = sum_t softmax(s)[h, t] row_scale[t] a[t], lse (Hq,) fp32) with
    s[h, t] = scale * (row_scale[t] * q_hat[h] . a[t] + bias_q[h] . bias_k[t])."""
    _require_cuda(q_hat, a, row_scale, bias_q, bias_k, workspace)
    hq, r = q_hat.shape
    s = a.shape[0]
    for name, x in (("q_hat", q_hat), ("a", a), ("bias_q", bias_q), ("bias_k", bias_k)):
        if x is not None and (x.dtype != torch.bfloat16 or x.stride(-1) != 1):
            raise _lib.XkvError(f"decode_absorbed: {name} must be bf16 with unit inner stride")
    if a.shape[1] != r or not q_hat.is_contiguous() or (bias_q is not None and not bias_q.is_contiguous()):
        raise _lib.XkvError("decode_absorbed: q_hat (Hq, r) / bias_q must be contiguous and match a (S, r)")
    if row_scale is not None and (row_scale.dtype != torch.float32 or not row_scale.is_contiguous() or row_scale.numel() < s):
        raise _lib.XkvError("decode_absorbed: row_scale must be a contiguous fp32 vector of S entries")
    lib = _lib.load()
    need = int(lib.xkv_decode_absorbed_workspace_bytes(hq, s, r))
    if workspace is None or workspace.numel() < need:
        workspace = torch.empty(need, dtype=torch.uint8, device=a.device)
    u = torch.empty(hq, r, dtype=torch.float32, device=a.device)
    lse = torch.empty(hq, dtype=torch.float32, device=a.device)
    check(lib.xkv_decode_absorbed(_ptr(q_hat), hq, _ptr(a), a.stride(0), r, s, _ptr(row_scale), _ptr(bias_q), _ptr(bias_k),
                                  bias_k.stride(0) if bias_k is not None else 0,
                                  bias_q.shape[1] if bias_q is not None else 0, C.c_float(scale), _ptr(u), _ptr(lse),
                                  C.c_void_p(workspace.data_ptr()), workspace.numel(), _stream()))
    return u, lse


def rope_bf16_(x: torch.Tensor, cos: torch.Tensor, sin: torch.Tensor) -> torch.Tensor:
    """In-place RoPE on token-major keys x (rows, H, D) bf16 with cos/sin (rows, D) bf16 (HF half-split)."""
    _require_cuda(x, cos, sin)
    rows, h, d = x.shape
    if x.stride(2) != 1 or x.stride(1) != d:
        raise _lib.XkvError("rope_bf16_: x must be (rows, H, D) with contiguous (H, D)")
    check(_lib.load().xkv_rope_bf16(_ptr(x), x.stride(0), rows, h, d, _ptr(cos), _ptr(sin), cos.stride(0), _stream()))
    return x


# ---------------------------------------------------------------------------------------------
# (4) append: project new token rows onto a group's right factor
# ---------------------------------------------------------------------------------------------
def append_project(x_new: torch.Tensor, v: torch.Tensor, out: Optional[torch.Tensor] = None,
                   workspace: Optional[torch.Tensor] = None) -> torch.Tensor:
    """a_new (T, r) = x_new (T, n) @ V (n, r), bf16 in / fp32 accumulate / bf16 out."""
    _require_cuda(x_new, v)
    t, n = x_new.shape
    r = v.shape[1]
    if x_new.dtype != torch.bfloat16 or v.dtype != torch.bfloat16 or x_new.stride(1) != 1 or v.stride(1) != 1:
        raise _lib.XkvError("append_project: bf16 operands with unit inner stride required")
    lib = _lib.load()
    need = int(lib.xkv_append_workspace_bytes(t, n, r))
    if workspace is None or workspace.numel() < need:
        workspace = torch.empty(need, dtype=torch.uint8, device=v.device)
    if out is None:
        out = torch.empty(t, r, dtype=torch.bfloat16, device=v.device)
    check(lib.xkv_append_project(_ptr(x_new), x_new.stride(0), t, _ptr(v), v.stride(0), n, r, _ptr(out), out.stride(0),
                                 C.c_void_p(workspace.data_ptr()), workspace.numel(), _stream()))
    return out


def append_project_many(xs: Sequence[torch.Tensor], vs: Sequence[torch.Tensor], outs: Sequence[torch.Tensor],
                        workspace: Optional[torch.Tensor] = None) -> None:
    """outs[i] (T, r_i) = xs[i] (T, n_i) @ vs[i] (n_i, r_i) for up to 4 projections in ONE launch (a group's K and V
    factor when decode tokens are folded)."""
    _require_cuda(*xs, *vs, *outs, workspace)
    lib = _lib.load()
    t = xs[0].shape[0]
    probs = (_lib.AppendProblem * len(xs))()
    need = 0
    for i, (x, v, o) in enumerate(zip(xs, vs, outs)):
        if (x.dtype != torch.bfloat16 or v.dtype != torch.bfloat16 or o.dtype != torch.bfloat16 or x.stride(1) != 1
                or v.stride(1) != 1 or o.stride(1) != 1 or x.shape[0] != t or x.shape[1] != v.shape[0]
                or tuple(o.shape) != (t, v.shape[1])):
            raise _lib.XkvError("append_project_many: bf16 (T, n) @ (n, r) -> (T, r) with unit inner strides required")
        probs[i].x_new, probs[i].V, probs[i].a_out = x.data_ptr(), v.data_ptr(), o.data_ptr()
        probs[i].ldx, probs[i].ldv, probs[i].lda = x.stride(0), v.stride(0), o.stride(0)
        probs[i].n, probs[i].r = v.shape[0], v.shape[1]
        need += int(lib.xkv_append_workspace_bytes(t, v.shape[0], v.shape[1]))
    if workspace is None or workspace.numel() < need:
        workspace = torch.empty(need, dtype=torch.uint8, device=vs[0].device)
    check(lib.xkv_append_project_batch(probs, len(xs), t, C.c_void_p(workspace.data_ptr()), workspace.numel(), _stream()))


# ---------------------------------------------------------------------------------------------
# SLERP / MiniCache branch
# ---------------------------------------------------------------------------------------------
def slerp_merge(x1: torch.Tensor, x2: torch.Tensor, t: float, gamma: float):
    """fake_minicache_merge (reference cache:93-100) on two (rows, d) bf16 matrices -> (e1, e2) bf16."""
    _require_cuda(x1, x2)
    if x1.dtype != torch.bfloat16 or x2.dtype != torch.bfloat16 or x1.shape != x2.shape or x1.stride() != x2.stride():
        raise _lib.XkvError("slerp_merge: two equally-shaped bf16 matrices required")
    if x1.stride(1) != 1:
        raise _lib.XkvError("slerp_merge: unit inner stride required")
    rows, d = x1.shape
    lib = _lib.load()
    ws = torch.empty(int(lib.xkv_slerp_workspace_bytes(rows)), dtype=torch.uint8, device=x1.device)
    e1 = torch.empty(rows, d, dtype=torch.bfloat16, device=x1.device)
    e2 = torch.empty_like(e1)
    check(lib.xkv_slerp_merge(_ptr(x1), _ptr(x2), rows, d, x1.stride(0), C.c_float(t), C.c_float(gamma), _ptr(e1),
                              _ptr(e2), e1.stride(0), C.c_void_p(ws.data_ptr()), ws.numel(), _stream()))
    return e1, e2
