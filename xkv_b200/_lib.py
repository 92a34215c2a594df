"""ctypes binding of the C-ABI library ``libxkv_b200.so`` (declared in ``include/xkv_b200.h``).

The library is the product: there is no CPU or PyTorch fallback.  If it is missing, ``load()``
raises, and every op in :mod:`xkv_b200.ops` fails loudly.
"""
from __future__ import annotations

import ctypes as C
import os
from typing import Optional

# XKV_B200_LIB: another build of the same library (same-box A/B measurements of a kernel change); default: the in-tree build
_LIB_PATH = os.environ.get("XKV_B200_LIB") or os.path.join(os.path.dirname(os.path.abspath(__file__)), "libxkv_b200.so")
_lib: Optional[C.CDLL] = None

MAX_GROUP_LAYERS = 16
MAX_GEMM_PROBLEMS = 16
MAX_BATCH = 16
FACTORIZE_SIGMA_COUNT = 128


class XkvError(RuntimeError):
    """Raised when a C-ABI call returns a non-zero status (mirrors the reference's Python exceptions)."""


class GemmProblem(C.Structure):
    """Mirror of ``xkv_gemm_problem`` (include/xkv_b200.h)."""

    _fields_ = [
        ("M", C.c_int32),
        ("N", C.c_int32),
        ("K", C.c_int32),
        ("num_terms", C.c_int32),
        ("a_mn_major", C.c_int32),
        ("b_mn_major", C.c_int32),
        ("A", C.c_void_p * 3),
        ("B", C.c_void_p * 3),
        ("lda", C.c_int64),
        ("ldb", C.c_int64),
        ("term_a", C.c_uint8 * 6),
        ("term_b", C.c_uint8 * 6),
        ("D", C.c_void_p),
        ("ldd", C.c_int64),
        ("out_bf16", C.c_int32),
        ("out_transposed", C.c_int32),
        ("sym_upper", C.c_int32),
        ("split_k", C.c_int32),
        ("split_stride", C.c_int64),
        ("accum_phases", C.c_int32),
        ("run_if", C.c_void_p),
        ("a_layers", C.c_int32),
        ("b_layers", C.c_int32),
        ("layer_cols", C.c_int32),
        ("A_layer", C.c_void_p * MAX_GROUP_LAYERS),
        ("B_layer", C.c_void_p * MAX_GROUP_LAYERS),
    ]


class AppendProblem(C.Structure):
    """Mirror of ``xkv_append_problem`` (include/xkv_b200.h)."""

    _fields_ = [("x_new", C.c_void_p), ("V", C.c_void_p), ("a_out", C.c_void_p), ("ldx", C.c_int64), ("ldv", C.c_int64),
                ("lda", C.c_int64), ("n", C.c_int32), ("r", C.c_int32)]


# name -> (restype, argtypes); every symbol include/xkv_b200.h declares must appear here
_vp, _i, _i64, _f, _sz = C.c_void_p, C.c_int, C.c_int64, C.c_float, C.c_size_t
_pp = C.POINTER(C.c_void_p)
SIGNATURES = {
    "xkv_last_error": (C.c_char_p, []),
    "xkv_version": (_i, []),
    "xkv_launch_count": (_i64, []),
    "xkv_pack_group": (_i, [_pp, _i, _i, _i, _i, _i, _i64, _i64, _i64, _vp, _vp]),
    "xkv_unpack_group": (_i, [_vp, _i, _i, _i, _i, _i, _i64, _i64, _i64, _pp, _vp]),
    "xkv_gemm_grouped": (_i, [C.POINTER(GemmProblem), _i, _vp]),
    "xkv_reduce_slabs": (_i, [_vp, _i, _i64, _i, _i, _i64, _i, _vp, _i64, _vp]),
    "xkv_reduce_slabs_batched": (_i, [_pp, _pp, _i, _i, _i64, _i, _i, _i64, _i, _i64, _vp]),
    "xkv_symmetrize_split_bf16": (_i, [_pp, _i, _i, _i64, _i, _i64, _pp, _pp, _pp, _i64, _vp]),
    "xkv_split_bf16_batched": (_i, [_pp, _pp, _pp, _pp, _i, _i, _i, _i64, _i64, _vp]),
    "xkv_split_bf16": (_i, [_vp, _i, _i, _i64, _vp, _vp, _vp, _i64, _vp]),
    "xkv_gram_packed_elems": (_sz, [_i]),
    "xkv_gram_pack_upper": (_i, [_vp, _i, _i64, _vp, _vp]),
    "xkv_gram_unpack_upper": (_i, [_vp, _i, _vp, _i64, _vp]),
    "xkv_fill_gaussian_bf16": (_i, [_vp, _i, _i, _i64, C.c_uint64, _vp]),
    "xkv_normalize_rows": (_i, [_pp, _pp, _pp, _pp, _i, _i, _i, _i64, _i64, _vp]),
    "xkv_shift_normalize_rows": (_i, [_pp, _pp, _vp, _pp, _i, _pp, _pp, _pp, _i, _i, _i, _i64, _i64, _vp]),
    "xkv_ritz_shift_update": (_i, [_pp, _i, _i, _i, _f, _vp, _vp]),
    "xkv_rdiag_update": (_i, [_pp, _pp, _i, _i, _i64, _vp]),
    "xkv_pass_flags": (_i, [_pp, _i, _i, _i64, C.c_float, _vp, _vp]),
    "xkv_set_launch_predicate": (None, [_vp]),
    "xkv_cholesky_inverse": (_i, [_pp, _pp, _i, _i, _i64, _f, _f, _vp]),
    "xkv_cholesky_inverse_limbs": (_i, [_pp, _pp, _pp, _pp, _pp, _i, _i, _i64, _i64, _f, _f, _vp]),
    "xkv_jacobi_eigh": (_i, [_pp, _pp, _pp, _i, _i, _i64, _i64, _i, _vp]),
    "xkv_convert_bf16": (_i, [_vp, _i, _i, _i64, _vp, _i64, _vp, _i64, _vp]),
    "xkv_sqrt_clamp": (_i, [_vp, _vp, _i, _vp]),
    "xkv_factorize_workspace_bytes": (_sz, [_i, _i, _i, _i]),
    "xkv_decode_workspace_bytes": (_sz, [_i, _i, _i, _i]),
    "xkv_decode_attention": (_i, [_vp, _i, _i, _i, _vp, _i64, _i, _vp, _i64, _vp, _i64, _i, _vp, _i64, _i, _vp, _vp, _i64,
                                  _vp, _vp, _i, _i64, _i64, _f, _vp, _vp, _sz, _vp]),
    "xkv_decode_attention_lse": (_i, [_vp, _i, _i, _i, _vp, _i64, _i, _vp, _i64, _vp, _i64, _i, _vp, _i64, _i, _vp, _vp,
                                      _i64, _vp, _vp, _i, _i64, _i64, _f, _vp, _vp, _sz, _vp, _vp]),
    "xkv_decode_attention_multi": (_i, [_vp, _i, _i, _i, _i, _vp, _i64, _i, _vp, _i64, _vp, _i64, _i, _vp, _i64, _i, _vp,
                                        _vp, _i64, _vp, _vp, _i, _i64, _i64, _f, _vp, _vp, _sz, _vp, _vp]),
    "xkv_decode_half_workspace_bytes": (_sz, [_i, _i, _i, _i]),
    "xkv_decode_attention_half": (_i, [_vp, _i, _i, _i, _i, _vp, _i64, _i, _vp, _i64, _vp, _i64, _i64, _vp, _i64, _i, _vp,
                                       _i64, _vp, _i64, _i64, _i, _vp, _vp, _i64, _vp, _vp, _i, _i64, _i64, _f, _vp, _vp,
                                       _sz, _vp, _vp]),
    "xkv_decode_absorbed_workspace_bytes": (_sz, [_i, _i, _i]),
    "xkv_decode_absorbed": (_i, [_vp, _i, _vp, _i64, _i, _i, _vp, _vp, _vp, _i64, _i, _f, _vp, _vp, _vp, _sz, _vp]),
    "xkv_decode_force_tiled": (None, [_i]),
    "xkv_decode_set_variant": (None, [_i]),
    "xkv_rope_bf16": (_i, [_vp, _i64, _i, _i, _i, _vp, _vp, _i64, _vp]),
    "xkv_append_workspace_bytes": (_sz, [_i, _i, _i]),
    "xkv_append_project": (_i, [_vp, _i64, _i, _vp, _i64, _i, _i, _vp, _i64, _vp, _sz, _vp]),
    "xkv_append_project_batch": (_i, [C.POINTER(AppendProblem), _i, _i, _vp, _sz, _vp]),
    "xkv_slerp_workspace_bytes": (_sz, [_i64]),
    "xkv_slerp_merge": (_i, [_vp, _vp, _i64, _i, _i64, _f, _f, _vp, _vp, _i64, _vp, _sz, _vp]),
    "xkv_gemm_problem_size": (C.c_size_t, []),
    "xkv_gemm_set_gram_pair": (None, [_i]),
    "xkv_factorize_groups": (_i, [_pp, _i, _i, _i, _i, _i64, _i, _pp, _pp, _pp, _pp, _vp, _sz, _pp, _vp]),
    "xkv_factorize_batch": (_i, [_pp, _i, _i, _i, _i64, _i, _pp, _pp, _pp, _pp, _pp, _i, _vp, _sz, _pp, _vp]),
}


def lib_path() -> str:
    return _LIB_PATH


def load() -> C.CDLL:
    """Load the shared library (once) and attach the prototypes."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(_LIB_PATH):
        raise XkvError(
            f"{_LIB_PATH} not found: build it with `python -c 'import __graft_entry__ as g; g.build()'` "
            "(or `make -C xkv_b200/csrc`). xkv_b200 has no CPU fallback."
        )
    lib = C.CDLL(_LIB_PATH)
    for name, (res, args) in SIGNATURES.items():
        fn = getattr(lib, name)
        fn.restype = res
        fn.argtypes = args
    _lib = lib
    return lib


def check(status: int) -> None:
    if status != 0:
        msg = load().xkv_last_error()
        raise XkvError(msg.decode() if msg else f"xkv call failed with status {status}")
