"""CPU: the C-ABI library loads without a GPU driver and exports every symbol include/xkv_b200.h declares."""
import os
import re

from xkv_b200 import _lib

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _declared_symbols():
    text = open(os.path.join(ROOT, "include", "xkv_b200.h")).read()
    return sorted(set(re.findall(r"XKV_API\s+[\w\s\*]+?\b(xkv_\w+)\s*\(", text)))


def test_library_exports_every_declared_symbol():
    lib = _lib.load()
    names = _declared_symbols()
    assert len(names) >= 20
    for name in names:
        assert hasattr(lib, name), f"{name} declared in include/xkv_b200.h but not exported"


def test_bindings_cover_the_header():
    assert sorted(_lib.SIGNATURES) == _declared_symbols()
    header = open(os.path.join(ROOT, "include", "xkv_b200.h")).read()
    for name in ("MAX_GROUP_LAYERS", "MAX_GEMM_PROBLEMS", "MAX_BATCH", "FACTORIZE_SIGMA_COUNT"):
        assert re.search(rf"#define XKV_{name} {getattr(_lib, name)}\b", header), name


def test_version_error_channel_and_host_queries():
    lib = _lib.load()
    assert lib.xkv_version() >= 100
    assert isinstance(lib.xkv_last_error(), bytes)
    assert lib.xkv_launch_count() >= 0
    # pure host arithmetic works without a device
    assert lib.xkv_factorize_workspace_bytes(1, 4096, 4096, 512) > 0
    assert lib.xkv_factorize_workspace_bytes(1, 64, 4096, 512) == 0      # rank > tokens
    assert b"rank" in lib.xkv_last_error()
    assert lib.xkv_decode_workspace_bytes(32, 65536, 16, 768) > 0
    # the ctypes mirror has the library's struct layout
    import ctypes as C

    assert lib.xkv_gemm_problem_size() == C.sizeof(_lib.GemmProblem)
