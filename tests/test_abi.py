"""CPU: the C-ABI library loads and exports exactly what include/vitb200.h declares, and the ctypes
signatures in vit/kernels/_lib.py agree with the header (no compute calls — there is no GPU here)."""
import ctypes
import os
import re

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
HEADER = os.path.join(ROOT, "include", "vitb200.h")

_CTYPE = {"int32_t": ctypes.c_int32, "int64_t": ctypes.c_int64, "float": ctypes.c_float, "uint32_t": ctypes.c_uint32}


def _declarations():
    text = re.sub(r"/\*.*?\*/", "", open(HEADER).read(), flags=re.S)
    decls = {}
    for m in re.finditer(r"\b(int|const char\*)\s+(vt_\w+)\s*\(([^)]*)\)\s*;", text):
        args = [a.strip() for a in m.group(3).split(",")] if m.group(3).strip() != "void" else []
        decls[m.group(2)] = args
    return decls


def _lib():
    from vit.kernels import _lib
    if not os.path.exists(_lib.lib_path()):
        import __graft_entry__
        __graft_entry__.build()
    return _lib


def test_header_declares_the_core_entry_points():
    names = set(_declarations())
    assert {"vt_layernorm", "vt_add", "vt_softmax", "vt_gemm_bf16", "vt_gemm_strided", "vt_flash_attn",
            "vt_gemm_bf16_ln", "vt_ln_fold", "vt_bgemm", "vt_pack_bf16", "vt_gemm_fp8", "vt_layernorm_fp8", "vt_quantize_rows_fp8", "vt_patch_embed_gemm", "vt_patching", "vt_embed_finalize", "vt_conv2d", "vt_pool_cls", "vt_pool_cls_allgather", "vt_version",
            "vt_status_string"} == names


def test_library_exports_every_declared_symbol():
    lib = _lib().load()
    for name in _declarations():
        assert hasattr(lib, name), f"{name} declared in vitb200.h but not exported"
    assert lib.vt_version() >= 100
    assert lib.vt_status_string(0) == b"ok"
    assert b"alignment" in lib.vt_status_string(-3)


def test_ctypes_signatures_match_header():
    mod = _lib()
    decls = _declarations()
    for name, argtypes in mod.SIGNATURES.items():
        args = decls[name]
        assert len(args) == len(argtypes), f"{name}: header has {len(args)} args, ctypes {len(argtypes)}"
        for a, ct in zip(args, argtypes):
            if "*" in a:
                assert ct in (ctypes.c_void_p, ctypes.POINTER(ctypes.c_int64)), f"{name}: {a}"
                if "int64_t*" in a.replace(" ", ""):
                    assert ct == ctypes.POINTER(ctypes.c_int64)
            else:
                base = a.split()[0]
                assert _CTYPE[base] == ct, f"{name}: {a} vs {ct}"
    assert set(mod.SIGNATURES) == {n for n in decls if n not in ("vt_version", "vt_status_string")}


def test_entry_points_refuse_cpu_tensors():
    """No CPU fallback: every public kernel entry point asserts on non-CUDA input."""
    import torch
    from vit import kernels
    x = torch.zeros(1, 4, 8)
    with pytest.raises(AssertionError):
        kernels.add(x, x)
    with pytest.raises(AssertionError):
        kernels.softmax(x)
    with pytest.raises(AssertionError):
        kernels.layernorm(x, torch.ones(8), torch.zeros(8), 1e-5)
    with pytest.raises(AssertionError):
        kernels.matmul(x, torch.zeros(8, 8))
    with pytest.raises(AssertionError):
        kernels.matmul3(x, torch.zeros(1, 8, 4))
    with pytest.raises(AssertionError):
        kernels.conv2d(torch.zeros(1, 3, 4, 4), torch.zeros(2, 3, 2, 2), torch.zeros(2))
    with pytest.raises(AssertionError):
        kernels.flash_attention(torch.zeros(1, 4, 3 * 64), 1)
