"""CPU: the any-resolution entry points — include/vitb200_resolution.h, the exports of libvitb200.so and the
RESOLUTION_SIGNATURES ctypes table agree in both directions and stay apart from vitb200.h's set — and the host-side
checks of ``interpolate_pos_encoding`` (no compute calls: there is no GPU here)."""
import ctypes
import os
import re

import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
HEADER = os.path.join(ROOT, "include", "vitb200_resolution.h")
CORE_HEADER = os.path.join(ROOT, "include", "vitb200.h")

_CTYPE = {"int32_t": ctypes.c_int32, "int64_t": ctypes.c_int64, "float": ctypes.c_float, "uint32_t": ctypes.c_uint32}


def _declarations(path):
    text = re.sub(r"/\*.*?\*/", "", open(path).read(), flags=re.S)
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


def test_resolution_header_declares_expected_entry_points():
    assert set(_declarations(HEADER)) == {"vt_patch_embed_gemm_hw", "vt_pos_embed_resample"}


def test_resolution_entry_points_are_not_in_the_core_header():
    assert not set(_declarations(HEADER)) & set(_declarations(CORE_HEADER))
    assert '#include "vitb200.h"' in open(HEADER).read()


def test_library_exports_every_resolution_symbol_and_ctypes_match():
    mod = _lib()
    lib = mod.load()
    decls = _declarations(HEADER)
    assert set(mod.RESOLUTION_SIGNATURES) == set(decls)
    assert not set(mod.RESOLUTION_SIGNATURES) & set(mod.SIGNATURES)
    for name, argtypes in mod.RESOLUTION_SIGNATURES.items():
        fn = getattr(lib, name)                     # exported
        assert fn.argtypes == argtypes and fn.restype == ctypes.c_int, f"{name}: not registered by load()"
        args = decls[name]
        assert len(args) == len(argtypes), f"{name}: header has {len(args)} args, ctypes {len(argtypes)}"
        for a, ct in zip(args, argtypes):
            if "*" in a:
                assert ct == ctypes.c_void_p, f"{name}: {a}"
            else:
                assert _CTYPE[a.split()[0]] == ct, f"{name}: {a} vs {ct}"


def test_patch_embed_gemm_hw_extends_the_square_signature():
    """Same arguments as vt_patch_embed_gemm with S split into H, W."""
    mod = _lib()
    sq = list(mod.SIGNATURES["vt_patch_embed_gemm"])
    hw = list(mod.RESOLUTION_SIGNATURES["vt_patch_embed_gemm_hw"])
    s_at = 11                                      # (pixels, dtype, w, ldw, bias, posb, out, stats, work, B, C, S, ...)
    assert hw == sq[:s_at] + [ctypes.c_int32, ctypes.c_int32] + sq[s_at + 1:]


def _tiny(arch="tiny-b"):
    from oracle import hf_oracle
    from vit.vit import VIT
    return VIT(**hf_oracle.vit_kwargs(arch))


def test_patch_grid_and_native_grid():
    from vit import packing
    emb = _tiny("tiny-h").embeddings                     # 14-pixel patches, 4 x 4 grid
    assert packing.native_grid(emb) == (4, 4)
    assert packing.patch_grid(emb, 56, 56) == (4, 4)
    assert packing.patch_grid(emb, 70, 100) == (5, 7)    # partial patches dropped like a stride-P convolution
    assert packing.patch_grid(emb, 14, 27) == (1, 1)


def test_interpolated_forward_checks_channels_and_minimum_size():
    model = _tiny()
    with pytest.raises(AssertionError, match="channels"):
        model(torch.zeros(1, 4, 64, 64), interpolate_pos_encoding=True)
    with pytest.raises(AssertionError, match="patch size"):
        model(torch.zeros(1, 3, 15, 64), interpolate_pos_encoding=True)
    with pytest.raises(AssertionError, match="patch size"):
        model.forward_uint8(torch.zeros(1, 64, 8, 3, dtype=torch.uint8), interpolate_pos_encoding=True)


def test_without_the_flag_a_wrong_size_raises_the_existing_assertion():
    model = _tiny()
    with pytest.raises(AssertionError, match=r"not matching with the model input size: \(3, 64, 64\)"):
        model(torch.zeros(1, 3, 64, 96))
    with pytest.raises(AssertionError, match=r"not matching with the model input size: \(64, 64, 3\)"):
        model.forward_uint8(torch.zeros(1, 64, 96, 3, dtype=torch.uint8))
    with pytest.raises(AssertionError, match="not matching with the model input size"):
        model.pooled(torch.zeros(1, 3, 96, 96))
