"""CPU: the ragged-batch entry points — include/vitb200_ragged.h, the exports of libvitb200.so and the RAGGED_SIGNATURES
ctypes table agree in both directions and stay apart from the core and resolution headers; the descriptor struct and
its ctypes mirror have the same fields; the packed layout and the host-side checks of ``VIT.forward_ragged`` (no
compute calls: there is no GPU here)."""
import ctypes
import os
import re

import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
HEADER = os.path.join(ROOT, "include", "vitb200_ragged.h")
CORE_HEADER = os.path.join(ROOT, "include", "vitb200.h")
RESOLUTION_HEADER = os.path.join(ROOT, "include", "vitb200_resolution.h")

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


def test_ragged_header_declares_expected_entry_points():
    assert set(_declarations(HEADER)) == {"vt_patch_embed_ragged_gather", "vt_gather_rows"}


def test_ragged_entry_points_are_not_in_the_other_headers():
    ragged = set(_declarations(HEADER))
    assert not ragged & set(_declarations(CORE_HEADER))
    assert not ragged & set(_declarations(RESOLUTION_HEADER))
    assert '#include "vitb200.h"' in open(HEADER).read()


def test_library_exports_every_ragged_symbol_and_ctypes_match():
    mod = _lib()
    lib = mod.load()
    decls = _declarations(HEADER)
    assert set(mod.RAGGED_SIGNATURES) == set(decls)
    assert not set(mod.RAGGED_SIGNATURES) & (set(mod.SIGNATURES) | set(mod.RESOLUTION_SIGNATURES))
    for name, argtypes in mod.RAGGED_SIGNATURES.items():
        fn = getattr(lib, name)                     # exported
        assert fn.argtypes == argtypes and fn.restype == ctypes.c_int, f"{name}: not registered by load()"
        args = decls[name]
        assert len(args) == len(argtypes), f"{name}: header has {len(args)} args, ctypes {len(argtypes)}"
        for a, ct in zip(args, argtypes):
            if "*" in a:
                assert ct == ctypes.c_void_p, f"{name}: {a}"
            else:
                assert _CTYPE[a.split()[0]] == ct, f"{name}: {a} vs {ct}"


def test_descriptor_struct_matches_its_ctypes_mirror():
    from vit.kernels import _lib
    text = re.sub(r"/\*.*?\*/", "", open(HEADER).read(), flags=re.S)
    body = re.search(r"typedef struct vt_ragged_image\s*\{(.*?)\}\s*vt_ragged_image\s*;", text, flags=re.S).group(1)
    fields = [re.match(r"\s*(.*?)\s*(\w+)$", f).groups() for f in body.split(";") if f.strip()]
    mirror = _lib.RaggedImage._fields_
    assert [name for _, name in fields] == [name for name, _ in mirror]
    for (ctype, name), (_, ct) in zip(fields, mirror):
        assert (ct == ctypes.c_void_p) if "*" in ctype else (_CTYPE[ctype] == ct), f"{name}: {ctype} vs {ct}"
    assert ctypes.sizeof(_lib.RaggedImage) == 40


def _tiny(arch="tiny-b", **kw):
    from oracle import hf_oracle
    from vit.vit import VIT
    return VIT(**hf_oracle.vit_kwargs(arch), **kw)


def test_layout_groups_images_by_token_count_and_keeps_caller_order_inside_a_group():
    from vit import packing
    grids = [(14, 14), (1, 1), (15, 15), (14, 14), (2, 3), (1, 1), (7, 28)]
    L = packing.RaggedLayout(grids)
    assert L.tokens == [197, 2, 226, 197, 7, 2, 197]
    assert L.order == [1, 5, 4, 0, 3, 6, 2]
    assert L.groups == [(0, 2, 2), (4, 1, 7), (11, 3, 197), (602, 1, 226)]
    assert L.rows == 828 == sum(L.tokens)
    for r0, count, n in L.groups:                     # every image of a group inside its range, ranges tile [0, M)
        members = [i for i in range(len(grids)) if r0 <= L.row0[i] < r0 + count * n]
        assert len(members) == count and all(L.tokens[i] == n for i in members)
    assert sorted(L.row0[i] for i in range(len(grids))) == [0, 2, 4, 11, 208, 405, 602]


def test_layout_chunks_stay_under_the_row_limit():
    from vit import packing
    L = packing.RaggedLayout([(14, 14), (1, 1), (15, 15), (14, 14), (2, 3), (1, 1)])
    assert L.chunks() == [L.order]
    chunks = L.chunks(400)
    assert chunks == [[1, 5, 4, 0], [3], [2]]
    assert [i for c in chunks for i in c] == L.order
    assert all(sum(L.tokens[i] for i in c) <= 400 for c in chunks)
    with pytest.raises(AssertionError):
        L.chunks(100)
    assert packing.RAGGED_MAX_ROWS == 2 ** 31 - 1


def test_ragged_input_checks_raise_before_any_launch():
    model = _tiny(add_pooling_layer=True, num_labels=5)       # 16-pixel patches, 3 channels, on the CPU
    ok = torch.zeros(3, 32, 48)
    calls = [model.forward_ragged, model.pooled, model.pooler_output, model.logits]
    for fn in calls:
        with pytest.raises(AssertionError, match="at least one image"):
            fn([])
        with pytest.raises(AssertionError, match="one dtype"):
            fn([ok, torch.zeros(3, 32, 32, dtype=torch.bfloat16)])
        with pytest.raises(AssertionError, match="channels"):
            fn([ok, torch.zeros(4, 32, 32)])
        with pytest.raises(AssertionError, match="channels"):
            fn([torch.zeros(32, 32, 1, dtype=torch.uint8)])
        with pytest.raises(AssertionError, match="smaller than one 16-pixel patch"):
            fn([ok, torch.zeros(3, 15, 64)])
        with pytest.raises(AssertionError, match="smaller than one 16-pixel patch"):
            fn([torch.zeros(64, 8, 3, dtype=torch.uint8)])
        with pytest.raises(AssertionError, match=r"expected \(C, H, W\)"):
            fn([torch.zeros(1, 3, 32, 32)])
        with pytest.raises(AssertionError, match="float32 / bfloat16"):
            fn([torch.zeros(3, 32, 32, dtype=torch.float16)])


def test_ragged_input_checks_do_not_touch_the_library(monkeypatch):
    """The assertions fire before anything reaches the kernel entry points."""
    from vit.kernels import _lib
    calls = []
    monkeypatch.setattr(_lib, "call", lambda name, *a: calls.append(name))
    model = _tiny()
    for bad in ([], [torch.zeros(3, 32, 32), torch.zeros(3, 8, 32)], [torch.zeros(2, 32, 32)]):
        with pytest.raises(AssertionError):
            model.forward_ragged(bad)
    assert calls == []
