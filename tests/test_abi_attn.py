"""CPU: the attention-probabilities entry point — include/vitb200_attn.h, the exports of libvitb200.so and the
ATTN_SIGNATURES ctypes table agree in both directions and stay apart from the other headers and tables; the host-side
refusals of ``output_hidden_states`` / ``output_attentions`` (no compute calls: there is no GPU here)."""
import ctypes
import os
import re

import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
HEADER = os.path.join(ROOT, "include", "vitb200_attn.h")
OTHER_HEADERS = [os.path.join(ROOT, "include", h)
                 for h in ("vitb200.h", "vitb200_resolution.h", "vitb200_ragged.h", "vitb200_mask.h")]

_CTYPE = {"int32_t": ctypes.c_int32, "int64_t": ctypes.c_int64, "float": ctypes.c_float}
NAMES = {"vt_attn_probs"}


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


def test_attn_header_declares_expected_entry_points():
    assert set(_declarations(HEADER)) == NAMES
    assert '#include "vitb200.h"' in open(HEADER).read()


def test_attn_entry_points_are_not_in_the_other_headers():
    for path in OTHER_HEADERS:
        assert not NAMES & set(_declarations(path)), path
    for path in OTHER_HEADERS:          # and the other headers' entry points are not declared here
        assert not set(_declarations(path)) & set(_declarations(HEADER)), path


def test_library_exports_every_attn_symbol_and_ctypes_match():
    mod = _lib()
    lib = mod.load()
    decls = _declarations(HEADER)
    assert set(mod.ATTN_SIGNATURES) == set(decls)
    assert not set(mod.ATTN_SIGNATURES) & (set(mod.SIGNATURES) | set(mod.RESOLUTION_SIGNATURES)
                                           | set(mod.RAGGED_SIGNATURES) | set(mod.MASK_SIGNATURES))
    for name, argtypes in mod.ATTN_SIGNATURES.items():
        fn = getattr(lib, name)                     # exported
        assert fn.argtypes == argtypes and fn.restype == ctypes.c_int, f"{name}: not registered by load()"
        args = decls[name]
        assert len(args) == len(argtypes), f"{name}: header has {len(args)} args, ctypes {len(argtypes)}"
        for a, ct in zip(args, argtypes):
            if "*" in a:
                assert ct == ctypes.c_void_p, f"{name}: {a}"
            else:
                assert _CTYPE[a.split()[0]] == ct, f"{name}: {a} vs {ct}"


def test_attn_probs_rejects_bad_arguments_without_a_launch():
    """Argument checks run on the host before anything touches the device (all pointers here are fake)."""
    mod = _lib()
    lib = mod.load()
    fake = 1 << 20
    assert lib.vt_attn_probs(None, fake, fake, 1, 1, 4, 64, 8, 32, 0.125, None) == -1
    assert lib.vt_attn_probs(fake, fake, fake, 0, 1, 4, 64, 8, 32, 0.125, None) == -1
    assert lib.vt_attn_probs(fake, fake, fake, 1, 1, 0, 64, 8, 32, 0.125, None) == -1
    assert lib.vt_attn_probs(fake, fake, fake, 1, 1, 4, 32, 8, 32, 0.125, None) == mod.VT_ERR_UNSUPPORTED
    assert lib.vt_attn_probs(fake, fake, fake, 1, 1, 4, 64, 8, 32, -0.125, None) == mod.VT_ERR_UNSUPPORTED
    assert lib.vt_attn_probs(fake, fake, fake, 1, 1, 4, 64, 12, 32, 0.125, None) == -3
    assert lib.vt_attn_probs(fake + 8, fake, fake, 1, 1, 4, 64, 8, 32, 0.125, None) == -3
    assert lib.vt_attn_probs(fake, fake, fake + 1, 1, 1, 4, 64, 8, 32, 0.125, None) == -3


def _tiny(arch="tiny-b", **kw):
    from oracle import hf_oracle
    from vit.vit import VIT
    return VIT(**hf_oracle.vit_kwargs(arch), **kw)


FLAGS = [dict(output_hidden_states=True), dict(output_attentions=True),
         dict(output_hidden_states=True, output_attentions=True)]


@pytest.mark.parametrize("flags", FLAGS)
def test_output_flags_are_refused_before_any_launch(monkeypatch, flags):
    from vit.kernels import _lib
    calls = []
    monkeypatch.setattr(_lib, "call", lambda name, *a: calls.append(name))
    model = _tiny(add_pooling_layer=True, num_labels=5, add_decoder=True)
    x = torch.zeros(2, 3, 64, 64)
    x8 = torch.zeros(2, 64, 64, 3, dtype=torch.uint8)
    with pytest.raises(AssertionError, match="list of images"):
        model([x[0], x[1]], **flags)
    with pytest.raises(AssertionError, match="list of images"):
        model.forward_uint8([x8[0], x8[1]], **flags)
    for name in ("pooled", "pooler_output", "logits"):
        for inp in (x, x8, [x[0], x[1]]):
            with pytest.raises(AssertionError, match=f"not supported by {name}"):
                getattr(model, name)(inp, **flags)
    with pytest.raises(AssertionError, match="not supported by masked_image_modeling"):
        model.masked_image_modeling(x, torch.zeros(2, 16, dtype=torch.bool), **flags)
    assert calls == []


def test_vit_output_fields():
    from vit.vit import VITOutput
    t = torch.zeros(1)
    out = VITOutput(t)
    assert out[0] is t and out.last_hidden_state is t
    assert out.hidden_states is None and out.attentions is None
    assert VITOutput._fields == ("last_hidden_state", "hidden_states", "attentions")
