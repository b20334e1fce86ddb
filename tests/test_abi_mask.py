"""CPU: the masked-input / masked-image-modeling entry points — include/vitb200_mask.h, the exports of libvitb200.so and
the MASK_SIGNATURES ctypes table agree in both directions and stay apart from the other headers; the state-dict keys of
``use_mask_token`` / ``add_decoder``; the loader against HF ``ViTForMaskedImageModeling``; the host-side checks of
``bool_masked_pos`` (no compute calls: there is no GPU here)."""
import ctypes
import os
import re

import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
HEADER = os.path.join(ROOT, "include", "vitb200_mask.h")
OTHER_HEADERS = [os.path.join(ROOT, "include", h) for h in ("vitb200.h", "vitb200_resolution.h", "vitb200_ragged.h")]

_CTYPE = {"int32_t": ctypes.c_int32, "int64_t": ctypes.c_int64, "float": ctypes.c_float, "uint32_t": ctypes.c_uint32}
NAMES = {"vt_patch_embed_masked_gather", "vt_embed_finalize_masked", "vt_mim_reconstruct"}


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


def test_mask_header_declares_expected_entry_points():
    assert set(_declarations(HEADER)) == NAMES
    assert '#include "vitb200.h"' in open(HEADER).read()


def test_mask_entry_points_are_not_in_the_other_headers():
    for path in OTHER_HEADERS:
        assert not NAMES & set(_declarations(path)), path


def test_library_exports_every_mask_symbol_and_ctypes_match():
    mod = _lib()
    lib = mod.load()
    decls = _declarations(HEADER)
    assert set(mod.MASK_SIGNATURES) == set(decls)
    assert not set(mod.MASK_SIGNATURES) & (set(mod.SIGNATURES) | set(mod.RESOLUTION_SIGNATURES)
                                           | set(mod.RAGGED_SIGNATURES))
    for name, argtypes in mod.MASK_SIGNATURES.items():
        fn = getattr(lib, name)                     # exported
        assert fn.argtypes == argtypes and fn.restype == ctypes.c_int, f"{name}: not registered by load()"
        args = decls[name]
        assert len(args) == len(argtypes), f"{name}: header has {len(args)} args, ctypes {len(argtypes)}"
        for a, ct in zip(args, argtypes):
            if "*" in a:
                assert ct == ctypes.c_void_p, f"{name}: {a}"
            else:
                assert _CTYPE[a.split()[0]] == ct, f"{name}: {a} vs {ct}"


def _tiny(arch="tiny-b", **kw):
    from oracle import hf_oracle
    from vit.vit import VIT
    return VIT(**hf_oracle.vit_kwargs(arch), **kw)


def test_state_dict_keys():
    base = _tiny()
    keys = list(base.state_dict())
    assert "embeddings.mask_token" not in keys and not any(k.startswith("decoder.") for k in keys)
    from oracle import hf_oracle
    from vit.vit import VIT
    assert len(VIT(**hf_oracle.vit_kwargs("vit-b16-224")).state_dict()) == 990

    masked = _tiny(use_mask_token=True).state_dict()
    assert set(masked) - set(keys) == {"embeddings.mask_token"} and set(keys) <= set(masked)
    assert masked["embeddings.mask_token"].shape == (1, 1, 128)

    for arch, stride, out in (("tiny-b", None, 16 * 16 * 3), ("tiny-h", None, 14 * 14 * 3), ("tiny-h", 16, 16 * 16 * 3)):
        kw = {} if stride is None else {"encoder_stride": stride}
        m = _tiny(arch, add_decoder=True, **kw)
        sd = m.state_dict()
        base_keys = set(_tiny(arch).state_dict())
        assert set(sd) - base_keys == {"embeddings.mask_token", "decoder.0.weight", "decoder.0.bias"}
        D = m.hidden_dim
        assert sd["decoder.0.weight"].shape == (out, D, 1, 1) and sd["decoder.0.bias"].shape == (out,)
        assert m.encoder_stride == (m.patch_size if stride is None else stride)


@pytest.mark.parametrize("stride", [14, 16])
def test_loader_copies_mask_token_and_decoder_from_hf(stride):
    from transformers import ViTConfig, ViTForMaskedImageModeling
    from oracle import hf_oracle
    from vit.utils import transfer_pretrained_weights
    torch.manual_seed(0)
    hf = ViTForMaskedImageModeling(ViTConfig(**hf_oracle.ARCHS["tiny-h"], encoder_stride=stride)).eval()
    with torch.no_grad():                          # HF zero-initialises the mask token and the conv bias
        hf.vit.embeddings.mask_token.normal_()
        hf.decoder[0].bias.normal_()
    model = _tiny("tiny-h", add_decoder=True, encoder_stride=stride)
    transfer_pretrained_weights(hf, model, verbose=False)
    assert torch.equal(model.embeddings.mask_token, hf.vit.embeddings.mask_token)
    assert torch.equal(model.decoder[0].weight, hf.decoder[0].weight)
    assert torch.equal(model.decoder[0].bias, hf.decoder[0].bias)
    assert torch.equal(model.embeddings.cls_token, hf.vit.embeddings.cls_token)


def test_mask_input_checks_raise_before_any_launch(monkeypatch):
    from vit.kernels import _lib
    calls = []
    monkeypatch.setattr(_lib, "call", lambda name, *a: calls.append(name))
    model = _tiny(add_pooling_layer=True, num_labels=5, add_decoder=True)   # 64 x 64, 16-pixel patches: 16 patches
    plain = _tiny(add_pooling_layer=True, num_labels=5)
    x = torch.zeros(2, 3, 64, 64)
    x8 = torch.zeros(2, 64, 64, 3, dtype=torch.uint8)
    good = torch.zeros(2, 16, dtype=torch.bool)
    fns = [lambda m, x_, k: m(x_, bool_masked_pos=k), lambda m, x_, k: m.pooled(x_, bool_masked_pos=k),
           lambda m, x_, k: m.pooler_output(x_, bool_masked_pos=k), lambda m, x_, k: m.logits(x_, bool_masked_pos=k),
           lambda m, x_, k: m.embeddings(x_, bool_masked_pos=k)]
    for fn in fns:
        with pytest.raises(AssertionError, match="use_mask_token"):
            fn(plain, x, good)
        with pytest.raises(AssertionError, match="torch.bool"):
            fn(model, x, good.to(torch.uint8))
        with pytest.raises(AssertionError, match="torch.bool"):
            fn(model, x, [[True] * 16] * 2)
        with pytest.raises(AssertionError, match=r"\(batch, patches\)"):
            fn(model, x, torch.zeros(2, 17, dtype=torch.bool))
        with pytest.raises(AssertionError, match=r"\(batch, patches\)"):
            fn(model, x, torch.zeros(3, 16, dtype=torch.bool))
        with pytest.raises(AssertionError, match="is on meta"):
            fn(model, x, good.to("meta"))
    for fn in fns[:4]:
        with pytest.raises(AssertionError, match="list of images"):
            fn(model, [x[0], x[1]], good)
    for fn in (model, model.embeddings):                  # an interpolated 3 x 5 grid has 15 patches
        with pytest.raises(AssertionError, match=r"\(batch, patches\) = \(2, 15\)"):
            fn(torch.zeros(2, 3, 48, 80), interpolate_pos_encoding=True, bool_masked_pos=good)
    with pytest.raises(AssertionError, match=r"\(batch, patches\)"):
        model.forward_uint8(x8, bool_masked_pos=torch.zeros(2, 15, dtype=torch.bool))
    with pytest.raises(AssertionError, match="torch.bool"):
        model.forward_uint8(x8, bool_masked_pos=good.float())
    with pytest.raises(AssertionError, match="use_mask_token"):
        plain.forward_uint8(x8, bool_masked_pos=good)
    with pytest.raises(AssertionError, match="use_mask_token"):
        plain.embeddings.forward_uint8(x8, bool_masked_pos=good)
    with pytest.raises(AssertionError, match="list of images"):
        model.forward_uint8([x8[0]], bool_masked_pos=good)
    assert calls == []


def test_masked_image_modeling_checks_raise_before_any_launch(monkeypatch):
    from vit.kernels import _lib
    calls = []
    monkeypatch.setattr(_lib, "call", lambda name, *a: calls.append(name))
    good = torch.zeros(2, 16, dtype=torch.bool)
    with pytest.raises(AssertionError, match="add_decoder"):
        _tiny(use_mask_token=True).masked_image_modeling(torch.zeros(2, 3, 64, 64), good)
    wide = _tiny("tiny-h", add_decoder=True, encoder_stride=16)         # HF's default stride with 14-pixel patches
    with pytest.raises(AssertionError, match="encoder_stride == patch_size"):
        wide.masked_image_modeling(torch.zeros(2, 3, 56, 56), torch.zeros(2, 16, dtype=torch.bool))
    model = _tiny(add_decoder=True)
    with pytest.raises(AssertionError, match="multiples of 16"):
        model.masked_image_modeling(torch.zeros(2, 3, 64, 70), torch.zeros(2, 16, dtype=torch.bool),
                                    interpolate_pos_encoding=True)
    with pytest.raises(AssertionError, match=r"\(batch, patches\)"):
        model.masked_image_modeling(torch.zeros(2, 3, 64, 64), torch.zeros(2, 4, dtype=torch.bool))
    with pytest.raises(AssertionError, match="not a list"):
        model.masked_image_modeling([torch.zeros(3, 64, 64)], good)
    assert calls == []
