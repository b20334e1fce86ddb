"""CPU: the prefix-token entry points (DeiT's distillation token) — include/vitb200_tokens.h, the exports of
libvitb200.so and the TOKENS_SIGNATURES ctypes table agree in both directions and stay apart from the other headers and
tables; every entry point refuses a prefix other than 1 or 2 and bad shapes before anything is launched; the state-dict
keys of ``distillation_token`` / ``distillation_head``; the loader against HF ``DeiTModel`` and its heads; the host-side
refusals (no compute calls: there is no GPU here)."""
import ctypes
import os
import re
from types import SimpleNamespace

import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
HEADER = os.path.join(ROOT, "include", "vitb200_tokens.h")
OTHER_HEADERS = [os.path.join(ROOT, "include", h) for h in
                 ("vitb200.h", "vitb200_resolution.h", "vitb200_ragged.h", "vitb200_mask.h", "vitb200_attn.h",
                  "vitb200_preprocess.h")]

_CTYPE = {"int32_t": ctypes.c_int32, "int64_t": ctypes.c_int64, "float": ctypes.c_float}
NAMES = {"vt_patch_embed_gemm_hw_prefix", "vt_patch_embed_masked_gather_prefix", "vt_patch_embed_ragged_gather_prefix",
         "vt_pos_embed_resample_prefix", "vt_embed_finalize_prefix", "vt_embed_finalize_masked_prefix"}
VT_ERR_ARG = -1


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


def test_tokens_header_declares_expected_entry_points():
    assert set(_declarations(HEADER)) == NAMES
    assert '#include "vitb200.h"' in open(HEADER).read()


def test_tokens_entry_points_are_not_in_the_other_headers_or_tables():
    for path in OTHER_HEADERS:
        assert not NAMES & set(_declarations(path)), path
    mod = _lib()
    for table in (mod.SIGNATURES, mod.RESOLUTION_SIGNATURES, mod.RAGGED_SIGNATURES, mod.MASK_SIGNATURES,
                  mod.ATTN_SIGNATURES, mod.PREPROCESS_SIGNATURES):
        assert not NAMES & set(table)


def test_library_exports_every_tokens_symbol_and_ctypes_match():
    mod = _lib()
    lib = mod.load()
    decls = _declarations(HEADER)
    assert set(mod.TOKENS_SIGNATURES) == set(decls)
    for name, argtypes in mod.TOKENS_SIGNATURES.items():
        fn = getattr(lib, name)                     # exported
        assert fn.argtypes == argtypes and fn.restype == ctypes.c_int, f"{name}: not registered by load()"
        args = decls[name]
        assert len(args) == len(argtypes), f"{name}: header has {len(args)} args, ctypes {len(argtypes)}"
        for a, ct in zip(args, argtypes):
            if "*" in a:
                assert ct == ctypes.c_void_p, f"{name}: {a}"
            else:
                assert _CTYPE[a.split()[0]] == ct, f"{name}: {a} vs {ct}"
        assert args[-2] == "int32_t prefix", name


def test_each_tokens_entry_point_is_an_existing_one_plus_prefix():
    mod = _lib()
    old = {**mod.SIGNATURES, **mod.RESOLUTION_SIGNATURES, **mod.RAGGED_SIGNATURES, **mod.MASK_SIGNATURES}
    for name, argtypes in mod.TOKENS_SIGNATURES.items():
        base = old[name[:-len("_prefix")]]
        assert argtypes == base[:-1] + [ctypes.c_int32, ctypes.c_void_p], name


_P = 4096    # stands for a device pointer: every call below must return before reading anything


def _calls(prefix, bad_shape=False):
    """(name, args) of every tokens entry point with a valid shape (or one bad dimension) and this prefix."""
    s = 0 if bad_shape else 1
    return [
        ("vt_patch_embed_gemm_hw_prefix",
         (_P, 1, _P, 768, _P, _P, _P, None, _P, 2, 3, 224 * s, 224, 16, 768, prefix, None)),
        ("vt_patch_embed_masked_gather_prefix",
         (_P, 1, _P, _P, _P, _P, 768, _P, 2, 3, 224, 224, 16, 768 * s, prefix, None)),
        ("vt_patch_embed_ragged_gather_prefix", (_P, 2, 1, 3, 16, _P, 768, _P, 768, 396 * s, prefix, None)),
        ("vt_pos_embed_resample_prefix", (_P, 0, _P, 768, 14, 24 * s, 24, prefix, None)),
        ("vt_embed_finalize_prefix", (_P, _P, _P, 2, 198 * s, 768, 0, prefix, None)),
        ("vt_embed_finalize_masked_prefix", (_P, _P, _P, _P, _P, 2, 198 * s, 768, 0, prefix, None)),
    ]


@pytest.mark.parametrize("prefix", [0, 3, -1, 1 << 20])
def test_bad_prefix_is_refused_before_any_launch(prefix):
    lib = _lib().load()
    for name, args in _calls(prefix):
        assert getattr(lib, name)(*args) == VT_ERR_ARG, name


@pytest.mark.parametrize("prefix", [1, 2])
def test_bad_shapes_are_refused_before_any_launch(prefix):
    lib = _lib().load()
    for name, args in _calls(prefix, bad_shape=True):
        assert getattr(lib, name)(*args) == VT_ERR_ARG, name
    # fewer tokens than prefix rows
    assert lib.vt_embed_finalize_prefix(_P, _P, _P, 2, 1, 768, 0, 2, None) == VT_ERR_ARG
    assert lib.vt_embed_finalize_masked_prefix(_P, _P, _P, _P, _P, 2, 1, 768, 0, 2, None) == VT_ERR_ARG


def _vit(arch="tiny-b", **kw):
    from oracle import hf_oracle
    from vit.vit import VIT
    return VIT(**hf_oracle.vit_kwargs(arch), **kw)


def test_state_dict_keys():
    base = _vit()
    keys = set(base.state_dict())
    assert len(_vit("vit-b16-224").state_dict()) == 990
    assert base.embeddings.num_prefix_tokens == 1 and base.embeddings.distillation_token is None
    assert base.cls_classifier is None and base.distillation_classifier is None

    deit = _vit(distillation_token=True)
    sd = deit.state_dict()
    assert set(sd) - keys == {"embeddings.distillation_token"} and keys <= set(sd)
    assert deit.embeddings.num_prefix_tokens == 2
    assert sd["embeddings.distillation_token"].shape == (1, 1, 128)
    assert sd["embeddings.position_embeddings"].shape == (1, 16 + 2, 128)
    assert len(_vit("vit-b16-224", distillation_token=True).state_dict()) == 991

    heads = _vit(distillation_token=True, distillation_head=True, num_labels=7).state_dict()
    assert set(heads) - set(sd) == {"cls_classifier.weight", "cls_classifier.bias", "distillation_classifier.weight",
                                    "distillation_classifier.bias"}
    for name in ("cls_classifier", "distillation_classifier"):
        assert heads[f"{name}.weight"].shape == (128, 7) and heads[f"{name}.bias"].shape == (7,)
    plain = _vit(distillation_token=True, num_labels=7).state_dict()
    assert set(plain) - set(sd) == {"classifier.weight", "classifier.bias"}


def _hf_models(arch, labels=5):
    from transformers import (DeiTConfig, DeiTForImageClassification, DeiTForImageClassificationWithTeacher,
                              DeiTModel)
    from oracle import hf_oracle
    torch.manual_seed(0)
    cfg = DeiTConfig(**hf_oracle.ARCHS[arch], num_labels=labels)
    models = [DeiTModel(cfg, add_pooling_layer=True, use_mask_token=True), DeiTForImageClassification(cfg),
              DeiTForImageClassificationWithTeacher(cfg)]
    for m in models:
        with torch.no_grad():                      # HF zero-initialises biases and the tokens
            for p in m.parameters():
                p.normal_()
    return models


def _expected(hf_sd, name, num_heads):
    """The HF tensor a destination key of this package holds (dense weights transposed, heads split)."""
    m = re.match(r"^encoder\.layer\.(\d+)\.attention\.attention\.(\d+)\.(query|key|value)\.(weight|bias)$", name)
    if m:
        full = hf_sd[f"encoder.layer.{m.group(1)}.attention.attention.{m.group(3)}.{m.group(4)}"]
        dh = full.shape[0] // num_heads
        h = int(m.group(2))
        return full[h * dh:(h + 1) * dh].t() if m.group(4) == "weight" else full[h * dh:(h + 1) * dh]
    src = {"embeddings.projection.weight": "embeddings.patch_embeddings.projection.weight",
           "embeddings.projection.bias": "embeddings.patch_embeddings.projection.bias"}.get(name, name)
    m = re.match(r"^encoder\.layer\.(\d+)\.(output|intermediate|attention\.output)\.(weight|bias)$", name)
    if m:
        src = f"encoder.layer.{m.group(1)}.{m.group(2)}.dense.{m.group(3)}"
    t = hf_sd[src]
    return t.t() if t.dim() == 2 and not name.startswith("embeddings") else t


@pytest.mark.parametrize("arch", ["tiny-b", "tiny-h"])
def test_loader_copies_every_tensor_of_hf_deit(arch):
    from vit.utils import transfer_pretrained_weights
    model, classifier, teacher = _hf_models(arch)
    cases = [(model, dict(add_pooling_layer=True, use_mask_token=True)), (classifier, dict(num_labels=5)),
             (teacher, dict(num_labels=5, distillation_head=True))]
    for hf, kw in cases:
        ours = _vit(arch, distillation_token=True, **kw)
        transfer_pretrained_weights(hf, ours, verbose=False)
        hf_sd = {re.sub(r"^deit\.", "", k): v for k, v in hf.state_dict().items()}
        sd = ours.state_dict()
        for name, t in sd.items():
            want = _expected(hf_sd, name, ours.num_heads)
            assert torch.equal(t, want), f"{type(hf).__name__}: {name}"
        assert torch.equal(sd["embeddings.distillation_token"], hf_sd["embeddings.distillation_token"])
        if hf is teacher:
            assert torch.equal(sd["cls_classifier.weight"], hf_sd["cls_classifier.weight"].t())
            assert torch.equal(sd["distillation_classifier.bias"], hf_sd["distillation_classifier.bias"])


def test_loader_refuses_a_token_mismatch():
    from transformers import ViTConfig, ViTModel
    from oracle import hf_oracle
    from vit.utils import transfer_pretrained_weights
    deit, _, teacher = _hf_models("tiny-b")
    for hf in (deit, teacher):
        plain = _vit()
        before = {k: v.clone() for k, v in plain.state_dict().items()}
        with pytest.raises(AssertionError, match="distillation_token=True"):
            transfer_pretrained_weights(hf, plain, verbose=False)
        assert all(torch.equal(v, before[k]) for k, v in plain.state_dict().items())
    vit_hf = ViTModel(ViTConfig(**hf_oracle.ARCHS["tiny-b"]), add_pooling_layer=False)
    with pytest.raises(AssertionError, match="distillation_token=True"):
        transfer_pretrained_weights(vit_hf, _vit(distillation_token=True), verbose=False)


def test_host_refusals_raise_before_any_launch(monkeypatch):
    from vit.kernels import _lib
    calls = []
    monkeypatch.setattr(_lib, "call", lambda name, *a: calls.append(name))
    with pytest.raises(AssertionError, match="num_labels"):
        _vit(distillation_token=True, distillation_head=True)
    with pytest.raises(AssertionError, match="distillation_token"):
        _vit(distillation_head=True, num_labels=5)
    mim = _vit(distillation_token=True, add_decoder=True)
    with pytest.raises(AssertionError, match="distillation_token"):
        mim.masked_image_modeling(torch.zeros(2, 3, 64, 64), torch.zeros(2, 16, dtype=torch.bool))
    with pytest.raises(AssertionError, match="distillation_token"):
        mim.masked_image_modeling(torch.zeros(2, 3, 64, 64))
    with pytest.raises(AssertionError, match="distillation_head"):
        _vit(distillation_token=True, num_labels=5).distillation_logits(torch.zeros(2, 3, 64, 64))
    teacher = _vit(distillation_token=True, distillation_head=True, num_labels=5)
    with pytest.raises(AssertionError, match="output_hidden_states"):
        teacher.distillation_logits(torch.zeros(2, 3, 64, 64), output_attentions=True)
    with pytest.raises(AssertionError, match="not matching"):
        teacher.distillation_logits(torch.zeros(2, 3, 64, 48))
    with pytest.raises(AssertionError, match=r"\(batch, patches\)"):      # the mask counts patches, not tokens
        _vit(distillation_token=True, use_mask_token=True)(torch.zeros(2, 3, 64, 64),
                                                         bool_masked_pos=torch.zeros(2, 18, dtype=torch.bool))
    assert calls == []


def test_data_parallel_out_dim_of_a_distillation_head_model():
    from vit.parallel import DataParallelVIT
    teacher = _vit(distillation_token=True, distillation_head=True, num_labels=24)
    assert DataParallelVIT._out_dim(SimpleNamespace(output="logits", model=teacher)) == 24
    assert DataParallelVIT._out_dim(SimpleNamespace(output="logits", model=_vit(num_labels=16))) == 16


def test_ragged_layout_counts_the_prefix_tokens():
    from vit import packing
    grids = [(14, 14), (1, 1), (3, 5), (14, 14)]
    one, two = packing.RaggedLayout(grids), packing.RaggedLayout(grids, 2)
    assert one.tokens == [197, 2, 16, 197] and two.tokens == [198, 3, 17, 198]
    assert two.order == one.order and two.rows == sum(two.tokens)
    assert two.groups == [(0, 1, 3), (3, 1, 17), (20, 2, 198)]


def test_default_model_builds_the_same_embedding_tables():
    """A ViT model's position tables are the ones of the single-CLS formula, bit for bit; a DeiT model's rows 0 and 1
    carry cls + pos[0] - bias and dist + pos[1] - bias, the other rows as for ViT."""
    from vit import packing
    g = torch.Generator().manual_seed(0)
    for tok in (False, True):
        m = _vit(distillation_token=tok, use_mask_token=True)
        with torch.no_grad():
            for p in m.embeddings.parameters():
                p.copy_(torch.randn(p.shape, generator=g))
        pk = packing.pack_embeddings(m.embeddings)
        pos = m.embeddings.position_embeddings.detach().float()[0]
        bias = m.embeddings.projection.bias.detach().float()
        want = pos.clone()
        want[0] += m.embeddings.cls_token.detach().float().reshape(-1) - bias
        if tok:
            want[1] += m.embeddings.distillation_token.detach().float().reshape(-1) - bias
        assert torch.equal(pk.posb16.view(torch.int16), want.bfloat16().view(torch.int16))
        assert pk.prefix32.shape == (m.embeddings.num_prefix_tokens, 128)
        assert torch.equal(pk.posm16, (pos + m.embeddings.mask_token.detach().float().reshape(-1) - bias).bfloat16())
