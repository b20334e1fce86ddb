"""CPU: CLIP image encoders — include/vitb200_clip.h, the exports of libvitb200.so and the CLIP_SIGNATURES ctypes table
agree in both directions and stay apart from the other headers and tables; unknown activation codes and widths
vt_layernorm_stats does not take are refused before anything is launched; a numpy restatement of the bf16 quick-GELU
epilogue (csrc/common.cuh: quick_gelu_bf16_x2) is within one bf16 ulp for every finite bf16 input; the loader against
random-init HF ``CLIPVisionModelWithProjection`` / ``CLIPModel``; the state-dict keys and the host-side refusals (no
compute calls: there is no GPU here)."""
import ctypes
import os
import re

import numpy as np
import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
HEADER = os.path.join(ROOT, "include", "vitb200_clip.h")
COMMON = os.path.join(ROOT, "vit.triton_b200", "csrc", "common.cuh")
OTHER_HEADERS = [os.path.join(ROOT, "include", h) for h in
                 ("vitb200.h", "vitb200_resolution.h", "vitb200_ragged.h", "vitb200_mask.h", "vitb200_attn.h",
                  "vitb200_preprocess.h", "vitb200_tokens.h")]
_CTYPE = {"int32_t": ctypes.c_int32, "int64_t": ctypes.c_int64, "float": ctypes.c_float}
NAMES = {"vt_layernorm_stats"}
VT_ERR_ARG, VT_ERR_UNSUPPORTED = -1, -4


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


# ---------------------------------------------------------------------------------------------------- ABI
def test_clip_header_declares_expected_entry_points_and_activation_codes():
    text = open(HEADER).read()
    assert set(_declarations(HEADER)) == NAMES
    assert '#include "vitb200.h"' in text
    codes = dict(re.findall(r"#define (VT_ACT_\w+) (\d+)", text))
    assert codes == {"VT_ACT_NONE": "0", "VT_ACT_GELU": "1", "VT_ACT_TANH": "2", "VT_ACT_QUICK_GELU": "3"}
    mod = _lib()
    for name, value in codes.items():
        assert getattr(mod, name) == int(value), name
    from vit.kernels import bgemm as bg
    assert (bg.ACT_NONE, bg.ACT_GELU, bg.ACT_TANH, bg.ACT_QUICK_GELU) == (0, 1, 2, 3)
    assert bg._ACT["quick_gelu"] == 3 and bg._ACT["gelu"] == 1


def test_clip_entry_points_are_not_in_the_other_headers_or_tables():
    for path in OTHER_HEADERS:
        assert not NAMES & set(_declarations(path)), path
    mod = _lib()
    for table in (mod.SIGNATURES, mod.RESOLUTION_SIGNATURES, mod.RAGGED_SIGNATURES, mod.MASK_SIGNATURES,
                  mod.ATTN_SIGNATURES, mod.PREPROCESS_SIGNATURES, mod.TOKENS_SIGNATURES):
        assert not NAMES & set(table)


def test_library_exports_every_clip_symbol_and_ctypes_match():
    mod = _lib()
    lib = mod.load()
    decls = _declarations(HEADER)
    assert set(mod.CLIP_SIGNATURES) == set(decls)
    for name, argtypes in mod.CLIP_SIGNATURES.items():
        fn = getattr(lib, name)
        assert fn.argtypes == argtypes and fn.restype == ctypes.c_int, f"{name}: not registered by load()"
        args = decls[name]
        assert len(args) == len(argtypes), f"{name}: header has {len(args)} args, ctypes {len(argtypes)}"
        for a, ct in zip(args, argtypes):
            if "*" in a:
                assert ct == ctypes.c_void_p, f"{name}: {a}"
            else:
                assert _CTYPE[a.split()[0]] == ct, f"{name}: {a} vs {ct}"


_P = 4096    # stands for a device pointer: every call below must return before reading anything


@pytest.mark.parametrize("act", [2, 4, -1, 1 << 20])
def test_unknown_activation_codes_are_refused_before_any_launch(act):
    mod = _lib()
    lib = mod.load()
    s4 = mod.i64x4(0, 0, 768, 1)
    for out_dtype in (mod.VT_BF16, mod.VT_F32):
        assert lib.vt_gemm_bf16(_P, 768, _P, 768, _P, 3072, out_dtype, _P, None, 0, 256, 3072, 768, act, None) \
            == VT_ERR_ARG
    assert lib.vt_gemm_bf16_ln(_P, 768, _P, 768, _P, 3072, _P, None, 0, 256, 3072, 768, act, _P, None, 768, 1e-5, None,
                               None) == VT_ERR_ARG
    for out_dtype in (mod.VT_BF16, mod.VT_E4M3):
        assert lib.vt_gemm_fp8(_P, 768, _P, 768, _P, 3072, out_dtype, _P, _P, None, 0, 256, 3072, 768, act, 1.0,
                               None) == VT_ERR_ARG
    assert lib.vt_gemm_strided(_P, _P, _P, None, 256, 64, 768, 1, 1, s4, s4, s4, 1.0, act, mod.VT_F32, None) == VT_ERR_ARG
    if act != 2:                                   # tanh is a vt_bgemm activation
        s3 = mod.i64x3(0, 0, 768)
        assert lib.vt_bgemm(_P, _P, _P, None, None, 256, 64, 768, 1, 1, s3, s3, mod.i64x3(0, 0, 64), 0, 1.0, act,
                            mod.VT_BF16, None) == VT_ERR_ARG


@pytest.mark.parametrize("dim,status", [(100, VT_ERR_ARG), (200, VT_ERR_ARG), (768 + 64, VT_ERR_ARG),
                                        (1408, VT_ERR_UNSUPPORTED), (0, VT_ERR_ARG)])
def test_layernorm_stats_refuses_widths_before_any_launch(dim, status):
    lib = _lib().load()
    assert lib.vt_layernorm_stats(_P, _P, _P, _P, _P, 10, dim, max(dim, 8), max(dim, 8), 1e-5, None) == status
    assert lib.vt_layernorm_stats(None, _P, _P, _P, _P, 10, 768, 768, 768, 1e-5, None) == VT_ERR_ARG
    assert lib.vt_layernorm_stats(_P, _P, _P, _P, None, 10, 768, 768, 768, 1e-5, None) == VT_ERR_ARG


# ---------------------------------------------------------------------------------------------------- bf16 quick GELU
def _epilogue_constants():
    """The fp32 constants of quick_gelu_bf16_x2 in csrc/common.cuh, in source order: the exponent scale, then the
    polynomial coefficients from the highest degree down."""
    text = open(COMMON).read()
    body = text[text.index("quick_gelu_bf16_x2(float2 x) {"):]
    body = body[:body.index("\n}\n")]
    return [np.float32(v) for v in re.findall(r"make_float2\((-?[0-9.]+)f, \1f\)", body)]


def _f32(v):
    return np.asarray(v, np.float64).astype(np.float32)


def _fma(a, b, c):
    # the product of two fp32 values is exact in fp64; one rounding of the sum to fp32
    return _f32(a.astype(np.float64) * b.astype(np.float64) + c.astype(np.float64))


def _ex2_approx_ftz(t):
    y = _f32(np.exp2(t.astype(np.float64)))
    return np.where(np.abs(y) < 2.0 ** -126, np.float32(0), y).astype(np.float32)


def _quick_gelu_bf16_restated(x):
    """quick_gelu_bf16_x2 in fp32 numpy, operation by operation."""
    arg, *coef = _epilogue_constants()
    a = np.abs(x)
    e2 = _ex2_approx_ftz(_f32(a * arg))
    e = _f32(e2 * e2)
    r = _fma(e, np.full_like(e, coef[0]), np.full_like(e, coef[1]))
    for c in coef[2:]:
        r = _fma(e, r, np.full_like(e, c))
    return _fma(_f32(a * e2), _f32(e2 * r), np.maximum(x, np.float32(0)))


def _rn_bf16(v):
    av = np.abs(v)
    ex = np.maximum(np.floor(np.log2(np.where(av > 0, av, 1.0))), -126)
    ulp = np.exp2(ex - 7)
    return np.round(v / ulp) * ulp


def _ordinal(v):
    b = _f32(v).view(np.int32) >> 16
    return np.where(b < 0, -(b & 0x7FFF), b).astype(np.int64)


def test_quick_gelu_bf16_restatement_within_one_ulp_for_every_bf16_input():
    """Constants read from the kernel source: -1.702 log2(e) / 2 and five polynomial coefficients."""
    consts = _epilogue_constants()
    assert len(consts) == 6 and abs(consts[0] + 1.702 * np.log2(np.e) / 2) < 1e-7
    x = (np.arange(1 << 16, dtype=np.uint32) << 16).view(np.float32)
    x = x[np.isfinite(x)]
    x64 = x.astype(np.float64)
    with np.errstate(over="ignore"):
        want = _rn_bf16(x64 / (1.0 + np.exp(-1.702 * x64)))
        got = _rn_bf16(_quick_gelu_bf16_restated(x).astype(np.float64))
    d = np.abs(_ordinal(got) - _ordinal(want))
    assert d.max() <= 1, f"{d.max()} ulp at x = {x[np.argmax(d)]}"
    # the polynomial alone: 1 / (1 + e) on [0, 1] to 3.0e-4 relative
    e = np.linspace(0, 1, 10001).astype(np.float32)
    r = np.full_like(e, consts[1])
    for c in consts[2:]:
        r = _fma(e, r, np.full_like(e, c))
    assert np.abs(-r.astype(np.float64) * (1 + e.astype(np.float64)) - 1).max() <= 3.0e-4


# ---------------------------------------------------------------------------------------------------- model and loader
def _tiny_cfg(**kw):
    from transformers import CLIPVisionConfig
    from vit import configs
    return CLIPVisionConfig(**{**configs.CLIP_ARCHS["tiny-clip-b16"], **kw}, layer_norm_eps=1e-5)


def _randomize(model, seed=0):
    g = torch.Generator().manual_seed(seed + 1)
    with torch.no_grad():
        for name, p in model.named_parameters():
            if name.endswith(".bias"):
                p.copy_(torch.randn(p.shape, generator=g) * 0.02)
            elif any(s in name for s in ("layer_norm", "layrnorm", "layernorm")) and name.endswith(".weight"):
                p.copy_(1.0 + torch.randn(p.shape, generator=g) * 0.02)
    return model


def _ours(**kw):
    from vit import configs
    from vit.vit import VIT
    return VIT(**{**configs.clip_kwargs("tiny-clip-b16"), **kw})


def _expected(hf_vision_sd, proj, model):
    """Our state dict restated from the HF vision tower's (``vision_model.`` stripped) one key at a time."""
    want = {}
    D = model.hidden_dim
    dh = D // model.num_heads
    s = hf_vision_sd
    want["embeddings.cls_token"] = s["embeddings.class_embedding"].reshape(1, 1, D)
    want["embeddings.position_embeddings"] = s["embeddings.position_embedding.weight"][None]
    want["embeddings.projection.weight"] = s["embeddings.patch_embedding.weight"]
    want["embeddings.projection.bias"] = torch.zeros(D)
    for ours, hf in (("pre_layernorm", "pre_layrnorm"), ("layernorm", "post_layernorm")):
        for kind in ("weight", "bias"):
            want[f"{ours}.{kind}"] = s[f"{hf}.{kind}"]
    for i in range(model.num_layers):
        p, q = f"encoder.layer.{i}.", f"encoder.layers.{i}."
        for proj_name, ours in (("q", "query"), ("k", "key"), ("v", "value")):
            w, b = s[f"{q}self_attn.{proj_name}_proj.weight"], s[f"{q}self_attn.{proj_name}_proj.bias"]
            for h in range(model.num_heads):
                want[f"{p}attention.attention.{h}.{ours}.weight"] = w[h * dh:(h + 1) * dh].t()
                want[f"{p}attention.attention.{h}.{ours}.bias"] = b[h * dh:(h + 1) * dh]
        for ours, hf in (("attention.output", "self_attn.out_proj"), ("intermediate", "mlp.fc1"), ("output", "mlp.fc2")):
            want[f"{p}{ours}.weight"] = s[f"{q}{hf}.weight"].t()
            want[f"{p}{ours}.bias"] = s[f"{q}{hf}.bias"]
        for ours, hf in (("layernorm_before", "layer_norm1"), ("layernorm_after", "layer_norm2")):
            for kind in ("weight", "bias"):
                want[f"{p}{ours}.{kind}"] = s[f"{q}{hf}.{kind}"]
    if model.visual_projection is not None:
        want["visual_projection.weight"] = proj.t()
    return want


@pytest.mark.parametrize("kind", ["with_projection", "clip_model"])
def test_loader_maps_every_vision_key(kind):
    from transformers import CLIPConfig, CLIPModel, CLIPVisionModelWithProjection
    from vit.utils import transfer_pretrained_weights
    torch.manual_seed(0)
    vcfg = _tiny_cfg()
    if kind == "with_projection":
        hf = _randomize(CLIPVisionModelWithProjection(vcfg))
    else:
        hf = _randomize(CLIPModel(CLIPConfig(vision_config=vcfg.to_dict(), projection_dim=vcfg.projection_dim,
                                             text_config=dict(hidden_size=32, intermediate_size=64, num_hidden_layers=1,
                                                              num_attention_heads=2))))
    sd = hf.state_dict()
    vision = {k[len("vision_model."):]: v for k, v in sd.items() if k.startswith("vision_model.")}
    model = _ours()
    transfer_pretrained_weights(hf, model, verbose=False)
    got = model.state_dict()
    want = _expected(vision, sd["visual_projection.weight"], model)
    assert set(got) == set(want)
    for k in got:
        assert torch.equal(got[k], want[k]), k
    untouched = [k for k, v in got.items() if torch.all(v == 0) and k != "embeddings.projection.bias"]
    assert not untouched, untouched
    # a projection in the checkpoint is ignored by a model built without one
    plain = _ours(projection_dim=None)
    transfer_pretrained_weights(hf, plain, verbose=False)
    assert "visual_projection.weight" not in plain.state_dict()
    assert torch.equal(plain.state_dict()["layernorm.weight"], want["layernorm.weight"])


def _unchanged(model, fn):
    before = {k: v.clone() for k, v in model.state_dict().items()}
    with pytest.raises(AssertionError) as exc:
        fn()
    after = model.state_dict()
    assert all(torch.equal(before[k], after[k]) for k in before), "a tensor was copied before the refusal"
    return str(exc.value)


def test_loader_refusals_name_the_argument():
    from transformers import CLIPVisionModel, CLIPVisionModelWithProjection, ViTConfig, ViTModel
    from oracle import hf_oracle
    from vit.utils import transfer_pretrained_weights
    from vit.vit import VIT
    torch.manual_seed(0)
    clip_hf = CLIPVisionModelWithProjection(_tiny_cfg())
    vit = VIT(**hf_oracle.vit_kwargs("tiny-b"))
    assert "clip=True" in _unchanged(vit, lambda: transfer_pretrained_weights(clip_hf, vit, verbose=False))
    vit_hf = ViTModel(ViTConfig(**hf_oracle.ARCHS["tiny-b"]), add_pooling_layer=False)
    clip = _ours()
    assert "clip=True" in _unchanged(clip, lambda: transfer_pretrained_weights(vit_hf, clip, verbose=False))
    gelu_hf = CLIPVisionModelWithProjection(_tiny_cfg(hidden_act="gelu"))
    assert "hidden_act" in _unchanged(clip, lambda: transfer_pretrained_weights(gelu_hf, clip, verbose=False))
    eps = _ours(layer_norm_eps=1e-6)
    assert "layer_norm_eps" in _unchanged(eps, lambda: transfer_pretrained_weights(clip_hf, eps, verbose=False))
    no_proj = CLIPVisionModel(_tiny_cfg())
    assert "projection_dim" in _unchanged(clip, lambda: transfer_pretrained_weights(no_proj, clip, verbose=False))
    transfer_pretrained_weights(no_proj, _ours(projection_dim=None), verbose=False)


def test_state_dict_keys():
    from oracle import hf_oracle
    from vit.vit import VIT
    base = set(VIT(**hf_oracle.vit_kwargs("tiny-b")).state_dict())
    same = set(VIT(**hf_oracle.vit_kwargs("tiny-b"), hidden_act="quick_gelu", layer_norm_eps=1e-6).state_dict())
    assert same == base
    clip = set(VIT(**hf_oracle.vit_kwargs("tiny-b"), clip=True).state_dict())
    assert clip == base | {"pre_layernorm.weight", "pre_layernorm.bias"}
    proj = VIT(**hf_oracle.vit_kwargs("tiny-b"), clip=True, projection_dim=48)
    assert set(proj.state_dict()) == clip | {"visual_projection.weight"}
    assert tuple(proj.visual_projection.weight.shape) == (128, 48)
    m = VIT(**hf_oracle.vit_kwargs("tiny-b"), hidden_act="quick_gelu", layer_norm_eps=1e-6)
    assert all(ln.eps == 1e-6 for ln in [m.layernorm] + [b.layernorm_before for b in m.encoder.layer])
    assert all(b.intermediate.activation == "quick_gelu" and b.act == 3 for b in m.encoder.layer)


@pytest.mark.parametrize("flag", [dict(use_mask_token=True), dict(add_decoder=True), dict(distillation_token=True),
                                  dict(add_pooling_layer=True), dict(num_labels=10)])
def test_clip_refuses_heads_hf_does_not_have(flag):
    with pytest.raises(AssertionError, match=next(iter(flag))):
        _ours(**flag)


def test_constructor_and_head_refusals():
    from oracle import hf_oracle
    from vit.parallel import DataParallelVIT
    from vit.vit import VIT
    with pytest.raises(AssertionError, match="hidden_act"):
        VIT(**hf_oracle.vit_kwargs("tiny-b"), hidden_act="relu")
    with pytest.raises(AssertionError, match="clip=True"):
        VIT(**hf_oracle.vit_kwargs("tiny-b"), projection_dim=64)
    clip = _ours()
    x = torch.zeros((1, 3, 64, 64))
    for method in (clip.logits, clip.distillation_logits, clip.masked_image_modeling):
        with pytest.raises(AssertionError):
            method(x)
    with pytest.raises(AssertionError, match="projection"):
        _ours(projection_dim=None).image_embeds(x)
    with pytest.raises(AssertionError, match="output_hidden_states"):
        clip.image_embeds(x, output_hidden_states=True)
    assert DataParallelVIT(clip, output="image_embeds")._out_dim() == 64
    with pytest.raises(AssertionError):
        DataParallelVIT(clip, output="embeds")


def test_clip_configs():
    from vit import configs
    for arch, (S, P, D) in {"clip-b32-224": (224, 32, 768), "clip-b16-224": (224, 16, 768),
                            "clip-l14-224": (224, 14, 1024), "clip-l14-336": (336, 14, 1024)}.items():
        kw = configs.clip_kwargs(arch)
        assert (kw["height"], kw["patch_size"], kw["hidden_dim"]) == (S, P, D)
        assert kw["clip"] and kw["hidden_act"] == "quick_gelu" and kw["layer_norm_eps"] == 1e-5
    assert not set(configs.CLIP_ARCHS) & set(configs.ARCHS)
