"""CPU: the attention-probabilities entry point — include/vitb200_attn.h, the exports of libvitb200.so and the
ATTN_SIGNATURES ctypes table agree in both directions and stay apart from the other headers and tables; the host-side
refusals of ``output_hidden_states`` / ``output_attentions`` (no compute calls: there is no GPU here)."""
import ctypes
import math
import os
import re

import numpy as np
import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
HEADER = os.path.join(ROOT, "include", "vitb200_attn.h")
OTHER_HEADERS = [os.path.join(ROOT, "include", h)
                 for h in ("vitb200.h", "vitb200_resolution.h", "vitb200_ragged.h", "vitb200_mask.h")]

_CTYPE = {"int32_t": ctypes.c_int32, "int64_t": ctypes.c_int64, "float": ctypes.c_float}
NAMES = {"vt_attn_probs"}
VT_ERR_ARG, VT_ERR_ALIGN = -1, -3      # include/vitb200.h


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


@pytest.mark.parametrize("scale", [-0.125, 0.0, -0.0, float("nan"), float("inf"), float("-inf")])
@pytest.mark.parametrize("N,dh", [(197, 64), (577, 64), (197, 80)])
def test_flash_attn_refuses_bad_scales_without_a_launch(N, dh, scale):
    """Both attention kernels take the row maximum of the raw scores and scale it afterwards, which is the maximum of
    the scaled logits only for scale > 0: any other scale is refused (before any driver call; the pointers are fake),
    and flash_attention takes the composed path, which is exact for every scale."""
    mod = _lib()
    lib = mod.load()
    fake = 1 << 20
    D = 2 * dh
    assert lib.vt_flash_attn(fake, fake, fake, fake, 1, 2, N, dh, 3 * D, 3 * D * N, D, D * N, scale,
                             None) == mod.VT_ERR_UNSUPPORTED


def test_flash_attn_rejects_bad_arguments_without_a_launch():
    mod = _lib()
    lib = mod.load()
    fake = 1 << 20
    args = [fake, fake, fake, fake, 1, 2, 197, 64, 384, 384 * 197, 128, 128 * 197, 0.125, None]

    def call(**kw):
        a = list(args)
        for i, v in kw.items():
            a[int(i[1:])] = v
        return lib.vt_flash_attn(*a)

    for i in range(4):
        assert call(**{f"a{i}": None}) == VT_ERR_ARG, f"null pointer {i}"
    assert call(a4=0) == VT_ERR_ARG and call(a5=0) == VT_ERR_ARG and call(a6=0) == VT_ERR_ARG
    for dh in (32, 48, 96, 128):
        assert call(a7=dh) == mod.VT_ERR_UNSUPPORTED, f"head dim {dh}"
    for N in (197, 577):
        for i in range(4):
            assert call(a6=N, **{f"a{i}": fake + 8}) == VT_ERR_ALIGN, f"N={N}: pointer {i} + 8 bytes"
        for i in range(8, 12):
            assert call(a6=N, **{f"a{i}": args[i] + 4}) == VT_ERR_ALIGN, f"N={N}: stride {i} + 4"


# ---------------------------------------------------------------------------------------------------- ex2_poly_x2
ATTN5 = os.path.join(ROOT, "vit.triton_b200", "csrc", "attn5_sm100.cu")
POLY_REL = 7.52e-5          # max relative error of the polynomial against 2^f on [-0.5, 0.5] (measured: 7.5146e-5)


def _attn5_source():
    return open(ATTN5).read()


def _poly_constants():
    """The fp32 constants of ex2_poly_x2 in source order: the rounding magic, its negation, -1, then the polynomial
    coefficients from the highest degree down."""
    body = _attn5_source()
    body = body[body.index("ex2_poly_x2(float2 x) {"):]
    body = body[:body.index("\n}\n")]
    return [np.float32(v) for v in re.findall(r"make_float2\((-?[0-9.]+)f, \1f\)", body)]


def _f32(v):
    return np.asarray(v, np.float64).astype(np.float32)


def _fma(a, b, c):
    # the product of two fp32 values is exact in fp64; one rounding of the sum to fp32
    return _f32(a.astype(np.float64) * np.float64(b) + np.asarray(c, np.float64))


def _poly(f, coef):
    p = _fma(f, coef[0], coef[1])
    for c in coef[2:]:
        p = _fma(p, f, c)
    return p


def _ex2_poly_restated(x):
    """ex2_poly_x2 in fp32 numpy, operation by operation: (result, n, f, poly(f))."""
    magic, neg_magic, minus_one, *coef = _poly_constants()
    x = np.asarray(x, np.float32)
    xf = _f32(x.astype(np.float64) + np.float64(magic))
    n = _f32(xf.astype(np.float64) + np.float64(neg_magic))
    f = _fma(n, minus_one, x)
    p = _poly(f, coef)
    r = (p.view(np.uint32) + (xf.view(np.uint32) << np.uint32(23))).view(np.float32)
    return r, n, f, p


def test_ex2_poly_constants():
    magic, neg_magic, minus_one, *coef = _poly_constants()
    assert magic == 1.5 * 2.0 ** 23 and neg_magic == -magic and minus_one == -1.0 and len(coef) == 4


def test_ex2_poly_relative_error_on_the_reduced_range():
    """2^f for f in [-0.5, 0.5]: every fp32 of the top binades (|f| in [0.25, 0.5], both ends and so both ties
    included) and a dense grid of the rest."""
    coef = _poly_constants()[3:]
    top = np.arange(np.float32(0.25).view(np.uint32), np.float32(0.5).view(np.uint32) + 1,
                    dtype=np.uint32).view(np.float32)
    f = np.concatenate([top, -top, np.linspace(-0.5, 0.5, 2_000_001).astype(np.float32)])
    rel = np.abs(_poly(f, coef).astype(np.float64) / np.exp2(f.astype(np.float64)) - 1)
    i = int(rel.argmax())
    assert rel[i] <= POLY_REL, f"relative error {rel[i]:.4e} at f = {f[i]!r}"
    assert rel[i] > 0.99 * POLY_REL, "the gate is far above the polynomial's error: tighten POLY_REL"
    assert "max relative error 7.52e-5" in _attn5_source(), "the comment of ex2_poly_x2 states another error"


def _valid(x):
    """Where the rounding and the exponent-field add of ex2_poly_x2 give exactly ldexp(poly(f), rint_even(x))."""
    r, n, f, p = _ex2_poly_restated(x)
    x64 = np.asarray(x, np.float64)
    n_even = np.round(x64)                          # numpy rounds half to even, like the fp32 add of the magic
    with np.errstate(invalid="ignore", over="ignore"):
        return (n.astype(np.float64) == n_even) & (f.astype(np.float64) == x64 - n_even) & \
            (r.astype(np.float64) == np.ldexp(p.astype(np.float64), n_even.astype(np.int64)))


def _admitted_argument_bound():
    """The largest |exp2 argument| the bounded path admits.  An item takes it when max|q|^2 * max|k|^2 * c^2 * M <= B^2
    (c = scale * log2 e, B = kLogitBound5, M = kBoundMargin5), with the squared norms accumulated by bf16 FMAs: eight
    chains of eight terms, each term one rounding of relative error at most 2^-8, so a computed sum of squares is at
    least (1 - 2^-8)^8 of the true one (the fp32 sum of the eight chains adds 8 * 2^-24).  By Cauchy-Schwarz
    |c q.k| <= c |q| |k| <= B / (sqrt(M) * low), low = (1 - 2^-8)^8 - 8 * 2^-24, and with m = 0 that is the
    argument (the fp32 score adds dh * 2^-23 relative, folded into the factor 1.001)."""
    src = _attn5_source()
    bound = float(re.search(r"constexpr float kLogitBound5 = ([0-9.]+)f;", src).group(1))
    margin = float(re.search(r"constexpr float kBoundMargin5 = ([0-9.]+)f;", src).group(1))
    low = (1 - 2.0 ** -8) ** 8 - 8 * 2.0 ** -24
    return 1.001 * bound / (math.sqrt(margin) * low)


def test_ex2_poly_rounding_and_exponent_add_are_exact():
    """On a fine grid and at every half-integer (ties go to even, as the fp32 add of 1.5 * 2^23 rounds): the result
    is exactly 2^rint(x) times the polynomial of the exact remainder, from x = -125.5 to 127.5."""
    x = np.concatenate([np.arange(-125.5 * 256, 127.5 * 256 + 1) / 256, np.arange(-251, 256) / 2,
                        [-125.75, 127.75]]).astype(np.float32)
    ok = _valid(x)
    assert ok.all(), f"not ldexp(poly(f), n) at x = {x[~ok][:8]}"


def test_ex2_poly_exponent_add_covers_the_bounded_path():
    """The exponent-field add is valid on (-126, 128) and only there: at x = -126 (n = -126 with poly < 1) the
    exponent field becomes 0, at x > 128 (n = 128, poly >= 1) it reaches 255.  The bounded path's arguments stay
    well inside: |x| <= kLogitBound5 / sqrt(kBoundMargin5) / (bf16 sums of squares at most 3.1 % low)."""
    assert not _valid(np.float32([-126.0, -126.25, -127.0, 128.25, 129.0])).any()
    assert _valid(np.float32([-125.984375, 128.0])).all()
    lim = _admitted_argument_bound()
    assert lim <= 0.75 * 126, f"the bounded path admits exp2 arguments up to {lim:.1f}: the exponent add is valid to 126"
    x = np.linspace(-lim, lim, 200_001).astype(np.float32)
    assert _valid(x).all()


def test_ex2_poly_bf16_rounding_equals_exp2():
    """bf16(ex2_poly_x2(x)) == bf16(2^x) wherever 2^x is farther than POLY_REL (relative) from a bf16 rounding
    midpoint; there the polynomial may round to the other side."""
    lim = _admitted_argument_bound()
    x = np.linspace(-lim, lim, 1_000_001).astype(np.float32)
    r = _ex2_poly_restated(x)[0].astype(np.float64)
    want = np.exp2(x.astype(np.float64))
    e = np.floor(np.log2(want))
    ulp = np.exp2(e - 7)
    mid = (np.floor(want / ulp) + 0.5) * ulp
    near = np.abs(want - mid) <= 1.01 * POLY_REL * want
    bad = (np.round(r / ulp) != np.round(want / ulp)) & ~near
    assert not bad.any(), f"bf16 rounding differs at x = {x[bad][:8]}"
    assert near.mean() < 0.05


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
