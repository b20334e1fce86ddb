"""GPU: CLIP image encoders — quick GELU in every GEMM epilogue, ``vt_layernorm_stats``, and ``VIT(clip=True)``.

Kernels: every finite bf16 input with |x| <= 16 through an identity-like GEMM (A holds x in column 0, every row of B is
e0, so out[m, n] = act(x_m)) on ``vt_gemm_bf16`` (both output dtypes), ``vt_bgemm`` and ``vt_gemm_strided``: bf16 outputs
within one bf16 ulp of the correctly rounded fp64 x * sigmoid(1.702 x), fp32 outputs within 2e-6 relative + 1e-7
absolute; ``vt_gemm_fp8`` (bf16 and e4m3 outputs) against a restatement of its quantisation; ``vt_gemm_bf16_ln`` (both
fold forms) against fp64.  Many tiles per CTA and guard rows around every output.  ``vt_layernorm_stats`` gives
``vt_layernorm``'s bits and per-group statistics matching fp64.  Model: parity with HF ``CLIPVisionModelWithProjection``
(fp32 on the CPU, eager attention) at the gates of tests/test_gpu_model.py (bf16 cosine >= 0.999 and max-abs <= 0.15,
fp32 <= 1e-3, FP8 cosine >= 0.995 and max-abs <= 0.5).  Properties: ragged lists, ``do_resize`` and CUDA-graph replay
give the plain call's bits; with the fold on a CLIP forward makes as many launches as the ViT forward of its shape."""
import functools

import numpy as np
import pytest
import torch
import torch.nn.functional as F

pytestmark = pytest.mark.gpu

DEV = "cuda:0"
GUARD = 3
CLIP_MEAN = (0.48145466, 0.4578275, 0.40821073)
CLIP_STD = (0.26862954, 0.26130258, 0.27577711)


# ---------------------------------------------------------------------------------------------------- references
def _bf16_inputs(limit=16.0):
    """Every finite bf16 value with |x| <= limit, as an fp32 CPU tensor."""
    x = torch.from_numpy((np.arange(1 << 16, dtype=np.uint32) << 16).view(np.float32).copy())
    return x[torch.isfinite(x) & (x.abs() <= limit)]


def _qgelu64(v):
    v = v.double()
    return v * torch.sigmoid(1.702 * v)


def _rn_bf16(v):
    """fp64 -> the correctly rounded bf16 value (as fp64), subnormals included."""
    v = v.double()
    ex = torch.floor(torch.log2(torch.where(v != 0, v.abs(), torch.ones_like(v)))).clamp_min(-126)
    ulp = torch.exp2(ex - 7)
    return torch.round(v / ulp) * ulp


def _ordinal(b16):
    """bf16 tensor -> integers in value order (adjacent bf16 values differ by one)."""
    b = b16.view(torch.int16).long()
    return torch.where(b < 0, -(b & 0x7FFF), b)


def _check_bf16(got, x, what):
    """Every column of got (M, N) bf16 within one ulp of the correctly rounded act(x_m)."""
    want = _rn_bf16(_qgelu64(x.double())).to(torch.bfloat16)         # exact: already a bf16 value
    d = (_ordinal(got.cpu()) - _ordinal(want)[:, None]).abs()
    worst = d.max().item()
    assert worst <= 1, f"{what}: {worst} ulp at x = {x[d.max(dim=1).values.argmax()].item()}"


def _check_f32(got, x, what):
    want = _qgelu64(x.double())[:, None]
    err = (got.cpu().double() - want).abs() - (2e-6 * want.abs() + 1e-7)
    assert err.max().item() <= 0, f"{what}: x = {x[err.max(dim=1).values.argmax()].item()}"


def _guarded(shape, dtype):
    rows = shape[0]
    buf = torch.full((rows + 2 * GUARD,) + tuple(shape[1:]), float("nan"), device=DEV, dtype=dtype)
    return buf, buf[GUARD:GUARD + rows]


def _guards_intact(buf):
    return bool(buf[:GUARD].isnan().all() and buf[-GUARD:].isnan().all())


# ---------------------------------------------------------------------------------------------------- quick GELU
K_ID = 128      # identity GEMM depth: x in column 0, zeros elsewhere
N_ID = 512


def _identity(x, dtype=torch.bfloat16, repeat=2):
    """(x repeated, A [M, K_ID], Bt [N_ID, K_ID]) of the identity-like GEMM out[m, n] = x_m."""
    xs = x.repeat(repeat)
    A = torch.zeros((xs.numel(), K_ID), dtype=dtype)
    A[:, 0] = xs
    Bt = torch.zeros((N_ID, K_ID), dtype=dtype)
    Bt[:, 0] = 1
    return xs, A.to(DEV), Bt.to(DEV)


@pytest.mark.parametrize("out_dtype", [torch.bfloat16, torch.float32])
def test_quick_gelu_gemm_bf16_every_bf16_input(out_dtype):
    """vt_gemm_bf16 with gelu = VT_ACT_QUICK_GELU: the 2-CTA kernel (bf16 out) and the 1-CTA kernel (fp32 out)."""
    from vit.kernels import _lib
    xs, A, Bt = _identity(_bf16_inputs())
    M = xs.numel()
    bias = torch.zeros(N_ID, device=DEV)
    buf, out = _guarded((M, N_ID), out_dtype)
    _lib.call("vt_gemm_bf16", A.data_ptr(), K_ID, Bt.data_ptr(), K_ID, out.data_ptr(), N_ID, _lib.dtype_code(out),
              bias.data_ptr(), None, 0, M, N_ID, K_ID, _lib.VT_ACT_QUICK_GELU, _lib.stream_ptr(A))
    torch.cuda.synchronize()
    assert _guards_intact(buf)
    (_check_bf16 if out_dtype == torch.bfloat16 else _check_f32)(out, xs, f"vt_gemm_bf16 {out_dtype}")


@pytest.mark.parametrize("out_dtype", [torch.bfloat16, torch.float32])
def test_quick_gelu_bgemm_every_bf16_input(out_dtype):
    from vit.kernels import bgemm as bg
    xs, A, Bt = _identity(_bf16_inputs())
    M = xs.numel()
    buf, out = _guarded((M, N_ID), out_dtype)
    bg.bgemm(A.data_ptr(), Bt.data_ptr(), out, out.data_ptr(), M, N_ID, K_ID, 1, 1, (0, 0, K_ID), (0, 0, K_ID),
             (0, 0, N_ID), act=bg.ACT_QUICK_GELU)
    torch.cuda.synchronize()
    assert _guards_intact(buf)
    (_check_bf16 if out_dtype == torch.bfloat16 else _check_f32)(out, xs, f"vt_bgemm {out_dtype}")


@pytest.mark.parametrize("dtype", [torch.bfloat16, torch.float32])
def test_quick_gelu_gemm_strided_every_bf16_input(dtype):
    from vit.kernels import _lib
    xs, A, Bt = _identity(_bf16_inputs(), dtype, repeat=1)
    M, N = xs.numel(), 64
    Bt = Bt[:N].contiguous()
    buf, out = _guarded((M, N), dtype)
    _lib.call("vt_gemm_strided", A.data_ptr(), Bt.data_ptr(), out.data_ptr(), None, M, N, K_ID, 1, 1,
              _lib.i64x4(0, 0, K_ID, 1), _lib.i64x4(0, 0, 1, K_ID), _lib.i64x4(0, 0, N, 1), 1.0,
              _lib.VT_ACT_QUICK_GELU, _lib.dtype_code(A), _lib.stream_ptr(A))
    torch.cuda.synchronize()
    assert _guards_intact(buf)
    (_check_bf16 if dtype == torch.bfloat16 else _check_f32)(out, xs, f"vt_gemm_strided {dtype}")


def _e4m3_ordinal(b):
    b = b.long()
    return torch.where(b >= 128, -(b - 128), b)


@pytest.mark.parametrize("out8", [False, True])
def test_quick_gelu_gemm_fp8_against_its_quantisation(out8):
    """vt_gemm_fp8: out = act(fma(acc, colscale_n, bias_n)) with acc = a_m (every finite e4m3 byte in column 0 of A, e0
    rows in B): bf16 output within one ulp of the correctly rounded act, e4m3 output (x out_scale) within one e4m3 step
    of the correctly rounded act * out_scale."""
    from vit.kernels import _lib
    codes = torch.tensor([b for b in range(256) if b not in (0x7F, 0xFF)], dtype=torch.uint8)
    a = codes.view(torch.float8_e4m3fn).double()
    rep = 64
    M, N, K = codes.numel() * rep, 512, 128
    A8 = torch.zeros((M, K), dtype=torch.uint8)
    A8[:, 0] = codes.repeat(rep)
    B8 = torch.zeros((N, K), dtype=torch.uint8)
    B8[:, 0] = 0x38                                                  # 1.0 in e4m3
    g = torch.Generator().manual_seed(17)
    scale = torch.linspace(0.002, 0.04, N, dtype=torch.float32)
    bias = (torch.rand((N,), generator=g, dtype=torch.float64) * 4 - 2).float()
    out_scale = 8.0
    # the epilogue's fma in fp32: a * s is exact in fp64 (4 + 24 bits), one rounding to fp32 after the add
    pre = (a.repeat(rep)[:, None] * scale.double()[None, :] + bias.double()[None, :]).float().double()
    A8d, B8d, sd, bd = A8.to(DEV), B8.to(DEV), scale.to(DEV), bias.to(DEV)
    if out8:
        buf = torch.full((M + 2 * GUARD, N), 0x7F, dtype=torch.uint8, device=DEV)
        out = buf[GUARD:GUARD + M]
    else:
        buf, out = _guarded((M, N), torch.bfloat16)
    _lib.call("vt_gemm_fp8", A8d.data_ptr(), K, B8d.data_ptr(), K, out.data_ptr(), N,
              _lib.VT_E4M3 if out8 else _lib.VT_BF16, bd.data_ptr(), sd.data_ptr(), None, 0, M, N, K,
              _lib.VT_ACT_QUICK_GELU, out_scale, _lib.stream_ptr(A8d))
    torch.cuda.synchronize()
    if out8:
        assert (buf[:GUARD] == 0x7F).all() and (buf[-GUARD:] == 0x7F).all()
        want = (_qgelu64(pre) * out_scale).to(torch.float8_e4m3fn).view(torch.uint8)
        d = (_e4m3_ordinal(out.cpu()) - _e4m3_ordinal(want)).abs()
        assert d.max().item() <= 1, f"e4m3 output: {d.max().item()} steps"
    else:
        assert _guards_intact(buf)
        want = _rn_bf16(_qgelu64(pre)).to(torch.bfloat16)
        d = (_ordinal(out.cpu()) - _ordinal(want)).abs()
        assert d.max().item() <= 1, f"bf16 output: {d.max().item()} ulp"


def _group_stats(xf):
    M, K = xf.shape
    xc = xf.view(M, K // 128, 128).double()
    m2 = ((xc - xc.mean(-1, keepdim=True)) ** 2).sum(-1)
    return torch.stack([xc.sum(-1), m2], dim=2).float().contiguous()


def _rel_err(got, want):
    return ((got.float() - want.float()).norm() / want.float().norm().clamp_min(1e-12)).item()


@pytest.mark.parametrize("M,K,N", [(197 * 64, 768, 3072), (300, 128, 512), (129, 1280, 264)])
@pytest.mark.parametrize("zero_sum", [False, True])
def test_quick_gelu_gemm_layernorm_fold(M, K, N, zero_sum):
    """vt_gemm_bf16_ln with quick GELU == quick_gelu(dense(LayerNorm(x))) in fp64, at the tolerance of the GELU fold
    tests of tests/test_gpu_kernels.py."""
    from vit import packing
    from vit.kernels import _lib
    torch.manual_seed(M + K)
    x = (2.0 * torch.randn(1, M, K, device=DEV) + 0.7).bfloat16()
    ln = torch.nn.LayerNorm(K, eps=1e-5).to(DEV)
    with torch.no_grad():
        ln.weight.copy_(1 + 0.2 * torch.randn(K, device=DEV))
        ln.bias.copy_(0.2 * torch.randn(K, device=DEV))
    w_nk = (torch.randn(N, K, device=DEV) / K ** 0.5).bfloat16()
    bias = torch.randn(N, device=DEV)
    w_fold, b_fold, colsum = packing.fold_layernorm(w_nk, bias, ln, zero_sum=zero_sum)
    xf = x.float()[0]
    got = packing.linear_ln(x, w_fold, b_fold, colsum, _group_stats(xf), 1e-5, gelu=_lib.VT_ACT_QUICK_GELU)
    want = F.layer_norm(xf.double(), (K,), ln.weight.double(), ln.bias.double(), 1e-5) @ w_nk.double().t() + bias.double()
    want = _qgelu64(want)
    assert _rel_err(got[0], want) <= 2 ** -7, f"rel err {_rel_err(got[0], want)}"


# ---------------------------------------------------------------------------------------------------- vt_layernorm_stats
@pytest.mark.parametrize("dim", [128, 384, 768, 1024, 1280])
def test_layernorm_stats_equals_layernorm_and_fp64_statistics(dim):
    from vit.kernels import _lib
    rows = 1003
    g = torch.Generator().manual_seed(dim)
    x = torch.randn((rows, dim), generator=g) * torch.logspace(-1, 1, rows)[:, None]
    x += torch.linspace(-50, 50, rows)[:, None]
    x[5::7, 3] = 300.0
    in_stride, out_stride = dim + 64, dim + 128
    xin = torch.full((rows, in_stride), float("nan"), dtype=torch.bfloat16)
    xin[:, :dim] = x.bfloat16()
    xin = xin.to(DEV)
    gamma = (1 + 0.2 * torch.randn((dim,), generator=g)).to(DEV, torch.bfloat16)
    beta = (0.2 * torch.randn((dim,), generator=g)).to(DEV, torch.bfloat16)
    buf_a, out_a = _guarded((rows, out_stride), torch.bfloat16)
    buf_b, out_b = _guarded((rows, out_stride), torch.bfloat16)
    sbuf, stats = _guarded((rows, dim // 128, 2), torch.float32)
    eps = 1e-5
    _lib.call("vt_layernorm", xin.data_ptr(), gamma.data_ptr(), beta.data_ptr(), out_a.data_ptr(), rows, dim, in_stride,
              out_stride, eps, _lib.VT_BF16, _lib.VT_BF16, _lib.stream_ptr(xin))
    _lib.call("vt_layernorm_stats", xin.data_ptr(), gamma.data_ptr(), beta.data_ptr(), out_b.data_ptr(),
              stats.data_ptr(), rows, dim, in_stride, out_stride, eps, _lib.stream_ptr(xin))
    torch.cuda.synchronize()
    assert _guards_intact(buf_a) and _guards_intact(buf_b) and _guards_intact(sbuf)
    assert out_b[:, dim:].isnan().all(), "columns past dim written"
    assert torch.equal(out_a[:, :dim].view(torch.int16), out_b[:, :dim].view(torch.int16))
    want = _group_stats(out_b[:, :dim].float().cpu()).double()
    got = stats.cpu().double()
    scale = out_b[:, :dim].float().cpu().abs().view(rows, dim // 128, 128).sum(-1).double()
    assert ((got[..., 0] - want[..., 0]).abs() <= 1e-6 * scale + 1e-6).all()
    assert ((got[..., 1] - want[..., 1]).abs() <= 1e-5 * want[..., 1] + 1e-6).all()


# ---------------------------------------------------------------------------------------------------- models
def _randomize(model, seed):
    """HF zero / one-initialises biases and LayerNorm affines (pre_layrnorm included): re-randomise them."""
    g = torch.Generator().manual_seed(seed + 1)
    with torch.no_grad():
        for name, p in model.named_parameters():
            if name.endswith(".bias"):
                p.copy_(torch.randn(p.shape, generator=g) * 0.02)
            elif any(s in name for s in ("layer_norm", "layrnorm", "layernorm")) and name.endswith(".weight"):
                p.copy_(1.0 + torch.randn(p.shape, generator=g) * 0.02)
            elif name.endswith(("position_embedding.weight", "position_embeddings")):
                p.copy_(torch.randn(p.shape, generator=g) * 0.1)
    return model


@functools.lru_cache(maxsize=None)
def _hf(arch):
    from transformers import CLIPVisionConfig, CLIPVisionModelWithProjection
    from vit import configs
    torch.manual_seed(0)
    cfg = CLIPVisionConfig(**configs.CLIP_ARCHS[arch], layer_norm_eps=configs.CLIP_LAYER_NORM_EPS,
                           attn_implementation="eager")
    return _randomize(CLIPVisionModelWithProjection(cfg).eval(), 0)


@functools.lru_cache(maxsize=None)
def _ours(arch, dtype):
    from vit import configs
    from vit.utils import transfer_pretrained_weights
    from vit.vit import VIT
    model = VIT(**configs.clip_kwargs(arch))
    transfer_pretrained_weights(_hf(arch), model, verbose=False)
    return model.to(device=DEV, dtype=dtype).eval()


def _hf_out(arch, x, interpolate=False):
    hf = _hf(arch)
    out = hf(pixel_values=x, output_hidden_states=True, output_attentions=True, interpolate_pos_encoding=interpolate)
    pooler = hf.vision_model.post_layernorm(out.last_hidden_state[:, 0])
    return out, pooler


def _x(batch, h, w, seed=5):
    g = torch.Generator().manual_seed(seed)
    return torch.randn((batch, 3, h, w), generator=g)


def _check(got, want, gate, what):
    got, want = got.float().cpu(), want.float()
    assert got.shape == want.shape, f"{what}: {tuple(got.shape)} vs {tuple(want.shape)}"
    assert torch.isfinite(got).all(), what
    err = (got - want).abs().max().item()
    cos = F.cosine_similarity(got.flatten(), want.flatten(), dim=0).item()
    print(f"{what}: max-abs {err:.3e} cosine {cos:.6f}")
    if gate == "fp32":
        assert err <= 1e-3, f"{what}: max-abs {err:.3e}"
    elif gate == "fp8":
        assert cos >= 0.995 and err <= 0.5, f"{what}: cosine {cos:.6f} max-abs {err:.4f}"
    else:
        assert cos >= 0.999 and err <= 0.15, f"{what}: cosine {cos:.6f} max-abs {err:.4f}"


class _Mode:
    def __init__(self, mode):
        self.mode = mode

    def __enter__(self):
        from vit import vit as V
        if self.mode == "fold_ln_before":
            V.set_layernorm_folding(True, mlp=False)
        elif self.mode == "no_fold":
            V.set_layernorm_folding(False)
        elif self.mode == "fp8":
            V.set_fp8(True)
        elif self.mode == "unfused":
            V.set_fused(False)

    def __exit__(self, *exc):
        from vit import vit as V
        V.set_layernorm_folding(True)
        V.set_fp8(False)
        V.set_fused(True)


ARCHS = ["tiny-clip-b16", "tiny-clip-h14", "tiny-clip-b32"]     # P 16 / 14 / 32, dh 64 / 80 / 64, D 128 / 160 / 256
MODES = ["fold", "fold_ln_before", "no_fold", "fp8", "fp32", "unfused"]


def _gate(dtype, mode):
    return "fp32" if dtype == torch.float32 else ("fp8" if mode == "fp8" else "bf16")


@pytest.mark.parametrize("mode", MODES)
@pytest.mark.parametrize("arch", ARCHS)
@torch.no_grad()
def test_outputs_match_hf(arch, mode):
    """last_hidden_state, pooler_output and image_embeds in every execution mode."""
    dtype = torch.float32 if mode in ("fp32", "unfused") else torch.bfloat16
    model = _ours(arch, dtype)
    S = model.height
    x = _x(3, S, S)
    want, pooler = _hf_out(arch, x)
    gate = _gate(dtype, mode)
    xd = x.to(DEV, dtype)
    with _Mode(mode):
        _check(model(xd), want.last_hidden_state, gate, f"{arch} {mode} last_hidden_state")
        _check(model.pooler_output(xd), pooler, gate, f"{arch} {mode} pooler_output")
        _check(model.image_embeds(xd), want.image_embeds, gate, f"{arch} {mode} image_embeds")


@pytest.mark.parametrize("mode", ["fold", "fp8", "fp32"])
@pytest.mark.parametrize("arch", ARCHS)
@torch.no_grad()
def test_hidden_states_and_attentions_match_hf(arch, mode):
    """Element 0 is pre_layrnorm's output, the last one last_hidden_state (no final LayerNorm)."""
    dtype = torch.float32 if mode == "fp32" else torch.bfloat16
    model = _ours(arch, dtype)
    x = _x(2, model.height, model.width, seed=7)
    want, _ = _hf_out(arch, x)
    assert len(want.attentions) == model.num_layers, "HF returned no attention maps (SDPA attention?)"
    with _Mode(mode):
        got = model(x.to(DEV, dtype), output_hidden_states=True, output_attentions=True)
    gate = _gate(dtype, mode)
    assert len(got.hidden_states) == len(want.hidden_states) and len(got.attentions) == len(want.attentions)
    for i, (a, b) in enumerate(zip(got.hidden_states, want.hidden_states)):
        _check(a, b, gate, f"{arch} {mode} hidden_states[{i}]")
    for i, (a, b) in enumerate(zip(got.attentions, want.attentions)):
        _check(a, b, gate, f"{arch} {mode} attentions[{i}]")
    assert torch.equal(got.hidden_states[-1], got.last_hidden_state)


@pytest.mark.parametrize("hw", [(96, 96), (48, 80)])
@pytest.mark.parametrize("dtype", [torch.bfloat16, torch.float32])
@torch.no_grad()
def test_interpolate_pos_encoding_matches_hf(hw, dtype):
    arch = "tiny-clip-b16"
    model = _ours(arch, dtype)
    x = _x(2, *hw, seed=hw[1])
    want, pooler = _hf_out(arch, x, interpolate=True)
    xd = x.to(DEV, dtype)
    gate = _gate(dtype, "fold")
    _check(model(xd, interpolate_pos_encoding=True), want.last_hidden_state, gate, f"interpolate {hw}")
    _check(model.image_embeds(xd, interpolate_pos_encoding=True), want.image_embeds, gate, f"interpolate {hw} embeds")


@pytest.mark.parametrize("arch", ARCHS)
@torch.no_grad()
def test_uint8_with_clip_constants_matches_hf(arch):
    model = _ours(arch, torch.bfloat16)
    S = model.height
    g = torch.Generator().manual_seed(9)
    x8 = torch.randint(0, 256, (3, S, S, 3), generator=g, dtype=torch.uint8)
    mean, std = torch.tensor(CLIP_MEAN), torch.tensor(CLIP_STD)
    xf = ((x8.float() / 255.0 - mean) / std).permute(0, 3, 1, 2).contiguous()
    want, _ = _hf_out(arch, xf)
    got = model.forward_uint8(x8.to(DEV), image_mean=CLIP_MEAN, image_std=CLIP_STD)
    _check(got, want.last_hidden_state, "bf16", f"{arch} uint8")


@pytest.mark.parametrize("dtype", [torch.bfloat16, torch.float32])
@torch.no_grad()
def test_vit_with_quick_gelu_and_eps_matches_hf(dtype):
    """hidden_act and layer_norm_eps are generic: a ViT built with them matches HF ViTModel at those config values."""
    from transformers import ViTConfig, ViTModel
    from oracle import hf_oracle
    from vit.utils import transfer_pretrained_weights
    from vit.vit import VIT
    torch.manual_seed(0)
    cfg = ViTConfig(**hf_oracle.ARCHS["tiny-b"], hidden_act="quick_gelu", layer_norm_eps=1e-6,
                    attn_implementation="eager")
    hf = _randomize(ViTModel(cfg, add_pooling_layer=False).eval(), 0)
    model = VIT(**hf_oracle.vit_kwargs("tiny-b"), hidden_act="quick_gelu", layer_norm_eps=1e-6)
    transfer_pretrained_weights(hf, model, verbose=False)
    model = model.to(DEV, dtype).eval()
    x = _x(2, 64, 64, seed=3)
    _check(model(x.to(DEV, dtype)), hf(pixel_values=x).last_hidden_state, _gate(dtype, "fold"), f"ViT quick_gelu {dtype}")


# ---------------------------------------------------------------------------------------------------- identities
@pytest.mark.parametrize("u8", [False, True])
@torch.no_grad()
def test_ragged_list_equals_each_images_own_call(u8):
    model = _ours("tiny-clip-b16", torch.bfloat16)
    sizes = [(64, 64), (48, 96), (80, 37), (64, 64), (16, 32)]
    g = torch.Generator().manual_seed(2)
    if u8:
        imgs = [torch.randint(0, 256, (h, w, 3), generator=g, dtype=torch.uint8).to(DEV) for h, w in sizes]
    else:
        imgs = [torch.randn((3, h, w), generator=g).to(DEV, torch.bfloat16) for h, w in sizes]
    own = model.forward_uint8 if u8 else model.forward
    got = model.forward_ragged(imgs)
    embeds = model.image_embeds(imgs)
    for i, img in enumerate(imgs):
        assert torch.equal(got[i], own(img[None], interpolate_pos_encoding=True)[0]), f"image {i} {sizes[i]}"
        assert torch.equal(embeds[i], model.image_embeds(img[None], interpolate_pos_encoding=True)[0]), f"image {i}"


@torch.no_grad()
def test_do_resize_equals_resize_then_call():
    from vit.kernels.resize import resize_uint8
    model = _ours("tiny-clip-b16", torch.bfloat16)
    g = torch.Generator().manual_seed(4)
    x8 = torch.randint(0, 256, (2, 100, 77, 3), generator=g, dtype=torch.uint8).to(DEV)
    r = resize_uint8(x8, 64, 64, 3)
    assert torch.equal(model.forward_uint8(x8, CLIP_MEAN, CLIP_STD, do_resize=True, resample=3),
                       model.forward_uint8(r, CLIP_MEAN, CLIP_STD))
    assert torch.equal(model.image_embeds(x8, do_resize=True, resample=3), model.image_embeds(r))


@torch.no_grad()
def test_cuda_graph_replay_equals_eager():
    from vit.utils import capture_cuda_graph
    model = _ours("tiny-clip-b16", torch.bfloat16)
    x = _x(8, 64, 64).to(DEV, torch.bfloat16)
    y = _x(8, 64, 64, seed=12).to(DEV, torch.bfloat16)
    static = x.clone()
    graph, out = capture_cuda_graph(model, static)
    graph2, out2 = capture_cuda_graph(model.image_embeds, static)
    for inp in (x, y):
        static.copy_(inp)
        graph.replay()
        graph2.replay()
        torch.cuda.synchronize()
        assert torch.equal(out, model(inp))
        assert torch.equal(out2, model.image_embeds(inp))


@torch.no_grad()
def test_clip_forward_makes_the_launches_of_vit(monkeypatch):
    """Fold on: pre_layernorm is one vt_layernorm_stats launch right after the patch embedding, block 0's QKV runs as
    vt_gemm_bf16_ln, and the forward makes as many launches as the ViT forward of the same shape (one LayerNorm added,
    the final one removed)."""
    from vit import configs
    from vit.kernels import _lib
    from vit.vit import VIT
    clip = _ours("tiny-clip-b16", torch.bfloat16)
    kw = {k: v for k, v in configs.clip_kwargs("tiny-clip-b16").items() if k not in ("clip", "projection_dim")}
    vit = VIT(**kw).to(DEV, torch.bfloat16).eval()
    x = _x(4, 64, 64).to(DEV, torch.bfloat16)
    clip(x), vit(x)                                        # build the packs
    names = []
    real = _lib.call
    monkeypatch.setattr(_lib, "call", lambda name, *a: (names.append(name), real(name, *a))[1])
    clip(x)
    clip_names = list(names)
    names.clear()
    vit(x)
    assert len(clip_names) == len(names), (clip_names, names)
    i = clip_names.index("vt_layernorm_stats")
    assert clip_names[:i] == names[:i] and clip_names[i + 1] == "vt_gemm_bf16_ln"
    assert names[-1] == "vt_layernorm" and clip_names.count("vt_layernorm") == 0


@torch.no_grad()
def test_data_parallel_image_embeds_world_size_one():
    from vit.parallel import DataParallelVIT
    model = _ours("tiny-clip-b16", torch.bfloat16)
    x = _x(4, 64, 64).to(DEV, torch.bfloat16)
    dp = DataParallelVIT(model, output="image_embeds")
    assert torch.equal(dp(x), model.image_embeds(x))
    assert torch.equal(DataParallelVIT(model, output="pooler")(x), model.pooler_output(x))
