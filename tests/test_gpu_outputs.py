"""GPU: ``output_hidden_states`` / ``output_attentions`` (HF ``ViTModel``'s flags) and the ``vt_attn_probs`` kernel.

Error bound of ``vt_attn_probs`` against a softmax in fp64 over the kernel's own bf16 Q and K.  Work in log2 units,
a_ij = c * q_i . k_j with c = scale * log2(e), m_i = max_j a_ij, A_ij = c * sum_d |q_id k_jd|, u = 2^-24:
  * the scores: products of bf16 values are exact in fp32; the dh-term fp32 accumulation is off by at most
    dh * u * A_ij (counted twice below, for the accumulation order of the tensor core);
  * the argument fma(s, c, -m) rounds once, u * (|a_ij| + |m_i|); an error of m_i itself is common to the whole row
    and cancels in the ratio;
  * exp2 (ex2.approx.ftz) has a relative error below 2^-21; the running sum of N terms (and, with several key blocks,
    the rescale factors) adds (N + blocks) * 2u, the reciprocal and the product 2u;
so before its one rounding to bf16 an element has the relative error
  E_i = 2 * ln2 * max_j (2 dh u A_ij + u (|a_ij| + |m_i|)) + 2^-20 + (N + 4) * 2u
(the factor 2: numerator and denominator), and the rounding adds at most half a bf16 ulp.  The gate is
  |p_ij - ref_ij| <= ulp_bf16(ref_ij) + 2 E_i ref_ij + 2^-126
(the last term: results below the fp32 normal range flush to zero), and |sum_j p_ij - 1| <= sum_j of the same bound.

The flags against eager HF (``attn_implementation="eager"``: HF's default SDPA attention returns no attention maps):
hidden states use the gates of test_gpu_model.py (bf16 cosine >= 0.999 and max-abs <= 0.15, fp32 max-abs <= 1e-3);
attentions fp32 max-abs <= 1e-3, bf16 per layer cosine >= 0.999 and max-abs <= 0.05."""
import functools
import math

import pytest
import torch
import torch.nn.functional as F

from oracle import hf_oracle

pytestmark = pytest.mark.gpu

DEV = "cuda:0"
GUARD = 13          # odd: the probabilities start 2 bytes past a 16-byte boundary, every span has a head and a tail
U = 2.0 ** -24


# ---------------------------------------------------------------------------------------------------- the kernel
def _qkv(B, N, H, dh, seed, pad=16):
    """bf16 (B, N, 3D) view of a (B, N, 3D + pad) buffer: Q and K random, the V third and the padding NaN."""
    g = torch.Generator().manual_seed(seed)
    D = H * dh
    buf = torch.full((B, N, 3 * D + pad), float("nan"), dtype=torch.bfloat16)
    buf[:, :, :2 * D] = (torch.randn((B, N, 2 * D), generator=g) * 1.5).to(torch.bfloat16)
    return buf.to(DEV)[:, :, :3 * D]


def _probs(qkv, H, dh, scale):
    """vt_attn_probs into the middle of a NaN-filled buffer: (probs (B, H, N, N), whole buffer)."""
    from vit.kernels import _lib
    B, N, D3 = qkv.shape
    total = B * H * N * N
    flat = torch.full((GUARD + total + GUARD,), float("nan"), dtype=torch.bfloat16, device=DEV)
    out = flat[GUARD:GUARD + total]
    _lib.call("vt_attn_probs", qkv.data_ptr(), qkv.data_ptr() + (D3 // 3) * 2, out.data_ptr(), B, H, N, dh,
              qkv.stride(1), qkv.stride(0), scale, _lib.stream_ptr(qkv))
    torch.cuda.synchronize()
    return out.view(B, H, N, N), flat


def _check_guards(flat, total):
    assert torch.isnan(flat[:GUARD]).all() and torch.isnan(flat[GUARD + total:]).all(), "a store left its span"


def _reference_and_bound(qkv, H, dh, scale):
    B, N, D3 = qkv.shape
    D = D3 // 3
    q = qkv[:, :, :D].double().reshape(B, N, H, dh).transpose(1, 2)
    k = qkv[:, :, D:2 * D].double().reshape(B, N, H, dh).transpose(1, 2)
    c = scale / math.log(2.0)
    a = c * (q @ k.transpose(-1, -2))
    A = c * (q.abs() @ k.abs().transpose(-1, -2))
    m = a.amax(-1, keepdim=True)
    ref = torch.softmax(a * math.log(2.0), dim=-1)
    arg = 2 * dh * U * A + U * (a.abs() + m.abs())
    E = 2 * math.log(2.0) * arg.amax(-1, keepdim=True) + 2.0 ** -20 + (N + 4) * 2 * U
    ulp = torch.exp2(torch.floor(torch.log2(ref.clamp_min(2.0 ** -126))) - 7)
    bound = ulp + 2 * E * ref + 2.0 ** -126
    return ref, bound


@pytest.mark.parametrize("dh", [64, 80])
@pytest.mark.parametrize("N", [1, 2, 17, 197, 257, 512, 513, 577, 1025, 2305])
def test_attn_probs_matches_fp64(N, dh):
    B, H = (2, 3) if N <= 577 else (1, 2)
    scale = 1.0 / math.sqrt(dh)
    qkv = _qkv(B, N, H, dh, seed=N * 7 + dh)
    got, flat = _probs(qkv, H, dh, scale)
    _check_guards(flat, got.numel())
    assert torch.isfinite(got).all()
    ref, bound = _reference_and_bound(qkv, H, dh, scale)
    err = (got.double() - ref).abs()
    worst = (err / bound).max().item()
    print(f"N={N} dh={dh}: max-abs {err.max().item():.3e}, worst error / bound {worst:.3f}")
    assert worst <= 1.0, f"N={N} dh={dh}: error / bound {worst:.3f}"
    rows = (got.double().sum(-1) - 1).abs()
    assert (rows <= bound.sum(-1)).all(), f"row sums off by {rows.max().item():.3e}"


@pytest.mark.parametrize("dh", [64, 80])
@pytest.mark.parametrize("N", [197, 577, 1025])
def test_attn_probs_peaked_rows(N, dh):
    """K = Q with large rows: every row's maximum is its own key, hundreds of log2 units above most others, so an
    exponential taken against anything but the row's true maximum (with several key blocks: the maximum of a later
    block) overflows fp32."""
    B, H = 1, 3
    D = H * dh
    qkv = _qkv(B, N, H, dh, seed=N + dh)
    g = torch.Generator().manual_seed(N)
    q = (torch.randn((B, N, D), generator=g) * 5).to(torch.bfloat16).to(DEV)
    qkv[:, :, :D] = q
    qkv[:, :, D:2 * D] = q
    scale = 1.0 / math.sqrt(dh)
    got, flat = _probs(qkv, H, dh, scale)
    _check_guards(flat, got.numel())
    assert torch.isfinite(got).all()
    ref, bound = _reference_and_bound(qkv, H, dh, scale)
    worst = ((got.double() - ref).abs() / bound).max().item()
    print(f"peaked N={N} dh={dh}: worst error / bound {worst:.3f}")
    assert worst <= 1.0, f"N={N} dh={dh}: error / bound {worst:.3f}"


def test_attn_probs_many_heads_and_repeatable():
    """B * H > 65535 work items at a small N; two calls give the same bits."""
    B, H, N, dh = 5462, 12, 2, 64
    qkv = _qkv(B, N, H, dh, seed=3)
    got, flat = _probs(qkv, H, dh, 0.125)
    _check_guards(flat, got.numel())
    again, _ = _probs(qkv, H, dh, 0.125)
    assert torch.equal(got, again)
    ref, bound = _reference_and_bound(qkv, H, dh, 0.125)
    assert ((got.double() - ref).abs() <= bound).all()


@pytest.mark.parametrize("N,dh", [(197, 64), (577, 64), (257, 80)])
def test_attn_probs_image_slice_equals_batch(N, dh):
    B, H = 3, 12
    qkv = _qkv(B, N, H, dh, seed=11)
    whole, _ = _probs(qkv, H, dh, 1.0 / math.sqrt(dh))
    for i in range(B):
        one, _ = _probs(qkv[i:i + 1], H, dh, 1.0 / math.sqrt(dh))
        assert torch.equal(one[0], whole[i]), f"image {i}"


# ---------------------------------------------------------------------------------------------------- models
def _randomize(model, seed):
    g = torch.Generator().manual_seed(seed + 1)
    with torch.no_grad():
        for name, p in model.named_parameters():
            if name.endswith(".bias"):
                p.copy_(torch.randn(p.shape, generator=g) * 0.02)
            elif "layernorm" in name and name.endswith(".weight"):
                p.copy_(1.0 + torch.randn(p.shape, generator=g) * 0.02)
            elif name.endswith("mask_token"):
                p.copy_(torch.randn(p.shape, generator=g) * 0.5)
    return model


@functools.lru_cache(maxsize=None)
def _hf(arch):
    from transformers import ViTConfig, ViTModel
    torch.manual_seed(0)
    cfg = ViTConfig(**hf_oracle.ARCHS[arch], attn_implementation="eager")
    return _randomize(ViTModel(cfg, add_pooling_layer=False, use_mask_token=True).eval(), 0)


@functools.lru_cache(maxsize=None)
def _ours(arch, dtype):
    from vit.utils import transfer_pretrained_weights
    from vit.vit import VIT
    model = VIT(**hf_oracle.vit_kwargs(arch), use_mask_token=True)
    transfer_pretrained_weights(_hf(arch), model, verbose=False)
    return model.to(device=DEV, dtype=dtype).eval()


def _pixels(batch, h, w, seed=5):
    g = torch.Generator().manual_seed(seed)
    return torch.randn((batch, 3, h, w), generator=g)


def _cos(a, b):
    return F.cosine_similarity(a.flatten().float(), b.flatten().float(), dim=0).item()


class _Mode:
    def __init__(self, mode):
        self.mode = mode

    def __enter__(self):
        from vit import vit as V
        if self.mode == "mlp_only":
            V.set_layernorm_folding(True, mlp=False)
        elif self.mode == "fold_off":
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


def _both(fn, x, **kw):
    """(flag-off result, result with both flags, hidden states only, attentions only)"""
    off = fn(x, **kw)
    on = fn(x, output_hidden_states=True, output_attentions=True, **kw)
    hs = fn(x, output_hidden_states=True, **kw)
    at = fn(x, output_attentions=True, **kw)
    return off, on, hs, at


MODES = ["fold", "mlp_only", "fold_off", "fp8", "uint8", "interp384", "mask", "fp32", "unfused"]


@pytest.mark.parametrize("mode", MODES)
@torch.no_grad()
def test_flags_leave_the_forward_bit_identical(mode):
    from vit.vit import VITOutput
    arch = "tiny-b" if mode == "fp32" else "vit-b16-224"
    dtype = torch.float32 if mode == "fp32" else torch.bfloat16
    model = _ours(arch, dtype)
    size = hf_oracle.ARCHS[arch]["image_size"]
    fn, kw = model, {}
    x = _pixels(2 if mode == "unfused" else 4, size, size).to(DEV, dtype)
    if mode == "uint8":
        g = torch.Generator().manual_seed(9)
        x = torch.randint(0, 256, (4, size, size, 3), generator=g, dtype=torch.uint8).to(DEV)
        fn = model.forward_uint8
    elif mode == "interp384":
        x = _pixels(2, 384, 384).to(DEV, dtype)
        kw = dict(interpolate_pos_encoding=True)
    elif mode == "mask":
        g = torch.Generator().manual_seed(7)
        kw = dict(bool_masked_pos=(torch.rand((4, 196), generator=g) < 0.6).to(DEV))
    with _Mode(mode):
        off, on, hs, at = _both(fn, x, **kw)
    torch.cuda.synchronize()
    L, H = model.num_layers, model.num_heads
    B, N, D = off.shape
    assert isinstance(off, torch.Tensor) and isinstance(on, VITOutput)
    for out in (on, hs, at):
        assert torch.equal(out.last_hidden_state, off), f"{mode}: flags changed the final hidden states"
        assert out[0] is out.last_hidden_state
    assert hs.attentions is None and at.hidden_states is None
    for out in (on, hs):
        assert len(out.hidden_states) == L + 1
        assert all(h.shape == (B, N, D) and h.dtype == dtype for h in out.hidden_states)
        assert torch.equal(model.layernorm(out.hidden_states[-1]), off)
    for out in (on, at):
        assert len(out.attentions) == L
        for a in out.attentions:
            assert a.shape == (B, H, N, N) and a.dtype == dtype and a.is_contiguous()
            assert torch.isfinite(a).all()
            assert ((a.float().sum(-1) - 1).abs() <= (0.02 if dtype == torch.bfloat16 else 1e-4)).all()
    for h1, h2 in zip(on.hidden_states, hs.hidden_states):
        assert torch.equal(h1, h2)
    for a1, a2 in zip(on.attentions, at.attentions):
        assert torch.equal(a1, a2)


def _check_hidden(got, want, dtype, what):
    got, want = got.float().cpu(), want.float()
    err, cos = (got - want).abs().max().item(), _cos(got, want)
    print(f"{what}: max-abs {err:.3e} cosine {cos:.6f}")
    if dtype == torch.bfloat16:
        assert cos >= 0.999 and err <= 0.15, f"{what}: cosine {cos:.6f} max-abs {err:.4f}"
    else:
        assert err <= 1e-3, f"{what}: max-abs {err:.3e}"


def _check_attn(got, want, dtype, what):
    got, want = got.float().cpu(), want.float()
    err, cos = (got - want).abs().max().item(), _cos(got, want)
    print(f"{what}: max-abs {err:.3e} cosine {cos:.6f}")
    if dtype == torch.bfloat16:
        assert cos >= 0.999 and err <= 0.05, f"{what}: cosine {cos:.6f} max-abs {err:.4f}"
    else:
        assert err <= 1e-3, f"{what}: max-abs {err:.3e}"


CASES = [("vit-b16-224", "bf16", 224), ("vit-b16-224", "bf16 384", 384), ("vit-b16-224", "bf16 512", 512),
         ("tiny-b", "fp32", 64), ("tiny-h", "fp32", 56), ("tiny-h", "bf16", 56), ("vit-b16-224", "bf16 mask", 224),
         ("tiny-b", "fp32 unfused", 64)]


@pytest.mark.parametrize("arch,kind,size", CASES)
@torch.no_grad()
def test_outputs_match_eager_hf(arch, kind, size):
    dtype = torch.float32 if kind.startswith("fp32") else torch.bfloat16
    model, hf = _ours(arch, dtype), _hf(arch)
    B = 2 if size > 224 else 3
    x = _pixels(B, size, size, seed=size)
    kw = dict(interpolate_pos_encoding=True) if size != hf_oracle.ARCHS[arch]["image_size"] else {}
    if "mask" in kind:
        g = torch.Generator().manual_seed(8)
        kw["bool_masked_pos"] = torch.rand((B, (size // model.patch_size) ** 2), generator=g) < 0.6
    want = hf(pixel_values=x, output_hidden_states=True, output_attentions=True, **kw)
    assert len(want.attentions) == model.num_layers, "HF returned no attention maps (SDPA attention?)"
    ours_kw = {k: (v.to(DEV) if torch.is_tensor(v) else v) for k, v in kw.items()}
    with _Mode("unfused" if "unfused" in kind else "fold"):
        got = model(x.to(DEV, dtype), output_hidden_states=True, output_attentions=True, **ours_kw)
    torch.cuda.synchronize()
    assert len(got.hidden_states) == len(want.hidden_states) and len(got.attentions) == len(want.attentions)
    for i, (g_, w_) in enumerate(zip(got.hidden_states, want.hidden_states)):
        _check_hidden(g_, w_, dtype, f"{arch} {kind} hidden_states[{i}]")
    for i, (g_, w_) in enumerate(zip(got.attentions, want.attentions)):
        _check_attn(g_, w_, dtype, f"{arch} {kind} attentions[{i}]")
    _check_hidden(got.last_hidden_state, want.last_hidden_state, dtype, f"{arch} {kind} last_hidden_state")


@torch.no_grad()
def test_graph_replay_with_both_flags_equals_eager():
    from vit.utils import capture_cuda_graph
    model = _ours("vit-b16-224", torch.bfloat16)
    fn = functools.partial(model, output_hidden_states=True, output_attentions=True)
    static = _pixels(4, 224, 224, seed=1).to(DEV, torch.bfloat16)
    graph, out = capture_cuda_graph(fn, static)
    x = _pixels(4, 224, 224, seed=2).to(DEV, torch.bfloat16)
    static.copy_(x)
    graph.replay()
    torch.cuda.synchronize()
    want = model(x, output_hidden_states=True, output_attentions=True)
    assert torch.equal(out.last_hidden_state, want.last_hidden_state)
    assert all(torch.equal(a, b) for a, b in zip(out.hidden_states, want.hidden_states))
    assert all(torch.equal(a, b) for a, b in zip(out.attentions, want.attentions))
