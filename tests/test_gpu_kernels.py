"""GPU parity of every kernel entry point against the torch op it stands for, on the reference's own
self-check shapes (SURVEY.md section 4) plus the model shapes (197/257/577 rows, D 768/1024/1280)
and ragged edge cases.  Tolerances are stated per test."""
import math

import pytest
import torch
import torch.nn.functional as F

pytestmark = pytest.mark.gpu


@pytest.fixture(autouse=True)
def _seed():
    torch.manual_seed(0)


def dev():
    return torch.device("cuda:0")


def rel_err(got, want):
    return ((got.float() - want.float()).norm() / want.float().norm().clamp_min(1e-12)).item()


# ------------------------------------------------------------------------------- layernorm (K4)
@pytest.mark.parametrize("shape", [(2, 25, 50), (4, 197, 768), (2, 257, 1280), (1, 577, 1024), (3, 7, 8), (1, 1, 4100)])
@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16])
def test_layernorm(shape, dtype):
    from vit.kernels import layernorm
    x = torch.randn(shape, device=dev()).to(dtype)
    w = (1 + 0.1 * torch.randn(shape[-1], device=dev())).to(dtype)
    b = (0.1 * torch.randn(shape[-1], device=dev())).to(dtype)
    got = layernorm(x, w, b, 1e-12)
    want = F.layer_norm(x.float(), (shape[-1],), w.float(), b.float(), 1e-12)
    assert got.dtype == dtype and got.shape == x.shape
    if dtype == torch.float32:
        assert (got - want).abs().max().item() <= 2e-5      # reference self-check: atol 1e-6 at (2,25,50)
    else:
        assert (got.float() - want).abs().max().item() <= 4e-2 and rel_err(got, want) <= 2 ** -7


def test_layernorm_module_and_mixed_output():
    from vit.kernels import LayerNormTriton, layernorm
    ln = LayerNormTriton(768, eps=1e-12).to(dev())
    x = torch.randn(2, 197, 768, device=dev())
    want = F.layer_norm(x, (768,), ln.weight, ln.bias, 1e-12)
    assert (ln(x) - want).abs().max().item() <= 2e-5
    got = layernorm(x, ln.weight.data, ln.bias.data, 1e-12, out_dtype=torch.bfloat16)
    assert got.dtype == torch.bfloat16 and rel_err(got, want) <= 2 ** -7


# ------------------------------------------------------------------------------- add (K5)
@pytest.mark.parametrize("shape", [(2, 2000, 5000), (4, 197, 768), (1, 3, 5), (1, 1, 1)])
@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16])
def test_add(shape, dtype):
    from vit.kernels import add
    a = torch.randn(shape, device=dev()).to(dtype)
    b = torch.randn(shape, device=dev()).to(dtype)
    got = add(a, b)
    assert torch.equal(got, a + b)       # one rounding of an exact fp32 sum: bit-exact with torch


def test_add_rejects_bad_inputs():
    from vit.kernels import add
    a = torch.randn(2, 4, 8, device=dev())
    with pytest.raises(AssertionError):
        add(a, torch.randn(2, 4, 4, device=dev()))
    with pytest.raises(AssertionError):
        add(a.transpose(1, 2), a.transpose(1, 2))
    with pytest.raises(AssertionError):
        add(a[0], a[0])


# ------------------------------------------------------------------------------- softmax (K6)
@pytest.mark.parametrize("shape", [(1, 1823, 781), (12, 197, 197), (2, 577, 577), (1, 1, 1), (2, 3, 33)])
@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16])
def test_softmax(shape, dtype):
    from vit.kernels import softmax
    x = torch.randint(0, 10, shape, device=dev()).to(dtype) if shape[1] == 1823 else (3 * torch.randn(shape, device=dev())).to(dtype)
    got = softmax(x)
    want = torch.softmax(x.float(), dim=-1)
    tol = 1e-6 if dtype == torch.float32 else 4e-3
    assert (got.float() - want).abs().max().item() <= tol


# ------------------------------------------------------------------------------- matmul (K1 + exact path)
@pytest.mark.parametrize("shape", [((4, 20, 30), (30, 10)), ((1, 197, 768), (768, 64)), ((2, 65, 129), (129, 77))])
@pytest.mark.parametrize("act", [None, "gelu"])
def test_matmul_fp32_exact(shape, act):
    from vit.kernels import matmul
    a = torch.randn(shape[0], device=dev())
    b = torch.randn(shape[1], device=dev())
    bias = torch.randn(shape[1][1], device=dev())
    got = matmul(a, b, bias, act)
    want = a.double() @ b.double() + bias.double()
    if act:
        want = F.gelu(want)
    # fp32 operands as six bf16 piece-products accumulated in fp32 on the tensor cores: 6 K adds per output,
    # so sqrt(6) x the rounding noise of an fp32 FMA loop (values here reach +-100)
    assert (got.double() - want).abs().max().item() <= 2.5e-4 * max(1.0, math.sqrt(shape[1][0]) / 4)


def test_matmul_fp32_strided_input():
    from vit.kernels import matmul
    a = torch.randn(3, 40, 24, device=dev()).transpose(1, 2)       # (3, 24, 40), non-contiguous
    b = torch.randn(64, 40, device=dev()).t()                       # (40, 64), non-contiguous
    got = matmul(a, b)
    # fp32 on the tensor cores: 3-piece bf16 split, ~2^-16 per product (values here reach +-25)
    assert (got.double() - a.double() @ b.double()).abs().max().item() <= 5e-4


GEMM_SHAPES = [
    (197, 768, 2304), (197 * 8, 768, 768), (197 * 8, 768, 3072), (197 * 4, 3072, 768),   # ViT-B layers
    (128, 64, 128), (1, 768, 768), (300, 264, 40), (129, 72, 264), (513, 1280, 1280),     # ragged M/N/K
]


@pytest.mark.parametrize("M,K,N", GEMM_SHAPES)
@pytest.mark.parametrize("act", [None, "gelu"])
def test_matmul_bf16_tensor_core(M, K, N, act):
    from vit.kernels import matmul
    a = torch.randn(1, M, K, device=dev()).bfloat16()
    w = (torch.randn(K, N, device=dev()) / math.sqrt(K)).bfloat16()
    bias = torch.randn(N, device=dev()).bfloat16()
    got = matmul(a, w, bias, act)
    want = a.float() @ w.float() + bias.float()
    if act:
        want = F.gelu(want)
    assert got.dtype == torch.bfloat16 and got.shape == (1, M, N)
    assert rel_err(got, want) <= 2 ** -7, f"rel err {rel_err(got, want)}"
    assert (got.float() - want).abs().max().item() <= 0.06


@pytest.mark.parametrize("M,K,N", [(197 * 6, 768, 768), (77, 3072, 768), (1000, 128, 136)])
@pytest.mark.parametrize("out_dtype", [torch.bfloat16, torch.float32])
def test_gemm_bf16_residual_epilogue(M, K, N, out_dtype):
    from vit import packing
    from vit.kernels import _lib
    x = torch.randn(1, M, K, device=dev()).bfloat16()
    w_nk = (torch.randn(N, K, device=dev()) / math.sqrt(K)).bfloat16()
    bias = torch.randn(N, device=dev())
    res = torch.randn(1, M, N, device=dev()).to(out_dtype)
    want = x.float() @ w_nk.float().t() + bias + res.float()
    if out_dtype == torch.bfloat16:
        got = packing.linear(x, w_nk, bias, residual=res)
    else:
        got = torch.empty(1, M, N, device=dev(), dtype=torch.float32)
        _lib.call("vt_gemm_bf16", x.data_ptr(), K, w_nk.data_ptr(), K, got.data_ptr(), N, _lib.VT_F32,
                  bias.data_ptr(), res.data_ptr(), N, M, N, K, 0, _lib.stream_ptr(x))
    tol = 2 ** -7 if out_dtype == torch.bfloat16 else 1e-5
    assert rel_err(got, want) <= tol, f"rel err {rel_err(got, want)}"


def test_gemm_bf16_in_place_residual():
    from vit.kernels import _lib
    M, K, N = 197 * 3, 768, 768
    x = torch.randn(M, K, device=dev()).bfloat16()
    w_nk = (torch.randn(N, K, device=dev()) / math.sqrt(K)).bfloat16()
    bias = torch.randn(N, device=dev())
    res = torch.randn(M, N, device=dev()).bfloat16()
    want = x.float() @ w_nk.float().t() + bias + res.float()
    _lib.call("vt_gemm_bf16", x.data_ptr(), K, w_nk.data_ptr(), K, res.data_ptr(), N, _lib.VT_BF16,
              bias.data_ptr(), res.data_ptr(), N, M, N, K, 0, _lib.stream_ptr(x))
    assert rel_err(res, want) <= 2 ** -7


def test_gemm_bf16_rejects_misaligned():
    from vit.kernels import _lib
    x = torch.randn(16, 12, device=dev()).bfloat16()
    w = torch.randn(16, 12, device=dev()).bfloat16()
    out = torch.empty(16, 16, device=dev()).bfloat16()
    with pytest.raises(_lib.KernelError):
        _lib.call("vt_gemm_bf16", x.data_ptr(), 12, w.data_ptr(), 12, out.data_ptr(), 16, _lib.VT_BF16,
                  None, None, 0, 16, 16, 12, 0, _lib.stream_ptr(x))


# ------------------------------------------------------------------------------- matmul3
@pytest.mark.parametrize("dtype,tol", [(torch.float32, 1e-2), (torch.bfloat16, 0.5)])
def test_matmul3(dtype, tol):
    from vit.kernels import matmul3
    a = torch.randn(4, 120, 760, device=dev()).to(dtype)
    b = torch.randn(4, 760, 500, device=dev()).to(dtype)
    got = matmul3(a, b, apply_scaling=True, scale_factor=1 / math.sqrt(760))
    want = (a.float() @ b.float()) / math.sqrt(760)
    assert (got.float() - want).abs().max().item() <= (1e-4 if dtype == torch.float32 else 0.03)
    with pytest.raises(AssertionError):
        matmul3(a[:1, :3], b[:1, :, :2])       # non-contiguous second operand, like the reference


# ------------------------------------------------------------------------------- batched tensor-core GEMM (vt_bgemm) + packing
@pytest.mark.parametrize("pieces,tol", [(1, 2 ** -7), (3, 3e-5), (6, 2e-6)])
@pytest.mark.parametrize("R,C", [(197, 64), (5, 197), (130, 777)])
def test_pack_split_reconstructs(pieces, tol, R, C):
    """vt_pack_bf16: the pieces of the A-side and B-side layouts multiply back to the fp32 product."""
    from vit.kernels import bgemm as bg
    x = torch.randn(3, 2, R, C, device=dev()) * torch.logspace(-3, 3, C, device=dev())
    cpad = bg.ceil8(C)
    a = bg.pack(x, x.data_ptr(), R, C, 3, 2, (2 * R * C, R * C, C, 1), pieces, pattern=0).view(3, 2, R, pieces, cpad).float()
    b = bg.pack(x, x.data_ptr(), R, C, 3, 2, (2 * R * C, R * C, C, 1), pieces, pattern=1).view(3, 2, R, pieces, cpad).float()
    assert (a[..., C:] == 0).all() and (b[..., C:] == 0).all()
    prod = (a[..., :C].double() * b[..., :C].double()).sum(dim=3)          # sum over the pieces = x * x
    want = x.double() ** 2
    assert ((prod - want).abs() / want.clamp_min(1e-30)).max().item() <= tol
    # transposed read through swapped strides
    t = bg.pack(x, x.data_ptr(), C, R, 3, 2, (2 * R * C, R * C, 1, C), 1).view(3, 2, C, bg.ceil8(R))[..., :R]
    assert torch.equal(t, x.transpose(2, 3).bfloat16())


@pytest.mark.parametrize("M,N,K,batch", [(197, 197, 64, 6), (197, 64, 200, 6), (128, 128, 64, 1), (300, 40, 768, 2), (1, 8, 8, 3),
                                         (257, 330, 520, 2)])
@pytest.mark.parametrize("b_mn", [False, True])
@pytest.mark.parametrize("out_dtype", [torch.bfloat16, torch.float32])
def test_bgemm_batched(M, N, K, batch, b_mn, out_dtype):
    """vt_bgemm on bf16 operands in place: batched, K-major and MN-major B, ragged M / N / K tails filled by
    TMA, scale + bias + residual epilogue, bf16 and fp32 output."""
    from vit.kernels import bgemm as bg
    if b_mn and N % 8:
        pytest.skip("MN-major rows need a multiple of 8 columns")
    a = torch.randn(batch, M, K, device=dev()).bfloat16()
    b = torch.randn(batch, K, N, device=dev()).bfloat16()
    bias = torch.randn(N, device=dev())
    res = torch.randn(batch, M, N, device=dev()).to(out_dtype)
    out = torch.empty(batch, M, N, device=dev(), dtype=out_dtype)
    if b_mn:
        bop, sB = b, (K * N, 0, N)
    else:
        bop, sB = b.transpose(1, 2).contiguous(), (N * K, 0, K)
    bg.bgemm(a.data_ptr(), bop.data_ptr(), out, out.data_ptr(), M, N, K, batch, 1, (M * K, 0, K), sB, (M * N, 0, N),
             bias32=bias, residual_ptr=res.data_ptr(), b_mn=b_mn, scale=0.25)
    want = 0.25 * (a.float() @ b.float()) + bias + res.float()
    tol = 2 ** -7 if out_dtype == torch.bfloat16 else 1e-5
    assert rel_err(out, want) <= tol, f"rel err {rel_err(out, want)}"


def test_bgemm_shared_weight_two_level_batch_and_activations():
    """Weights shared by all batches (batch strides 0), (outer, inner) batch levels with separate output
    strides (the attention context layout), GELU and tanh epilogues."""
    from vit.kernels import bgemm as bg
    Bo, Bi, M, N, K = 2, 3, 70, 64, 96
    a = torch.randn(Bo, Bi, M, K, device=dev()).bfloat16()
    w = torch.randn(N, K, device=dev()).bfloat16() / math.sqrt(K)
    bias = torch.randn(N, device=dev())
    for act, fn in ((bg.ACT_NONE, lambda t: t), (bg.ACT_GELU, F.gelu), (bg.ACT_TANH, torch.tanh)):
        out = torch.zeros(Bo, M, Bi * N, device=dev())                        # [outer, row, inner * N]: like (B, N, H * dh)
        bg.bgemm(a.data_ptr(), w.data_ptr(), out, out.data_ptr(), M, N, K, Bo, Bi, (Bi * M * K, M * K, K), (0, 0, K),
                 (M * Bi * N, N, Bi * N), bias32=bias, act=act)
        want = fn(a.float() @ w.float().t() + bias).permute(0, 2, 1, 3).reshape(Bo, M, Bi * N)
        assert (out - want).abs().max().item() <= 2e-5


def test_bgemm_rejects_misaligned():
    from vit.kernels import _lib, bgemm as bg
    a = torch.randn(4, 12, device=dev()).bfloat16()
    out = torch.empty(4, 4, device=dev())
    with pytest.raises(_lib.KernelError):
        bg.bgemm(a.data_ptr(), a.data_ptr(), out, out.data_ptr(), 4, 4, 12, 1, 1, (0, 0, 12), (0, 0, 12), (0, 0, 4))


@pytest.mark.parametrize("dtype,tol", [(torch.float32, 1e-4), (torch.bfloat16, 3e-2)])
@pytest.mark.parametrize("shape", [((4, 197, 64), (4, 64, 197)), ((4, 197, 197), (4, 197, 64)), ((2, 50, 128), (2, 128, 256))])
def test_matmul3_reference_shapes_on_tensor_cores(dtype, tol, shape):
    """matmul3 on the reference's own call shapes (vit/vit.py:66-72: q k^T with 197 keys, P v) — odd row
    lengths take the packing pass, aligned bf16 operands are consumed in place (MN-major B)."""
    from vit.kernels import matmul3
    a = torch.randn(*shape[0], device=dev()).to(dtype)
    b = torch.randn(*shape[1], device=dev()).to(dtype)
    got = matmul3(a, b, apply_scaling=True, scale_factor=0.125)
    want = 0.125 * (a.double() @ b.double())
    assert got.dtype == dtype and got.shape == want.shape
    assert (got.double() - want).abs().max().item() <= tol * max(1.0, want.abs().max().item() / 4)


def test_fp32_matmul_split_accuracy(monkeypatch):
    """fp32 ``matmul`` on the tensor cores: the 3-piece split (default, ~2^-16 per product, SURVEY.md 7.2) and
    the 6-piece one, both far inside what one TF32 pass (the reference's tl.dot, ~1e-3 here) gives."""
    from vit.kernels import matmul
    a = torch.randn(2, 197, 768, device=dev())
    w = torch.randn(768, 3072, device=dev()) / math.sqrt(768)
    b = torch.randn(3072, device=dev())
    want = F.gelu(a.double() @ w.double() + b.double())
    errs = {}
    for pieces in ("6", "3"):
        monkeypatch.setenv("VT_FP32_SPLIT", pieces)
        errs[pieces] = (matmul(a, w, b, "gelu").double() - want).abs().max().item()
    monkeypatch.setenv("VT_EXACT_FP32", "1")
    errs["simt"] = (matmul(a, w, b, "gelu").double() - want).abs().max().item()
    # measured on B200: 3 pieces 3.2e-5, 6 pieces 5.3e-5, FP32 pipe 6e-6.  The six-piece split is NOT better than
    # the three-piece one on this hardware: the tensor core adds into its fp32 accumulator with truncation, and
    # 6 K such adds lose more than the products dropped by the three-piece split (DESIGN.md section 4)
    assert errs["6"] <= 1.5e-4 and errs["3"] <= 1.5e-4 and errs["simt"] <= 1e-5, errs


# ------------------------------------------------------------------------------- attention (K3)
def _attn_ref(qkv, H):
    B, N, D3 = qkv.shape
    D = D3 // 3
    dh = D // H
    q, k, v = qkv.float().split(D, dim=2)
    q = q.view(B, N, H, dh).transpose(1, 2)
    k = k.view(B, N, H, dh).transpose(1, 2)
    v = v.view(B, N, H, dh).transpose(1, 2)
    p = torch.softmax(q @ k.transpose(-1, -2) / math.sqrt(dh), dim=-1)
    return (p @ v).transpose(1, 2).reshape(B, N, D)


@pytest.mark.parametrize("B,H,N", [(2, 12, 197), (1, 2, 17), (1, 1, 128), (1, 1, 129), (2, 3, 256), (1, 16, 257), (2, 12, 577), (1, 1, 1), (1, 2, 16)])
def test_flash_attention_bf16(B, H, N):
    from vit.kernels import flash_attention
    qkv = torch.randn(B, N, 3 * H * 64, device=dev()).bfloat16()
    got = flash_attention(qkv, H)
    want = _attn_ref(qkv, H)
    assert got.shape == (B, N, H * 64) and got.dtype == torch.bfloat16
    assert torch.isfinite(got.float()).all()
    assert (got.float() - want).abs().max().item() <= 2e-2, f"max err {(got.float() - want).abs().max().item()}"
    assert rel_err(got, want) <= 1e-2


@pytest.mark.parametrize("B,H,N", [(2, 16, 257), (1, 2, 17), (1, 1, 128), (1, 3, 500), (1, 1, 1), (2, 2, 208), (1, 2, 209)])
def test_flash_attention_bf16_head_dim_80(B, H, N):
    """ViT-H heads (dh = 80): 64-column SWIZZLE_128B + 16-column SWIZZLE_32B operand tiles."""
    from vit.kernels import flash_attention
    qkv = torch.randn(B, N, 3 * H * 80, device=dev()).bfloat16()
    got = flash_attention(qkv, H)
    want = _attn_ref(qkv, H)
    assert got.shape == (B, N, H * 80) and torch.isfinite(got.float()).all()
    assert (got.float() - want).abs().max().item() <= 2e-2, f"max err {(got.float() - want).abs().max().item()}"
    assert rel_err(got, want) <= 1e-2


@pytest.mark.parametrize("B,H,N,gain", [(2, 3, 577, 1.0), (1, 2, 209, 1.0), (3, 2, 416, 1.0), (1, 2, 577, 8.0),
                                        (1, 1, 417, 1.0), (5, 7, 257, 1.0), (148, 2, 209, 1.0), (1, 1, 1000, 1.0)])
def test_flash_attention_two_group_kernel_multiblock(B, H, N, gain):
    """attn5mb (default for head dim 64, N > 208): the two-group kernel on sequences of several KV
    blocks (online softmax).  Item counts
    per CTA that are odd, one, or zero for the second group are all covered by the shapes."""
    from vit.kernels import flash_attention
    qkv = (gain * torch.randn(B, N, 3 * H * 64, device=dev())).bfloat16()
    got = flash_attention(qkv, H)
    want = _attn_ref(qkv, H)
    assert torch.isfinite(got.float()).all()
    assert rel_err(got, want) <= (1e-2 if gain == 1.0 else 2e-2)
    sub = flash_attention(qkv[:1].contiguous(), H)
    assert torch.equal(sub, got[:1])


@pytest.mark.parametrize("B,H,N,gain", [(5, 7, 197, 8.0), (1, 1, 200, 1.0), (2, 2, 48, 1.0), (3, 5, 197, 1.0), (1, 2, 130, 1.0),
                                        (2, 2, 64, 1.0), (150, 1, 197, 1.0)])
def test_flash_attention_two_group_kernel_single_block(B, H, N, gain):
    """attn5 (default for head dim 64, N <= 208): peaky logits, one and two query tiles, odd item counts
    per CTA; images and heads are independent, so a sub-batch gives bit-identical rows."""
    from vit.kernels import flash_attention
    qkv = (gain * torch.randn(B, N, 3 * H * 64, device=dev())).bfloat16()
    got = flash_attention(qkv, H)
    assert torch.isfinite(got.float()).all()
    assert rel_err(got, _attn_ref(qkv, H)) <= (1e-2 if gain == 1.0 else 2e-2)
    sub = flash_attention(qkv[:1].contiguous(), H)
    assert torch.equal(sub, got[:1])


@pytest.mark.parametrize("B,H,N,dh", [(3, 6, 197, 64), (2, 4, 100, 64), (40, 12, 197, 64), (3, 6, 577, 64), (2, 5, 257, 80),
                                       (1, 3, 1000, 64)])
def test_flash_attention_bounded_logit_path_vs_exact_path(B, H, N, dh):
    """attn5 skips the row-max pass for (image, head) items whose logits are bounded by |q||k| (Cauchy-Schwarz,
    csrc/attn5_sm100.cu kLogitBound5) and keeps the exact two-pass softmax for the others (the multi-block kernel
    always takes the exact online step: its shapes are here so the switch stays harmless for them).  Heads with gains
    0.5 ... 8 put both kinds of item (and the threshold region, gain 2) into ONE launch, alternating inside a CTA;
    softmax is shift-invariant, so the two paths must agree to rounding — and with the fp32 reference."""
    import ctypes
    from vit.kernels import _lib, flash_attention
    lib = _lib.load()
    lib.vt_debug_set_attn_bound.argtypes = [ctypes.c_int]
    lib.vt_debug_set_attn_bound.restype = None
    gains = torch.tensor([0.5, 8.0, 1.0, 2.0, 4.0, 1.5, 2.2, 0.1, 3.0, 1.0, 6.0, 2.0], device=dev())[:H]
    qkv = torch.randn(B, N, 3, H, dh, device=dev())
    qkv[:, :, :2] *= gains.view(1, 1, 1, H, 1)
    qkv[B // 2, :, 0, 0] *= 30.0          # one image whose first head is far over the bound
    if N > 208:                           # multi-block kernel: one KV block over the bound, the others under it
        qkv[0, 300 % N:, 1, H - 1] *= 40.0
    qkv = qkv.view(B, N, 3 * H * dh).bfloat16()
    want = _attn_ref(qkv, H)
    try:
        lib.vt_debug_set_attn_bound(1)
        fast = flash_attention(qkv, H)
        lib.vt_debug_set_attn_bound(0)
        exact = flash_attention(qkv, H)
    finally:
        lib.vt_debug_set_attn_bound(-1)
    assert torch.isfinite(fast.float()).all() and torch.isfinite(exact.float()).all()
    assert rel_err(exact, want) <= 2e-2
    assert rel_err(fast, want) <= 2e-2
    # path against path: one bf16 rounding of P and of the output apart
    assert (fast.float() - exact.float()).abs().max().item() <= 3e-2
    assert rel_err(fast, exact) <= 1e-2


def test_flash_attention_bounded_logit_path_zero_and_constant_rows():
    """All-zero q / k (every logit 0) and constant keys: the unshifted exponentials are exactly 1."""
    from vit.kernels import flash_attention
    qkv = torch.randn(2, 197, 3, 2, 64, device=dev())
    qkv[0, :, 0] = 0.0
    qkv[1, :, 1] = 0.25
    qkv = qkv.view(2, 197, 3 * 2 * 64).bfloat16()
    got = flash_attention(qkv, 2)
    assert rel_err(got, _attn_ref(qkv, 2)) <= 1e-2


def test_flash_attention_peaky_scores():
    """Large logits: the online max subtraction must keep exp() in range."""
    from vit.kernels import flash_attention
    qkv = (8 * torch.randn(1, 577, 3 * 2 * 64, device=dev())).bfloat16()
    got = flash_attention(qkv, 2)
    want = _attn_ref(qkv, 2)
    assert torch.isfinite(got.float()).all()
    assert rel_err(got, want) <= 2e-2


@pytest.mark.parametrize("dtype,H,dh", [(torch.float32, 2, 64), (torch.float32, 2, 80), (torch.bfloat16, 2, 80)])
def test_attention_exact_path(dtype, H, dh):
    from vit.kernels import flash_attention
    qkv = torch.randn(2, 57, 3 * H * dh, device=dev()).to(dtype)
    got = flash_attention(qkv, H)
    D = H * dh
    q, k, v = qkv.float().split(D, dim=2)
    sh = lambda t: t.view(2, 57, H, dh).transpose(1, 2)
    want = (torch.softmax(sh(q) @ sh(k).transpose(-1, -2) / math.sqrt(dh), -1) @ sh(v)).transpose(1, 2).reshape(2, 57, D)
    # fp32: the two contractions run as 3-piece bf16 splits on the tensor cores (~2^-16 per product)
    assert (got.float() - want).abs().max().item() <= (1e-4 if dtype == torch.float32 else 3e-2)


# ------------------------------------------------------------------------------- conv2d / patching / patch-embed (K2)
def test_patching_matches_unfold():
    from vit.kernels import patching
    img = torch.arange(2 * 3 * 32 * 32, device=dev(), dtype=torch.float32).view(2, 3, 32, 32)
    got = patching(img, 16)
    want = img.unfold(2, 16, 16).unfold(3, 16, 16).permute(0, 2, 3, 1, 4, 5).contiguous().view(2, -1, 3 * 256)
    assert torch.equal(got, want)


@pytest.mark.parametrize("kshape", [(512, 3, 16, 16), (40, 3, 14, 14), (8, 3, 4, 2)])
def test_conv2d_fp32(kshape):
    from vit.kernels import conv2d, Conv2DTriton
    x = torch.randint(0, 10, (4, 3, 224, 224), device=dev()).float()
    w = torch.randn(kshape, device=dev()) * 0.05
    b = torch.randn(kshape[0], device=dev())
    got = conv2d(x, w, b)
    want = F.conv2d(x.double(), w.double(), b.double(), stride=kshape[2:]).float()
    assert got.shape == want.shape
    assert (got - want).abs().max().item() <= 2e-3
    mod = Conv2DTriton(3, kshape[0], tuple(kshape[2:])).to(dev())
    with torch.no_grad():
        mod.weight.copy_(w)
        mod.bias.copy_(b)
    assert torch.equal(mod(x), got)


@pytest.mark.parametrize("S,P,D,B", [(224, 16, 768, 3), (384, 16, 768, 1), (224, 14, 1280, 2), (64, 16, 128, 5), (56, 14, 160, 2)])
@pytest.mark.parametrize("pix_dtype", [torch.float32, torch.bfloat16])
def test_patch_embed_fused(S, P, D, B, pix_dtype):
    from vit.vit import Embeddings
    n = (S // P) ** 2
    emb = Embeddings(P, n, 3 * P * P, D).to(dev())
    with torch.no_grad():
        for p_ in emb.parameters():
            p_.copy_(torch.randn_like(p_) * 0.05)
    emb = emb.to(torch.bfloat16)
    x = torch.randn(B, 3, S, S, device=dev()).to(pix_dtype)
    got = emb(x)
    xb = x.bfloat16().float()
    tok = F.conv2d(xb, emb.projection.weight.float(), emb.projection.bias.float(), stride=P).flatten(2).transpose(1, 2)
    want = torch.cat([emb.cls_token.float().expand(B, -1, -1), tok], 1) + emb.position_embeddings.float()
    assert got.shape == (B, n + 1, D) and got.dtype == torch.bfloat16
    assert rel_err(got, want) <= 2 ** -7, f"rel err {rel_err(got, want)}"
    assert (got.float() - want).abs().max().item() <= 0.05
    if D % 128 == 0:
        # the same launch with the row statistics for the LayerNorm folded into block 0's QKV GEMM
        stats = torch.full((B * (n + 1), D // 128, 2), float("nan"), device=dev())
        again = emb(x, stats)
        assert torch.equal(again, got)
        wc = want.reshape(B * (n + 1), D // 128, 128)
        assert torch.allclose(stats[..., 0], wc.sum(-1), rtol=1e-3, atol=2e-2)
        assert torch.allclose(stats[..., 1], (wc - wc.mean(-1, keepdim=True)).pow(2).sum(-1), rtol=1e-3, atol=2e-2)


@pytest.mark.parametrize("S,P,D,B", [(224, 16, 768, 3), (64, 16, 128, 5), (56, 14, 160, 2), (224, 14, 1280, 1), (96, 32, 64, 2)])
def test_patch_embed_uint8_nhwc(S, P, D, B):
    """Raw uint8 NHWC pixels with the image processor's rescale / normalise folded into the operands
    == conv2d over the normalised NCHW pixels (8-byte vector gather for P*3 % 8 == 0, scalar otherwise)."""
    from vit.vit import Embeddings
    n = (S // P) ** 2
    emb = Embeddings(P, n, 3 * P * P, D).to(dev())
    with torch.no_grad():
        for p_ in emb.parameters():
            p_.copy_(torch.randn_like(p_) * 0.05)
    emb = emb.to(torch.bfloat16)
    mean, std = (0.485, 0.456, 0.406), (0.229, 0.224, 0.225)
    x = torch.randint(0, 256, (B, S, S, 3), device=dev(), dtype=torch.uint8)
    got = emb.forward_uint8(x, mean, std, 1.0 / 255.0)
    xn = (x.float() / 255.0 - torch.tensor(mean, device=dev())) / torch.tensor(std, device=dev())
    tok = F.conv2d(xn.permute(0, 3, 1, 2), emb.projection.weight.float(), emb.projection.bias.float(), stride=P)
    tok = tok.flatten(2).transpose(1, 2)
    want = torch.cat([emb.cls_token.float().expand(B, -1, -1), tok], 1) + emb.position_embeddings.float()
    assert got.shape == (B, n + 1, D) and got.dtype == torch.bfloat16
    assert rel_err(got, want) <= 2 ** -7, f"rel err {rel_err(got, want)}"
    # second call hits the packing cache; changing a weight invalidates it
    assert torch.equal(emb.forward_uint8(x, mean, std, 1.0 / 255.0), got)
    with torch.no_grad():
        emb.projection.bias.add_(1.0)
    assert not torch.equal(emb.forward_uint8(x, mean, std, 1.0 / 255.0), got)


def test_pool_cls():
    from vit.kernels import _lib
    x = torch.randn(5, 197, 768, device=dev()).bfloat16()
    out = torch.empty(5, 768, device=dev(), dtype=torch.bfloat16)
    _lib.call("vt_pool_cls", x.data_ptr(), out.data_ptr(), 5, 768, x.stride(0), _lib.VT_BF16, _lib.stream_ptr(x))
    assert torch.equal(out, x[:, 0, :])


# ------------------------------------------------------------------------------- LayerNorm folded into the GEMM
def _group_stats(xf):
    """(M, K) fp32 -> (M, K/128, 2): (sum, M2 about the group's own mean) — the rowstats layout of vt_gemm_bf16_ln."""
    M, K = xf.shape
    xc = xf.view(M, K // 128, 128).double()
    m2 = ((xc - xc.mean(-1, keepdim=True)) ** 2).sum(-1)
    return torch.stack([xc.sum(-1), m2], dim=2).float().contiguous()


def _ln_module(K):
    ln = torch.nn.LayerNorm(K, eps=1e-12).to(dev())
    with torch.no_grad():
        ln.weight.copy_(1 + 0.2 * torch.randn(K, device=dev()))
        ln.bias.copy_(0.2 * torch.randn(K, device=dev()))
    return ln


@pytest.mark.parametrize("M,K,N", [(197 * 5, 768, 2304), (300, 128, 512), (129, 1280, 264), (260, 384, 640), (70, 1536, 256)])
@pytest.mark.parametrize("gelu", [False, True])
@pytest.mark.parametrize("zero_sum", [False, True])
def test_gemm_layernorm_fold(M, K, N, gelu, zero_sum):
    """vt_gemm_bf16_ln == dense(LayerNorm(x)) with the normalisation applied in the epilogue; the folded
    operands come from the pack kernel (vt_ln_fold)."""
    from vit import packing
    x = (2.0 * torch.randn(1, M, K, device=dev()) + 0.7).bfloat16()
    ln = _ln_module(K)
    w_nk = (torch.randn(N, K, device=dev()) / math.sqrt(K)).bfloat16()
    bias = torch.randn(N, device=dev())
    w_fold, b_fold, colsum = packing.fold_layernorm(w_nk, bias, ln, zero_sum=zero_sum)
    if zero_sum:      # mean term inside the weights (rows sum to zero), no column-sum operand
        assert colsum is None
        assert w_fold.double().sum(dim=1).abs().max().item() <= 2e-3 * w_fold.float().abs().mean().item()
    xf = x.float()[0]
    got = packing.linear_ln(x, w_fold, b_fold, colsum, _group_stats(xf), 1e-12, gelu=gelu)
    want = F.layer_norm(xf, (K,), ln.weight, ln.bias, 1e-12) @ w_nk.float().t() + bias
    if gelu:
        want = F.gelu(want)
    assert rel_err(got[0], want) <= 2 ** -7, f"rel err {rel_err(got[0], want)}"


@pytest.mark.parametrize("K,N", [(128, 96), (768, 2304), (1280, 520), (5120, 128)])
@pytest.mark.parametrize("zero_sum", [False, True])
def test_ln_fold_kernel_matches_restatement(K, N, zero_sum):
    """vt_ln_fold (csrc/ln_fold.cu) against the torch restatement of the same algorithm
    (oracle/fold_restatement.py): identical bias, weights identical up to tie-breaking of equal prices,
    row sums at the 1e-6 level, no element more than one extra ulp away from its exact value."""
    from oracle import fold_restatement
    from vit import packing
    torch.manual_seed(K + N)
    ln = _ln_module(K)
    w_nk = (torch.randn(N, K, device=dev()) / math.sqrt(K)).bfloat16()
    bias = torch.randn(N, device=dev())
    w_fold, b_fold, colsum = packing.fold_layernorm(w_nk, bias, ln, zero_sum=zero_sum)
    again = packing.fold_layernorm(w_nk, bias, ln, zero_sum=zero_sum)
    assert torch.equal(w_fold, again[0]) and torch.equal(b_fold, again[1])        # deterministic
    if not zero_sum:
        w_ref, b_ref, c_ref = fold_restatement.fold_layernorm_colsum(w_nk, bias, ln)
        assert torch.equal(w_fold, w_ref)
        assert torch.allclose(b_fold, b_ref, rtol=1e-5, atol=1e-5)
        assert torch.allclose(colsum, w_fold.double().sum(dim=1).float(), rtol=0, atol=1e-6)
        return
    w_ref, b_ref = fold_restatement.fold_layernorm_zero_sum(w_nk, bias, ln)
    assert torch.allclose(b_fold, b_ref, rtol=1e-5, atol=1e-5)
    scale = w_fold.float().abs().mean().item()
    assert w_fold.double().sum(dim=1).abs().max().item() <= 2e-3 * scale
    assert w_fold.double().sum(dim=1).abs().max().item() <= 4 * w_ref.double().sum(dim=1).abs().max().item() + 1e-5 * scale
    exact = w_nk.float() * ln.weight.detach()[None, :]
    exact = exact - exact.double().mean(dim=1, keepdim=True).float()       # the kernel's row mean is an fp64 sum
    ulp = torch.exp2(torch.floor(torch.log2(exact.abs().clamp_min(1e-30))) - 7.0)
    # rounding (0.5 ulp) + one move (1 ulp, 2 at a binade edge); the absolute slack covers elements so close to
    # zero that the last bit of the row mean is many of their own ulps
    ratio = ((w_fold.float() - exact).abs() - 1e-8).clamp_min(0) / ulp
    assert ratio.max().item() <= 2.6, f"element {ratio.argmax().item()} is {ratio.max().item()} ulp from its exact value"
    # the two implementations pick (almost) the same elements: added squared error within 10 %
    e_k = (w_fold.float() - exact).pow(2).sum().item()
    e_r = (w_ref.float() - exact).pow(2).sum().item()
    assert e_k <= 1.1 * e_r + 1e-12, (e_k, e_r)
    assert (w_fold != w_ref).float().mean().item() <= 0.02


def _stats_of(x):
    """Row statistics of x (1, M, K) bf16 as the GEMM epilogue writes them: out = 0 @ W^T + 0 + x."""
    from vit import packing
    _, M, K = x.shape
    zeros = torch.zeros(1, M, 64, device=x.device, dtype=torch.bfloat16)
    w0 = torch.zeros(K, 64, device=x.device, dtype=torch.bfloat16)
    b0 = torch.zeros(K, device=x.device)
    stats = torch.full((M, K // 128, 2), float("nan"), device=x.device)
    out = packing.linear_res_stats(zeros, w0, b0, x, stats)
    assert torch.equal(out, x)
    return stats


OUTLIER_CASES = ["massive_channels", "large_mean_100", "large_mean_1000", "near_constant", "constant", "mixed"]


def _outlier_rows(case, M, K):
    g = torch.Generator(device="cpu").manual_seed(sum(map(ord, case)))
    x = torch.randn(M, K, generator=g)
    if case == "massive_channels":          # a few channels at +-50..200 in every row (real ViT checkpoints)
        for ch, v in ((3, 60.0), (K // 2 + 1, -120.0), (K - 5, 200.0), (130 % K, -50.0)):
            x[:, ch] = v * (1 + 0.05 * torch.randn(M, generator=g))
    elif case == "large_mean_100":          # |mean| / std = 100
        x = 0.5 * x + 50.0
    elif case == "large_mean_1000":         # |mean| / std = 1000: one-pass E[x^2] - mean^2 has no digits left
        x = 0.1 * x - 100.0
    elif case == "near_constant":           # spread of a few bf16 ulps around a constant
        x = 1.0 + 0.01 * x
    elif case == "constant":                # variance exactly 0: LN(x) = beta
        x = torch.full((M, K), 3.25)
        x[M // 2:] = 0.0
    elif case == "mixed":                   # every row different: offsets, scales and planted channels
        x = x * torch.logspace(-2, 2, M)[:, None] + torch.linspace(-300, 300, M)[:, None]
        x[::3, 7] = 1000.0
    return x


@pytest.mark.parametrize("case", OUTLIER_CASES)
@pytest.mark.parametrize("K,N", [(768, 512), (1280, 264)])
@pytest.mark.parametrize("gelu", [False, True])
def test_gemm_layernorm_fold_outliers(case, K, N, gelu):
    """The LayerNorm fold on the activations real checkpoints produce and the benign tests do not: massive
    channels, rows with |mean| >> std, near-constant and constant rows.  Statistics come from the GEMM
    epilogue itself (vt_gemm_bf16_ln stats_out); the oracle is F.layer_norm -> dense in fp32 on the same
    bf16 inputs (reference: centred two-pass variance, vit/kernels/layernorm.py:51-85)."""
    from vit import packing
    M = 333
    torch.manual_seed(11)
    x = _outlier_rows(case, M, K).to(dev()).bfloat16()[None]
    ln = _ln_module(K)
    w_nk = (torch.randn(N, K, device=dev()) / math.sqrt(K)).bfloat16()
    bias = torch.randn(N, device=dev())
    w_fold, b_fold, _ = packing.fold_layernorm(w_nk, bias, ln)
    stats = _stats_of(x)
    xf = x.float()[0]
    ref_stats = _group_stats(xf)
    assert torch.allclose(stats[..., 0], ref_stats[..., 0], rtol=1e-5, atol=1e-3)
    assert torch.allclose(stats[..., 1], ref_stats[..., 1], rtol=1e-3, atol=1e-6), \
        f"M2 max rel err {((stats[..., 1] - ref_stats[..., 1]).abs() / ref_stats[..., 1].clamp_min(1e-20)).max().item()}"
    got = packing.linear_ln(x, w_fold, b_fold, None, stats, 1e-12, gelu=gelu).float()[0]
    want = F.layer_norm(xf.double(), (K,), ln.weight.double(), ln.bias.double(), 1e-12).float() @ w_nk.float().t() + bias
    if gelu:
        want = F.gelu(want)
    assert torch.isfinite(got).all()
    # per row: the folded result is as good as bf16 rounding of the exact result allows
    row_err = (got - want).norm(dim=1) / want.norm(dim=1).clamp_min(1e-6)
    assert row_err.max().item() <= 2 ** -6, f"{case}: worst row rel err {row_err.max().item()} (row {row_err.argmax().item()})"
    assert rel_err(got, want) <= 2 ** -7, f"{case}: rel err {rel_err(got, want)}"


@pytest.mark.parametrize("case", ["massive_channels", "large_mean_100", "mixed"])
def test_patch_embed_stats_outliers_against_parameters(case):
    """Row statistics written by the patch-embedding epilogue when the position / bias table carries large
    offsets and planted channels (the rows of block 0's folded layernorm_before)."""
    from vit.vit import Embeddings
    torch.manual_seed(5)
    P, S, D, B = 16, 64, 256, 3
    n = (S // P) ** 2
    emb = Embeddings(P, n, 3 * P * P, D).to(dev(), torch.bfloat16)
    with torch.no_grad():
        emb.projection.weight.copy_(torch.randn_like(emb.projection.weight) * 0.02)
        emb.projection.bias.copy_(torch.randn_like(emb.projection.bias) * 0.02)
        emb.cls_token.copy_(torch.randn_like(emb.cls_token))
        pos = _outlier_rows(case, n + 1, D).to(dev())
        emb.position_embeddings.copy_(pos[None].bfloat16())
    x = torch.randn(B, 3, S, S, device=dev()).bfloat16()
    plain = emb(x)
    stats = torch.full((B * (n + 1), D // 128, 2), float("nan"), device=dev())
    again = emb(x, stats)
    assert torch.equal(plain, again)
    # the kernel's statistics are those of the fp32 values BEFORE the bf16 rounding of the output
    pk = emb.packed()
    from vit.kernels.patching import patching
    patches = patching(x, P).float()                                     # (B, n, K)
    tok = patches @ pk.w[:, :pk.K].float().t()                           # (B, n, D)
    posb = emb.position_embeddings.detach().float()[0].clone()           # pos + (row 0: cls, rows >= 1: conv bias)
    posb[0] += emb.cls_token.detach().float().reshape(-1)
    posb[1:] += emb.projection.bias.detach().float()
    full = torch.cat([torch.zeros(B, 1, D, device=dev()), tok], dim=1) + posb[None]
    ref = _group_stats(full.reshape(B * (n + 1), D))
    st, rf = stats.view(B, n + 1, -1, 2), ref.view(B, n + 1, -1, 2)
    assert torch.allclose(st[:, 1:, :, 0], rf[:, 1:, :, 0], rtol=1e-4, atol=5e-2)
    assert torch.allclose(st[:, 1:, :, 1], rf[:, 1:, :, 1], rtol=2e-3, atol=1e-3)
    # CLS rows: the two-launch form adds the conv bias to a bf16 table entry (cls + pos[0] - bias): one bf16 rounding
    # of the entry — below the rounding of the bf16 output itself
    ulp_row = 2.0 ** -8 * full[:, 0].abs().amax().item()
    assert torch.allclose(st[:, 0, :, 0], rf[:, 0, :, 0], rtol=1e-4, atol=128 * ulp_row + 5e-2)
    assert torch.allclose(st[:, 0, :, 1], rf[:, 0, :, 1], rtol=2e-2, atol=128 * ulp_row * full[:, 0].abs().amax().item() + 1e-3)


def test_gemm_row_stats_output():
    from vit import packing
    M, K, N = 197 * 3 + 5, 3072, 768
    x = torch.randn(1, M, K, device=dev()).bfloat16()
    w_nk = (torch.randn(N, K, device=dev()) / math.sqrt(K)).bfloat16()
    bias = torch.randn(N, device=dev())
    res = torch.randn(1, M, N, device=dev()).bfloat16()
    stats = torch.full((M, N // 128, 2), float("nan"), device=dev())
    got = packing.linear_res_stats(x, w_nk, bias, res, stats)
    want = x.float()[0] @ w_nk.float().t() + bias + res.float()[0]
    assert rel_err(got[0], want) <= 2 ** -7
    wc = want.view(M, N // 128, 128)
    assert torch.allclose(stats[..., 0], wc.sum(-1), rtol=1e-3, atol=2e-2)
    assert torch.allclose(stats[..., 1], (wc - wc.mean(-1, keepdim=True)).pow(2).sum(-1), rtol=1e-3, atol=2e-2)
    again = torch.empty_like(stats)
    packing.linear_res_stats(x, w_nk, bias, res, again)
    assert torch.equal(stats, again)          # no atomics: bit-reproducible


# ------------------------------------------------------------------------------- pool + peer all-gather (K7)
def test_pool_cls_allgather_single_rank_protocol():
    """vt_pool_cls_allgather with world = 1 (the rank is its own peer): the step counter lives in device
    memory (identical launches step after step), rows land in gather buffer step mod 4 and in the local
    output, the flag counter advances by blocks-per-peer each step; then the split PUT / GET form: GET
    with lag 1 returns the step before the last PUT, lag 0 the last one."""
    import ctypes
    from vit.kernels import _lib
    B, N, D = 37, 5, 768
    flags = torch.zeros(1, dtype=torch.int32, device=dev())
    ctrl = torch.zeros(2, dtype=torch.int32, device=dev())
    bufs = torch.full((4, B, D), float("nan"), device=dev(), dtype=torch.bfloat16)
    out = torch.full((B, D), float("nan"), device=dev(), dtype=torch.bfloat16)
    flag_tab = (ctypes.c_void_p * 1)(flags.data_ptr())
    out_tab = (ctypes.c_void_p * 4)(*[bufs[b].data_ptr() for b in range(4)])

    def launch(x, o, mode, lag):
        _lib.call("vt_pool_cls_allgather", _lib.ptr(x), B, D, x.stride(0) if x is not None else D, _lib.VT_BF16,
                  ctypes.cast(out_tab, ctypes.c_void_p), ctypes.cast(flag_tab, ctypes.c_void_p), 0, 1,
                  ctrl.data_ptr(), _lib.ptr(o), mode, lag, _lib.stream_ptr(bufs))

    seen = []
    for step in (1, 2, 3, 4, 5):
        x = torch.randn(B, N, D, device=dev()).bfloat16()
        launch(x, out, _lib.VT_PG_PUT | _lib.VT_PG_GET, 0)
        torch.cuda.synchronize()
        assert torch.equal(out, x[:, 0, :]) and torch.equal(bufs[step & 3], x[:, 0, :])
        assert ctrl.tolist() == [step, 0]
        seen.append(int(flags.item()))
    assert all(b - a == seen[0] for a, b in zip(seen, seen[1:])) and seen[0] >= 1
    # split form, continuing from step 5
    xs = [torch.randn(B, N, D, device=dev()).bfloat16() for _ in range(3)]
    launch(xs[0], None, _lib.VT_PG_PUT, 0)                 # step 6
    launch(xs[1], None, _lib.VT_PG_PUT, 0)                 # step 7
    launch(None, out, _lib.VT_PG_GET, 1)                   # collects step 6
    torch.cuda.synchronize()
    assert torch.equal(out, xs[0][:, 0, :]) and ctrl.tolist() == [7, 0]
    launch(xs[2], None, _lib.VT_PG_PUT, 0)                 # step 8
    launch(None, out, _lib.VT_PG_GET, 1)                   # collects step 7
    torch.cuda.synchronize()
    assert torch.equal(out, xs[1][:, 0, :])
    launch(None, out, _lib.VT_PG_GET, 0)                   # drains step 8
    torch.cuda.synchronize()
    assert torch.equal(out, xs[2][:, 0, :])
    with pytest.raises(_lib.KernelError):                  # PUT needs rows
        launch(None, out, _lib.VT_PG_PUT | _lib.VT_PG_GET, 0)
    with pytest.raises(_lib.KernelError):                  # GET needs somewhere to put them
        launch(None, None, _lib.VT_PG_GET, 0)


def test_pool_cls_allgather_graph_replay():
    """The gather launch has no per-step argument: captured once into a CUDA graph, every replay is the
    next step (world = 1)."""
    import ctypes
    from vit.kernels import _lib
    B, N, D = 16, 3, 256
    flags = torch.zeros(1, dtype=torch.int32, device=dev())
    ctrl = torch.zeros(2, dtype=torch.int32, device=dev())
    bufs = torch.zeros((4, B, D), device=dev(), dtype=torch.bfloat16)
    out = torch.zeros((B, D), device=dev(), dtype=torch.bfloat16)
    x = torch.randn(B, N, D, device=dev()).bfloat16()
    flag_tab = (ctypes.c_void_p * 1)(flags.data_ptr())
    out_tab = (ctypes.c_void_p * 4)(*[bufs[b].data_ptr() for b in range(4)])
    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph, stream=side):
        _lib.call("vt_pool_cls_allgather", x.data_ptr(), B, D, x.stride(0), _lib.VT_BF16,
                  ctypes.cast(out_tab, ctypes.c_void_p), ctypes.cast(flag_tab, ctypes.c_void_p), 0, 1,
                  ctrl.data_ptr(), out.data_ptr(), _lib.VT_PG_PUT | _lib.VT_PG_GET, 0, _lib.stream_ptr(x))
    for step in (1, 2, 3, 4, 5, 6):
        x.copy_(torch.randn(B, N, D, device=dev()).bfloat16())
        graph.replay()
        torch.cuda.synchronize()
        assert torch.equal(out, x[:, 0, :]) and torch.equal(bufs[step & 3], x[:, 0, :]) and ctrl.tolist() == [step, 0]


# ------------------------------------------------------------------------------- FP8 path (VT_FP8, kind::f8f6f4)
def _e4m3(t):
    return t.to(torch.float8_e4m3fn)


@pytest.mark.parametrize("M,N,K", [(197 * 3, 2304, 768), (300, 128, 3072), (129, 640, 1280), (64, 264, 512)])
@pytest.mark.parametrize("mode", ["plain", "gelu", "res", "gelu_fp8out"])
def test_gemm_fp8(M, N, K, mode):
    """vt_gemm_fp8 against the same e4m3 operands multiplied in fp32 (the kernel's arithmetic is exact up to fp32
    accumulation: products of e4m3 values are exact), column scales, bias, GELU, residual, e4m3 output."""
    from vit import packing
    if mode == "gelu_fp8out" and N % 128:
        pytest.skip("e4m3 output needs N % 128 == 0")
    x = torch.randn(1, M, K, device=dev())
    w = (torch.randn(N, K, device=dev()) / math.sqrt(K)).bfloat16()
    bias = torch.randn(N, device=dev())
    res = torch.randn(1, M, N, device=dev()).bfloat16()
    x8 = _e4m3(x * 16.0)
    w8, scales = packing.quantize_weight_fp8(w)
    # the pack kernel's quantisation is the nearest-e4m3 rounding of w / (amax / 448)
    want_w8 = _e4m3(w.float() / (w.float().abs().amax(dim=1, keepdim=True) / 448.0))
    assert (w8.view(torch.float8_e4m3fn).float() != want_w8.float()).float().mean().item() <= 3e-3   # ties of w * (1 / s) vs w / s (7e-4 of the elements on the CPU too)
    assert torch.allclose(scales, w.float().abs().amax(dim=1) / 448.0)
    colscale = (scales / 16.0).contiguous()
    ref = (x8.float()[0] @ w8.view(torch.float8_e4m3fn).float().t()) * colscale + bias
    got = packing.linear_fp8(x8.view(torch.uint8), w8, colscale, bias, gelu=mode.startswith("gelu"),
                             residual=res if mode == "res" else None, out_fp8=mode == "gelu_fp8out", out_scale=8.0)
    if mode.startswith("gelu"):
        ref = F.gelu(ref)
    if mode == "res":
        ref = ref + res.float()[0]
    if mode == "gelu_fp8out":
        got = got.view(torch.float8_e4m3fn).float()[0] / 8.0
        assert rel_err(got, ref) <= 0.04          # e4m3 rounding of the output: 2^-4 relative per element
    else:
        assert rel_err(got[0], ref) <= 2 ** -7, f"rel err {rel_err(got[0], ref)}"
    # and the quantised product is a fair approximation of the bf16 layer itself
    full = x[0] @ w.float().t() + bias
    if mode == "plain":
        assert rel_err(got[0], full) <= 0.06


@pytest.mark.parametrize("rows,dim", [(197 * 2, 768), (77, 1024), (33, 1280), (5, 128)])
def test_layernorm_fp8(rows, dim):
    from vit import packing
    x = (torch.randn(1, rows, dim, device=dev()) * 3 + 0.5).bfloat16()
    ln = _ln_module(dim).to(torch.bfloat16)
    got = packing.layernorm_fp8(x, ln).view(torch.float8_e4m3fn).float()[0] / 16.0
    want = F.layer_norm(x.float()[0], (dim,), ln.weight.float(), ln.bias.float(), ln.eps)
    assert (got - want).abs().max().item() <= 2 ** -4 * want.abs().max().item() + 1e-3
    assert rel_err(got, want) <= 0.04
