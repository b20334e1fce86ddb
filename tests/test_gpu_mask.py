"""GPU: ``bool_masked_pos`` and the masked image modeling head (HF ``ViTModel(use_mask_token=True)`` and
``ViTForMaskedImageModeling``).

Kernels: the masked gather against ``F.unfold`` and the selected position rows, ``vt_embed_finalize_masked`` against a
torch restatement, ``vt_mim_reconstruct`` against ``F.pixel_shuffle``, all bit for bit, and its loss against an fp64
restatement.  Model: an all-false mask equals the unmasked call bit for bit on every path; random and all-true masks
against HF at the gates of tests/test_gpu_model.py (bf16 cosine >= 0.999 and max-abs <= 0.15, fp32 <= 1e-3); batch
independence; graph replay with a new mask copied in; the heads; the reconstruction and loss against HF.  HF
zero-initialises the mask token, the decoder bias and the other biases, so they are re-randomised here."""
import functools

import pytest
import torch
import torch.nn.functional as F

from oracle import hf_oracle

pytestmark = pytest.mark.gpu

DEV = "cuda:0"
NAN_GUARD = 3


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
def _hf_model(arch, pooling=False):
    from transformers import ViTConfig, ViTModel
    torch.manual_seed(0)
    return _randomize(ViTModel(ViTConfig(**hf_oracle.ARCHS[arch]), add_pooling_layer=pooling,
                               use_mask_token=True).eval(), 0)


@functools.lru_cache(maxsize=None)
def _hf_mim(arch, stride):
    from transformers import ViTConfig, ViTForMaskedImageModeling
    torch.manual_seed(0)
    return _randomize(ViTForMaskedImageModeling(ViTConfig(**hf_oracle.ARCHS[arch], encoder_stride=stride)).eval(), 0)


def _ours(hf, arch, dtype, **kw):
    from vit.utils import transfer_pretrained_weights
    from vit.vit import VIT
    model = VIT(**hf_oracle.vit_kwargs(arch), **kw)
    transfer_pretrained_weights(hf, model, verbose=False)
    return model.to(device=DEV, dtype=dtype).eval()


@functools.lru_cache(maxsize=None)
def _b16(dtype):
    return _ours(_hf_model("vit-b16-224"), "vit-b16-224", dtype, use_mask_token=True)


def _pixels(batch, h, w, seed=5):
    g = torch.Generator().manual_seed(seed)
    return torch.randn((batch, 3, h, w), generator=g)


def _mask(batch, n, seed=7, ratio=0.6):
    g = torch.Generator().manual_seed(seed)
    return torch.rand((batch, n), generator=g) < ratio


def _cos(a, b):
    return F.cosine_similarity(a.flatten().float(), b.flatten().float(), dim=0).item()


def _check(got, want, dtype, what):
    got, want = got.float().cpu(), want.float().cpu()
    assert got.shape == want.shape, f"{what}: {tuple(got.shape)} vs {tuple(want.shape)}"
    assert torch.isfinite(got).all(), what
    err, cos = (got - want).abs().max().item(), _cos(got, want)
    print(f"{what}: max-abs {err:.3e} cosine {cos:.6f}")
    if dtype == torch.bfloat16:
        assert cos >= 0.999 and err <= 0.15, f"{what}: cosine {cos:.6f} max-abs {err:.4f}"
    else:
        assert err <= 1e-3, f"{what}: max-abs {err:.3e}"


# ---------------------------------------------------------------------------------------------------- kernels
def _unfold_rows(x, P, nhwc):
    """(B, n, K) bf16 patch rows in the gather's order: (c, i, j) for NCHW, (i, j, c) for NHWC."""
    if nhwc:
        B, H, W, C = x.shape
        u = F.unfold(x.permute(0, 3, 1, 2).float(), P, stride=P)          # (B, C*P*P, n), (c, i, j)
        n = u.shape[2]
        return u.reshape(B, C, P, P, n).permute(0, 4, 2, 3, 1).reshape(B, n, P * P * C).bfloat16()
    return F.unfold(x.float(), P, stride=P).transpose(1, 2).bfloat16()


@pytest.mark.parametrize("hw", [(64, 64), (48, 70), (80, 37)])       # square; non-square + odd W (scalar loads)
@pytest.mark.parametrize("pix", ["f32", "bf16", "u8"])
def test_masked_gather_matches_unfold(pix, hw):
    from vit.kernels import _lib
    B, C, P, D = 3, 3, 16, 136
    H, W = hw
    gh, gw = H // P, W // P
    n = gh * gw
    N = n + 1
    K = C * P * P
    ldw = K + 8                                            # padding columns must come out zero
    g = torch.Generator().manual_seed(H * 100 + W)
    if pix == "u8":
        x = torch.randint(0, 256, (B, H, W, C), generator=g, dtype=torch.uint8)
        code = _lib.VT_U8
    else:
        x = torch.randn((B, C, H, W), generator=g).to(torch.float32 if pix == "f32" else torch.bfloat16)
        code = _lib.VT_F32 if pix == "f32" else _lib.VT_BF16
    mask = _mask(B, n, seed=H + W)
    mask[0, 0] = True
    mask[1, -1] = False
    pos = torch.randn((N, D), generator=g).bfloat16()
    posm = torch.randn((N, D), generator=g).bfloat16()
    rows = B * N
    patches = torch.full((rows + 2 * NAN_GUARD, ldw), float("nan"), dtype=torch.bfloat16, device=DEV)
    table = torch.full((rows + 2 * NAN_GUARD, D), float("nan"), dtype=torch.bfloat16, device=DEV)
    xd, md, pd, pmd = x.to(DEV), mask.to(DEV), pos.to(DEV), posm.to(DEV)
    _lib.call("vt_patch_embed_masked_gather", xd.data_ptr(), code, md.data_ptr(), pd.data_ptr(), pmd.data_ptr(),
              patches[NAN_GUARD:].data_ptr(), ldw, table[NAN_GUARD:].data_ptr(), B, C, H, W, P, D,
              _lib.stream_ptr(xd))
    torch.cuda.synchronize()
    patches, table = patches.cpu(), table.cpu()
    for buf in (patches, table):
        assert buf[:NAN_GUARD].isnan().all() and buf[-NAN_GUARD:].isnan().all(), "guard rows overwritten"
    got_p = patches[NAN_GUARD:-NAN_GUARD].view(B, N, ldw)
    got_t = table[NAN_GUARD:-NAN_GUARD].view(B, N, D)
    want_p = torch.zeros((B, N, ldw), dtype=torch.bfloat16)
    want_p[:, 1:, :K] = _unfold_rows(x, P, pix == "u8").masked_fill(mask[:, :, None], 0)
    want_t = pos[None].repeat(B, 1, 1)
    want_t[:, 1:][mask] = posm[1:].expand(B, n, D)[mask]
    assert torch.equal(got_p.view(torch.int16), want_p.view(torch.int16))
    assert torch.equal(got_t.view(torch.int16), want_t.view(torch.int16))


@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16])
def test_embed_finalize_masked_matches_torch(dtype):
    from vit.kernels import _lib
    B, N, D = 5, 21, 100
    g = torch.Generator().manual_seed(3)
    x = torch.randn((B, N, D), generator=g).to(dtype)
    pos, cls, mt = (torch.randn(s, generator=g).to(dtype) for s in ((N, D), (D,), (D,)))
    mask = _mask(B, N - 1, seed=4)
    want = torch.empty_like(x)
    want[:, 0] = (cls.float() + pos[0].float()).to(dtype)
    body = torch.where(mask[:, :, None], mt.expand(B, N - 1, D), x[:, 1:])
    want[:, 1:] = (body.float() + pos[1:].float()).to(dtype)
    xd = x.to(DEV)
    pd, cd, md, maskd = pos.to(DEV), cls.to(DEV), mt.to(DEV), mask.to(DEV)
    _lib.call("vt_embed_finalize_masked", xd.data_ptr(), pd.data_ptr(), cd.data_ptr(), md.data_ptr(), maskd.data_ptr(),
              B, N, D, _lib.dtype_code(xd), _lib.stream_ptr(xd))
    assert torch.equal(xd.cpu(), want)


def _loss64(pixels, rec, mask, s, u8, mean=(0.5, 0.5, 0.5), std=(0.5, 0.5, 0.5), rescale=1 / 255):
    px = pixels.double()
    if u8:
        m, sd = torch.tensor(mean, dtype=torch.float64), torch.tensor(std, dtype=torch.float64)
        px = ((px * rescale - m) / sd).permute(0, 3, 1, 2)
    B, C = rec.shape[:2]
    gh, gw = rec.shape[2] // s, rec.shape[3] // s
    mpix = mask.reshape(B, gh, gw).repeat_interleave(s, 1).repeat_interleave(s, 2)[:, None].double()
    return ((px - rec.double()).abs() * mpix).sum() / (mpix.sum() + 1e-5) / C


@pytest.mark.parametrize("grid", [(4, 4, 16), (3, 5, 16), (4, 4, 14), (2, 7, 14)])     # (gh, gw, s)
@pytest.mark.parametrize("dtype,pix", [(torch.float32, "f32"), (torch.bfloat16, "bf16"), (torch.bfloat16, "u8"),
                                       (torch.float32, "u8")])
def test_mim_reconstruct_matches_pixel_shuffle_and_fp64_loss(grid, dtype, pix):
    from vit import packing
    from vit.kernels import _lib
    gh, gw, s = grid
    B, C = 6, 3
    n = gh * gw
    g = torch.Generator().manual_seed(gh * 31 + gw * 7 + s)
    dec = torch.randn((B, 1 + n, s * s * C), generator=g).to(dtype)
    want = F.pixel_shuffle(dec[:, 1:].transpose(1, 2).reshape(B, s * s * C, gh, gw), s)
    loss, rec = packing.mim_reconstruct(dec.to(DEV), gh, gw, s, C)
    assert loss is None and rec.dtype == dtype
    assert torch.equal(rec.cpu(), want), "reconstruction differs from F.pixel_shuffle"

    H, W = gh * s, gw * s
    if pix == "u8":
        pixels = torch.randint(0, 256, (B, H, W, C), generator=g, dtype=torch.uint8)
        code, norm = _lib.VT_U8, torch.tensor([0.485, 0.456, 0.406, 0.229, 0.224, 0.225], device=DEV)
    else:
        pixels = torch.randn((B, C, H, W), generator=g).to(torch.float32 if pix == "f32" else torch.bfloat16)
        code, norm = _lib.dtype_code(pixels), None
    mask = _mask(B, n, seed=gh + gw)
    args = (dec.to(DEV), gh, gw, s, C, pixels.to(DEV), code, norm, 1 / 255, mask.to(DEV))
    loss, rec = packing.mim_reconstruct(*args)
    loss2, _ = packing.mim_reconstruct(*args)
    assert loss.shape == () and loss.dtype == torch.float32 and loss.device.type == "cuda"
    assert torch.equal(rec.cpu(), want)
    kw = dict(mean=(0.485, 0.456, 0.406), std=(0.229, 0.224, 0.225)) if pix == "u8" else {}
    ref = _loss64(pixels, rec.cpu(), mask, s, pix == "u8", **kw).item()
    got = loss.item()
    assert abs(got - ref) <= 1e-5 * abs(ref), f"loss {got!r} vs fp64 {ref!r}"
    assert torch.equal(loss.view(torch.int32), loss2.view(torch.int32)), "the loss changed between two calls"


# ---------------------------------------------------------------------------------------------------- all-false mask
@torch.no_grad()
def _all_false_equal(model, x, interp=False, u8=False):
    B = x.shape[0]
    H, W = (x.shape[1], x.shape[2]) if u8 else (x.shape[2], x.shape[3])
    n = (H // model.patch_size) * (W // model.patch_size)
    none = torch.zeros((B, n), dtype=torch.bool, device=DEV)
    fn = model.forward_uint8 if u8 else model.forward
    kw = dict(interpolate_pos_encoding=True) if interp else {}
    want = fn(x, **kw)
    got = fn(x, bool_masked_pos=none, **kw)
    assert torch.equal(got, want), f"all-false mask differs from the unmasked call: {(got.float() - want.float()).abs().max()}"


@pytest.mark.parametrize("mode", ["fold", "ln_before_only", "no_fold", "fp8"])
def test_all_false_mask_equals_unmasked_bit_for_bit(mode):
    from vit import vit as V
    model = _b16(torch.bfloat16)
    try:
        if mode == "ln_before_only":
            V.set_layernorm_folding(True, mlp=False)
        elif mode == "no_fold":
            V.set_layernorm_folding(False)
        elif mode == "fp8":
            V.set_fp8(True)
        x = _pixels(4, 224, 224).to(DEV, torch.bfloat16)
        _all_false_equal(model, x)
        _all_false_equal(model, _pixels(3, 240, 250).to(DEV), interp=True)
        g = torch.Generator().manual_seed(9)
        x8 = torch.randint(0, 256, (3, 224, 224, 3), generator=g, dtype=torch.uint8).to(DEV)
        _all_false_equal(model, x8, u8=True)
        x8 = torch.randint(0, 256, (2, 240, 250, 3), generator=g, dtype=torch.uint8).to(DEV)
        _all_false_equal(model, x8, interp=True, u8=True)
    finally:
        V.set_layernorm_folding(True)
        V.set_fp8(False)


def test_all_false_mask_equals_unmasked_fp32_and_unfused():
    from vit import vit as V
    hf = _hf_model("tiny-b")
    model = _ours(hf, "tiny-b", torch.float32, use_mask_token=True)
    _all_false_equal(model, _pixels(3, 64, 64).to(DEV))
    _all_false_equal(model, _pixels(3, 48, 80).to(DEV), interp=True)
    try:
        V.set_fused(False)
        _all_false_equal(model, _pixels(3, 64, 64).to(DEV))
        _all_false_equal(_b16(torch.bfloat16), _pixels(2, 224, 224).to(DEV, torch.bfloat16))
    finally:
        V.set_fused(True)


# ---------------------------------------------------------------------------------------------------- vs HF ViTModel
@torch.no_grad()
def _vs_hf(model, hf, x, mask, dtype, what, interp=False):
    want = hf(pixel_values=x, bool_masked_pos=mask, interpolate_pos_encoding=interp).last_hidden_state
    got = model(x.to(DEV, dtype), bool_masked_pos=mask.to(DEV), interpolate_pos_encoding=interp)
    _check(got, want, dtype, what)


@pytest.mark.parametrize("kind", ["random", "all_true"])
def test_vit_b16_masked_matches_hf(kind):
    hf = _hf_model("vit-b16-224")
    model = _b16(torch.bfloat16)
    x = _pixels(4, 224, 224)
    mask = _mask(4, 196) if kind == "random" else torch.ones((4, 196), dtype=torch.bool)
    _vs_hf(model, hf, x, mask, torch.bfloat16, f"ViT-B/16 224 {kind}")
    x = _pixels(2, 384, 384, seed=6)
    mask = _mask(2, 576, seed=8) if kind == "random" else torch.ones((2, 576), dtype=torch.bool)
    _vs_hf(model, hf, x, mask, torch.bfloat16, f"ViT-B/16 384 interpolated {kind}", interp=True)


@pytest.mark.parametrize("arch", ["tiny-b", "tiny-h"])
@pytest.mark.parametrize("kind", ["random", "all_true"])
def test_tiny_fp32_masked_matches_hf(arch, kind):
    hf = _hf_model(arch)
    model = _ours(hf, arch, torch.float32, use_mask_token=True)
    size = hf_oracle.ARCHS[arch]["image_size"]
    n = (size // hf_oracle.ARCHS[arch]["patch_size"]) ** 2
    mask = _mask(4, n) if kind == "random" else torch.ones((4, n), dtype=torch.bool)
    _vs_hf(model, hf, _pixels(4, size, size), mask, torch.float32, f"{arch} fp32 {kind}")


def test_unfused_masked_matches_hf():
    from vit import vit as V
    try:
        V.set_fused(False)
        hf = _hf_model("tiny-b")
        model = _ours(hf, "tiny-b", torch.float32, use_mask_token=True)
        _vs_hf(model, hf, _pixels(3, 64, 64), _mask(3, 16), torch.float32, "tiny-b fp32 unfused")
        _vs_hf(_b16(torch.bfloat16), _hf_model("vit-b16-224"), _pixels(2, 224, 224), _mask(2, 196), torch.bfloat16,
               "ViT-B/16 bf16 unfused")
    finally:
        V.set_fused(True)


# ---------------------------------------------------------------------------------------------------- properties
@torch.no_grad()
def test_masked_batch_independence():
    model = _b16(torch.bfloat16)
    x = _pixels(64, 224, 224, seed=12).to(DEV, torch.bfloat16)
    mask = _mask(64, 196, seed=13).to(DEV)
    full = model(x, bool_masked_pos=mask)
    for i in range(64):
        assert torch.equal(model(x[i:i + 1], bool_masked_pos=mask[i:i + 1]), full[i:i + 1]), f"image {i}"


@torch.no_grad()
def test_masked_graph_replay_takes_a_new_mask():
    model = _b16(torch.bfloat16)
    x = _pixels(8, 224, 224, seed=14).to(DEV, torch.bfloat16)
    static_mask = _mask(8, 196, seed=15).to(DEV)
    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):
        for _ in range(2):
            model(x, bool_masked_pos=static_mask)
    torch.cuda.current_stream().wait_stream(side)
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        out = model(x, bool_masked_pos=static_mask)
    new_mask = _mask(8, 196, seed=16).to(DEV)
    static_mask.copy_(new_mask)
    graph.replay()
    torch.cuda.synchronize()
    want = model(x, bool_masked_pos=new_mask)
    assert torch.equal(out, want)
    assert not torch.equal(want, model(x, bool_masked_pos=_mask(8, 196, seed=15).to(DEV)))


@torch.no_grad()
def test_heads_take_the_mask():
    hf = _hf_model("tiny-b", pooling=True)
    model = _ours(hf, "tiny-b", torch.bfloat16, use_mask_token=True, add_pooling_layer=True, num_labels=7)
    with torch.no_grad():
        model.classifier.weight.normal_(0, 0.05)
        model.classifier.bias.normal_(0, 0.05)
    model.invalidate_packed()
    x = _pixels(5, 64, 64).to(DEV, torch.bfloat16)
    mask = _mask(5, 16).to(DEV)
    hidden = model(x, bool_masked_pos=mask)
    assert not torch.equal(hidden, model(x))
    cls = hidden[:, 0].float()
    assert torch.equal(model.pooled(x, bool_masked_pos=mask), hidden[:, 0])
    pool = model.pooler_output(x, bool_masked_pos=mask).float()
    want = torch.tanh(cls @ model.pooler.dense.weight.float() + model.pooler.dense.bias.float())
    assert (pool - want).abs().max().item() <= 2e-2
    hf_pool = hf(pixel_values=x.float().cpu(), bool_masked_pos=mask.cpu()).pooler_output
    _check(pool, hf_pool, torch.bfloat16, "tiny-b pooler_output masked vs HF")
    logits = model.logits(x, bool_masked_pos=mask).float()
    want = cls @ model.classifier.weight.float() + model.classifier.bias.float()
    assert (logits - want).abs().max().item() <= 2e-2


# ---------------------------------------------------------------------------------------------------- vs HF MIM
@torch.no_grad()
def _mim_vs_hf(arch, stride, dtype, batch, with_mask, what):
    hf = _hf_mim(arch, stride)
    model = _ours(hf, arch, dtype, add_decoder=True, encoder_stride=stride)
    size = hf_oracle.ARCHS[arch]["image_size"]
    n = (size // hf_oracle.ARCHS[arch]["patch_size"]) ** 2
    x = _pixels(batch, size, size, seed=21)
    mask = _mask(batch, n, seed=22) if with_mask else None
    want = hf(pixel_values=x, bool_masked_pos=mask)
    loss, rec = model.masked_image_modeling(x.to(DEV, dtype), None if mask is None else mask.to(DEV))
    _check(rec, want.reconstruction, dtype, f"{what} reconstruction")
    if mask is None:
        assert loss is None and want.loss is None
        return
    got, ref = loss.item(), want.loss.item()
    rel = abs(got - ref) / abs(ref)
    print(f"{what} loss {got:.6f} vs HF {ref:.6f}: relative {rel:.2e}")
    assert rel <= (5e-3 if dtype == torch.bfloat16 else 1e-4), f"{what}: loss {got} vs {ref}"


@pytest.mark.parametrize("dtype", [torch.bfloat16, torch.float32])
def test_vit_b16_mim_matches_hf(dtype):
    _mim_vs_hf("vit-b16-224", 16, dtype, 4, True, f"ViT-B/16 MIM {dtype}")
    _mim_vs_hf("vit-b16-224", 16, dtype, 2, False, f"ViT-B/16 MIM {dtype} no mask")


def test_tiny_h_mim_matches_hf():
    _mim_vs_hf("tiny-h", 14, torch.float32, 4, True, "tiny-h MIM stride 14")
    _mim_vs_hf("tiny-h", 16, torch.float32, 4, False, "tiny-h MIM stride 16 (HF default)")


@torch.no_grad()
def test_mim_uint8_loss_matches_normalised_float_input():
    hf = _hf_mim("tiny-b", 16)
    model = _ours(hf, "tiny-b", torch.bfloat16, add_decoder=True)      # uint8 input runs on bf16 models
    g = torch.Generator().manual_seed(23)
    x8 = torch.randint(0, 256, (3, 64, 64, 3), generator=g, dtype=torch.uint8)
    mask = _mask(3, 16, seed=24)
    xf = ((x8.float() / 255.0 - 0.5) / 0.5).permute(0, 3, 1, 2).contiguous()
    want = hf(pixel_values=xf, bool_masked_pos=mask)
    loss, rec = model.masked_image_modeling(x8.to(DEV), mask.to(DEV))
    _check(rec, want.reconstruction, torch.bfloat16, "tiny-b MIM uint8 reconstruction")
    rel = abs(loss.item() - want.loss.item()) / abs(want.loss.item())
    print(f"tiny-b MIM uint8 loss {loss.item():.6f} vs HF {want.loss.item():.6f}: relative {rel:.2e}")
    assert rel <= 5e-3
