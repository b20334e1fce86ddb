"""GPU: running a checkpoint at any input resolution (``interpolate_pos_encoding=True``), against HF ``ViTModel`` called
with the same flag.

Kernels: the bicubic position-table resample against F.interpolate, the rectangular patch gather through the whole
patch embedding against F.conv2d, the square entry point's call against the rectangular one's.  Model: the gates of tests/test_gpu_model.py (bf16
cosine >= 0.999 and max-abs <= 0.15, fp32 <= 1e-3 for ViT-B and <= 1e-4 for the tiny shapes, FP8 cosine >= 0.995 and
max-abs <= 0.5) at non-native sizes, square, rectangular and not divisible by the patch size.  Properties: bit
equality at the native size, batch independence, chunking of very large batches, graph replay (also of graphs whose
grids left the cache), the per-grid cache and its invalidation, the tensor-core attention at every tested token count."""
import functools

import pytest
import torch
import torch.nn.functional as F

from oracle import hf_oracle

pytestmark = pytest.mark.gpu

DEV = "cuda:0"


def _build(arch, dtype, hf=None, **kw):
    from vit.utils import transfer_pretrained_weights
    from vit.vit import VIT
    hf = hf or hf_oracle.build_hf(arch, seed=0)
    model = VIT(**hf_oracle.vit_kwargs(arch), **kw)
    transfer_pretrained_weights(hf, model, verbose=False)
    return model.to(device=DEV, dtype=dtype).eval(), hf


@functools.lru_cache(maxsize=None)
def _hf(arch):
    return hf_oracle.build_hf(arch, seed=0)


@functools.lru_cache(maxsize=None)
def _b16(dtype):
    return _build("vit-b16-224", dtype, _hf("vit-b16-224"))[0]


def _input(batch, h, w, seed=11):
    g = torch.Generator().manual_seed(seed)
    return torch.randn((batch, 3, h, w), generator=g)


@torch.no_grad()
def _hf_interp(hf, x):
    return hf(pixel_values=x, interpolate_pos_encoding=True).last_hidden_state


def _cos(a, b):
    return F.cosine_similarity(a.flatten().float(), b.flatten().float(), dim=0).item()


def _check_bf16(got, want, what=""):
    assert got.shape == want.shape, f"{what}: {tuple(got.shape)} vs {tuple(want.shape)}"
    assert torch.isfinite(got).all()
    cos, err = _cos(got, want), (got - want).abs().max().item()
    assert cos >= 0.999 and err <= 0.15, f"{what}: cosine {cos:.6f} max-abs {err:.4f}"


# ---------------------------------------------------------------------------------------------------- kernels
GRIDS = [(14, 24, 24), (14, 10, 10), (14, 14, 20), (14, 7, 37), (14, 32, 32), (4, 1, 1), (4, 6, 9)]


@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16])
@pytest.mark.parametrize("g_in,gh,gw", GRIDS)
def test_pos_resample_matches_interpolate(g_in, gh, gw, dtype):
    from vit import packing
    g = torch.Generator().manual_seed(g_in * 1000 + gh * 37 + gw)
    D = 200                                                  # not a multiple of the block size
    pos = (torch.randn((1 + g_in * g_in, D), generator=g) * 3.0).to(DEV, dtype)
    got = packing.resample_pos_table(pos, g_in, gh, gw)
    src = pos.float()
    grid = src[1:].reshape(1, g_in, g_in, D).permute(0, 3, 1, 2)
    want = F.interpolate(grid, size=(gh, gw), mode="bicubic", align_corners=False).permute(0, 2, 3, 1).reshape(-1, D)
    assert got.dtype == torch.float32 and got.shape == (1 + gh * gw, D)
    assert torch.equal(got[0], src[0])
    tol = 1e-5 * max(1.0, src.abs().max().item())
    assert (got[1:] - want).abs().max().item() <= tol
    same = packing.resample_pos_table(pos, g_in, g_in, g_in)
    assert torch.equal(same, src), "the same-size resample must reproduce the table exactly"


def _emb_reference(emb, x_f32, hf_table):
    """F.conv2d on the cropped image (bf16-rounded operands, fp32 sums) + CLS + the HF-interpolated table."""
    P = emb.patch_size
    H, W = x_f32.shape[2] // P * P, x_f32.shape[3] // P * P
    xc = x_f32[:, :, :H, :W]
    w = emb.projection.weight.float()
    tok = F.conv2d(xc, w, emb.projection.bias.float(), stride=P).flatten(2).transpose(1, 2)
    cls = emb.cls_token.float().expand(x_f32.shape[0], -1, -1)
    return torch.cat([cls, tok], dim=1) + hf_table.to(x_f32.device)


@pytest.mark.parametrize("hw", [(96, 128), (70, 230), (130, 40)])        # vector path, scalar path (W % 8 != 0), crops
@pytest.mark.parametrize("pix", ["f32", "bf16", "u8"])
def test_rectangular_patch_embedding_matches_conv2d(pix, hw):
    hf = _hf("tiny-b")
    model, _ = _build("tiny-b", torch.bfloat16, hf)
    emb = model.embeddings
    H, W = hw
    P = emb.patch_size
    n = (H // P) * (W // P)
    table = hf.embeddings.interpolate_pos_encoding(torch.zeros(1, 1 + n, emb.hidden_dim), H, W).detach()
    g = torch.Generator().manual_seed(H * W)
    with torch.no_grad():
        if pix == "u8":
            x_u8 = torch.randint(0, 256, (3, H, W, 3), generator=g, dtype=torch.uint8)
            got = emb.forward_uint8(x_u8.to(DEV), interpolate_pos_encoding=True).float()
            x = ((x_u8.float() / 255.0 - 0.5) / 0.5).permute(0, 3, 1, 2).contiguous().to(DEV)
        else:
            x = torch.randn((3, 3, H, W), generator=g).to(DEV, torch.float32 if pix == "f32" else torch.bfloat16)
            got = emb(x, interpolate_pos_encoding=True).float()
            x = x.bfloat16().float()                      # the gather rounds pixels to bf16
        want = _emb_reference(emb, x, table[0])
    assert got.shape == (3, 1 + n, emb.hidden_dim)
    err = (got - want).abs()
    assert (err <= 2e-2 + 1e-2 * want.abs()).all(), f"max-abs {err.max().item():.4f}"


@pytest.mark.parametrize("pix", ["f32", "bf16", "u8"])
@pytest.mark.parametrize("S", [64, 224])
def test_square_entry_point_equals_hw_entry_point(pix, S):
    """Both entry points accept the same square call and agree bit for bit, with and without row statistics.  The
    square entry point forwards to the rectangular one, so this pins the ABI contract only; that its output is
    the same as before rests on the unchanged patch-embedding and model parity tests (test_gpu_kernels.py,
    test_gpu_model.py)."""
    from vit.kernels import _lib
    g = torch.Generator().manual_seed(S)
    P, C, D, B = 16, 3, 256, 3
    K = C * P * P
    n_tok = (S // P) ** 2 + 1
    w = (torch.randn((D, K), generator=g) * 0.03).to(DEV, torch.bfloat16)
    bias = (torch.randn((D,), generator=g) * 0.1).to(DEV)
    posb = (torch.randn((n_tok, D), generator=g) * 0.1).to(DEV, torch.bfloat16)
    if pix == "u8":
        x, code = torch.randint(0, 256, (B, S, S, C), generator=g, dtype=torch.uint8).to(DEV), _lib.VT_U8
    else:
        x = torch.randn((B, C, S, S), generator=g).to(DEV, torch.float32 if pix == "f32" else torch.bfloat16)
        code = _lib.dtype_code(x)
    stream = _lib.stream_ptr(x)
    outs = []
    for name in ("vt_patch_embed_gemm", "vt_patch_embed_gemm_hw"):
        for with_stats in (False, True):
            out = torch.empty((B, n_tok, D), device=DEV, dtype=torch.bfloat16)
            stats = torch.empty((B * n_tok, D // 128, 2), device=DEV) if with_stats else None
            work = torch.empty((B, (n_tok + 31) // 32 * 32, K), device=DEV, dtype=torch.bfloat16)
            size = (S,) if name == "vt_patch_embed_gemm" else (S, S)
            _lib.call(name, x.data_ptr(), code, w.data_ptr(), K, bias.data_ptr(), posb.data_ptr(), out.data_ptr(),
                      _lib.ptr(stats), work.data_ptr(), B, C, *size, P, D, stream)
            outs.append((out, stats))
    torch.cuda.synchronize()
    assert torch.equal(outs[0][0], outs[2][0]) and torch.equal(outs[1][0], outs[3][0])
    assert torch.equal(outs[1][1], outs[3][1])


# ---------------------------------------------------------------------------------------------------- model vs HF
B16_SIZES = [(384, 384), (160, 160), (224, 384), (240, 250), (512, 512)]


@pytest.mark.parametrize("hw", B16_SIZES)
def test_vit_b16_224_bf16_at_other_resolutions_matches_hf(hw):
    model = _b16(torch.bfloat16)
    x = _input(2, *hw)
    want = _hf_interp(_hf("vit-b16-224"), x)
    with torch.no_grad():
        got = model(x.to(DEV, torch.bfloat16), interpolate_pos_encoding=True).float().cpu()
    _check_bf16(got, want, f"{hw}")
    for i in range(2):
        assert _cos(got[i], want[i]) >= 0.999


def test_vit_b16_224_fp32_batch1_384x256_matches_hf():
    model = _b16(torch.float32)
    x = _input(1, 384, 256)
    want = _hf_interp(_hf("vit-b16-224"), x)
    with torch.no_grad():
        got = model(x.to(DEV), interpolate_pos_encoding=True).cpu()
    assert got.shape == want.shape == (1, 385, 768)
    assert (got - want).abs().max().item() <= 1e-3


@pytest.mark.parametrize("arch,hw", [("tiny-b", (48, 80)), ("tiny-b", (100, 70)),
                                     ("tiny-h", (42, 70)), ("tiny-h", (90, 60))])
def test_tiny_fp32_at_other_resolutions_matches_hf(arch, hw):
    """dh 64 and P = 16 (tiny-b), dh 80 and P = 14 (tiny-h)."""
    model, hf = _build(arch, torch.float32, _hf(arch))
    x = _input(2, *hw)
    want = _hf_interp(hf, x)
    with torch.no_grad():
        got = model(x.to(DEV), interpolate_pos_encoding=True).cpu()
    assert got.shape == want.shape
    assert (got - want).abs().max().item() <= 1e-4


def test_layernorm_fold_off_matches_hf():
    from vit import vit as vit_mod
    model = _b16(torch.bfloat16)
    x = _input(2, 224, 384)
    want = _hf_interp(_hf("vit-b16-224"), x)
    vit_mod.set_layernorm_folding(False)
    try:
        with torch.no_grad():
            got = model(x.to(DEV, torch.bfloat16), interpolate_pos_encoding=True).float().cpu()
    finally:
        vit_mod.set_layernorm_folding(True)
    _check_bf16(got, want, "fold off")


def test_fp8_path_matches_hf():
    from vit import vit as vit_mod
    model = _b16(torch.bfloat16)
    x = _input(2, 288, 512)
    want = _hf_interp(_hf("vit-b16-224"), x)
    before = vit_mod.fp8_enabled()
    vit_mod.set_fp8(True)
    try:
        with torch.no_grad():
            got = model(x.to(DEV, torch.bfloat16), interpolate_pos_encoding=True).float().cpu()
    finally:
        vit_mod.set_fp8(before)
    assert got.shape == want.shape and torch.isfinite(got).all()
    cos, err = _cos(got, want), (got - want).abs().max().item()
    assert cos >= 0.995 and err <= 0.5, f"cosine {cos:.6f} max-abs {err:.4f}"


def test_uint8_nhwc_256x384_matches_hf_image_processor():
    import numpy as np
    from transformers import ViTImageProcessor
    model = _b16(torch.bfloat16)
    g = torch.Generator().manual_seed(7)
    x_u8 = torch.randint(0, 256, (2, 256, 384, 3), generator=g, dtype=torch.uint8)
    proc = ViTImageProcessor(do_resize=False)
    pixel_values = proc(images=list(np.asarray(x_u8)), return_tensors="pt")["pixel_values"]
    assert pixel_values.shape == (2, 3, 256, 384)
    want = _hf_interp(_hf("vit-b16-224"), pixel_values)
    with torch.no_grad():
        got = model.forward_uint8(x_u8.to(DEV), interpolate_pos_encoding=True).float().cpu()
        pooled = model.pooled(x_u8.to(DEV), interpolate_pos_encoding=True).float().cpu()
    _check_bf16(got, want, "uint8 256x384")
    assert torch.equal(pooled, got[:, 0, :])


def test_pooler_and_logits_heads_match_hf():
    from transformers import ViTConfig, ViTForImageClassification, ViTModel
    from vit.utils import transfer_pretrained_weights
    from vit.vit import VIT
    arch = "tiny-b"
    x = _input(3, 80, 112)
    torch.manual_seed(3)
    hf = ViTModel(ViTConfig(**hf_oracle.ARCHS[arch]), add_pooling_layer=True).eval()
    torch.manual_seed(5)
    hfc = ViTForImageClassification(ViTConfig(**hf_oracle.ARCHS[arch], num_labels=40)).eval()
    with torch.no_grad():
        hf.pooler.dense.bias.copy_(torch.randn_like(hf.pooler.dense.bias) * 0.1)
        hfc.classifier.weight.copy_(torch.randn_like(hfc.classifier.weight) * 0.1)
        hfc.classifier.bias.copy_(torch.randn_like(hfc.classifier.bias) * 0.1)
        want_pool = hf(pixel_values=x, interpolate_pos_encoding=True).pooler_output
        want_logits = hfc(pixel_values=x, interpolate_pos_encoding=True).logits
    for dtype, tol_p, tol_l in ((torch.float32, 1e-4, 1e-4), (torch.bfloat16, 3e-2, 5e-2)):
        mp = VIT(**hf_oracle.vit_kwargs(arch), add_pooling_layer=True)
        transfer_pretrained_weights(hf, mp, verbose=False)
        mc = VIT(**hf_oracle.vit_kwargs(arch), num_labels=40)
        transfer_pretrained_weights(hfc, mc, verbose=False)
        mp, mc = mp.to(DEV, dtype).eval(), mc.to(DEV, dtype).eval()
        with torch.no_grad():
            got_pool = mp.pooler_output(x.to(DEV, dtype), interpolate_pos_encoding=True).float().cpu()
            got_logits = mc.logits(x.to(DEV, dtype), interpolate_pos_encoding=True).float().cpu()
        assert (got_pool - want_pool).abs().max().item() <= tol_p, f"{dtype} pooler"
        assert got_logits.shape == (3, 40) and (got_logits - want_logits).abs().max().item() <= tol_l, f"{dtype} logits"


# ---------------------------------------------------------------------------------------------------- properties
@pytest.mark.parametrize("arch,dtype", [("vit-b16-224", torch.bfloat16), ("tiny-b", torch.float32),
                                        ("vit-b16-224", torch.float32)])
def test_native_size_with_the_flag_is_bit_identical(arch, dtype):
    model = _b16(dtype) if arch == "vit-b16-224" else _build(arch, dtype, _hf(arch))[0]
    x = hf_oracle.make_input(arch, 2).to(DEV, dtype)
    with torch.no_grad():
        plain = model(x)
        interp = model(x, interpolate_pos_encoding=True)
    assert torch.equal(plain, interp)
    assert model.embeddings.interpolate_pos_encoding(x.shape[2], x.shape[3]) is model.embeddings.position_embeddings


def test_batch_independence_288x512():
    model = _b16(torch.bfloat16)
    x = _input(64, 288, 512, seed=5).to(DEV, torch.bfloat16)
    with torch.no_grad():
        full = model(x, interpolate_pos_encoding=True)
        for lo in (0, 30, 60):
            part = model(x[lo:lo + 4].contiguous(), interpolate_pos_encoding=True)
            assert torch.equal(full[lo:lo + 4], part), f"images {lo}..{lo + 3} differ between batch 64 and batch 4"


def test_cuda_graph_replay_equals_eager_224x384():
    from vit.utils import capture_cuda_graph
    model = _b16(torch.bfloat16)
    model.invalidate_packed()                   # the graph's warm-up builds the 14 x 24 tables
    x = _input(4, 224, 384).to(DEV, torch.bfloat16)
    static_in = torch.zeros_like(x)
    graph, static_out = capture_cuda_graph(functools.partial(model, interpolate_pos_encoding=True), static_in)
    static_in.copy_(x)
    graph.replay()
    torch.cuda.synchronize()
    with torch.no_grad():
        eager = model(x, interpolate_pos_encoding=True)
    assert torch.equal(static_out, eager)


def test_graphs_at_more_resolutions_than_the_cache_keeps_stay_valid():
    """A captured graph reads its grid's tables through raw addresses: they must outlive the grid's eviction from the
    cache.  Graphs at more grids than the cache keeps, then eager forwards at further grids (every captured grid is
    evicted and its memory would be reused), then every graph is replayed against its eager output."""
    from vit import packing
    from vit.utils import capture_cuda_graph
    model, _ = _build("tiny-b", torch.bfloat16, _hf("tiny-b"))          # native grid 4 x 4 (64 x 64)
    fn = functools.partial(model, interpolate_pos_encoding=True)
    sizes = [(48, 48), (48, 80), (80, 48), (96, 96), (32, 112), (112, 64)]
    assert len(sizes) > packing.POS_GRIDS_KEPT
    graphs = []
    for i, hw in enumerate(sizes):
        x = _input(2, *hw, seed=20 + i).to(DEV, torch.bfloat16)
        static_in = torch.zeros_like(x)
        graph, static_out = capture_cuda_graph(fn, static_in)
        with torch.no_grad():
            want = model(x, interpolate_pos_encoding=True).clone()
        graphs.append((hw, graph, static_in, x, static_out, want))
    with torch.no_grad():
        for i, hw in enumerate([(32, 128), (48, 112), (80, 96), (96, 80), (112, 48), (128, 32)]):
            model(_input(2, *hw, seed=40 + i).to(DEV, torch.bfloat16), interpolate_pos_encoding=True)
    assert not set(model.embeddings.__dict__["_pos_grids"]) & {packing.patch_grid(model.embeddings, *hw) for hw in sizes}
    for hw, graph, static_in, x, static_out, want in graphs:
        static_in.copy_(x)
        graph.replay()
        torch.cuda.synchronize()
        assert torch.equal(static_out, want), f"graph captured at {hw} no longer equals eager"


def test_large_batch_at_a_small_grid_is_chunked():
    """More than 65535 images at a 2 x 2 grid: the patch embedding runs in chunks of at most 65535 images."""
    model, _ = _build("tiny-b", torch.bfloat16, _hf("tiny-b"))
    g = torch.Generator().manual_seed(9)
    x = torch.randn((65536 + 100, 3, 32, 40), generator=g).to(DEV, torch.bfloat16)
    with torch.no_grad():
        full = model(x, interpolate_pos_encoding=True)
        for lo in (0, 65532, 65536 + 96):
            part = model(x[lo:lo + 4].contiguous(), interpolate_pos_encoding=True)
            assert torch.equal(full[lo:lo + 4], part), f"images {lo}..{lo + 3} differ"


def test_alternating_resolutions_use_the_right_tables():
    from vit import packing
    model = _b16(torch.bfloat16)
    x384 = _input(2, 384, 384).to(DEV, torch.bfloat16)
    x224 = hf_oracle.make_input("vit-b16-224", 2).to(DEV, torch.bfloat16)
    with torch.no_grad():
        a = model(x384, interpolate_pos_encoding=True).clone()
        b = model(x224, interpolate_pos_encoding=True).clone()
        c = model(x384, interpolate_pos_encoding=True).clone()
        # more grids than the cache keeps, then back to 384
        for s in (160, 192, 256, 288, 320, 352):
            model(_input(1, s, s).to(DEV, torch.bfloat16), interpolate_pos_encoding=True)
        assert len(model.embeddings.__dict__["_pos_grids"]) <= packing.POS_GRIDS_KEPT
        d = model(x384, interpolate_pos_encoding=True)
        plain = model(x224)
    assert a.shape == (2, 577, 768) and b.shape == (2, 197, 768)
    assert torch.equal(a, c) and torch.equal(a, d)
    assert torch.equal(b, plain)


def test_parameter_changes_reach_the_interpolated_tables():
    """An in-place change of the position table (version bump) and a load_state_dict are both seen."""
    from vit.utils import transfer_pretrained_weights
    hf = hf_oracle.build_hf("tiny-b", seed=0)
    model, _ = _build("tiny-b", torch.bfloat16, hf)
    x = _input(2, 80, 48)
    with torch.no_grad():
        _check_bf16(model(x.to(DEV, torch.bfloat16), interpolate_pos_encoding=True).float().cpu(), _hf_interp(hf, x),
                    "before")
        hf.embeddings.position_embeddings.mul_(-2.0)
        model.embeddings.position_embeddings.mul_(-2.0)
        _check_bf16(model(x.to(DEV, torch.bfloat16), interpolate_pos_encoding=True).float().cpu(), _hf_interp(hf, x),
                    "after an in-place change")
        hf2 = hf_oracle.build_hf("tiny-b", seed=4)
        transfer_pretrained_weights(hf2, model, verbose=False)
        _check_bf16(model(x.to(DEV, torch.bfloat16), interpolate_pos_encoding=True).float().cpu(), _hf_interp(hf2, x),
                    "after load_state_dict")


@pytest.mark.parametrize("hw,tokens", [((160, 160), 101), ((240, 250), 226), ((224, 384), 337), ((384, 256), 385),
                                       ((384, 384), 577), ((288, 512), 577), ((512, 512), 1025)])
def test_attention_stays_on_the_tensor_core_kernel(hw, tokens):
    from vit.kernels import _lib
    model = _b16(torch.bfloat16)
    x = _input(1, *hw).to(DEV, torch.bfloat16)
    names = []
    _lib.event_hook = lambda name, before, args: names.append(name) if before else None
    try:
        with torch.no_grad():
            out = model(x, interpolate_pos_encoding=True)
    finally:
        _lib.event_hook = None
    assert out.shape == (1, tokens, 768)
    assert names.count("vt_flash_attn") == 12
    assert "vt_softmax" not in names and "vt_bgemm" not in names, names


def test_data_parallel_wrapper_passes_the_flag():
    from vit.parallel import DataParallelVIT
    model = _b16(torch.bfloat16)
    x = _input(3, 224, 320).to(DEV, torch.bfloat16)
    dp = DataParallelVIT(model, interpolate_pos_encoding=True)
    assert dp.world_size == 1
    with torch.no_grad():
        got = dp(x)
        want = model.pooled(x, interpolate_pos_encoding=True)
    assert torch.equal(got, want)
