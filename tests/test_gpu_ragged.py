"""GPU: images of different resolutions in one batch (``VIT.forward_ragged``, list inputs of ``pooled`` /
``pooler_output`` / ``logits``).

Kernels: the ragged patch gather against a torch restatement (F.unfold on the cropped image, the position rows), bit
for bit, into NaN-filled buffers with guard rows, with an unaligned image and an unaligned position table; the
row gather.  Embedding: every image's embeddings and row
statistics equal its own ``interpolate_pos_encoding=True`` patch embedding bit for bit.  Model: the ragged forward of
ViT-B/16@224 in bf16 equals one ``model(x[None], interpolate_pos_encoding=True)`` call per image bit for bit, with the
LayerNorm fold on, with only ``layernorm_before`` folded, with the fold off, with FP8, and from uint8 pixels through the
heads; the list holds the native grid, a one-patch image, 240x250, 384x256, 512x512 (1025 tokens, the multi-block
attention kernel), grids repeated apart from each other, more grids than the position-table cache keeps, and enough
rows for many GEMM tiles.  HF ``ViTModel(interpolate_pos_encoding=True)`` per image at the gates of
tests/test_gpu_model.py (bf16 cosine >= 0.999 and max-abs <= 0.15, fp32 <= 1e-3); fp32 and unfused lists equal
per-image calls."""
import functools

import pytest
import torch
import torch.nn.functional as F

from oracle import hf_oracle

pytestmark = pytest.mark.gpu

DEV = "cuda:0"

# 12 images, 8 distinct grids (more than packing.POS_GRIDS_KEPT), (224, 224) / (240, 250) / (384, 256) repeated apart
SIZES = [(224, 224), (16, 16), (240, 250), (384, 256), (512, 512), (160, 160), (224, 224), (96, 320), (240, 250),
         (20, 31), (384, 256), (128, 128)]


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


@functools.lru_cache(maxsize=None)
def _b16_heads():
    """ViT-B/16 bf16 with a pooler and a 40-class classifier (random head weights)."""
    from vit.utils import transfer_pretrained_weights
    from vit.vit import VIT
    model = VIT(**hf_oracle.vit_kwargs("vit-b16-224"), add_pooling_layer=True, num_labels=40)
    transfer_pretrained_weights(_hf("vit-b16-224"), model, verbose=False)
    g = torch.Generator().manual_seed(9)
    with torch.no_grad():
        for p in (model.pooler.dense.weight, model.pooler.dense.bias, model.classifier.weight, model.classifier.bias):
            p.copy_(torch.randn(p.shape, generator=g) * 0.05)
    return model.to(device=DEV, dtype=torch.bfloat16).eval()


def _images(sizes, dtype=torch.float32, seed=3, repeat=1):
    g = torch.Generator().manual_seed(seed)
    out = []
    for _ in range(repeat):
        for h, w in sizes:
            if dtype == torch.uint8:
                out.append(torch.randint(0, 256, (h, w, 3), generator=g, dtype=torch.uint8).to(DEV))
            else:
                out.append(torch.randn((3, h, w), generator=g).to(DEV, dtype))
    return out


def _per_image(model, images, **kw):
    with torch.no_grad():
        if images[0].dtype == torch.uint8:
            return [model.forward_uint8(x[None], interpolate_pos_encoding=True, **kw)[0] for x in images]
        return [model(x[None], interpolate_pos_encoding=True)[0] for x in images]


def _assert_equal_lists(got, want, what):
    assert len(got) == len(want)
    for i, (a, b) in enumerate(zip(got, want)):
        assert a.shape == b.shape, f"{what}: image {i} {tuple(a.shape)} vs {tuple(b.shape)}"
        if not torch.equal(a, b):
            bad = (a.float() - b.float()).abs()
            raise AssertionError(f"{what}: image {i} ({tuple(a.shape)}) differs from its own call: "
                                 f"{int((bad > 0).sum())} elements, max {bad.max().item():.3g}")


def _cos(a, b):
    return F.cosine_similarity(a.flatten().float(), b.flatten().float(), dim=0).item()


# ---------------------------------------------------------------------------------------------------- kernels
def _gather_reference(img, P, u8):
    """bf16 [n, K] patch rows of one image: (c, i, j) order via F.unfold for NCHW, (i, j, c) for NHWC."""
    if u8:
        H, W, C = img.shape
        gh, gw = H // P, W // P
        x = img[:gh * P, :gw * P].float().reshape(gh, P, gw, P, C).permute(0, 2, 1, 3, 4).reshape(gh * gw, P * P * C)
    else:
        C, H, W = img.shape
        gh, gw = H // P, W // P
        x = F.unfold(img[:, :gh * P, :gw * P].float()[None], P, stride=P)[0].t()
    return x.to(torch.bfloat16)


@pytest.mark.parametrize("pix", ["f32", "bf16", "u8"])
def test_ragged_gather_matches_unfold_and_position_rows(pix):
    from vit import packing
    from vit.kernels import _lib
    P, C, D, guard = 16, 3, 136, 5
    K = C * P * P
    ldw = K + 16                                              # zero padding columns past K
    sizes = [(32, 48), (70, 37), (16, 16), (50, 64), (33, 21), (64, 40)]   # odd W: the scalar loads
    g = torch.Generator().manual_seed(len(pix))
    imgs, tables, keep = [], [], []
    for n, (h, w) in enumerate(sizes):
        if pix == "u8":
            img = torch.randint(0, 256, (h, w, C), generator=g, dtype=torch.uint8).to(DEV)
        else:
            dt = torch.float32 if pix == "f32" else torch.bfloat16
            img = torch.randn((C, h, w), generator=g).to(DEV, dt)
            if n == 3:                                        # an image at an address that is not 16-byte aligned
                flat = torch.empty((img.numel() + 1,), device=DEV, dtype=dt)
                flat[1:].copy_(img.flatten())
                keep.append(flat)
                img = flat[1:].view(C, h, w)
        imgs.append(img)
        table = (torch.randn((1 + (h // P) * (w // P), D), generator=g) * 0.1).to(DEV, torch.bfloat16)
        if n == 4:                                            # a position table that is not 16-byte aligned
            flat = torch.empty((table.numel() + 1,), device=DEV, dtype=torch.bfloat16)
            flat[1:].copy_(table.flatten())
            keep.append(flat)
            table = flat[1:].view(table.shape)
        tables.append(table)
    layout = packing.RaggedLayout([(h // P, w // P) for h, w in sizes])
    # caller order on purpose (not layout.order): the kernel only needs consecutive row ranges
    row0, rows = [], 0
    for t in layout.tokens:
        row0.append(rows)
        rows += t
    desc = (_lib.RaggedImage * len(imgs))()
    for i, (im, (h, w)) in enumerate(zip(imgs, sizes)):
        desc[i] = _lib.RaggedImage(im.data_ptr(), tables[i].data_ptr(), row0[i], h, w, layout.tokens[i], 0)
    desc_dev = torch.frombuffer(bytearray(bytes(desc)), dtype=torch.uint8).to(DEV)
    patches = torch.full((rows + 2 * guard, ldw), float("nan"), device=DEV, dtype=torch.bfloat16)
    table = torch.full((rows + 2 * guard, D), float("nan"), device=DEV, dtype=torch.bfloat16)
    code = _lib.VT_U8 if pix == "u8" else _lib.dtype_code(imgs[0])
    _lib.call("vt_patch_embed_ragged_gather", desc_dev.data_ptr(), len(imgs), code, C, P, patches[guard:].data_ptr(),
              ldw, table[guard:].data_ptr(), D, rows, _lib.stream_ptr(patches))
    torch.cuda.synchronize()
    assert torch.isnan(patches[:guard]).all() and torch.isnan(patches[guard + rows:]).all()
    assert torch.isnan(table[:guard]).all() and torch.isnan(table[guard + rows:]).all()
    for i, im in enumerate(imgs):
        r = guard + row0[i]
        n = layout.tokens[i]
        want = torch.zeros((n, ldw), device=DEV, dtype=torch.bfloat16)
        want[1:, :K] = _gather_reference(im, P, pix == "u8")
        assert torch.equal(patches[r:r + n], want), f"image {i} {tuple(im.shape)}: patch rows differ"
        assert torch.equal(table[r:r + n], tables[i]), f"image {i}: position rows differ"


@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16])
def test_gather_rows(dtype):
    from vit import packing
    g = torch.Generator().manual_seed(1)
    x = torch.randn((700, 200), generator=g).to(DEV, dtype)
    rows = [5, 0, 699, 5, 311, 42]
    got = packing.gather_rows(x, rows)
    assert torch.equal(got, x[rows])


@pytest.mark.parametrize("u8", [False, True])
@pytest.mark.parametrize("with_stats", [False, True])
def test_ragged_embedding_equals_each_images_own_call(u8, with_stats):
    """Embeddings and row statistics of every image: the ragged gather + plain GEMM with the per-row table as residual
    against the gather + token-mode GEMM of the image's own call, bit for bit."""
    from vit import packing
    model = _b16(torch.bfloat16)
    emb = model.embeddings
    D = emb.hidden_dim
    imgs = _images(SIZES, torch.uint8 if u8 else torch.float32, seed=4)
    grids, _ = packing.check_ragged(emb, imgs)
    layout = packing.RaggedLayout(grids)
    stats = torch.full((layout.rows, D // 128, 2), float("nan"), device=DEV) if with_stats else None
    with torch.no_grad():
        packed = packing.patch_embed_ragged(emb, imgs, layout, stats, u8)[0]
        for i, x in enumerate(imgs):
            n = layout.tokens[i]
            own_stats = torch.full((n, D // 128, 2), float("nan"), device=DEV) if with_stats else None
            if u8:
                own = emb.forward_uint8(x[None], stats_out=own_stats, interpolate_pos_encoding=True)[0]
            else:
                own = emb(x[None], own_stats, interpolate_pos_encoding=True)[0]
            r = layout.row0[i]
            assert torch.equal(packed[r:r + n], own), f"image {i} {tuple(x.shape)}: embeddings differ"
            if with_stats:
                assert torch.equal(stats[r:r + n], own_stats), f"image {i}: row statistics differ"


# ---------------------------------------------------------------------------------------------------- model
def _fold_mode(mode):
    from vit import vit as vit_mod
    if mode == "fold":
        vit_mod.set_layernorm_folding(True)
    elif mode == "fold_ln_before":
        vit_mod.set_layernorm_folding(True, mlp=False)
    elif mode == "no_fold":
        vit_mod.set_layernorm_folding(False)
    vit_mod.set_fp8(mode == "fp8")


@pytest.mark.parametrize("mode,pix", [("fold", torch.float32), ("fold", torch.bfloat16),
                                      ("fold_ln_before", torch.bfloat16), ("no_fold", torch.bfloat16),
                                      ("fp8", torch.bfloat16)])
def test_ragged_forward_equals_per_image_calls(mode, pix):
    from vit import packing
    from vit import vit as vit_mod
    model = _b16(torch.bfloat16)
    imgs = _images(SIZES, pix, seed=5, repeat=2)                     # 24 images, M = 5864 rows
    fp8_before = vit_mod.fp8_enabled()
    try:
        _fold_mode(mode)
        with torch.no_grad():
            got = model.forward_ragged(imgs)
        want = _per_image(model, imgs)
    finally:
        vit_mod.set_layernorm_folding(True)
        vit_mod.set_fp8(fp8_before)
    assert len(got) == len(imgs) and sum(t.shape[0] for t in got) == 5864
    assert len({t.untyped_storage().data_ptr() for t in got}) == 1, "views into one packed buffer"
    assert len({packing.patch_grid(model.embeddings, x.shape[1], x.shape[2]) for x in imgs}) > packing.POS_GRIDS_KEPT
    _assert_equal_lists(got, want, mode)
    assert got[4].shape == (1025, 768) and got[1].shape == (2, 768)


def test_ragged_uint8_through_the_heads_equals_per_image_calls():
    model = _b16_heads()
    imgs = _images(SIZES, torch.uint8, seed=6)
    mean, std = (0.485, 0.456, 0.406), (0.229, 0.224, 0.225)
    with torch.no_grad():
        hidden = model.forward_ragged(imgs, image_mean=mean, image_std=std)
        want_hidden = _per_image(model, imgs, image_mean=mean, image_std=std)
        pooled = model.pooled(imgs)
        pooler = model.pooler_output(imgs)
        logits = model.logits(imgs)
        want_pooled = [model.pooled(x[None], interpolate_pos_encoding=True)[0] for x in imgs]
        want_pooler = [model.pooler_output(x[None], interpolate_pos_encoding=True)[0] for x in imgs]
        want_logits = [model.logits(x[None], interpolate_pos_encoding=True)[0] for x in imgs]
    _assert_equal_lists(hidden, want_hidden, "uint8 hidden states")
    assert pooled.shape == (len(imgs), 768) and pooler.shape == (len(imgs), 768) and logits.shape == (len(imgs), 40)
    _assert_equal_lists(list(pooled), want_pooled, "pooled")
    _assert_equal_lists(list(pooler), want_pooler, "pooler_output")
    _assert_equal_lists(list(logits), want_logits, "logits")


HF_SIZES = [(224, 224), (240, 250), (16, 16), (384, 256), (96, 320)]


@torch.no_grad()
def _hf_per_image(images):
    hf = _hf("vit-b16-224")
    return [hf(pixel_values=x[None].float().cpu(), interpolate_pos_encoding=True).last_hidden_state[0] for x in images]


def test_ragged_bf16_matches_hf_per_image():
    imgs = _images(HF_SIZES, torch.float32, seed=7)
    want = _hf_per_image(imgs)
    with torch.no_grad():
        got = _b16(torch.bfloat16).forward_ragged([x.bfloat16() for x in imgs])
    for i, (a, b) in enumerate(zip(got, want)):
        a = a.float().cpu()
        assert a.shape == b.shape and torch.isfinite(a).all()
        cos, err = _cos(a, b), (a - b).abs().max().item()
        assert cos >= 0.999 and err <= 0.15, f"image {i} {HF_SIZES[i]}: cosine {cos:.6f} max-abs {err:.4f}"


def test_ragged_fp32_matches_hf_and_per_image_calls():
    model = _b16(torch.float32)
    imgs = _images(HF_SIZES, torch.float32, seed=8)
    want = _hf_per_image(imgs)
    with torch.no_grad():
        got = model.forward_ragged(imgs)
        pooled = model.pooled(imgs)
    _assert_equal_lists(got, _per_image(model, imgs), "fp32")
    for i, (a, b) in enumerate(zip(got, want)):
        assert a.dtype == torch.float32 and (a.cpu() - b).abs().max().item() <= 1e-3, f"image {i} {HF_SIZES[i]}"
    assert torch.equal(pooled, torch.stack([h[0] for h in got]))


def test_ragged_unfused_equals_per_image_calls():
    from vit import vit as vit_mod
    model, _ = _build("tiny-b", torch.bfloat16, _hf("tiny-b"))
    imgs = _images([(64, 64), (48, 80), (16, 16), (100, 70), (48, 80)], torch.bfloat16, seed=9)
    vit_mod.set_fused(False)
    try:
        with torch.no_grad():
            got = model.forward_ragged(imgs)
        want = _per_image(model, imgs)
    finally:
        vit_mod.set_fused(True)
    _assert_equal_lists(got, want, "unfused")


def test_repeating_a_list_of_many_grids_resamples_nothing():
    """A list with more non-native grids than ``packing.POS_GRIDS_KEPT`` keeps all of them cached: the second call of the
    same list launches no ``vt_pos_embed_resample``, and still gives the same result."""
    from vit import packing
    from vit.kernels import _lib
    model = _b16(torch.bfloat16)
    model.embeddings.invalidate_packed()
    sizes = [(240, 250), (384, 256), (160, 160), (96, 320), (128, 128), (288, 224), (224, 224)]
    imgs = _images(sizes, torch.bfloat16, seed=10)
    assert len({(h // 16, w // 16) for h, w in sizes} - {(14, 14)}) > packing.POS_GRIDS_KEPT
    names = []
    hook_before = _lib.event_hook
    _lib.event_hook = lambda name, before, args: names.append(name) if before else None
    try:
        with torch.no_grad():
            first = model.forward_ragged(imgs)
            n_first = names.count("vt_pos_embed_resample")
            names.clear()
            second = model.forward_ragged(imgs)
    finally:
        _lib.event_hook = hook_before
    assert n_first == 6 and names.count("vt_pos_embed_resample") == 0
    _assert_equal_lists(second, [t.clone() for t in first], "second call")
