"""GPU: ``resize_uint8`` (vt_resize_u8 / vt_resize_u8_list) against PIL.Image.resize byte for byte, and
``do_resize=True`` on ``forward_uint8`` and the heads against the same calls on PIL-resized images, bit for bit.

The expected bytes are PIL 12's: BILINEAR / BICUBIC of L (C = 1) and RGB (C = 3) images.  Model-level results are also
compared with HF's default ViTImageProcessor (torchvision backend, which differs from PIL by a grey level on a fraction
of a percent of the values) and ViTImageProcessorPil + ViTModel / ViTForImageClassification on the CPU."""
import functools

import numpy as np
import pytest
import torch
import torch.nn.functional as F
from PIL import Image

from oracle import hf_oracle

pytestmark = pytest.mark.gpu

DEV = "cuda:0"
S = 224
SIZES = [(1, 1), (1, 300), (300, 1), (16, 16), (8000, 60), (97, 1201), (375, 500), (223, 225), (224, 100),
         (224, 224), (17, 300), (1000, 37)]


def _pil(img: np.ndarray, oh: int, ow: int, resample: int) -> np.ndarray:
    """(H, W, C) uint8 -> PIL.Image.resize to (oh, ow), (oh, ow, C)."""
    C = img.shape[2]
    out = np.asarray(Image.fromarray(img[..., 0] if C == 1 else img, "L" if C == 1 else "RGB").resize((ow, oh), resample))
    return out.reshape(oh, ow, C)


def _images(rng, sizes, C):
    return [rng.integers(0, 256, (h, w, C), dtype=np.uint8) for h, w in sizes]


def _check(got: torch.Tensor, imgs, oh, ow, resample):
    got = got.cpu().numpy()
    assert got.shape == (len(imgs), oh, ow, imgs[0].shape[2])
    for i, img in enumerate(imgs):
        want = _pil(img, oh, ow, resample)
        if not np.array_equal(got[i], want):
            bad = np.argwhere(got[i] != want)
            pytest.fail(f"image {i} {img.shape[:2]} -> {(oh, ow)} resample {resample}: {len(bad)} bytes differ, "
                        f"first at {bad[0].tolist()}: {got[i][tuple(bad[0])]} vs {want[tuple(bad[0])]}")


@pytest.mark.parametrize("resample", [2, 3])
@pytest.mark.parametrize("C", [1, 3])
def test_batch_and_list_equal_pil(resample, C):
    from vit.kernels import resize_uint8
    rng = np.random.default_rng(10 * resample + C)
    for h, w in SIZES:
        imgs = _images(rng, [(h, w)] * 2, C)
        x = torch.from_numpy(np.stack(imgs)).to(DEV)
        got = resize_uint8(x, S, S, resample)
        if (h, w) == (S, S):
            assert got is x                                # PIL's copy: nothing launched
        _check(got, imgs, S, S, resample)
    for oh, ow in [(S, S), (384, 300), (7, 513), (1, 1)]:
        imgs = _images(rng, SIZES, C)
        got = resize_uint8([torch.from_numpy(i).to(DEV) for i in imgs], oh, ow, resample)
        _check(got, imgs, oh, ow, resample)


def test_strided_batches_and_other_output_sizes():
    from vit.kernels import resize_uint8
    rng = np.random.default_rng(3)
    base = torch.from_numpy(rng.integers(0, 256, (3, 301, 403, 3), dtype=np.uint8)).to(DEV)
    views = [base[:, 1:, 2:], base[::2], base[:1], base.permute(0, 2, 1, 3)]
    for v in views:
        for oh, ow in [(S, S), (100, 500), (301, 97)]:
            imgs = list(v.cpu().numpy())
            _check(resize_uint8(v, oh, ow, 3), imgs, oh, ow, 3)


def test_thousand_random_sizes_in_one_list():
    from vit.kernels import resize_uint8
    rng = np.random.default_rng(11)
    sizes = [(int(rng.integers(1, 700)), int(rng.integers(1, 700))) for _ in range(1000)]
    imgs = _images(rng, sizes, 3)
    dev = [torch.from_numpy(i).to(DEV) for i in imgs]
    for resample in (2, 3):
        got = resize_uint8(dev, S, S, resample)
        _check(got, imgs, S, S, resample)
        assert torch.equal(resize_uint8(dev, S, S, resample), got)          # same bits on a second call


def test_batch_past_two_gigabytes():
    """41 images of 4000 x 4500 x 3: the last one starts 2.16 GB into the batch (64-bit pixel offsets)."""
    from vit.kernels import resize_uint8
    rng = np.random.default_rng(5)
    first, last = _images(rng, [(4000, 4500)] * 2, 3)
    x = torch.empty((41, 4000, 4500, 3), dtype=torch.uint8, device=DEV)
    assert x[40].data_ptr() - x.data_ptr() > 2 ** 31
    x[0].copy_(torch.from_numpy(first))
    x[40].copy_(torch.from_numpy(last))
    for resample in (2, 3):
        got = resize_uint8(x, S, S, resample)
        _check(got[[0, 40]], [first, last], S, S, resample)
    lst = resize_uint8([x[40], x[0]], S, S, 2)
    _check(lst, [last, first], S, S, 2)
    del x
    torch.cuda.empty_cache()


def test_guard_bytes_around_the_output(monkeypatch):
    """Both entry points write exactly the (B, out_h, out_w, C) output: the kernel's output pointer is redirected into a
    buffer with sentinel bytes in front and behind."""
    from vit.kernels import _lib, resize_uint8
    guard = 4096
    real = _lib.call
    seen = {}

    def redirect(name, *args):
        args = list(args)
        pos = {"vt_resize_u8": 10, "vt_resize_u8_list": 4}[name]
        n = seen["bytes"]
        buf = torch.full((n + 2 * guard + 1,), 0xA5, dtype=torch.uint8, device=DEV)
        args[pos] = buf.data_ptr() + guard + 1           # odd address on purpose
        seen["buf"] = buf
        real(name, *args)

    rng = np.random.default_rng(8)
    for C in (1, 3):
        imgs = _images(rng, [(97, 1201), (1, 1), (8000, 60), (333, 17)], C)
        for oh, ow in [(S, S), (5, 3)]:
            seen["bytes"] = len(imgs) * oh * ow * C
            monkeypatch.setattr(_lib, "call", redirect)
            resize_uint8([torch.from_numpy(i).to(DEV) for i in imgs], oh, ow, 3)
            x = torch.from_numpy(np.stack(_images(rng, [(150, 171)] * 3, C))).to(DEV)
            buf_list = seen["buf"]
            seen["bytes"] = 3 * oh * ow * C
            resize_uint8(x, oh, ow, 2)
            buf_batch = seen["buf"]
            monkeypatch.setattr(_lib, "call", real)
            for buf, n, src, r in ((buf_list, len(imgs), imgs, 3), (buf_batch, 3, list(x.cpu().numpy()), 2)):
                host = buf.cpu().numpy()
                body = n * oh * ow * C
                assert (host[:guard + 1] == 0xA5).all() and (host[guard + 1 + body:] == 0xA5).all()
                _check(torch.from_numpy(host[guard + 1:guard + 1 + body].reshape(n, oh, ow, C)), src, oh, ow, r)


# ------------------------------------------------------------------------------------------------------ the model
def _randomize(model, seed):
    g = torch.Generator().manual_seed(seed + 1)
    with torch.no_grad():
        for name, p in model.named_parameters():
            if name.endswith(".bias"):
                p.copy_(torch.randn(p.shape, generator=g) * 0.02)
            elif "layernorm" in name and name.endswith(".weight"):
                p.copy_(1.0 + torch.randn(p.shape, generator=g) * 0.02)
            elif name.endswith("mask_token"):
                p.copy_(torch.randn(p.shape, generator=g) * 0.02)
    return model.eval()


@functools.lru_cache(maxsize=None)
def _hf_cls():
    from transformers import ViTConfig, ViTForImageClassification
    torch.manual_seed(0)
    return _randomize(ViTForImageClassification(ViTConfig(**hf_oracle.ARCHS["vit-b16-224"], num_labels=50)), 0)


@functools.lru_cache(maxsize=None)
def _b16():
    from vit.utils import transfer_pretrained_weights
    from vit.vit import VIT
    model = VIT(**hf_oracle.vit_kwargs("vit-b16-224"), num_labels=50, add_pooling_layer=True, use_mask_token=True)
    transfer_pretrained_weights(_hf_cls(), model, verbose=False)
    with torch.no_grad():
        g = torch.Generator().manual_seed(4)
        model.pooler.dense.weight.copy_(torch.randn(model.pooler.dense.weight.shape, generator=g) * 0.03)
        model.embeddings.mask_token.copy_(torch.randn(model.embeddings.mask_token.shape, generator=g) * 0.02)
    return model.to(device=DEV, dtype=torch.bfloat16).eval()


def _photos(seed, sizes):
    rng = np.random.default_rng(seed)
    return _images(rng, sizes, 3)


def _pil_batch(imgs, resample):
    return torch.from_numpy(np.stack([_pil(i, S, S, resample) for i in imgs])).to(DEV)


MIXED = [(375, 500), (97, 1201), (224, 224), (480, 640), (17, 300)]


@pytest.mark.parametrize("mode", ["fold", "ln_before_only", "no_fold", "fp8"])
def test_forward_uint8_do_resize_equals_pil_resized(mode):
    from vit import vit as V
    model = _b16()
    imgs = _photos(1, MIXED)
    lst = [torch.from_numpy(i).to(DEV) for i in imgs]
    batch = torch.from_numpy(np.stack(_photos(2, [(375, 500)] * 3))).to(DEV)
    try:
        if mode == "ln_before_only":
            V.set_layernorm_folding(True, mlp=False)
        elif mode == "no_fold":
            V.set_layernorm_folding(False)
        elif mode == "fp8":
            V.set_fp8(True)
        with torch.no_grad():
            for resample in (2, 3):
                want = model.forward_uint8(_pil_batch(imgs, resample))
                assert torch.equal(model.forward_uint8(lst, do_resize=True, resample=resample), want)
                want_b = model.forward_uint8(_pil_batch(list(batch.cpu().numpy()), resample))
                assert torch.equal(model.forward_uint8(batch, do_resize=True, resample=resample), want_b)
            pil = _pil_batch(imgs, 2)
            mask = torch.rand((len(imgs), 196), generator=torch.Generator().manual_seed(3)) < 0.5
            mask = mask.to(DEV)
            kw = dict(output_hidden_states=True, output_attentions=True, bool_masked_pos=mask)
            want = model.forward_uint8(pil, **kw)
            got = model.forward_uint8(lst, do_resize=True, **kw)
            assert torch.equal(got.last_hidden_state, want.last_hidden_state)
            assert all(torch.equal(a, b) for a, b in zip(got.hidden_states, want.hidden_states))
            assert all(torch.equal(a, b) for a, b in zip(got.attentions, want.attentions))
            assert len(got.hidden_states) == 13 and len(got.attentions) == 12
            # already the model's size: the same bits as without do_resize
            assert torch.equal(model.forward_uint8(pil, do_resize=True), model.forward_uint8(pil))
    finally:
        V.set_layernorm_folding(True)
        V.set_fp8(False)


def test_heads_of_a_mixed_size_list_equal_pil_resized():
    model = _b16()
    imgs = _photos(6, MIXED + [(1, 1), (8000, 60)])
    lst = [torch.from_numpy(i).to(DEV) for i in imgs]
    with torch.no_grad():
        for resample in (2, 3):
            pil = _pil_batch(imgs, resample)
            for name in ("logits", "pooled", "pooler_output"):
                fn = getattr(model, name)
                assert torch.equal(fn(lst, do_resize=True, resample=resample), fn(pil)), name
        # without do_resize a list still means a ragged batch (each image at its own size)
        ragged = model.pooled(lst[:4])
        assert ragged.shape == (4, model.hidden_dim)
        assert torch.equal(ragged[2], model.pooled(lst[2][None])[0])


def test_cuda_graph_of_forward_uint8_with_do_resize():
    from vit.utils import capture_cuda_graph
    model = _b16()
    fwd = functools.partial(model.forward_uint8, do_resize=True)
    static = torch.from_numpy(np.stack(_photos(7, [(375, 500)] * 4))).to(DEV)
    graph, out = capture_cuda_graph(fwd, static)
    for seed in (8, 9):
        imgs = _photos(seed, [(375, 500)] * 4)
        static.copy_(torch.from_numpy(np.stack(imgs)))
        graph.replay()
        torch.cuda.synchronize()
        with torch.no_grad():
            assert torch.equal(out, model.forward_uint8(_pil_batch(imgs, 2)))


def _cos(a, b):
    return F.cosine_similarity(a.flatten().float(), b.flatten().float(), dim=0).item()


def test_against_hf_default_image_processor_and_models():
    """HF's default ViTImageProcessor (torchvision resize) and ViTImageProcessorPil + ViTModel /
    ViTForImageClassification on the CPU in fp32, against do_resize=True in bf16 on the GPU.  Hidden states: the suite's
    bf16 gate (cosine >= 0.999) against both processors.  Logits of the random 50-class head: their bf16 error is the
    forward's, not the resize's, so the torchvision-processed result must be as close as the PIL-processed one (the same
    pixels as ours), within 5e-4 of cosine."""
    from transformers import ViTImageProcessor
    from transformers.models.vit.image_processing_pil_vit import ViTImageProcessorPil
    imgs = _photos(12, MIXED)
    hf = _hf_cls()
    model = _b16()
    lst = [torch.from_numpy(i).to(DEV) for i in imgs]
    pv = {"torchvision": ViTImageProcessor()(images=imgs, return_tensors="pt")["pixel_values"],
          "PIL": ViTImageProcessorPil()(images=imgs, return_tensors="pt")["pixel_values"]}
    with torch.no_grad():
        got_h = model.forward_uint8(lst, do_resize=True).float().cpu()
        got_l = model.logits(lst, do_resize=True).float().cpu()
        want = {name: (hf.vit(pixel_values=x).last_hidden_state, hf(pixel_values=x).logits) for name, x in pv.items()}
    res = {"processor pixel max-abs torchvision vs PIL": (pv["torchvision"] - pv["PIL"]).abs().max().item()}
    for name, (h, lg) in want.items():
        res[f"hidden cos ({name})"] = _cos(got_h, h)
        res[f"hidden max-abs ({name})"] = (got_h - h).abs().max().item()
        res[f"logits cos ({name})"] = _cos(got_l, lg)
        res[f"logits max-abs ({name})"] = (got_l - lg).abs().max().item()
    print("do_resize vs HF:", {k: round(v, 6) for k, v in res.items()})
    assert res["hidden cos (torchvision)"] >= 0.999 and res["hidden cos (PIL)"] >= 0.999, res
    assert abs(res["logits cos (torchvision)"] - res["logits cos (PIL)"]) <= 5e-4, res
