"""GPU: DeiT — a distillation token after CLS (``VIT(distillation_token=True)``), the teacher head
(``distillation_head=True``, ``VIT.distillation_logits``), and the prefix-token entry points of include/vitb200_tokens.h.

Kernels: every ``_prefix`` entry point at prefix 1 equals the entry point it generalises bit for bit; at prefix 2 the
gathers, the table rows, the resample and the finalize equal torch restatements bit for bit, with guard rows around
every output untouched.  Model: parity with HF ``DeiTModel`` / ``DeiTForImageClassification`` /
``DeiTForImageClassificationWithTeacher`` (fp32 on the CPU) at the gates of tests/test_gpu_model.py (bf16 cosine >=
0.999 and max-abs <= 0.15, fp32 <= 1e-3, FP8 cosine >= 0.995 and max-abs <= 0.5).  Properties: an all-false mask, a
ragged list, ``do_resize`` and CUDA-graph replay give the bits of the plain call; the teacher head is one ``vt_bgemm``."""
import functools

import pytest
import torch
import torch.nn.functional as F

from oracle import hf_oracle

pytestmark = pytest.mark.gpu

DEV = "cuda:0"
GUARD = 3          # NaN rows before and after every kernel output


# ---------------------------------------------------------------------------------------------------- kernels
def _pixels(B, H, W, C, pix, g):
    from vit.kernels import _lib
    if pix == "u8":
        return torch.randint(0, 256, (B, H, W, C), generator=g, dtype=torch.uint8).to(DEV), _lib.VT_U8
    x = torch.randn((B, C, H, W), generator=g).to(DEV, torch.float32 if pix == "f32" else torch.bfloat16)
    return x, _lib.dtype_code(x)


def _unfold(x, P, u8):
    """bf16 [B, n, K] patch rows: (c, i, j) order via F.unfold for NCHW, (i, j, c) for NHWC."""
    if u8:
        B, H, W, C = x.shape
        gh, gw = H // P, W // P
        r = x[:, :gh * P, :gw * P].float().reshape(B, gh, P, gw, P, C).permute(0, 1, 3, 2, 4, 5)
        return r.reshape(B, gh * gw, P * P * C).bfloat16()
    B, C, H, W = x.shape
    return F.unfold(x[:, :, :H // P * P, :W // P * P].float(), P, stride=P).transpose(1, 2).bfloat16()


def _guarded(shape, dtype):
    """(buffer with GUARD NaN rows on each side, the inner view)"""
    rows = shape[0]
    buf = torch.full((rows + 2 * GUARD,) + tuple(shape[1:]), float("nan"), device=DEV, dtype=dtype)
    return buf, buf[GUARD:GUARD + rows]


def _guards_intact(buf):
    return bool(buf[:GUARD].isnan().all() and buf[-GUARD:].isnan().all())


def _bits(t):
    return t.view(torch.int16) if t.dtype == torch.bfloat16 else t.view(torch.int32)


def _embed_gemm(name, x, code, w, bias, posb, B, C, H, W, P, D, prefix=None, stats=False):
    """(out, stats, workspace) of vt_patch_embed_gemm_hw[_prefix]: out and workspace guarded."""
    from vit.kernels import _lib
    n_tok = (H // P) * (W // P) + (1 if prefix is None else prefix)
    tok_pad = (n_tok + 31) // 32 * 32
    K = w.shape[1]
    out_buf, out = _guarded((B * n_tok, D), torch.bfloat16)
    work_buf, work = _guarded((B * tok_pad, K), torch.bfloat16)
    st = torch.empty((B * n_tok, D // 128, 2), device=DEV) if stats else None
    args = [x.data_ptr(), code, w.data_ptr(), K, bias.data_ptr(), posb.data_ptr(), out.data_ptr(), _lib.ptr(st),
            work.data_ptr(), B, C, H, W, P, D]
    _lib.call(name, *args, *([] if prefix is None else [prefix]), _lib.stream_ptr(x))
    torch.cuda.synchronize()
    assert _guards_intact(out_buf) and _guards_intact(work_buf), f"{name}: guard rows overwritten"
    return out.view(B, n_tok, D), st, work.view(B, tok_pad, K)


EMBED_SHAPES = [(64, 64), (48, 70), (80, 37)]     # square; non-square; non-square with W * C % 8 != 0 (scalar loads)


@pytest.mark.parametrize("hw", EMBED_SHAPES)
@pytest.mark.parametrize("pix", ["f32", "bf16", "u8"])
def test_patch_embed_gemm_prefix(pix, hw):
    """Prefix 1 == vt_patch_embed_gemm_hw (output, row statistics, workspace).  Prefix 2: workspace rows 0, 1 zero and
    F.unfold rows at 2 + p; output rows 2.. equal the prefix-1 rows 1.., rows 0 and 1 the prefix-1 row 0 (all zero
    patch rows + bias + the same table row)."""
    g = torch.Generator().manual_seed(hw[0] * 7 + hw[1])
    B, C, P, D = 3, 3, 16, 256
    H, W = hw
    K = C * P * P
    n = (H // P) * (W // P)
    x, code = _pixels(B, H, W, C, pix, g)
    w = (torch.randn((D, K), generator=g) * 0.03).to(DEV, torch.bfloat16)
    bias = (torch.randn((D,), generator=g) * 0.1).to(DEV)
    posb1 = (torch.randn((1 + n, D), generator=g) * 0.1).to(DEV, torch.bfloat16)
    old = _embed_gemm("vt_patch_embed_gemm_hw", x, code, w, bias, posb1, B, C, H, W, P, D, stats=True)
    one = _embed_gemm("vt_patch_embed_gemm_hw_prefix", x, code, w, bias, posb1, B, C, H, W, P, D, prefix=1, stats=True)
    for a, b in zip(old, one):
        assert torch.equal(_bits(a), _bits(b))

    posb2 = torch.cat([posb1[:1], posb1[:1], posb1[1:]])
    out2, _, work2 = _embed_gemm("vt_patch_embed_gemm_hw_prefix", x, code, w, bias, posb2, B, C, H, W, P, D, prefix=2)
    want = torch.zeros_like(work2)
    want[:, 2:2 + n, :K] = _unfold(x.cpu(), P, pix == "u8").to(DEV)
    assert torch.equal(_bits(work2), _bits(want))
    assert torch.equal(_bits(out2[:, 2:]), _bits(old[0][:, 1:]))
    assert torch.equal(_bits(out2[:, 0]), _bits(old[0][:, 0])) and torch.equal(_bits(out2[:, 1]), _bits(old[0][:, 0]))


def _mask(B, n, seed):
    g = torch.Generator().manual_seed(seed)
    return torch.rand((B, n), generator=g) < 0.5


def _masked_gather(name, x, code, mask, pos, posm, B, C, H, W, P, D, ldw, prefix=None):
    from vit.kernels import _lib
    N = (H // P) * (W // P) + (1 if prefix is None else prefix)
    p_buf, patches = _guarded((B * N, ldw), torch.bfloat16)
    t_buf, table = _guarded((B * N, D), torch.bfloat16)
    md = mask.to(DEV)
    _lib.call(name, x.data_ptr(), code, md.data_ptr(), pos.data_ptr(), posm.data_ptr(), patches.data_ptr(), ldw,
              table.data_ptr(), B, C, H, W, P, D, *([] if prefix is None else [prefix]), _lib.stream_ptr(x))
    torch.cuda.synchronize()
    assert _guards_intact(p_buf) and _guards_intact(t_buf), f"{name}: guard rows overwritten"
    return patches.view(B, N, ldw).cpu(), table.view(B, N, D).cpu()


@pytest.mark.parametrize("hw", EMBED_SHAPES)
@pytest.mark.parametrize("pix", ["f32", "bf16", "u8"])
def test_masked_gather_prefix(pix, hw):
    g = torch.Generator().manual_seed(hw[0] + hw[1])
    B, C, P, D = 3, 3, 16, 136
    H, W = hw
    K = C * P * P
    ldw = K + 8
    n = (H // P) * (W // P)
    x, code = _pixels(B, H, W, C, pix, g)
    mask = _mask(B, n, seed=H * W)
    mask[0, 0], mask[1, -1] = True, True
    pos = (torch.randn((2 + n, D), generator=g) * 0.1).to(DEV, torch.bfloat16)
    posm = (torch.randn((2 + n, D), generator=g) * 0.1).to(DEV, torch.bfloat16)
    old = _masked_gather("vt_patch_embed_masked_gather", x, code, mask, pos, posm, B, C, H, W, P, D, ldw)
    one = _masked_gather("vt_patch_embed_masked_gather_prefix", x, code, mask, pos, posm, B, C, H, W, P, D, ldw, 1)
    for a, b in zip(old, one):
        assert torch.equal(_bits(a), _bits(b))

    patches, table = _masked_gather("vt_patch_embed_masked_gather_prefix", x, code, mask, pos, posm, B, C, H, W, P, D,
                                    ldw, 2)
    want_p = torch.zeros((B, 2 + n, ldw), dtype=torch.bfloat16)
    want_p[:, 2:, :K] = _unfold(x.cpu(), P, pix == "u8").masked_fill(mask[:, :, None], 0)
    want_t = pos.cpu()[None].repeat(B, 1, 1)
    want_t[:, 2:][mask] = posm.cpu()[2:].expand(B, n, D)[mask]
    assert torch.equal(_bits(patches), _bits(want_p))
    assert torch.equal(_bits(table), _bits(want_t))


def _ragged(imgs, tables, grids, prefix, code, C, P, D, ldw):
    from vit import packing
    from vit.kernels import _lib
    layout = packing.RaggedLayout(grids, 1 if prefix is None else prefix)
    desc = (_lib.RaggedImage * len(imgs))()
    row0, rows = [], 0
    for t in layout.tokens:
        row0.append(rows)
        rows += t
    for i, im in enumerate(imgs):
        h, w = (im.shape[0], im.shape[1]) if code == _lib.VT_U8 else (im.shape[1], im.shape[2])
        desc[i] = _lib.RaggedImage(im.data_ptr(), tables[i].data_ptr(), row0[i], h, w, layout.tokens[i], 0)
    desc_dev = torch.frombuffer(bytearray(bytes(desc)), dtype=torch.uint8).to(DEV)
    p_buf, patches = _guarded((rows, ldw), torch.bfloat16)
    t_buf, table = _guarded((rows, D), torch.bfloat16)
    name = "vt_patch_embed_ragged_gather" + ("" if prefix is None else "_prefix")
    _lib.call(name, desc_dev.data_ptr(), len(imgs), code, C, P, patches.data_ptr(), ldw, table.data_ptr(), D, rows,
              *([] if prefix is None else [prefix]), _lib.stream_ptr(patches))
    torch.cuda.synchronize()
    assert _guards_intact(p_buf) and _guards_intact(t_buf), f"{name}: guard rows overwritten"
    return patches.cpu(), table.cpu(), row0, layout.tokens


@pytest.mark.parametrize("pix", ["f32", "bf16", "u8"])
def test_ragged_gather_prefix(pix):
    from vit.kernels import _lib
    P, C, D = 16, 3, 136
    K = C * P * P
    ldw = K + 16
    sizes = [(32, 48), (70, 37), (16, 16), (50, 64), (33, 21)]
    g = torch.Generator().manual_seed(len(pix) + 1)
    imgs, tables = [], []
    for h, w in sizes:
        if pix == "u8":
            imgs.append(torch.randint(0, 256, (h, w, C), generator=g, dtype=torch.uint8).to(DEV))
        else:
            imgs.append(torch.randn((C, h, w), generator=g).to(DEV, torch.float32 if pix == "f32" else torch.bfloat16))
        tables.append((torch.randn((2 + (h // P) * (w // P), D), generator=g) * 0.1).to(DEV, torch.bfloat16))
    grids = [(h // P, w // P) for h, w in sizes]
    code = _lib.VT_U8 if pix == "u8" else _lib.dtype_code(imgs[0])
    old = _ragged(imgs, tables, grids, None, code, C, P, D, ldw)
    one = _ragged(imgs, tables, grids, 1, code, C, P, D, ldw)
    assert torch.equal(_bits(old[0]), _bits(one[0])) and torch.equal(_bits(old[1]), _bits(one[1]))

    patches, table, row0, tokens = _ragged(imgs, tables, grids, 2, code, C, P, D, ldw)
    for i, im in enumerate(imgs):
        r, n = row0[i], tokens[i]
        want = torch.zeros((n, ldw), dtype=torch.bfloat16)
        want[2:, :K] = _unfold(im.cpu()[None], P, pix == "u8")[0]
        assert torch.equal(_bits(patches[r:r + n]), _bits(want)), f"image {i}: patch rows differ"
        assert torch.equal(_bits(table[r:r + n]), _bits(tables[i].cpu())), f"image {i}: position rows differ"


@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16])
@pytest.mark.parametrize("grid", [(24, 24), (10, 15), (14, 14), (3, 1)])
def test_pos_resample_prefix(dtype, grid):
    from vit.kernels import _lib
    g = torch.Generator().manual_seed(grid[0] * 31 + grid[1])
    g_in, D = 14, 200
    gh, gw = grid
    pos2 = torch.randn((2 + g_in * g_in, D), generator=g).to(DEV, dtype)
    pos1 = torch.cat([pos2[:1], pos2[2:]])

    def run(name, pos, prefix):
        n = (1 if prefix is None else prefix) + gh * gw
        buf, out = _guarded((n, D), torch.float32)
        _lib.call(name, pos.data_ptr(), _lib.dtype_code(pos), out.data_ptr(), D, g_in, gh, gw,
                  *([] if prefix is None else [prefix]), _lib.stream_ptr(pos))
        torch.cuda.synchronize()
        assert _guards_intact(buf), f"{name}: guard rows overwritten"
        return out.cpu()

    old = run("vt_pos_embed_resample", pos1, None)
    assert torch.equal(_bits(old), _bits(run("vt_pos_embed_resample_prefix", pos1, 1)))
    two = run("vt_pos_embed_resample_prefix", pos2, 2)
    assert torch.equal(_bits(two[:2]), _bits(pos2[:2].float().cpu()))
    assert torch.equal(_bits(two[2:]), _bits(old[1:]))


@pytest.mark.parametrize("masked", [False, True])
@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16])
def test_embed_finalize_prefix(dtype, masked):
    from vit.kernels import _lib
    B, n, D = 5, 19, 100
    g = torch.Generator().manual_seed(3 + masked)
    x0 = torch.randn((B, 2 + n, D), generator=g).to(dtype)
    pos = torch.randn((2 + n, D), generator=g).to(dtype)
    rows = torch.randn((2, D), generator=g).to(dtype)
    mt = torch.randn((D,), generator=g).to(dtype)
    mask = _mask(B, n, seed=4)

    def run(name, x, prefix, pos_, rows_, mask_):
        buf, xd = _guarded((x.shape[0] * x.shape[1], D), dtype)
        xd.copy_(x.reshape(-1, D))
        N = x.shape[1]
        pd, rd, md, kd = pos_.to(DEV), rows_.contiguous().to(DEV), mt.to(DEV), mask_.contiguous().to(DEV)
        tail = ([] if prefix is None else [prefix]) + [_lib.stream_ptr(xd)]
        if masked:
            _lib.call(name, xd.data_ptr(), pd.data_ptr(), rd.data_ptr(), md.data_ptr(), kd.data_ptr(), B, N, D,
                      _lib.dtype_code(xd), *tail)
        else:
            _lib.call(name, xd.data_ptr(), pd.data_ptr(), rd.data_ptr(), B, N, D, _lib.dtype_code(xd), *tail)
        torch.cuda.synchronize()
        assert _guards_intact(buf), f"{name}: guard rows overwritten"
        return xd.view(B, N, D).cpu()

    base = "vt_embed_finalize_masked" if masked else "vt_embed_finalize"
    x1, pos1 = torch.cat([x0[:, :1], x0[:, 2:]], 1), torch.cat([pos[:1], pos[2:]])
    old = run(base, x1, None, pos1, rows[0], mask)
    assert torch.equal(_bits(old), _bits(run(base + "_prefix", x1, 1, pos1, rows[:1], mask)))

    got = run(base + "_prefix", x0, 2, pos, rows, mask)
    want = torch.empty_like(x0)
    want[:, :2] = (rows.float() + pos[:2].float()).to(dtype)
    body = torch.where(mask[:, :, None], mt.expand(B, n, D), x0[:, 2:]) if masked else x0[:, 2:]
    want[:, 2:] = (body.float() + pos[2:].float()).to(dtype)
    assert torch.equal(_bits(got), _bits(want))


# ---------------------------------------------------------------------------------------------------- models
LABELS = 10


def _randomize(model, seed):
    """HF zero-initialises biases, LayerNorm affines, the tokens and the position table: re-randomise them."""
    g = torch.Generator().manual_seed(seed + 1)
    with torch.no_grad():
        for name, p in model.named_parameters():
            if name.endswith(".bias"):
                p.copy_(torch.randn(p.shape, generator=g) * 0.02)
            elif "layernorm" in name and name.endswith(".weight"):
                p.copy_(1.0 + torch.randn(p.shape, generator=g) * 0.02)
            elif name.endswith(("cls_token", "distillation_token", "mask_token")):
                p.copy_(torch.randn(p.shape, generator=g) * 0.5)
            elif name.endswith("position_embeddings"):
                p.copy_(torch.randn(p.shape, generator=g) * 0.1)
            elif "classifier" in name:
                p.copy_(torch.randn(p.shape, generator=g) * 0.1)
    return model


@functools.lru_cache(maxsize=None)
def _hf(arch, kind="model"):
    from transformers import (DeiTConfig, DeiTForImageClassification, DeiTForImageClassificationWithTeacher,
                              DeiTModel)
    torch.manual_seed(0)
    cfg = DeiTConfig(**hf_oracle.ARCHS[arch], num_labels=LABELS, attn_implementation="eager")
    if kind == "model":
        m = DeiTModel(cfg, add_pooling_layer=True, use_mask_token=True)
    elif kind == "classifier":
        m = DeiTForImageClassification(cfg)
    else:
        m = DeiTForImageClassificationWithTeacher(cfg)
    return _randomize(m.eval(), 0)


_KW = {"model": dict(add_pooling_layer=True, use_mask_token=True), "classifier": dict(num_labels=LABELS),
       "teacher": dict(num_labels=LABELS, distillation_head=True)}


@functools.lru_cache(maxsize=None)
def _ours(arch, dtype, kind="model"):
    from vit.utils import transfer_pretrained_weights
    from vit.vit import VIT
    model = VIT(**hf_oracle.vit_kwargs(arch), distillation_token=True, **_KW[kind])
    transfer_pretrained_weights(_hf(arch, kind), model, verbose=False)
    return model.to(device=DEV, dtype=dtype).eval()


def _x(batch, h, w, seed=5):
    g = torch.Generator().manual_seed(seed)
    return torch.randn((batch, 3, h, w), generator=g)


def _cos(a, b):
    return F.cosine_similarity(a.flatten().float(), b.flatten().float(), dim=0).item()


def _check(got, want, gate, what):
    got, want = got.float().cpu(), want.float()
    assert got.shape == want.shape, f"{what}: {tuple(got.shape)} vs {tuple(want.shape)}"
    assert torch.isfinite(got).all(), what
    err, cos = (got - want).abs().max().item(), _cos(got, want)
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


ARCHS = ["tiny-b", "tiny-h", "vit-b16-224"]
MODES = ["fold", "fold_ln_before", "no_fold", "fp8", "fp32", "unfused"]


@pytest.mark.parametrize("mode", MODES)
@pytest.mark.parametrize("arch", ARCHS)
@torch.no_grad()
def test_last_hidden_state_matches_hf(arch, mode):
    dtype = torch.float32 if mode in ("fp32", "unfused") else torch.bfloat16
    model, hf = _ours(arch, dtype), _hf(arch)
    S = hf_oracle.ARCHS[arch]["image_size"]
    x = _x(2, S, S)
    want = hf(pixel_values=x).last_hidden_state
    with _Mode(mode):
        got = model(x.to(DEV, dtype))
    assert got.shape[1] == 2 + (S // model.patch_size) ** 2
    _check(got, want, "fp32" if dtype == torch.float32 else ("fp8" if mode == "fp8" else "bf16"), f"{arch} {mode}")


@pytest.mark.parametrize("arch", ARCHS)
@torch.no_grad()
def test_uint8_pooler_and_masks_match_hf(arch):
    """uint8 pixels, pooler_output and random masks (DeiTModel(use_mask_token=True))."""
    model, hf = _ours(arch, torch.bfloat16), _hf(arch)
    S = hf_oracle.ARCHS[arch]["image_size"]
    g = torch.Generator().manual_seed(9)
    x8 = torch.randint(0, 256, (3, S, S, 3), generator=g, dtype=torch.uint8)
    xf = ((x8.float() / 255.0 - 0.5) / 0.5).permute(0, 3, 1, 2).contiguous()
    _check(model.forward_uint8(x8.to(DEV)), hf(pixel_values=xf).last_hidden_state, "bf16", f"{arch} uint8")
    x = _x(3, S, S, seed=6)
    out = hf(pixel_values=x)
    _check(model.pooler_output(x.to(DEV, torch.bfloat16)), out.pooler_output, "bf16", f"{arch} pooler_output")
    mask = _mask(3, (S // model.patch_size) ** 2, seed=S)
    want = hf(pixel_values=x, bool_masked_pos=mask).last_hidden_state
    _check(model(x.to(DEV, torch.bfloat16), bool_masked_pos=mask.to(DEV)), want, "bf16", f"{arch} mask")
    x32 = _ours(arch, torch.float32)
    _check(x32(x.to(DEV), bool_masked_pos=mask.to(DEV)), want, "fp32", f"{arch} fp32 mask")


@pytest.mark.parametrize("hw", [(384, 384), (160, 288)])
@torch.no_grad()
def test_interpolate_pos_encoding_matches_hf(hw):
    model, hf = _ours("vit-b16-224", torch.bfloat16), _hf("vit-b16-224")
    x = _x(2, *hw, seed=hw[1])
    want = hf(pixel_values=x, interpolate_pos_encoding=True).last_hidden_state
    got = model(x.to(DEV, torch.bfloat16), interpolate_pos_encoding=True)
    _check(got, want, "bf16", f"interpolate {hw}")
    x32 = _ours("tiny-b", torch.float32)
    xt = _x(2, hw[0] // 4, hw[1] // 4, seed=hw[0])
    want = _hf("tiny-b")(pixel_values=xt, interpolate_pos_encoding=True).last_hidden_state
    _check(x32(xt.to(DEV), interpolate_pos_encoding=True), want, "fp32", f"tiny-b fp32 interpolate {hw}")


@pytest.mark.parametrize("arch,dtype", [("tiny-b", torch.float32), ("tiny-h", torch.bfloat16),
                                        ("vit-b16-224", torch.bfloat16)])
@torch.no_grad()
def test_hidden_states_and_attentions_match_eager_hf(arch, dtype):
    model, hf = _ours(arch, dtype), _hf(arch)
    S = hf_oracle.ARCHS[arch]["image_size"]
    x = _x(2, S, S, seed=7)
    want = hf(pixel_values=x, output_hidden_states=True, output_attentions=True)
    assert len(want.attentions) == model.num_layers, "HF returned no attention maps (SDPA attention?)"
    got = model(x.to(DEV, dtype), output_hidden_states=True, output_attentions=True)
    gate = "fp32" if dtype == torch.float32 else "bf16"
    assert len(got.hidden_states) == len(want.hidden_states) and len(got.attentions) == len(want.attentions)
    for i, (a, b) in enumerate(zip(got.hidden_states, want.hidden_states)):
        _check(a, b, gate, f"{arch} hidden_states[{i}]")
    for i, (a, b) in enumerate(zip(got.attentions, want.attentions)):
        _check(a, b, gate, f"{arch} attentions[{i}]")
    _check(got.last_hidden_state, want.last_hidden_state, gate, f"{arch} last_hidden_state")


@pytest.mark.parametrize("dtype", [torch.bfloat16, torch.float32])
@pytest.mark.parametrize("arch", ARCHS)
@torch.no_grad()
def test_heads_match_hf(arch, dtype):
    """``logits`` against DeiTForImageClassification, the three fields of ``distillation_logits`` against
    DeiTForImageClassificationWithTeacher, and ``logits`` of the teacher model is the mean."""
    gate = "fp32" if dtype == torch.float32 else "bf16"
    S = hf_oracle.ARCHS[arch]["image_size"]
    x = _x(4, S, S, seed=8)
    xd = x.to(DEV, dtype)
    _check(_ours(arch, dtype, "classifier").logits(xd), _hf(arch, "classifier")(pixel_values=x).logits, gate,
           f"{arch} logits")
    teacher = _ours(arch, dtype, "teacher")
    want = _hf(arch, "teacher")(pixel_values=x)
    got = teacher.distillation_logits(xd)
    for field in ("logits", "cls_logits", "distillation_logits"):
        _check(getattr(got, field), getattr(want, field), gate, f"{arch} {field}")
    assert torch.equal(teacher.logits(xd), got.logits)


# ---------------------------------------------------------------------------------------------------- identities
@torch.no_grad()
def test_all_false_mask_equals_unmasked_call():
    model = _ours("vit-b16-224", torch.bfloat16)
    x = _x(3, 224, 224).to(DEV, torch.bfloat16)
    none = torch.zeros((3, 196), dtype=torch.bool, device=DEV)
    assert torch.equal(model(x, bool_masked_pos=none), model(x))
    x8 = torch.randint(0, 256, (3, 224, 224, 3), dtype=torch.uint8).to(DEV)
    assert torch.equal(model.forward_uint8(x8, bool_masked_pos=none), model.forward_uint8(x8))


@pytest.mark.parametrize("u8", [False, True])
@torch.no_grad()
def test_ragged_list_equals_each_images_own_call(u8):
    model = _ours("vit-b16-224", torch.bfloat16)
    teacher = _ours("vit-b16-224", torch.bfloat16, "teacher")
    sizes = [(224, 224), (160, 96), (240, 250), (224, 224), (48, 64)]
    g = torch.Generator().manual_seed(2)
    if u8:
        imgs = [torch.randint(0, 256, (h, w, 3), generator=g, dtype=torch.uint8).to(DEV) for h, w in sizes]
    else:
        imgs = [torch.randn((3, h, w), generator=g).to(DEV, torch.bfloat16) for h, w in sizes]
    own = model.forward_uint8 if u8 else model.forward
    got = model.forward_ragged(imgs)
    for i, img in enumerate(imgs):
        want = own(img[None], interpolate_pos_encoding=True)[0]
        assert got[i].shape[0] == 2 + (sizes[i][0] // 16) * (sizes[i][1] // 16)
        assert torch.equal(got[i], want), f"image {i} {sizes[i]}"
    pooled = model.pooler_output(imgs)
    heads = teacher.distillation_logits(imgs)
    for i, img in enumerate(imgs):
        assert torch.equal(pooled[i], model.pooler_output(img[None], interpolate_pos_encoding=True)[0])
        one = teacher.distillation_logits(img[None], interpolate_pos_encoding=True)
        for field in range(3):
            assert torch.equal(heads[field][i], one[field][0]), f"image {i} field {field}"


@torch.no_grad()
def test_do_resize_equals_resize_then_call():
    from vit.kernels.resize import resize_uint8
    model = _ours("vit-b16-224", torch.bfloat16)
    teacher = _ours("vit-b16-224", torch.bfloat16, "teacher")
    g = torch.Generator().manual_seed(4)
    x8 = torch.randint(0, 256, (2, 300, 257, 3), generator=g, dtype=torch.uint8).to(DEV)
    r = resize_uint8(x8, 224, 224, 2)
    assert torch.equal(model.forward_uint8(x8, do_resize=True), model.forward_uint8(r))
    got, want = teacher.distillation_logits(x8, do_resize=True), teacher.distillation_logits(r)
    assert all(torch.equal(a, b) for a, b in zip(got, want))


@torch.no_grad()
def test_cuda_graph_replay_equals_eager():
    from vit.utils import capture_cuda_graph
    model = _ours("vit-b16-224", torch.bfloat16)
    teacher = _ours("vit-b16-224", torch.bfloat16, "teacher")
    x = _x(8, 224, 224).to(DEV, torch.bfloat16)
    y = _x(8, 224, 224, seed=12).to(DEV, torch.bfloat16)
    static = x.clone()
    graph, out = capture_cuda_graph(model, static)
    fn = lambda t: torch.cat(teacher.distillation_logits(t), dim=1)   # noqa: E731
    graph2, out2 = capture_cuda_graph(fn, static)
    for inp in (x, y):
        static.copy_(inp)
        graph.replay()
        graph2.replay()
        torch.cuda.synchronize()
        assert torch.equal(out, model(inp))
        assert torch.equal(out2, fn(inp))


@pytest.mark.parametrize("dtype", [torch.bfloat16, torch.float32])
@torch.no_grad()
def test_teacher_head_is_one_bgemm_after_the_encoder(monkeypatch, dtype):
    from vit.kernels import _lib
    teacher = _ours("tiny-b", dtype, "teacher")
    x = _x(3, 64, 64).to(DEV, dtype)
    teacher.distillation_logits(x)                         # builds the packed head
    names = []
    real = _lib.call
    monkeypatch.setattr(_lib, "call", lambda name, *a: (names.append(name), real(name, *a))[1])
    teacher(x)
    encoder = list(names)
    names.clear()
    got = teacher.distillation_logits(x)
    head = names[len(encoder):]
    assert names[:len(encoder)] == encoder
    assert head == (["vt_bgemm"] if dtype == torch.bfloat16 else ["vt_pack_bf16", "vt_bgemm"])
    base = got.cls_logits.untyped_storage().data_ptr()
    assert all(t.untyped_storage().data_ptr() == base for t in got)
    # a changed classifier is noticed, and invalidate_packed drops the pack
    bias = teacher.distillation_classifier.bias
    saved = bias.detach().clone()
    with torch.no_grad():
        bias.add_(1.0)
    try:
        moved = teacher.distillation_logits(x)
        assert torch.allclose(moved.distillation_logits.float(), got.distillation_logits.float() + 1.0, atol=0.07)
    finally:
        with torch.no_grad():
            bias.copy_(saved)
    teacher.invalidate_packed()
    assert "_teacher_packed" not in teacher.__dict__
