"""Weight packing for the fused execution path.

The module tree keeps the reference's parameter layout (per-head (D, dh) query/key/value matrices,
(in, out) dense weights — vit/vit.py:25-35,38-53; 990 state-dict keys for ViT-B).  The tensor-core
kernels want something else: ONE K-major [3D, D] matrix for Q, K and V of all heads, K-major
[out, in] matrices for the other dense layers, fp32 biases, and the position embedding pre-added to
the CLS token / conv bias.  This module derives those once and caches them per module; the cache is
dropped when the module is moved / cast (``_apply``), when a state-dict is loaded, or when any
source parameter's storage pointer or version counter changes (in-place ops, optimizer steps,
``p.data = new``).  Writes THROUGH ``p.data`` (``p.data.copy_()``, ``p.data.normal_()``, EMA updates)
bump no version counter and cannot be seen without reading the device: call ``VIT.invalidate_packed()``
after them.
"""
import ctypes
import math
from collections import OrderedDict
from types import SimpleNamespace
from typing import Optional

import torch

import os

from .kernels import _lib, bgemm as bg


class PackedMixin:
    """Gives a module lazily built, automatically invalidated ``packed(kind, *args)`` namespaces.

    ``kind`` selects a builder ``_build_packed[_<kind>]`` and its source list
    ``_packed_sources[_<kind>]`` (default: every parameter of the module).  ``args`` go to the builder and are part of
    the cache key: one namespace per kind is kept, built for the last ``args``."""

    def _packed_sources(self):
        return list(self.parameters())

    @staticmethod
    def _packed_key(params):
        return tuple((p.data_ptr(), p._version) for p in params)

    def packed(self, kind: str = "", *args):
        states = self.__dict__.setdefault("_packed_states", {})
        state = states.get(kind)
        if state is not None:
            params, key, value = state
            if key == (args, self._packed_key(params)):
                return value
        suffix = f"_{kind}" if kind else ""
        params = getattr(self, "_packed_sources" + suffix, self._packed_sources)()
        with torch.no_grad():
            value = getattr(self, "_build_packed" + suffix)(*args)
        states[kind] = (params, (args, self._packed_key(params)), value)
        return value

    def invalidate_packed(self):
        self.__dict__.pop("_packed_states", None)

    def _apply(self, fn, *args, **kwargs):
        self.invalidate_packed()
        return super()._apply(fn, *args, **kwargs)

    def _load_from_state_dict(self, *args, **kwargs):
        self.invalidate_packed()
        return super()._load_from_state_dict(*args, **kwargs)


def _nk(weight_in_out: torch.Tensor) -> torch.Tensor:
    """(in, out) -> contiguous [out, in]: the K-major operand layout."""
    return weight_in_out.detach().t().contiguous()


def pack_attention(mha) -> SimpleNamespace:
    heads = mha.attention
    wq = torch.cat([h.query.weight.detach() for h in heads], dim=1)
    wk = torch.cat([h.key.weight.detach() for h in heads], dim=1)
    wv = torch.cat([h.value.weight.detach() for h in heads], dim=1)
    bq = torch.cat([h.query.bias.detach() for h in heads])
    bk = torch.cat([h.key.bias.detach() for h in heads])
    bv = torch.cat([h.value.bias.detach() for h in heads])
    return SimpleNamespace(
        wqkv=_nk(torch.cat([wq, wk, wv], dim=1)),          # [3D, D]
        bqkv=torch.cat([bq, bk, bv]).float().contiguous(),  # [3D] fp32
        wo=_nk(mha.output.weight),                          # [D, D]
        bo=mha.output.bias.detach().float().contiguous(),
    )


def pack_mlp(block) -> SimpleNamespace:
    return SimpleNamespace(
        w1=_nk(block.intermediate.weight),                  # [F, D]
        b1=block.intermediate.bias.detach().float().contiguous(),
        w2=_nk(block.output.weight),                        # [D, F]
        b2=block.output.bias.detach().float().contiguous(),
    )


def fold_layernorm(w_nk: torch.Tensor, bias32: torch.Tensor, ln, zero_sum: bool = True) -> tuple:
    """Fold y = LN(x) into the dense layer that consumes it (one launch of ``vt_ln_fold``, csrc/ln_fold.cu):

        LN(x) @ W^T + b = rstd * (x @ (W * gamma)^T) - rstd * mean * colsum(W * gamma) + (b + W @ beta).

    ``zero_sum`` (the default packing) moves the mean term INTO the weights: every row of W * gamma is
    shifted by its own mean, so  x @ W'^T = x @ (W * gamma)^T - mean(x) * colsum  comes out of the GEMM
    itself and the epilogue is  rstd * acc + (b + W @ beta)  — no column-sum operand, one FMA per element
    less; the bf16 rounding residue of each row sum (~3e-3 for a 768-wide row) is cancelled in the kernel
    by re-rounding the elements closest to a rounding tie the other way (left: ~1e-6).
    Returns (W' bf16 [N, K], b' fp32 [N], colsum fp32 [N] or None for the zero-sum form)."""
    assert w_nk.is_cuda and w_nk.dtype == torch.bfloat16 and w_nk.is_contiguous(), \
        "LayerNorm folding runs on CUDA bf16 K-major weights (there is no CPU path)"
    N, K = w_nk.shape
    gamma = ln.weight.detach().float().contiguous()
    beta = ln.bias.detach().float().contiguous()
    bias32 = bias32.contiguous()
    w_out = torch.empty_like(w_nk)
    b_out = torch.empty((N,), device=w_nk.device, dtype=torch.float32)
    colsum = None if zero_sum else torch.empty((N,), device=w_nk.device, dtype=torch.float32)
    _lib.call("vt_ln_fold", w_nk.data_ptr(), K, bias32.data_ptr(), gamma.data_ptr(), beta.data_ptr(),
              w_out.data_ptr(), K, b_out.data_ptr(), _lib.ptr(colsum), N, K, 1 if zero_sum else 0,
              _lib.stream_ptr(w_nk))
    return w_out, b_out, colsum


def pack_block_folded(block) -> SimpleNamespace:
    """Both LayerNorms of one encoder block folded into the GEMMs that consume them, zero-sum form:
    layernorm_before -> fused QKV weights, layernorm_after -> fc1 weights (two ``vt_ln_fold`` launches)."""
    att = block.attention.packed()
    mlp = block.packed()
    wqkv, bqkv, _ = fold_layernorm(att.wqkv, att.bqkv, block.layernorm_before)
    w1, b1, _ = fold_layernorm(mlp.w1, mlp.b1, block.layernorm_after)
    return SimpleNamespace(wqkv=wqkv, bqkv=bqkv, cqkv=None, w1=w1, b1=b1, c1=None)


# ------------------------------------------------------------------------------------------------ FP8 (optional)
FP8_ACT_SCALE = 16.0     # LayerNorm outputs are quantised as e4m3(y * scale), scale <= 16 (fp8_ln_scale)
FP8_MID_SCALE = 8.0      # GELU outputs (fc2's operand) as e4m3(g * 8), saturating at |g| = 56
FP8_LN_MAX_DIM = 2048    # vt_layernorm_fp8 keeps a row in registers: at most 8 16-byte vectors per lane


def fp8_supported(x: torch.Tensor, dim: int, mlp_dim: int) -> bool:
    return (x.is_cuda and x.dtype == torch.bfloat16 and dim % 16 == 0 and dim <= FP8_LN_MAX_DIM
            and mlp_dim % 128 == 0)


def fp8_ln_scale(ln) -> float:
    """Activation scale of the e4m3 output of LayerNorm ``ln``: the largest power of two <= FP8_ACT_SCALE at which no
    element can saturate.  Every output element satisfies |gamma_i y_i + beta_i| <= B = max|gamma| sqrt(D - 1) +
    max|beta|, because a normalised row has |y_i| <= sqrt(D - 1) (Samuelson's inequality); B * (1 + 2^-10) * scale
    <= 448 leaves room for the kernel's fp32 rounding of y.  A power of two changes no e4m3 code that stays in the
    normal range, so a LayerNorm with B <= 28 / (1 + 2^-10) keeps the scale 16."""
    gamma = ln.weight.detach().double()
    beta = ln.bias.detach().double()
    bound = gamma.abs().max().item() * math.sqrt(gamma.numel() - 1) + beta.abs().max().item()
    if bound == 0.0:
        return FP8_ACT_SCALE
    return min(FP8_ACT_SCALE, 2.0 ** math.floor(math.log2(448.0 / (bound * (1.0 + 2.0 ** -10)))))


def quantize_weight_fp8(w_nk: torch.Tensor) -> tuple:
    """bf16 [N, K] K-major weight -> (e4m3 bytes [N, K], fp32 per-output-channel scales [N])."""
    assert w_nk.is_cuda and w_nk.dtype == torch.bfloat16 and w_nk.is_contiguous()
    N, K = w_nk.shape
    w8 = torch.empty((N, K), device=w_nk.device, dtype=torch.uint8)
    scales = torch.empty((N,), device=w_nk.device, dtype=torch.float32)
    _lib.call("vt_quantize_rows_fp8", w_nk.data_ptr(), K, w8.data_ptr(), K, scales.data_ptr(), N, K,
              _lib.stream_ptr(w_nk))
    return w8, scales


def pack_block_fp8(block) -> SimpleNamespace:
    """e4m3 weights of the QKV / fc1 / fc2 layers of one block with their per-channel dequantisation scales,
    the activation scales already divided out (the GEMM epilogue is acc * colscale + bias); ``ln1_scale`` /
    ``ln2_scale`` are the e4m3 scales of layernorm_before / layernorm_after (fp8_ln_scale)."""
    att = block.attention.packed()
    mlp = block.packed()
    wqkv8, sqkv = quantize_weight_fp8(att.wqkv)
    w18, s1 = quantize_weight_fp8(mlp.w1)
    w28, s2 = quantize_weight_fp8(mlp.w2)
    ln1_scale = fp8_ln_scale(block.layernorm_before)
    ln2_scale = fp8_ln_scale(block.layernorm_after)
    return SimpleNamespace(wqkv8=wqkv8, cqkv=(sqkv / ln1_scale).contiguous(), w18=w18,
                           c1=(s1 / ln2_scale).contiguous(), w28=w28, c2=(s2 / FP8_MID_SCALE).contiguous(),
                           ln1_scale=ln1_scale, ln2_scale=ln2_scale)


def layernorm_fp8(x: torch.Tensor, ln, scale: float = FP8_ACT_SCALE) -> torch.Tensor:
    """(B, N, D) bf16 -> e4m3(LN(x) * scale) as uint8 (B, N, D): LayerNorm with the GEMM operand's quantisation fused."""
    B, N, D = x.shape
    out = torch.empty((B, N, D), device=x.device, dtype=torch.uint8)
    if out.numel():
        _lib.call("vt_layernorm_fp8", x.data_ptr(), ln.weight.data_ptr(), ln.bias.data_ptr(), out.data_ptr(), B * N, D,
                  D, D, float(ln.eps), float(scale), _lib.stream_ptr(x))
    return out


def linear_fp8(x8: torch.Tensor, w8: torch.Tensor, colscale: torch.Tensor, bias32: torch.Tensor, gelu: int = 0,
               residual: Optional[torch.Tensor] = None, out_fp8: bool = False, out_scale: float = 1.0) -> torch.Tensor:
    """out = act((x8 @ w8^T) * colscale + bias) (+ residual) on tcgen05.mma kind::f8f6f4; x8 / w8 are e4m3 bytes.
    ``gelu``: the activation code (``_lib.VT_ACT_*``: 0 none, 1 exact GELU, 3 quick GELU; False / True are 0 / 1)."""
    B, N, K = x8.shape
    n_out = w8.shape[0]
    out = torch.empty((B, N, n_out), device=x8.device, dtype=torch.uint8 if out_fp8 else torch.bfloat16)
    if out.numel():
        _lib.call("vt_gemm_fp8", x8.data_ptr(), K, w8.data_ptr(), K, out.data_ptr(), n_out,
                  _lib.VT_E4M3 if out_fp8 else _lib.VT_BF16, bias32.data_ptr(), colscale.data_ptr(),
                  _lib.ptr(residual), n_out, B * N, n_out, K, int(gelu), float(out_scale), _lib.stream_ptr(x8))
    return out


def _posb16(pos32: torch.Tensor, prefix32: torch.Tensor, bias32: torch.Tensor) -> torch.Tensor:
    """bf16 [N, D] position table of the two-launch patch embedding (``vt_patch_embed_gemm``): the GEMM adds the
    conv bias to EVERY row, so row t < prefix (CLS, distillation token: zero patch rows) carries
    token_t + pos[t] - bias, with ``prefix32`` the fp32 [prefix, D] token rows (``prefix_rows32``)."""
    t = pos32.clone()
    t[:prefix32.shape[0]] += prefix32 - bias32
    return t.to(torch.bfloat16).contiguous()


def prefix_tokens(emb) -> list:
    """The learned tokens in front of the patches, (1, 1, D) each: [cls_token], or [cls_token, distillation_token]."""
    return [emb.cls_token] if emb.distillation_token is None else [emb.cls_token, emb.distillation_token]


def prefix_rows32(emb) -> torch.Tensor:
    """fp32 [prefix, D] rows of the tokens in front of the patches, [cls; dist]."""
    return torch.cat([t.detach().float().reshape(1, -1) for t in prefix_tokens(emb)])


def _posm16(pos32: torch.Tensor, mask_token: Optional[torch.Tensor], bias32: torch.Tensor) -> Optional[torch.Tensor]:
    """bf16 [N, D] table of masked patches (``vt_patch_embed_masked_gather``): a masked patch's row is zero, so the GEMM
    gives bias + this row, which must come out as mask_token + pos.  One rounding from fp32; the prefix rows are not
    read.  None for a model without a mask token."""
    if mask_token is None:
        return None
    return (pos32 + mask_token.detach().float().reshape(-1) - bias32).to(torch.bfloat16).contiguous()


def pixel_format(image_mean, image_std, rescale_factor: float) -> tuple:
    """The pixel format of raw uint8 NHWC pixels with these image-processor constants: (mean, std, rescale) as floats.
    Every embedding function takes a format ``fmt``: None for float NCHW pixels, or this key."""
    return tuple(float(m) for m in image_mean), tuple(float(v) for v in image_std), float(rescale_factor)


def pixel_dims(x: torch.Tensor, fmt: Optional[tuple]) -> tuple:
    """(B, C, H, W) of a pixel batch of format ``fmt``: (B, C, H, W) float pixels, or (B, H, W, C) raw uint8 ones."""
    if fmt is None:
        return tuple(x.shape)
    B, H, W, C = x.shape
    return B, C, H, W


def pack_embeddings(emb, fmt: Optional[tuple] = None) -> SimpleNamespace:
    """Patch-projection operands for pixels of format ``fmt``: the bf16 | fp32 weight ``w`` [D, ldw] (K = C*P*P columns,
    zero padding to a multiple of 8), the fp32 bias ``bias32`` [D], the fp32 prefix-token rows ``prefix32`` [prefix, D]
    and the bf16 position tables ``posb16`` / ``posm16`` of the trained grid.  Float pixels: the conv weight in the
    reference's (c, i, j) order and the conv bias.

    Raw uint8 NHWC pixels (``fmt`` = ``pixel_format``): the image processor's ``(x * rescale - mean_c) / std_c`` (HF
    ViTImageProcessor: 1/255, 0.5, 0.5) is folded into the operands, so the kernel multiplies bytes:

        sum_k w[d,k] * (x_k * r - mean_c) / std_c  =  sum_k (w[d,k] * r / std_c) * x_k  -  sum_k w[d,k] * mean_c / std_c

    The weight is re-ordered from the reference's (c, i, j) to (i, j, c) — a patch row of an NHWC image is P*C
    contiguous bytes — and scaled in fp32 before the single rounding to the model's dtype; the constant term is
    subtracted from the conv bias."""
    w = emb.projection.weight.detach()                         # [D, C, P, P]
    D, C = w.shape[0], w.shape[1]
    K = w[0].numel()
    kpad = (K + 7) // 8 * 8
    bias32 = emb.projection.bias.detach().float().contiguous()
    if fmt is not None:
        image_mean, image_std, rescale_factor = fmt
        w32 = w.float()
        mean = torch.as_tensor(image_mean, dtype=torch.float32, device=w.device).reshape(1, C, 1, 1)
        std = torch.as_tensor(image_std, dtype=torch.float32, device=w.device).reshape(1, C, 1, 1)
        bias32 = (bias32 - (w32 * (mean / std)).sum(dim=(1, 2, 3))).contiguous()
        w = (w32 * (rescale_factor / std)).permute(0, 2, 3, 1).to(w.dtype)
    w2d = torch.zeros((D, kpad), device=w.device, dtype=w.dtype)
    w2d[:, :K] = w.reshape(D, K)
    pos = emb.position_embeddings.detach().float()[0]          # [N, D]
    prefix32 = prefix_rows32(emb)
    return SimpleNamespace(w=w2d, ldw=kpad, K=K, bias32=bias32, prefix32=prefix32,
                           posb16=_posb16(pos, prefix32, bias32), posm16=_posm16(pos, emb.mask_token, bias32))


def pack_teacher_head(cls_head, dist_head, pieces: int) -> SimpleNamespace:
    """DeiT's two classifiers (``LinearWithBias``, weight (D, L)) as ONE GEMM over each image's rows 0 and 1 (2D
    contiguous elements): the K-major [3L, 2D] weight [[Wc, 0], [0, Wd], [Wc / 2, Wd / 2]] packed for ``bg.dense_rows``
    with ``pieces`` (``w``), and the fp32 bias [bc, bd, (bc + bd) / 2] (``bias32``).  The outputs are the cls logits,
    the distillation logits and their mean; halving is exact."""
    wc = cls_head.weight.detach().t()                          # [L, D]
    wd = dist_head.weight.detach().t()
    L, D = wc.shape
    w = torch.zeros((3 * L, 2 * D), device=wc.device, dtype=wc.dtype)
    w[:L, :D] = wc
    w[L:2 * L, D:] = wd
    w[2 * L:, :D] = wc / 2
    w[2 * L:, D:] = wd / 2
    bc = cls_head.bias.detach().float()
    bd = dist_head.bias.detach().float()
    return SimpleNamespace(w=bg.pack_weight_nk(w, pieces), pieces=pieces, labels=L,
                           bias32=torch.cat([bc, bd, (bc + bd) / 2]).contiguous())


def embed_pack(emb, fmt: Optional[tuple] = None) -> SimpleNamespace:
    """``pack_embeddings(emb, fmt)``, cached on the module (``PackedMixin.packed``): the float pack and the pack of one
    set of uint8 constants at a time, rebuilt when a source parameter's storage pointer or version counter changes."""
    return emb.packed() if fmt is None else emb.packed("u8", fmt)


STATS_COLS = 128   # columns per (sum, M2) partial of the row statistics (VT_LN_STATS_COLS in include/vitb200.h)
LN_STATS_MAX_DIM = 1280   # widest row vt_layernorm_stats takes (include/vitb200_clip.h)


def folding_supported(x: torch.Tensor, dim: int, mlp_dim: int) -> bool:
    """LayerNorm folding runs on the bf16 tensor-core GEMM only."""
    return x.is_cuda and x.dtype == torch.bfloat16 and dim % STATS_COLS == 0 and mlp_dim % 8 == 0


def linear_ln(x: torch.Tensor, w_fold: torch.Tensor, b_fold: torch.Tensor, colsum: Optional[torch.Tensor],
              rowstats: torch.Tensor, eps: float, gelu: int = 0) -> torch.Tensor:
    """out = act(LN(x) @ W^T + b) computed as a GEMM on the un-normalised x with the normalisation
    applied per row in the epilogue; ``rowstats`` is the (M, K/128, 2) fp32 table of per-128-column
    (sum, M2) partials of x's rows written by ``linear_res_stats`` (or ``layernorm_stats``).  ``gelu``: the activation
    code, as for ``linear``."""
    B, N, K = x.shape
    n_out = w_fold.shape[0]
    out = torch.empty((B, N, n_out), device=x.device, dtype=x.dtype)
    _lib.call("vt_gemm_bf16_ln", x.data_ptr(), K, w_fold.data_ptr(), K, out.data_ptr(), n_out,
              b_fold.data_ptr(), None, 0, B * N, n_out, K, int(gelu), rowstats.data_ptr(),
              _lib.ptr(colsum), K, float(eps), None, _lib.stream_ptr(x))
    return out


def layernorm_stats(x: torch.Tensor, ln, stats_out: torch.Tensor) -> torch.Tensor:
    """LayerNorm ``ln`` of bf16 (B, N, D) rows that also writes every output row's per-128-column (sum, M2) partials
    into the (B * N, D/128, 2) fp32 ``stats_out`` for the LayerNorm folded into the next GEMM (``vt_layernorm_stats``:
    the same bits as ``ln(x)``)."""
    B, N, D = x.shape
    x = x.contiguous()
    out = torch.empty_like(x)
    _lib.call("vt_layernorm_stats", x.data_ptr(), ln.weight.data_ptr(), ln.bias.data_ptr(), out.data_ptr(),
              stats_out.data_ptr(), B * N, D, D, D, float(ln.eps), _lib.stream_ptr(x))
    return out


def linear_res_stats(x: torch.Tensor, w_nk: torch.Tensor, bias32: torch.Tensor, residual: torch.Tensor,
                     stats_out: torch.Tensor) -> torch.Tensor:
    """out = x @ W^T + b + residual, also writing every output row's per-128-column (sum, M2) partials
    into the (M, N/128, 2) fp32 ``stats_out`` for the LayerNorm folded into the next GEMM."""
    B, N, K = x.shape
    n_out = w_nk.shape[0]
    out = torch.empty((B, N, n_out), device=x.device, dtype=x.dtype)
    _lib.call("vt_gemm_bf16_ln", x.data_ptr(), K, w_nk.data_ptr(), K, out.data_ptr(), n_out,
              bias32.data_ptr(), residual.data_ptr(), n_out, B * N, n_out, K, 0, None, None, 0, 0.0,
              stats_out.data_ptr(), _lib.stream_ptr(x))
    return out


def linear(x: torch.Tensor, w_nk: torch.Tensor, bias32: torch.Tensor, gelu: int = 0,
           residual: Optional[torch.Tensor] = None) -> torch.Tensor:
    """out = epi(x @ w_nk^T + bias) over the flattened (B*N, K) activation.  ``gelu``: the activation code of the
    epilogue (``_lib.VT_ACT_*``: 0 none, 1 exact GELU, 3 quick GELU; False / True are 0 / 1).

    bf16 -> tcgen05 GEMM with bias / GELU / residual fused into the epilogue;
    fp32 -> exact FP32-pipe GEMM (bias / GELU fused, residual added by the add kernel).
    """
    B, N, K = x.shape
    n_out = w_nk.shape[0]
    out = torch.empty((B, N, n_out), device=x.device, dtype=x.dtype)
    M = B * N
    if M == 0:
        return out
    stream = _lib.stream_ptr(x)
    if x.dtype == torch.bfloat16 and K % 8 == 0 and n_out % 8 == 0:
        _lib.call("vt_gemm_bf16", x.data_ptr(), K, w_nk.data_ptr(), K, out.data_ptr(), n_out,
                  _lib.VT_BF16, bias32.data_ptr(), _lib.ptr(residual), n_out, M, n_out, K,
                  int(gelu), stream)
        return out

    if os.environ.get("VT_EXACT_FP32") == "1":      # FP32-pipe kernel, A/B comparisons only
        bias = bias32 if x.dtype == torch.float32 else bias32.to(x.dtype)
        code = _lib.dtype_code(x)
        step = 65535 * 64
        for m0 in range(0, M, step):
            mm = min(step, M - m0)
            es = x.element_size()
            _lib.call("vt_gemm_strided", x.data_ptr() + m0 * K * es, w_nk.data_ptr(),
                      out.data_ptr() + m0 * n_out * es, bias.data_ptr(), mm, n_out, K, 1, 1,
                      _lib.i64x4(0, 0, K, 1), _lib.i64x4(0, 0, 1, K), _lib.i64x4(0, 0, n_out, 1),
                      1.0, int(gelu), code, stream)
        if residual is not None:
            _lib.call("vt_add", out.data_ptr(), residual.data_ptr(), out.data_ptr(), out.numel(), code, stream)
        return out

    # fp32 model (and bf16 layers whose widths are not multiples of 8): tensor cores through vt_bgemm —
    # fp32 operands split into bf16 pieces (kernels/bgemm.py), bias / GELU / residual fused
    pieces = 1 if x.dtype == torch.bfloat16 else bg.split_pieces()
    wp = split_weight(w_nk, pieces)
    bg.dense_rows(x, x.data_ptr(), M, K, K, wp, pieces, n_out, bias32, int(gelu), out,
                  out.data_ptr(), n_out, residual_ptr=_lib.ptr(residual))
    return out


# packed (split) forms of K-major weights, keyed on the packed tensor itself: the [N, K] matrices in the
# PackedMixin namespaces are rebuilt (new tensors) whenever a source parameter changes, so entries die
# with them
_split_cache = {}


def split_weight(w_nk: torch.Tensor, pieces: int) -> torch.Tensor:
    key = (id(w_nk), pieces)
    hit = _split_cache.get(key)
    if hit is not None and hit[0]() is w_nk:
        return hit[1]
    import weakref
    if len(_split_cache) > 1024:
        for k in [k for k, v in _split_cache.items() if v[0]() is None]:
            del _split_cache[k]
    value = bg.pack_weight_nk(w_nk, pieces)
    _split_cache[key] = (weakref.ref(w_nk), value)
    return value


def _embed_batch_step(n_patches: int) -> int:
    """Images per patch-embedding launch: the gather's grid is (token rows, images), at most 65535 images."""
    return min(65535, 65535 * 128 // n_patches)


def _embed_call(stats, b0, n_tok, dim, pk, pos, pixels_ptr, pix_code, out_ptr, nb, C, H, W, P, stream, device,
                interpolate, prefix):
    """Patch embedding of images b0 .. b0 + nb: gather + 2-CTA GEMM in token mode with the bf16 position table ``pos``;
    row statistics of those images go into ``stats`` when given.  ``vt_patch_embed_gemm`` for a square input at the
    model's size with one prefix token, ``vt_patch_embed_gemm_hw`` (``_prefix``) for any (H, W) with ``interpolate`` or
    ``prefix`` tokens in front of the patches."""
    s_ptr = None if stats is None else stats.data_ptr() + b0 * n_tok * (dim // STATS_COLS) * 2 * 4
    tok_pad = (n_tok + 31) // 32 * 32
    work = torch.empty((nb, tok_pad, pk.ldw), device=device, dtype=torch.bfloat16)
    if interpolate or prefix != 1:
        _lib.call_prefix("vt_patch_embed_gemm_hw", prefix, pixels_ptr, pix_code, pk.w.data_ptr(), pk.ldw,
                         pk.bias32.data_ptr(), pos.data_ptr(), out_ptr, s_ptr, work.data_ptr(), nb, C, H, W, P, dim,
                         stream)
    else:
        _lib.call("vt_patch_embed_gemm", pixels_ptr, pix_code, pk.w.data_ptr(), pk.ldw, pk.bias32.data_ptr(),
                  pos.data_ptr(), out_ptr, s_ptr, work.data_ptr(), nb, C, H, P, dim, stream)


def patch_embed(emb, x: torch.Tensor, fmt: Optional[tuple] = None, stats: Optional[torch.Tensor] = None,
                interpolate: bool = False, mask: Optional[torch.Tensor] = None) -> torch.Tensor:
    """Pixels of format ``fmt`` -> token embeddings (B, prefix + n, D) including CLS (and distillation token) and
    position embeddings, prefix = ``emb.num_prefix_tokens``.  ``fmt`` None:
    float pixels (B, C, S, S); ``pixel_format``: raw uint8 NHWC pixels (B, S, S, C), rescale + normalise + patch
    projection in the same launches (bf16 models on the tensor-core path only).
    ``stats``: optional (B * (prefix + n), D/128, 2) fp32 buffer for the row statistics the LayerNorm folded
    into the first QKV GEMM consumes (bf16 tensor-core path only).  ``interpolate``: pixels at any
    H, W >= patch size, n = (H // P) * (W // P), position table resampled to that grid (``pos_grid``).
    ``mask``: checked bool_masked_pos (B, n): masked patches take the mask token (``embed_masked`` on the bf16
    tensor-core path, ``vt_embed_finalize_masked`` on the others)."""
    w = emb.projection.weight
    D = emb.hidden_dim
    if fmt is None:
        B, C, H, W = x.shape
    else:
        assert x.is_cuda and x.dtype == torch.uint8 and x.dim() == 4, \
            f"Raw pixels need to be a CUDA uint8 (B, H, W, C) tensor, provided: {x.dtype}, {tuple(x.shape)}"
        assert w.dtype == torch.bfloat16 and D % 8 == 0, \
            "The fused uint8 input path runs on the bf16 tensor-core kernels only"
        B, C, H, W = pixel_dims(x, fmt)
        if interpolate:
            check_any_size(emb, C, H, W)
        else:
            assert H == W and C == emb.channels, f"Image size {tuple(x.shape[1:])} not matching with the model input size"
    pk = embed_pack(emb, fmt)
    P = emb.patch_size
    n = emb.num_patches
    grid = None                                            # patch grid of an interpolated input, None = the model's own
    if interpolate:
        grid = patch_grid(emb, H, W)
        n = grid[0] * grid[1]
    tensor_core = fmt is not None or (w.dtype == torch.bfloat16 and D % 8 == 0
                                      and x.dtype in (torch.float32, torch.bfloat16))
    if tensor_core:
        pos = grid_table(emb, grid, fmt, False)
        posm = None if mask is None else grid_table(emb, grid, fmt, True)
    else:
        pos = emb.position_embeddings if grid is None or grid == native_grid(emb) else pos_grid(emb, *grid).pos
    prefix = emb.num_prefix_tokens
    n_tok = prefix + n
    x = x.contiguous()
    out = torch.empty((B, n_tok, D), device=x.device, dtype=w.dtype)
    if B == 0:
        return out
    stream = _lib.stream_ptr(x)

    if tensor_core:
        code = _lib.dtype_code(x) if fmt is None else _lib.VT_U8
        if mask is not None:
            embed_masked(emb, x, code, H, W, mask, pk, pos, posm, out, stats)
            return out
        step = _embed_batch_step(n)
        for b0 in range(0, B, step):
            nb = min(step, B - b0)
            _embed_call(stats, b0, n_tok, D, pk, pos, x[b0:].data_ptr(), code, out[b0:].data_ptr(), nb, C, H, W, P,
                        stream, x.device, interpolate, prefix)
        return out
    assert stats is None, "Row statistics come out of the bf16 tensor-core patch embedding only"

    # fp32 / odd-width path: im2col rows, tensor-core GEMM (fp32 operands split into bf16 pieces) straight
    # into rows prefix .. prefix + n - 1 of every image, then the prefix tokens and position embeddings
    from .kernels.patching import patching
    if x.dtype != w.dtype:
        x = x.to(w.dtype)
    if interpolate and (H % P or W % P):
        x = x[:, :, :H // P * P, :W // P * P]               # the pixels no patch covers (patching() copies)
    patches = patching(x, P)
    K = pk.K
    code = _lib.dtype_code(out)
    es = out.element_size()
    if os.environ.get("VT_EXACT_FP32") == "1":
        bias = pk.bias32 if w.dtype == torch.float32 else emb.projection.bias.detach().contiguous()
        for b0 in range(0, B, 32768):
            nb = min(32768, B - b0)
            _lib.call("vt_gemm_strided", patches[b0:].data_ptr(), pk.w.data_ptr(),
                      out[b0:].data_ptr() + prefix * D * es, bias.data_ptr(), n, D, K, nb, 1,
                      _lib.i64x4(n * K, 0, K, 1), _lib.i64x4(0, 0, 1, pk.ldw), _lib.i64x4(n_tok * D, 0, D, 1),
                      1.0, 0, code, stream)
    else:
        pieces = 1 if w.dtype == torch.bfloat16 else bg.split_pieces()
        wp = split_weight(pk.w, pieces)                    # [D, pieces * ldw]: pk.w rows are already padded to 8
        a = bg.pack(patches, patches.data_ptr(), n, K, B, 1, (n * K, 0, K, 1), pieces, pattern=0)
        kk = a.shape[2]
        bg.bgemm(a.data_ptr(), wp.data_ptr(), out, out.data_ptr() + prefix * D * es, n, D, kk, B, 1, (n * kk, 0, kk),
                 (0, 0, kk), (n_tok * D, 0, D), bias32=pk.bias32)
    finalize_embeddings(emb, out, pos, mask)
    return out


def finalize_embeddings(emb, out: torch.Tensor, pos: torch.Tensor, mask: Optional[torch.Tensor]) -> None:
    """Prefix-token rows and position add of embeddings (B, N, D) whose rows prefix.. hold the patch projections, in
    place: ``vt_embed_finalize``, or ``vt_embed_finalize_masked`` (masked patches take the mask token) with a mask."""
    B, n_tok, D = out.shape
    code, stream = _lib.dtype_code(out), _lib.stream_ptr(out)
    rows = emb.prefix_rows()
    if mask is None:
        _lib.call_prefix("vt_embed_finalize", emb.num_prefix_tokens, out.data_ptr(), pos.data_ptr(), rows.data_ptr(), B,
                         n_tok, D, code, stream)
    else:
        _lib.call_prefix("vt_embed_finalize_masked", emb.num_prefix_tokens, out.data_ptr(), pos.data_ptr(),
                         rows.data_ptr(), emb.mask_token.data_ptr(), mask.contiguous().data_ptr(), B, n_tok, D, code,
                         stream)


# ------------------------------------------------------------------------------------------------ bool_masked_pos
def check_mask(emb, mask, x, n_patches: int) -> None:
    """Host-side checks of a ``bool_masked_pos`` for pixels ``x`` with ``n_patches`` patches per image, before anything
    is launched."""
    assert getattr(emb, "mask_token", None) is not None, \
        "bool_masked_pos needs a model built with use_mask_token=True (or add_decoder=True)"
    assert not isinstance(x, (list, tuple)), "bool_masked_pos is not supported with a list of images (ragged batch)"
    assert isinstance(mask, torch.Tensor) and mask.dtype == torch.bool, \
        f"bool_masked_pos must be a torch.bool tensor, provided: {getattr(mask, 'dtype', type(mask))}"
    assert tuple(mask.shape) == (x.shape[0], n_patches), \
        f"bool_masked_pos must be (batch, patches) = {(x.shape[0], n_patches)}, provided: {tuple(mask.shape)}"
    assert mask.device == x.device, f"bool_masked_pos is on {mask.device}, the pixels on {x.device}"


def embed_masked(emb, x: torch.Tensor, pix_code: int, H: int, W: int, mask: torch.Tensor, pk, pos: torch.Tensor,
                 posm: torch.Tensor, out: torch.Tensor, stats: Optional[torch.Tensor]) -> None:
    """Patch embedding with bool_masked_pos into ``out`` (B, N, D) (bf16 tensor-core path): per chunk of images one
    ``vt_patch_embed_masked_gather`` (unpadded patch rows, masked ones zero, and a per-row table of ``pos`` / ``posm``
    rows) and one plain-mode ``vt_gemm_bf16_ln`` with that table as its residual (and the row statistics into
    ``stats``): the epilogue of the token-mode GEMM, so an all-false mask gives the unmasked call's output bit for
    bit."""
    B, n_tok, D = out.shape
    x = x.contiguous()
    mask = mask.contiguous()
    stream = _lib.stream_ptr(out)
    step = min(65535, RAGGED_MAX_ROWS // n_tok)           # the gather's grid.y and the GEMM's 32-bit row count
    for b0 in range(0, B, step):
        nb = min(step, B - b0)
        rows = nb * n_tok
        patches = torch.empty((rows, pk.ldw), device=out.device, dtype=torch.bfloat16)
        table = torch.empty((rows, D), device=out.device, dtype=torch.bfloat16)
        _lib.call_prefix("vt_patch_embed_masked_gather", emb.num_prefix_tokens, x[b0:].data_ptr(), pix_code,
                         mask[b0:].data_ptr(), pos.data_ptr(), posm.data_ptr(), patches.data_ptr(), pk.ldw,
                         table.data_ptr(), nb, emb.channels, H, W, emb.patch_size, D, stream)
        s_ptr = None if stats is None else stats[b0 * n_tok:].data_ptr()
        _lib.call("vt_gemm_bf16_ln", patches.data_ptr(), pk.ldw, pk.w.data_ptr(), pk.ldw, out[b0:].data_ptr(), D,
                  pk.bias32.data_ptr(), table.data_ptr(), D, rows, D, pk.ldw, 0, None, None, 0, 0.0, s_ptr, stream)


def mim_reconstruct(dec: torch.Tensor, gh: int, gw: int, s: int, channels: int, pixels: Optional[torch.Tensor] = None,
                    pix_code: int = 0, norm: Optional[torch.Tensor] = None, rescale: float = 1.0,
                    mask: Optional[torch.Tensor] = None) -> tuple:
    """Decoder output (B, 1 + gh * gw, s * s * C) -> (loss or None, reconstruction (B, C, gh * s, gw * s)) with one
    ``vt_mim_reconstruct`` (PixelShuffle(s) of the patch rows; with ``mask`` also the masked L1 loss against
    ``pixels``, a 0-dim fp32 device tensor, reduced in a fixed order)."""
    B = dec.shape[0]
    dec = dec.contiguous()
    rec = torch.empty((B, channels, gh * s, gw * s), device=dec.device, dtype=dec.dtype)
    loss = partial = None
    if mask is not None:
        loss = torch.empty((), device=dec.device, dtype=torch.float32)
        partial = torch.empty((B * gh * gw,), device=dec.device, dtype=torch.float32)
        pixels = pixels.contiguous()
        mask = mask.contiguous()
    if B:
        _lib.call("vt_mim_reconstruct", dec.data_ptr(), rec.data_ptr(), _lib.dtype_code(dec), B, channels, gh, gw, s,
                  _lib.ptr(pixels), pix_code, _lib.ptr(norm), float(rescale), _lib.ptr(mask), _lib.ptr(partial),
                  _lib.ptr(loss), _lib.stream_ptr(dec))
    elif loss is not None:
        loss.zero_()
    return loss, rec


# ------------------------------------------------------------------------------------------------ any input resolution
POS_GRIDS_KEPT = 4     # resampled position tables kept per Embeddings module, least recently used dropped first


def patch_grid(emb, height: int, width: int) -> tuple:
    """(gh, gw) patch grid of an input: a stride-P convolution drops the last H % P rows and W % P columns."""
    return height // emb.patch_size, width // emb.patch_size


def native_grid(emb) -> tuple:
    """(g0, g0): the patch grid the position table was trained for."""
    g0 = math.isqrt(emb.num_patches)
    assert g0 * g0 == emb.num_patches, f"Position table of {emb.num_patches} patches is not a square grid"
    return g0, g0


def check_any_size(emb, channels: int, height: int, width: int) -> None:
    P = emb.patch_size
    assert channels == emb.channels and height >= P and width >= P, \
        f"Image size {(channels, height, width)} needs {emb.channels} channels and sides of at least the patch size {P}"


def resample_pos_table(pos: torch.Tensor, g_in: int, gh: int, gw: int, prefix: int = 1) -> torch.Tensor:
    """[prefix + g_in^2, D] position table (fp32 | bf16, CUDA) -> fp32 [prefix + gh * gw, D]: the ``prefix`` rows of
    the tokens in front of the patches (CLS, distillation token) copied, the grid resampled bicubically like HF
    ``ViTEmbeddings`` / ``DeiTEmbeddings.interpolate_pos_encoding`` (one ``vt_pos_embed_resample`` launch)."""
    assert pos.is_cuda and pos.dim() == 2 and pos.shape[0] == prefix + g_in * g_in, \
        f"Expected a CUDA [{prefix} + {g_in}^2, D] position table, provided: {tuple(pos.shape)} on {pos.device}"
    pos = pos.contiguous()
    out = torch.empty((prefix + gh * gw, pos.shape[1]), device=pos.device, dtype=torch.float32)
    _lib.call_prefix("vt_pos_embed_resample", prefix, pos.data_ptr(), _lib.dtype_code(pos), out.data_ptr(),
                     pos.shape[1], g_in, gh, gw, _lib.stream_ptr(pos))
    return out


class PosGrid:
    """Position tables of one non-native patch grid, all derived from one resample of the model's table:
    ``pos32`` fp32 [prefix + n, D]; ``pos`` (1, prefix + n, D) in the model's dtype (``Embeddings.interpolate_pos_encoding``
    and ``vt_embed_finalize`` of the fp32 / unfused paths); ``table`` the bf16 tables of the tensor-core patch embedding
    for each pixel format.  A table, once built, is never replaced while this object lives: CUDA graphs keep
    reading it (see ``pos_grid``)."""

    def __init__(self, emb, gh: int, gw: int):
        source = emb.position_embeddings.detach()
        self.pos32 = resample_pos_table(source[0], native_grid(emb)[0], gh, gw, emb.num_prefix_tokens)
        self.pos = self.pos32.to(source.dtype)[None]
        self._tables = {}

    def table(self, emb, fmt: Optional[tuple], masked: bool) -> torch.Tensor:
        """bf16 table for pixels of format ``fmt`` (the pack ``embed_pack(emb, fmt)``): of every token (row t < prefix =
        token_t + pos[t] - the pack's bias), or with ``masked`` of masked patches (mask_token + pos - the pack's bias,
        ``embed_masked``)."""
        table = self._tables.get((fmt, masked))
        if table is None:
            _assert_not_capturing()
            pk = embed_pack(emb, fmt)
            with torch.no_grad():
                if masked:
                    table = _posm16(self.pos32, emb.mask_token, pk.bias32)
                else:
                    table = _posb16(self.pos32, pk.prefix32, pk.bias32)
            self._tables[(fmt, masked)] = table
        return table


def _assert_not_capturing() -> None:
    assert not torch.cuda.is_current_stream_capturing(), \
        "the position tables of a new input resolution are built outside CUDA-graph capture: run the interpolated " \
        "forward once at that resolution first (capture_cuda_graph's warm-up does)"


def pos_grid(emb, gh: int, gw: int, keep: int = POS_GRIDS_KEPT) -> PosGrid:
    """Cached ``PosGrid`` of the (gh, gw) patch grid.  Dropped with the module's packs (``_apply``, ``load_state_dict``,
    ``VIT.invalidate_packed``) and rebuilt when a source parameter's storage pointer or version counter changes; the
    last ``keep`` grids are kept (a ragged batch passes the number of grids it uses, so that repeating the list finds
    every table in the cache).

    A CUDA graph captured at a resolution holds the raw addresses of that grid's tables, so a ``PosGrid`` read during
    capture is also referenced from ``_pos_grids_in_graphs`` for the life of the module: dropping it from the cache
    (eviction, invalidation) never frees memory a captured graph still reads."""
    cache = emb.__dict__.setdefault("_pos_grids", OrderedDict())
    stamp = emb._packed_key(emb._packed_sources())
    hit = cache.get((gh, gw))
    if hit is not None and hit[0] == stamp:
        cache.move_to_end((gh, gw))
        if torch.cuda.is_current_stream_capturing():
            emb.__dict__.setdefault("_pos_grids_in_graphs", {})[id(hit[1])] = hit[1]
        return hit[1]
    if hit is not None:
        cache.clear()                                      # every entry was derived from the old parameters
    _assert_not_capturing()
    with torch.no_grad():
        value = PosGrid(emb, gh, gw)
    cache[(gh, gw)] = (stamp, value)
    while len(cache) > keep:
        cache.popitem(last=False)
    return value


def grid_table(emb, grid: Optional[tuple], fmt: Optional[tuple], masked: bool,
               keep: int = POS_GRIDS_KEPT) -> torch.Tensor:
    """bf16 [prefix + gh * gw, D] position table of the tensor-core patch embedding for patch grid ``grid`` (None: the
    model's own) and pixels of format ``fmt``; with ``masked`` the table of masked patches.  The pack's ``posb16`` /
    ``posm16`` at the trained grid, else ``PosGrid.table`` of the resampled grid; ``keep``: grids ``pos_grid`` keeps."""
    if grid is None or grid == native_grid(emb):
        pk = embed_pack(emb, fmt)
        return pk.posm16 if masked else pk.posb16
    return pos_grid(emb, *grid, keep=keep).table(emb, fmt, masked)


# ------------------------------------------------------------------------------------------------ ragged batches
RAGGED_MAX_ROWS = 2 ** 31 - 1    # packed rows per embedding launch: the GEMM's row count is a 32-bit integer


class RaggedLayout:
    """Where the images of a ragged batch go in the packed (M, D) activation.  Images are grouped by token count, so
    that images with the same count occupy one contiguous row range (one attention call each); inside a group they keep
    the caller's order.  ``order``: caller indices in packed order; ``row0[i]`` / ``tokens[i]``: first row (CLS) and
    token count of caller image i, ``prefix`` tokens in front of its patches; ``groups``: (first row, images, tokens) per
    distinct token count; ``rows`` = M."""

    def __init__(self, grids, prefix: int = 1):
        self.grids = [tuple(g) for g in grids]
        self.prefix = prefix
        self.tokens = [prefix + gh * gw for gh, gw in self.grids]
        self.order = sorted(range(len(self.grids)), key=lambda i: (self.tokens[i], i))
        self.row0 = [0] * len(self.grids)
        self.groups = []
        row = 0
        for i in self.order:
            n = self.tokens[i]
            self.row0[i] = row
            if self.groups and self.groups[-1][2] == n:
                r0, count, _ = self.groups[-1]
                self.groups[-1] = (r0, count + 1, n)
            else:
                self.groups.append((row, 1, n))
            row += n
        self.rows = row

    def chunks(self, max_rows: int = RAGGED_MAX_ROWS) -> list:
        """Consecutive runs of ``order`` of at most ``max_rows`` packed rows each: one patch-embedding launch pair each
        (the gather and the embedding GEMM take a 32-bit row count).  This covers the embedding only; the encoder runs
        over all M rows at once, like a batched forward of M rows."""
        out, cur, rows = [], [], 0
        for i in self.order:
            n = self.tokens[i]
            assert n <= max_rows, f"an image of {n} tokens exceeds {max_rows} rows"
            if cur and rows + n > max_rows:
                out.append(cur)
                cur, rows = [], 0
            cur.append(i)
            rows += n
        if cur:
            out.append(cur)
        return out


def check_ragged(emb, images) -> tuple:
    """Host-side checks of a ragged batch, before anything is launched: a non-empty list of (C, H, W) float32 / bfloat16
    or (H, W, C) uint8 tensors of one dtype, on one device, with the model's channel count and sides of at least one
    patch.  Returns (patch grids, uint8?)."""
    assert isinstance(images, (list, tuple)), f"A ragged batch is a list of images, provided: {type(images)}"
    assert len(images) > 0, "A ragged batch needs at least one image"
    dtype, device = images[0].dtype, images[0].device
    assert dtype in (torch.float32, torch.bfloat16, torch.uint8), \
        f"Images need to be float32 / bfloat16 (C, H, W) or uint8 (H, W, C), provided: {dtype}"
    u8 = dtype == torch.uint8
    grids = []
    for i, img in enumerate(images):
        assert isinstance(img, torch.Tensor) and img.dtype == dtype, \
            f"All images of a ragged batch need one dtype: image 0 is {dtype}, image {i} {getattr(img, 'dtype', type(img))}"
        assert img.device == device, f"All images of a ragged batch need one device: image {i} is on {img.device}"
        assert img.dim() == 3, f"Image {i}: expected {'(H, W, C)' if u8 else '(C, H, W)'}, provided: {tuple(img.shape)}"
        C, H, W = (img.shape[2], img.shape[0], img.shape[1]) if u8 else tuple(img.shape)
        assert C == emb.channels, f"Image {i} has {C} channels, the model {emb.channels}"
        assert H >= emb.patch_size and W >= emb.patch_size, \
            f"Image {i} of size {(H, W)} is smaller than one {emb.patch_size}-pixel patch"
        grids.append(patch_grid(emb, H, W))
    return grids, u8


def _to_device_async(host_bytes: bytes, device) -> torch.Tensor:
    """Bytes -> a device uint8 tensor: staged in pinned host memory, one cudaMemcpyAsync on the current stream (the
    pinned block is not reused before the copy has run)."""
    pinned = torch.empty((len(host_bytes),), dtype=torch.uint8, pin_memory=True)
    ctypes.memmove(pinned.data_ptr(), host_bytes, len(host_bytes))
    dev = torch.empty((len(host_bytes),), dtype=torch.uint8, device=device)
    dev.copy_(pinned, non_blocking=True)
    return dev


def patch_embed_ragged(emb, images, layout: RaggedLayout, stats: Optional[torch.Tensor] = None, u8: bool = False,
                       image_mean=(0.5, 0.5, 0.5), image_std=(0.5, 0.5, 0.5),
                       rescale_factor: float = 1.0 / 255.0) -> torch.Tensor:
    """Images of different sizes (raw uint8 ones with these image-processor constants when ``u8``) -> packed token
    embeddings (1, M, D) in ``layout``'s row order: per chunk of at most
    ``RAGGED_MAX_ROWS`` rows one ``vt_patch_embed_ragged_gather`` (patch rows + per-row position table) and one
    ``vt_gemm_bf16_ln`` over the packed rows with the table as its residual (and ``stats``, (M, D/128, 2) fp32, the row
    statistics for block 0's folded LayerNorm).  Every image's rows equal its own ``interpolate_pos_encoding=True``
    call's bit for bit (bf16 tensor-core path only)."""
    w = emb.projection.weight
    D = emb.hidden_dim
    assert w.is_cuda and w.dtype == torch.bfloat16 and D % 8 == 0, \
        "The ragged patch embedding runs on the bf16 tensor-core kernels only"
    fmt = pixel_format(image_mean, image_std, rescale_factor) if u8 else None
    pk = embed_pack(emb, fmt)
    device = images[0].device
    # every grid's table is held here until the launches are enqueued, and the cache keeps at least this list's grids:
    # a list of many aspect ratios, run again, finds all of its tables instead of resampling each one per call
    grids = list(dict.fromkeys(layout.grids))
    keep = max(POS_GRIDS_KEPT, len(grids))
    tables = {g: grid_table(emb, g, fmt, False, keep) for g in grids}
    pixels = [img.contiguous() for img in images]
    code = _lib.dtype_code(pixels[0]) if fmt is None else _lib.VT_U8
    out = torch.empty((1, layout.rows, D), device=device, dtype=w.dtype)
    stream = _lib.stream_ptr(out)
    for chunk in layout.chunks():
        base = layout.row0[chunk[0]]
        rows = sum(layout.tokens[i] for i in chunk)
        desc = (_lib.RaggedImage * len(chunk))()
        for j, i in enumerate(chunk):
            _, _, h, wd = pixel_dims(pixels[i][None], fmt)
            desc[j] = _lib.RaggedImage(pixels[i].data_ptr(), tables[layout.grids[i]].data_ptr(),
                                       layout.row0[i] - base, h, wd, layout.tokens[i], 0)
        desc_dev = _to_device_async(bytes(desc), device)
        patches = torch.empty((rows, pk.ldw), device=device, dtype=torch.bfloat16)
        table = torch.empty((rows, D), device=device, dtype=torch.bfloat16)
        _lib.call_prefix("vt_patch_embed_ragged_gather", layout.prefix, desc_dev.data_ptr(), len(chunk), code,
                         emb.channels, emb.patch_size, patches.data_ptr(), pk.ldw, table.data_ptr(), D, rows, stream)
        s_ptr = None if stats is None else stats[base:].data_ptr()
        _lib.call("vt_gemm_bf16_ln", patches.data_ptr(), pk.ldw, pk.w.data_ptr(), pk.ldw, out[0, base:].data_ptr(), D,
                  pk.bias32.data_ptr(), table.data_ptr(), D, rows, D, pk.ldw, 0, None, None, 0, 0.0, s_ptr, stream)
    return out


def ragged_attention(qkv: torch.Tensor, num_heads: int, scale: float, groups) -> torch.Tensor:
    """Attention of a packed ragged batch (1, M, 3D): one ``flash_attention`` per group of images with the same token
    count ((first row, images, tokens), ``RaggedLayout.groups``), each over its contiguous row range."""
    from .kernels import flash_attention
    _, M, D3 = qkv.shape
    out = torch.empty((1, M, D3 // 3), device=qkv.device, dtype=qkv.dtype)
    for row0, count, n_tok in groups:
        rows = slice(row0, row0 + count * n_tok)
        flash_attention(qkv[0, rows].view(count, n_tok, D3), num_heads, scale,
                        out=out[0, rows].view(count, n_tok, D3 // 3))
    return out


def gather_rows(x: torch.Tensor, rows) -> torch.Tensor:
    """(len(rows), D) = x[rows, :] of a (M, D) CUDA tensor: one ``vt_gather_rows`` launch (index list uploaded like the
    ragged descriptors)."""
    assert x.is_cuda and x.dim() == 2 and x.stride(1) == 1
    out = torch.empty((len(rows), x.shape[1]), device=x.device, dtype=x.dtype)
    if not rows:
        return out
    idx = _to_device_async(bytes((ctypes.c_int64 * len(rows))(*rows)), x.device)
    _lib.call("vt_gather_rows", x.data_ptr(), x.stride(0), idx.data_ptr(), out.data_ptr(), out.stride(0), len(rows),
              x.shape[1], _lib.dtype_code(x), _lib.stream_ptr(x))
    return out
