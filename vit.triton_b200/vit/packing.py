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
    """Gives a module lazily built, automatically invalidated ``packed(kind)`` namespaces.

    ``kind`` selects a builder ``_build_packed[_<kind>]`` and its source list
    ``_packed_sources[_<kind>]`` (default: every parameter of the module)."""

    def _packed_sources(self):
        return list(self.parameters())

    @staticmethod
    def _packed_key(params):
        return tuple((p.data_ptr(), p._version) for p in params)

    def packed(self, kind: str = ""):
        states = self.__dict__.setdefault("_packed_states", {})
        state = states.get(kind)
        if state is not None:
            params, key, value = state
            if self._packed_key(params) == key:
                return value
        suffix = f"_{kind}" if kind else ""
        params = getattr(self, "_packed_sources" + suffix, self._packed_sources)()
        with torch.no_grad():
            value = getattr(self, "_build_packed" + suffix)()
        states[kind] = (params, self._packed_key(params), value)
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
FP8_ACT_SCALE = 16.0     # LayerNorm outputs are quantised as e4m3(y * 16): |LN(x)| <= sqrt(dim - 1), 448 / 16 = 28
FP8_MID_SCALE = 8.0      # GELU outputs (fc2's operand) as e4m3(g * 8), saturating at |g| = 56


def fp8_supported(x: torch.Tensor, dim: int, mlp_dim: int) -> bool:
    return x.is_cuda and x.dtype == torch.bfloat16 and dim % 16 == 0 and mlp_dim % 128 == 0


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
    the activation scales already divided out (the GEMM epilogue is acc * colscale + bias)."""
    att = block.attention.packed()
    mlp = block.packed()
    wqkv8, sqkv = quantize_weight_fp8(att.wqkv)
    w18, s1 = quantize_weight_fp8(mlp.w1)
    w28, s2 = quantize_weight_fp8(mlp.w2)
    return SimpleNamespace(wqkv8=wqkv8, cqkv=(sqkv / FP8_ACT_SCALE).contiguous(), w18=w18,
                           c1=(s1 / FP8_ACT_SCALE).contiguous(), w28=w28, c2=(s2 / FP8_MID_SCALE).contiguous())


def layernorm_fp8(x: torch.Tensor, ln, scale: float = FP8_ACT_SCALE) -> torch.Tensor:
    """(B, N, D) bf16 -> e4m3(LN(x) * scale) as uint8 (B, N, D): LayerNorm with the GEMM operand's quantisation fused."""
    B, N, D = x.shape
    out = torch.empty((B, N, D), device=x.device, dtype=torch.uint8)
    if out.numel():
        _lib.call("vt_layernorm_fp8", x.data_ptr(), ln.weight.data_ptr(), ln.bias.data_ptr(), out.data_ptr(), B * N, D,
                  D, D, float(ln.eps), float(scale), _lib.stream_ptr(x))
    return out


def linear_fp8(x8: torch.Tensor, w8: torch.Tensor, colscale: torch.Tensor, bias32: torch.Tensor, gelu: bool = False,
               residual: Optional[torch.Tensor] = None, out_fp8: bool = False, out_scale: float = 1.0) -> torch.Tensor:
    """out = act((x8 @ w8^T) * colscale + bias) (+ residual) on tcgen05.mma kind::f8f6f4; x8 / w8 are e4m3 bytes."""
    B, N, K = x8.shape
    n_out = w8.shape[0]
    out = torch.empty((B, N, n_out), device=x8.device, dtype=torch.uint8 if out_fp8 else torch.bfloat16)
    if out.numel():
        _lib.call("vt_gemm_fp8", x8.data_ptr(), K, w8.data_ptr(), K, out.data_ptr(), n_out,
                  _lib.VT_E4M3 if out_fp8 else _lib.VT_BF16, bias32.data_ptr(), colscale.data_ptr(),
                  _lib.ptr(residual), n_out, B * N, n_out, K, 1 if gelu else 0, float(out_scale), _lib.stream_ptr(x8))
    return out


def _posb16(pos32: torch.Tensor, cls_token: torch.Tensor, bias32: torch.Tensor) -> torch.Tensor:
    """bf16 [N, D] position table of the two-launch patch embedding (``vt_patch_embed_gemm``): the GEMM adds the
    conv bias to EVERY row, so row 0 (CLS: a zero patch row) carries cls + pos[0] - bias."""
    t = pos32.clone()
    t[0] += cls_token.detach().float().reshape(-1) - bias32
    return t.to(torch.bfloat16).contiguous()


def _posm16(pos32: torch.Tensor, mask_token: Optional[torch.Tensor], bias32: torch.Tensor) -> Optional[torch.Tensor]:
    """bf16 [N, D] table of masked patches (``vt_patch_embed_masked_gather``): a masked patch's row is zero, so the GEMM
    gives bias + this row, which must come out as mask_token + pos.  One rounding from fp32; row 0 is not read.  None
    for a model without a mask token."""
    if mask_token is None:
        return None
    return (pos32 + mask_token.detach().float().reshape(-1) - bias32).to(torch.bfloat16).contiguous()


def pack_embeddings(emb) -> SimpleNamespace:
    w = emb.projection.weight.detach()
    D = w.shape[0]
    K = w[0].numel()
    kpad = (K + 7) // 8 * 8
    w2d = torch.zeros((D, kpad), device=w.device, dtype=w.dtype)
    w2d[:, :K] = w.reshape(D, K)
    pos = emb.position_embeddings.detach().float()[0]          # [N, D]
    posb = pos.clone()
    posb[0] += emb.cls_token.detach().float().reshape(-1)
    posb[1:] += emb.projection.bias.detach().float()
    bias32 = emb.projection.bias.detach().float().contiguous()
    return SimpleNamespace(w=w2d, ldw=kpad, K=K, posb=posb.contiguous(), bias32=bias32,
                           posb16=_posb16(pos, emb.cls_token, bias32), posm16=_posm16(pos, emb.mask_token, bias32))


def pack_embeddings_u8(emb, image_mean, image_std, rescale_factor: float) -> SimpleNamespace:
    """Patch projection for RAW uint8 NHWC pixels: the image processor's
    ``(x * rescale_factor - mean_c) / std_c`` (HF ViTImageProcessor: 1/255, 0.5, 0.5) is folded into
    the operands, so the kernel multiplies bytes:

        sum_k w[d,k] * (x_k * r - mean_c) / std_c  =  sum_k (w[d,k] * r / std_c) * x_k  -  sum_k w[d,k] * mean_c / std_c

    The weight is re-ordered from the reference's (c, i, j) to (i, j, c) — a patch row of an NHWC
    image is P*C contiguous bytes — and scaled in fp32 before the single rounding to bf16; the
    constant term joins the conv bias in the fp32 position/bias table."""
    w = emb.projection.weight.detach().float()                 # [D, C, P, P]
    D, C = w.shape[0], w.shape[1]
    mean = torch.as_tensor(image_mean, dtype=torch.float32, device=w.device).reshape(1, C, 1, 1)
    std = torch.as_tensor(image_std, dtype=torch.float32, device=w.device).reshape(1, C, 1, 1)
    w_scaled = w * (float(rescale_factor) / std)
    offset = (w * (mean / std)).sum(dim=(1, 2, 3))              # [D]
    K = w[0].numel()
    kpad = (K + 7) // 8 * 8
    w2d = torch.zeros((D, kpad), device=w.device, dtype=emb.projection.weight.dtype)
    w2d[:, :K] = w_scaled.permute(0, 2, 3, 1).reshape(D, K).to(w2d.dtype)
    pos = emb.position_embeddings.detach().float()[0]
    posb = pos.clone()
    posb[0] += emb.cls_token.detach().float().reshape(-1)
    posb[1:] += emb.projection.bias.detach().float() - offset
    bias32 = (emb.projection.bias.detach().float() - offset).contiguous()
    return SimpleNamespace(w=w2d, ldw=kpad, K=K, posb=posb.contiguous(), bias32=bias32,
                           posb16=_posb16(pos, emb.cls_token, bias32), posm16=_posm16(pos, emb.mask_token, bias32))


def u8_pack(emb, image_mean, image_std, rescale_factor: float) -> tuple:
    """(key, pack) of ``pack_embeddings_u8`` for these image-processor constants, cached on the module (one set of
    constants at a time) and rebuilt when a source parameter's storage pointer or version counter changes."""
    key = (tuple(float(m) for m in image_mean), tuple(float(v) for v in image_std), float(rescale_factor))
    cache = emb.__dict__.setdefault("_u8_pack", {})
    params = emb._packed_sources()
    stamp = emb._packed_key(params)
    hit = cache.get(key)
    if hit is None or hit[0] != stamp:
        with torch.no_grad():
            hit = (stamp, pack_embeddings_u8(emb, image_mean, image_std, rescale_factor))
        cache.clear()
        cache[key] = hit
    return key, hit[1]


def patch_embed_u8(emb, x: torch.Tensor, image_mean, image_std, rescale_factor: float,
                   stats: Optional[torch.Tensor] = None, interpolate: bool = False,
                   mask: Optional[torch.Tensor] = None) -> torch.Tensor:
    """Raw uint8 NHWC pixels (B, S, S, C) -> token embeddings (B, n+1, D), rescale + normalise + patch
    projection + CLS + position embeddings in ONE kernel (bf16 models on the tensor-core path).
    ``interpolate``: any (B, H, W, C) with H, W >= patch size, position table resampled to its patch grid
    (``pos_grid``).  ``mask``: checked bool_masked_pos (B, n), masked patches take the mask token (``embed_masked``)."""
    w = emb.projection.weight
    assert x.is_cuda and x.dtype == torch.uint8 and x.dim() == 4, \
        f"Raw pixels need to be a CUDA uint8 (B, H, W, C) tensor, provided: {x.dtype}, {tuple(x.shape)}"
    assert w.dtype == torch.bfloat16 and emb.hidden_dim % 8 == 0, \
        "The fused uint8 input path runs on the bf16 tensor-core kernels only"
    B, S, S2, C = x.shape
    if interpolate:
        check_any_size(emb, C, S, S2)
    else:
        assert S == S2 and C == emb.channels, f"Image size {tuple(x.shape[1:])} not matching with the model input size"
    _, pk = u8_pack(emb, image_mean, image_std, rescale_factor)
    x = x.contiguous()
    n = emb.num_patches
    hw = posb16 = None
    posm16 = pk.posm16
    if interpolate:
        grid = patch_grid(emb, S, S2)
        n = grid[0] * grid[1]
        hw = (S, S2)
        if grid != native_grid(emb):
            pg = pos_grid(emb, *grid)
            posb16 = pg.token_table_u8(emb, image_mean, image_std, rescale_factor)
            if mask is not None:
                posm16 = pg.mask_table_u8(emb, image_mean, image_std, rescale_factor)
    n_tok = n + 1
    out = torch.empty((B, n_tok, emb.hidden_dim), device=x.device, dtype=w.dtype)
    if B == 0:
        return out
    if mask is not None:
        embed_masked(emb, x, _lib.VT_U8, S, S2, mask, pk, pk.posb16 if posb16 is None else posb16, posm16, out, stats)
        return out
    stream = _lib.stream_ptr(x)
    step = _embed_batch_step(n)
    for b0 in range(0, B, step):
        nb = min(step, B - b0)
        _embed_call(stats, b0, n_tok, emb.hidden_dim, pk, x[b0:].data_ptr(), _lib.VT_U8, out[b0:].data_ptr(), nb, C, S,
                    emb.patch_size, stream, x.device, hw=hw, posb16=posb16)
    return out


STATS_COLS = 128   # columns per (sum, M2) partial of the row statistics (VT_LN_STATS_COLS in include/vitb200.h)


def folding_supported(x: torch.Tensor, dim: int, mlp_dim: int) -> bool:
    """LayerNorm folding runs on the bf16 tensor-core GEMM only."""
    return x.is_cuda and x.dtype == torch.bfloat16 and dim % STATS_COLS == 0 and mlp_dim % 8 == 0


def linear_ln(x: torch.Tensor, w_fold: torch.Tensor, b_fold: torch.Tensor, colsum: Optional[torch.Tensor],
              rowstats: torch.Tensor, eps: float, gelu: bool = False) -> torch.Tensor:
    """out = act(LN(x) @ W^T + b) computed as a GEMM on the un-normalised x with the normalisation
    applied per row in the epilogue; ``rowstats`` is the (M, K/128, 2) fp32 table of per-128-column
    (sum, M2) partials of x's rows written by ``linear_res_stats``."""
    B, N, K = x.shape
    n_out = w_fold.shape[0]
    out = torch.empty((B, N, n_out), device=x.device, dtype=x.dtype)
    _lib.call("vt_gemm_bf16_ln", x.data_ptr(), K, w_fold.data_ptr(), K, out.data_ptr(), n_out,
              b_fold.data_ptr(), None, 0, B * N, n_out, K, 1 if gelu else 0, rowstats.data_ptr(),
              _lib.ptr(colsum), K, float(eps), None, _lib.stream_ptr(x))
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


def linear(x: torch.Tensor, w_nk: torch.Tensor, bias32: torch.Tensor, gelu: bool = False,
           residual: Optional[torch.Tensor] = None) -> torch.Tensor:
    """out = epi(x @ w_nk^T + bias) over the flattened (B*N, K) activation.

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
                  1 if gelu else 0, stream)
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
                      1.0, 1 if gelu else 0, code, stream)
        if residual is not None:
            _lib.call("vt_add", out.data_ptr(), residual.data_ptr(), out.data_ptr(), out.numel(), code, stream)
        return out

    # fp32 model (and bf16 layers whose widths are not multiples of 8): tensor cores through vt_bgemm —
    # fp32 operands split into bf16 pieces (kernels/bgemm.py), bias / GELU / residual fused
    pieces = 1 if x.dtype == torch.bfloat16 else bg.split_pieces()
    wp = split_weight(w_nk, pieces)
    bg.dense_rows(x, x.data_ptr(), M, K, K, wp, pieces, n_out, bias32, bg.ACT_GELU if gelu else bg.ACT_NONE, out,
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


def _two_launch_embed() -> bool:
    """Gather + token-mode GEMM (default) or round 1's single kernel (VT_PATCH_EMBED=1, A/B measurements)."""
    return os.environ.get("VT_PATCH_EMBED", "2") != "1"


def _embed_call(stats, b0, n_tok, dim, pk, pixels_ptr, pix_code, out_ptr, nb, C, S, P, stream, device, hw=None,
                posb16=None):
    """Patch embedding of images b0 .. b0 + nb: ``vt_patch_embed_gemm`` (gather + 2-CTA GEMM in token mode), or the
    single-kernel ``vt_patch_embed[_stats]``; row statistics of those images go into ``stats`` when given.
    ``hw`` = (H, W): an input at any resolution, ``vt_patch_embed_gemm_hw`` with the position table ``posb16``
    (None: the packed one) — always the two-launch form, the single kernel takes square native inputs only."""
    s_ptr = None if stats is None else stats.data_ptr() + b0 * n_tok * (dim // STATS_COLS) * 2 * 4
    if hw is not None:
        tok_pad = (n_tok + 31) // 32 * 32
        work = torch.empty((nb, tok_pad, pk.ldw), device=device, dtype=torch.bfloat16)
        posb16 = pk.posb16 if posb16 is None else posb16
        _lib.call("vt_patch_embed_gemm_hw", pixels_ptr, pix_code, pk.w.data_ptr(), pk.ldw, pk.bias32.data_ptr(),
                  posb16.data_ptr(), out_ptr, s_ptr, work.data_ptr(), nb, C, hw[0], hw[1], P, dim, stream)
        return
    if _two_launch_embed():
        tok_pad = (n_tok + 31) // 32 * 32
        work = torch.empty((nb, tok_pad, pk.ldw), device=device, dtype=torch.bfloat16)
        _lib.call("vt_patch_embed_gemm", pixels_ptr, pix_code, pk.w.data_ptr(), pk.ldw, pk.bias32.data_ptr(),
                  pk.posb16.data_ptr(), out_ptr, s_ptr, work.data_ptr(), nb, C, S, P, dim, stream)
        return
    if stats is None:
        _lib.call("vt_patch_embed", pixels_ptr, pix_code, pk.w.data_ptr(), pk.ldw, pk.posb.data_ptr(), out_ptr,
                  _lib.VT_BF16, nb, C, S, P, dim, stream)
    else:
        _lib.call("vt_patch_embed_stats", pixels_ptr, pix_code, pk.w.data_ptr(), pk.ldw, pk.posb.data_ptr(), out_ptr,
                  _lib.VT_BF16, s_ptr, nb, C, S, P, dim, stream)


def patch_embed(emb, x: torch.Tensor, stats: Optional[torch.Tensor] = None, interpolate: bool = False,
                mask: Optional[torch.Tensor] = None) -> torch.Tensor:
    """Pixels (B, C, S, S) -> token embeddings (B, n+1, D) including CLS and position embeddings.
    ``stats``: optional (B * (n+1), D/128, 2) fp32 buffer for the row statistics the LayerNorm folded
    into the first QKV GEMM consumes (bf16 tensor-core path only).  ``interpolate``: pixels (B, C, H, W) at any
    H, W >= patch size, n = (H // P) * (W // P), position table resampled to that grid (``pos_grid``).
    ``mask``: checked bool_masked_pos (B, n): masked patches take the mask token (``embed_masked`` on the bf16
    tensor-core path, ``vt_embed_finalize_masked`` on the others)."""
    pk = emb.packed()
    w = emb.projection.weight
    B, C, S, S2 = x.shape
    P = emb.patch_size
    D = emb.hidden_dim
    n = emb.num_patches
    grid = None                                            # resampled tables, None = the model's own
    if interpolate:
        gh, gw = patch_grid(emb, S, S2)
        n = gh * gw
        if (gh, gw) != native_grid(emb):
            grid = pos_grid(emb, gh, gw)
    n_tok = n + 1
    x = x.contiguous()
    out = torch.empty((B, n_tok, D), device=x.device, dtype=w.dtype)
    if B == 0:
        return out
    stream = _lib.stream_ptr(x)

    if w.dtype == torch.bfloat16 and D % 8 == 0 and x.dtype in (torch.float32, torch.bfloat16):
        if mask is not None:
            pos, posm = (pk.posb16, pk.posm16) if grid is None else (grid.token_table(emb), grid.mask_table(emb))
            embed_masked(emb, x, _lib.dtype_code(x), S, S2, mask, pk, pos, posm, out, stats)
            return out
        hw = (S, S2) if interpolate else None
        posb16 = None if grid is None else grid.token_table(emb)
        step = _embed_batch_step(n)
        for b0 in range(0, B, step):
            nb = min(step, B - b0)
            _embed_call(stats, b0, n_tok, D, pk, x[b0:].data_ptr(), _lib.dtype_code(x), out[b0:].data_ptr(), nb, C, S, P,
                        stream, x.device, hw=hw, posb16=posb16)
        return out
    assert stats is None, "Row statistics come out of the bf16 tensor-core patch embedding only"

    # fp32 / odd-width path: im2col rows, tensor-core GEMM (fp32 operands split into bf16 pieces) straight
    # into rows 1..n of every image, then CLS / position embeddings
    from .kernels.patching import patching
    if x.dtype != w.dtype:
        x = x.to(w.dtype)
    if interpolate and (S % P or S2 % P):
        x = x[:, :, :S // P * P, :S2 // P * P]             # the pixels no patch covers (patching() copies)
    patches = patching(x, P)
    K = pk.K
    code = _lib.dtype_code(out)
    es = out.element_size()
    if os.environ.get("VT_EXACT_FP32") == "1":
        bias = pk.bias32 if w.dtype == torch.float32 else emb.projection.bias.detach().contiguous()
        for b0 in range(0, B, 32768):
            nb = min(32768, B - b0)
            _lib.call("vt_gemm_strided", patches[b0:].data_ptr(), pk.w.data_ptr(),
                      out[b0:].data_ptr() + D * es, bias.data_ptr(), n, D, K, nb, 1,
                      _lib.i64x4(n * K, 0, K, 1), _lib.i64x4(0, 0, 1, pk.ldw), _lib.i64x4(n_tok * D, 0, D, 1),
                      1.0, 0, code, stream)
    else:
        pieces = 1 if w.dtype == torch.bfloat16 else bg.split_pieces()
        wp = split_weight(pk.w, pieces)                    # [D, pieces * ldw]: pk.w rows are already padded to 8
        a = bg.pack(patches, patches.data_ptr(), n, K, B, 1, (n * K, 0, K, 1), pieces, pattern=0)
        kk = a.shape[2]
        bg.bgemm(a.data_ptr(), wp.data_ptr(), out, out.data_ptr() + D * es, n, D, kk, B, 1, (n * kk, 0, kk),
                 (0, 0, kk), (n_tok * D, 0, D), bias32=pk.bias32)
    pos = emb.position_embeddings if grid is None else grid.pos
    finalize_embeddings(emb, out, pos, mask)
    return out


def finalize_embeddings(emb, out: torch.Tensor, pos: torch.Tensor, mask: Optional[torch.Tensor]) -> None:
    """CLS row and position add of embeddings (B, N, D) whose rows 1.. hold the patch projections, in place:
    ``vt_embed_finalize``, or ``vt_embed_finalize_masked`` (masked patches take the mask token) with a mask."""
    B, n_tok, D = out.shape
    code, stream = _lib.dtype_code(out), _lib.stream_ptr(out)
    if mask is None:
        _lib.call("vt_embed_finalize", out.data_ptr(), pos.data_ptr(), emb.cls_token.data_ptr(), B, n_tok, D, code,
                  stream)
    else:
        _lib.call("vt_embed_finalize_masked", out.data_ptr(), pos.data_ptr(), emb.cls_token.data_ptr(),
                  emb.mask_token.data_ptr(), mask.contiguous().data_ptr(), B, n_tok, D, code, stream)


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
        _lib.call("vt_patch_embed_masked_gather", x[b0:].data_ptr(), pix_code, mask[b0:].data_ptr(), pos.data_ptr(),
                  posm.data_ptr(), patches.data_ptr(), pk.ldw, table.data_ptr(), nb, emb.channels, H, W,
                  emb.patch_size, D, stream)
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


def resample_pos_table(pos: torch.Tensor, g_in: int, gh: int, gw: int) -> torch.Tensor:
    """[1 + g_in^2, D] position table (fp32 | bf16, CUDA) -> fp32 [1 + gh * gw, D]: row 0 copied, the grid resampled
    bicubically like HF ``ViTEmbeddings.interpolate_pos_encoding`` (one ``vt_pos_embed_resample`` launch)."""
    assert pos.is_cuda and pos.dim() == 2 and pos.shape[0] == 1 + g_in * g_in, \
        f"Expected a CUDA [1 + {g_in}^2, D] position table, provided: {tuple(pos.shape)} on {pos.device}"
    pos = pos.contiguous()
    out = torch.empty((1 + gh * gw, pos.shape[1]), device=pos.device, dtype=torch.float32)
    _lib.call("vt_pos_embed_resample", pos.data_ptr(), _lib.dtype_code(pos), out.data_ptr(), pos.shape[1], g_in, gh, gw,
              _lib.stream_ptr(pos))
    return out


class PosGrid:
    """Position tables of one non-native patch grid, all derived from one resample of the model's table:
    ``pos32`` fp32 [1 + n, D]; ``pos`` (1, 1 + n, D) in the model's dtype (``Embeddings.interpolate_pos_encoding``,
    and ``vt_embed_finalize`` of the fp32 / unfused paths); ``token_table`` / ``token_table_u8`` the bf16 tables of
    the two-launch patch embedding (row 0 = cls + pos[0] - the pack's bias); ``mask_table`` / ``mask_table_u8`` those
    of masked patches (mask_token + pos - the pack's bias, ``embed_masked``).  A table, once built, is never replaced
    while this object lives: CUDA graphs keep reading it (see ``pos_grid``)."""

    def __init__(self, emb, gh: int, gw: int):
        source = emb.position_embeddings.detach()
        self.pos32 = resample_pos_table(source[0], native_grid(emb)[0], gh, gw)
        self.pos = self.pos32.to(source.dtype)[None]
        self._plain = None
        self._u8 = {}
        self._plain_masked = None
        self._u8_masked = {}

    def token_table(self, emb) -> torch.Tensor:
        """bf16 table for pixels in NCHW (the pack ``emb.packed()``)."""
        if self._plain is None:
            _assert_not_capturing()
            with torch.no_grad():
                self._plain = _posb16(self.pos32, emb.cls_token, emb.packed().bias32)
        return self._plain

    def token_table_u8(self, emb, image_mean, image_std, rescale_factor: float) -> torch.Tensor:
        """bf16 table for raw uint8 NHWC pixels with these image-processor constants (the pack ``u8_pack``)."""
        key, pk = u8_pack(emb, image_mean, image_std, rescale_factor)
        table = self._u8.get(key)
        if table is None:
            _assert_not_capturing()
            with torch.no_grad():
                table = self._u8[key] = _posb16(self.pos32, emb.cls_token, pk.bias32)
        return table

    def mask_table(self, emb) -> torch.Tensor:
        """bf16 table of masked patches for pixels in NCHW (the pack ``emb.packed()``)."""
        if self._plain_masked is None:
            _assert_not_capturing()
            with torch.no_grad():
                self._plain_masked = _posm16(self.pos32, emb.mask_token, emb.packed().bias32)
        return self._plain_masked

    def mask_table_u8(self, emb, image_mean, image_std, rescale_factor: float) -> torch.Tensor:
        """bf16 table of masked patches for raw uint8 NHWC pixels with these image-processor constants."""
        key, pk = u8_pack(emb, image_mean, image_std, rescale_factor)
        table = self._u8_masked.get(key)
        if table is None:
            _assert_not_capturing()
            with torch.no_grad():
                table = self._u8_masked[key] = _posm16(self.pos32, emb.mask_token, pk.bias32)
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


# ------------------------------------------------------------------------------------------------ ragged batches
RAGGED_MAX_ROWS = 2 ** 31 - 1    # packed rows per embedding launch: the GEMM's row count is a 32-bit integer


class RaggedLayout:
    """Where the images of a ragged batch go in the packed (M, D) activation.  Images are grouped by token count, so
    that images with the same count occupy one contiguous row range (one attention call each); inside a group they keep
    the caller's order.  ``order``: caller indices in packed order; ``row0[i]`` / ``tokens[i]``: first row (CLS) and
    token count of caller image i; ``groups``: (first row, images, tokens) per distinct token count; ``rows`` = M."""

    def __init__(self, grids):
        self.grids = [tuple(g) for g in grids]
        self.tokens = [1 + gh * gw for gh, gw in self.grids]
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


def _ragged_table(emb, grid, u8: bool, image_mean, image_std, rescale_factor: float, keep: int) -> torch.Tensor:
    """bf16 [1 + gh * gw, D] position table of one grid for the ragged gather: the one the image's own
    interpolate_pos_encoding=True call reads (the packed table at the trained grid).  ``keep``: grids ``pos_grid``
    keeps."""
    if u8:
        if grid == native_grid(emb):
            return u8_pack(emb, image_mean, image_std, rescale_factor)[1].posb16
        return pos_grid(emb, *grid, keep=keep).token_table_u8(emb, image_mean, image_std, rescale_factor)
    if grid == native_grid(emb):
        return emb.packed().posb16
    return pos_grid(emb, *grid, keep=keep).token_table(emb)


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
    """Images of different sizes -> packed token embeddings (1, M, D) in ``layout``'s row order: per chunk of at most
    ``RAGGED_MAX_ROWS`` rows one ``vt_patch_embed_ragged_gather`` (patch rows + per-row position table) and one
    ``vt_gemm_bf16_ln`` over the packed rows with the table as its residual (and ``stats``, (M, D/128, 2) fp32, the row
    statistics for block 0's folded LayerNorm).  Every image's rows equal its own ``interpolate_pos_encoding=True``
    call's bit for bit (bf16 tensor-core path only)."""
    w = emb.projection.weight
    D = emb.hidden_dim
    assert w.is_cuda and w.dtype == torch.bfloat16 and D % 8 == 0, \
        "The ragged patch embedding runs on the bf16 tensor-core kernels only"
    pk = u8_pack(emb, image_mean, image_std, rescale_factor)[1] if u8 else emb.packed()
    device = images[0].device
    # every grid's table is held here until the launches are enqueued, and the cache keeps at least this list's grids:
    # a list of many aspect ratios, run again, finds all of its tables instead of resampling each one per call
    grids = list(dict.fromkeys(layout.grids))
    keep = max(POS_GRIDS_KEPT, len(grids))
    tables = {g: _ragged_table(emb, g, u8, image_mean, image_std, rescale_factor, keep) for g in grids}
    pixels = [img.contiguous() for img in images]
    code = _lib.VT_U8 if u8 else _lib.dtype_code(pixels[0])
    out = torch.empty((1, layout.rows, D), device=device, dtype=w.dtype)
    stream = _lib.stream_ptr(out)
    for chunk in layout.chunks():
        base = layout.row0[chunk[0]]
        rows = sum(layout.tokens[i] for i in chunk)
        desc = (_lib.RaggedImage * len(chunk))()
        for j, i in enumerate(chunk):
            shape = pixels[i].shape
            h, wd = (shape[0], shape[1]) if u8 else (shape[1], shape[2])
            desc[j] = _lib.RaggedImage(pixels[i].data_ptr(), tables[layout.grids[i]].data_ptr(),
                                       layout.row0[i] - base, h, wd, layout.tokens[i], 0)
        desc_dev = _to_device_async(bytes(desc), device)
        patches = torch.empty((rows, pk.ldw), device=device, dtype=torch.bfloat16)
        table = torch.empty((rows, D), device=device, dtype=torch.bfloat16)
        _lib.call("vt_patch_embed_ragged_gather", desc_dev.data_ptr(), len(chunk), code, emb.channels, emb.patch_size,
                  patches.data_ptr(), pk.ldw, table.data_ptr(), D, rows, stream)
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
