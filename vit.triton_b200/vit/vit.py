"""ViT encoder — host-side module tree with the reference's public API (vit/vit.py:25-247).

Class names, constructor arguments, parameter names / shapes (hence state-dict keys) and forward
signatures are those of cmeraki/vit.triton so this file drops in for the reference's; what runs
underneath is different.  Each ``Transformer`` block executes as SEVEN launches (six with the default
LayerNorm fold: ``layernorm_before`` of blocks 1.. runs inside the QKV GEMM's epilogue) of hand-written
sm_100a kernels over the flattened (B*N, D) activation:

    LN1 -> QKV GEMM (all heads, one launch) -> fused attention -> out-proj GEMM (+bias +residual)
        -> LN2 -> fc1 GEMM (+bias +GELU) -> fc2 GEMM (+bias +residual)

instead of the reference's 79 Triton launches + 24 torch copies per block (SURVEY.md 3.1).  The
per-head ``SelfAttention`` / ``LinearWithBias`` modules still exist, own the parameters and can be
run stand-alone (``set_fused(False)`` runs the whole model that way, which is what per-module
forward-hook comparisons against HuggingFace need).

Differences from the reference that are deliberate (SURVEY.md appendix C): the patch projection has
``hidden_dim`` output channels (the reference passes ``patch_dim``, equal only for ViT-B/16), the MLP
width can be set, and dtype / device follow the parameters instead of module-level globals.
"""
import math
import os
from types import SimpleNamespace
from typing import NamedTuple, Optional, Tuple

import torch
from torch import nn

from . import packing
from .kernels import (
    matmul,
    softmax,
    add,
    matmul3,
    LayerNormTriton,
    Conv2DTriton,
    flash_attention,
)
from .kernels import _lib
from .kernels.layernorm import layernorm

_FUSED = True
# Both LayerNorms of a block are folded into the GEMM that consumes them: the normalisation is applied
# per row in that GEMM's epilogue (zero-sum folded weights, packing.fold_layernorm / csrc/ln_fold.cu) and the row
# statistics come out of the epilogue of the GEMM that PRODUCES the row (fc2 of the previous block /
# the patch embedding for layernorm_before, the out-proj for layernorm_after).  Measured in one process
# under the sustained power cap (tools/fold_ab.py): 9.19 / 9.01 / 8.76 ms per forward with no fold / only
# layernorm_before / both — 24 launches and 3.7 GB of activation traffic less per forward.
_FOLD_LN = True
_FOLD_LN_MLP = True    # layernorm_after -> fc1 fold (statistics from the out-proj epilogue), see set_layernorm_folding


# Optional FP8 path (SURVEY.md 8f-3; off by default and off the bf16 headline metric; VT_FP8=1 or set_fp8(True)):
# the QKV, fc1 and fc2 GEMMs of every block run on e4m3 operands (tcgen05.mma kind::f8f6f4): the LayerNorms write
# e4m3 directly, fc1's epilogue writes e4m3 for fc2, weights are quantised per output channel at pack time; the
# attention, the out-projection, the residual stream and the final LayerNorm stay bf16.
_FP8 = os.environ.get("VT_FP8", "0") == "1"


def set_fp8(enabled: bool) -> None:
    global _FP8
    _FP8 = bool(enabled)


def fp8_enabled() -> bool:
    return _FP8


def set_fused(enabled: bool) -> None:
    """Toggle the fused per-block execution (default on).  Off = one kernel entry point per
    reference op, heads processed one by one, every sub-module's forward() is really called."""
    global _FUSED
    _FUSED = bool(enabled)


def fused_enabled() -> bool:
    return _FUSED


def set_layernorm_folding(enabled: bool, mlp: bool = True) -> None:
    """Toggle folding of the LayerNorms into the GEMM epilogues (default: both ON, see the note at _FOLD_LN;
    only affects the fused bf16 path).  ``mlp=False`` keeps layernorm_after as a kernel (6 launches per
    block), ``enabled=False`` both (7 launches per block instead of 5)."""
    global _FOLD_LN, _FOLD_LN_MLP
    _FOLD_LN = bool(enabled)
    _FOLD_LN_MLP = bool(enabled and mlp)


class LinearWithBias(nn.Module):
    """y = act(x @ weight + bias); weight is stored (in, out) like the reference (vit.py:25-35)."""

    def __init__(self, input_dim: int, output_dim: int, activation: Optional[str] = None):
        super().__init__()
        self.weight = nn.Parameter(torch.zeros(input_dim, output_dim))
        self.bias = nn.Parameter(torch.zeros(output_dim))
        self.activation = activation

    def forward(self, x) -> torch.Tensor:
        return matmul(x, self.weight, self.bias, self.activation)


class SelfAttention(nn.Module):
    """One attention head (reference vit.py:38-74).  Stand-alone forward = three projections,
    scaled scores, softmax, weighted sum — each through its kernel entry point."""

    def __init__(self, d_in: int, d_out: int, dropout: int = 0):
        super().__init__()
        self.d_in = d_in
        self.d_out = d_out
        self.query = LinearWithBias(self.d_in, self.d_out)
        self.key = LinearWithBias(self.d_in, self.d_out)
        self.value = LinearWithBias(self.d_in, self.d_out)

    def forward(self, x: torch.Tensor, probs: Optional[list] = None) -> torch.Tensor:
        """``probs``: a list that receives this head's attention probabilities (B, N, N)."""
        q = self.query(x)
        k_t = self.key(x).transpose(1, 2).contiguous()
        v = self.value(x)
        p = softmax(matmul3(q, k_t, apply_scaling=True, scale_factor=1 / math.sqrt(self.d_out)))
        if probs is not None:
            probs.append(p)
        return matmul3(p, v)


def _attention(qkv: torch.Tensor, num_heads: int, scale: float, groups=None, attn: Optional[list] = None) -> torch.Tensor:
    """Fused attention of (B, N, 3D) rows, or of a packed ragged batch (1, M, 3D) when ``groups`` is given.  ``attn``: a
    list that receives the attention probabilities (B, H, N, N) (not with ``groups``)."""
    if groups is None:
        return flash_attention(qkv, num_heads, scale, probs=attn)
    assert attn is None, "attention probabilities are not supported for a list of images"
    return packing.ragged_attention(qkv, num_heads, scale, groups)


class MultiHeadAttention(packing.PackedMixin, nn.Module):
    """All heads + output projection (reference vit.py:77-111)."""

    def __init__(self, num_heads: int, d_in: int, d_out: int):
        super().__init__()
        assert d_in % num_heads == 0, f'Input dimension should be equally divided amongst all heads. d_in%num_heads needs to be 0. Current: {d_in%num_heads}'
        assert d_in / num_heads == d_out, f'`d_out` is not equal to `d_in/num_heads`. Current: {d_in/num_heads}, {d_out}'
        self.num_heads = num_heads
        self.d_in = d_in
        self.d_out = d_out
        self.attention = nn.ModuleList([SelfAttention(d_in=d_in, d_out=d_out) for _ in range(self.num_heads)])
        self.output = LinearWithBias(self.d_in, self.d_in)

    def forward(self, x: torch.Tensor, residual: Optional[torch.Tensor] = None, groups=None,
                attn: Optional[list] = None) -> torch.Tensor:
        """x: (B, N, D).  ``residual`` (fused path only) is added in the out-projection epilogue.  ``groups`` (fused path
        only): x is a packed ragged batch (1, M, D), attention per group of images (``packing.RaggedLayout.groups``).
        ``attn``: a list that receives the attention probabilities of all heads, (B, H, N, N)."""
        if not (_FUSED and x.is_cuda):
            assert residual is None
            heads_out = torch.empty_like(x)
            heads_probs = None if attn is None else []
            for i, head in enumerate(self.attention):
                heads_out[:, :, i * self.d_out:(i + 1) * self.d_out] = head(x, heads_probs)
            if attn is not None:
                attn.append(torch.stack(heads_probs, dim=1))
            return self.output(heads_out)

        pk = self.packed()
        B, N, D = x.shape
        x = x.contiguous()
        qkv = packing.linear(x, pk.wqkv, pk.bqkv)
        ctx = _attention(qkv, self.num_heads, 1.0 / math.sqrt(self.d_out), groups, attn)
        return packing.linear(ctx, pk.wo, pk.bo, residual=residual)

    def _build_packed(self):
        return packing.pack_attention(self)


class Transformer(packing.PackedMixin, nn.Module):
    """Pre-LN encoder block (reference vit.py:114-149): res = x + MHA(LN1(x));
    out = res + W2 . GELU(W1 . LN2(res)).  LayerNorm eps is 1e-12 like HF ViT."""

    def __init__(self, num_heads: int, d_in: int, d_out: int, mlp_dim: Optional[int] = None):
        super().__init__()
        self.num_heads = num_heads
        self.d_in = d_in
        self.d_out = d_out
        self.mlp_dim = 4 * self.d_in if mlp_dim is None else mlp_dim

        self.layernorm_before = LayerNormTriton(self.d_in, eps=1e-12)
        self.attention = MultiHeadAttention(self.num_heads, self.d_in, self.d_out)
        self.intermediate = LinearWithBias(self.d_in, self.mlp_dim, activation='gelu')
        self.output = LinearWithBias(self.mlp_dim, self.d_in)
        self.layernorm_after = LayerNormTriton(self.d_in, eps=1e-12)

    def forward(self, x, groups=None, attn: Optional[list] = None):
        """``attn``: a list that receives the block's attention probabilities (B, H, N, N)."""
        if not (_FUSED and x.is_cuda):
            assert groups is None
            res = add(self.attention(self.layernorm_before(x), attn=attn), x)
            out = self.output(self.intermediate(self.layernorm_after(res)))
            return add(out, res)

        pk = self.packed()
        x = x.contiguous()
        res = self.attention(self.layernorm_before(x), residual=x, groups=groups, attn=attn)
        mid = packing.linear(self.layernorm_after(res), pk.w1, pk.b1, gelu=True)
        return packing.linear(mid, pk.w2, pk.b2, residual=res)

    def _packed_sources(self):
        return [self.intermediate.weight, self.intermediate.bias, self.output.weight, self.output.bias]

    def _build_packed(self):
        return packing.pack_mlp(self)

    def _packed_sources_folded(self):
        return list(self.parameters())

    def _build_packed_folded(self):
        return packing.pack_block_folded(self)

    def _packed_sources_fp8(self):
        return list(self.parameters())

    def _build_packed_fp8(self):
        return packing.pack_block_fp8(self)

    def forward_fp8(self, x: torch.Tensor, groups=None, attn: Optional[list] = None) -> torch.Tensor:
        """Block forward with the QKV / fc1 / fc2 GEMMs on e4m3 operands (7 launches; see the note at _FP8).
        ``groups``, ``attn``: as for ``MultiHeadAttention.forward``."""
        att = self.attention.packed()
        mlp = self.packed()
        q8 = self.packed("fp8")
        x = x.contiguous()
        qkv = packing.linear_fp8(packing.layernorm_fp8(x, self.layernorm_before), q8.wqkv8, q8.cqkv, att.bqkv)
        ctx = _attention(qkv, self.num_heads, 1.0 / math.sqrt(self.d_out), groups, attn)
        res = packing.linear(ctx, att.wo, att.bo, residual=x)
        mid8 = packing.linear_fp8(packing.layernorm_fp8(res, self.layernorm_after), q8.w18, q8.c1, mlp.b1, gelu=True,
                                  out_fp8=True, out_scale=packing.FP8_MID_SCALE)
        return packing.linear_fp8(mid8, q8.w28, q8.c2, mlp.b2, residual=res)

    def forward_folded(self, x: torch.Tensor, ln1_stats: Optional[torch.Tensor], groups=None,
                       attn: Optional[list] = None):
        """Block forward with layernorm_before folded into the QKV GEMM (bf16 only).

        ``ln1_stats``: (M, D/128, 2) fp32 per-128-column (sum, M2) partials of x's rows, written by the
        previous block's last GEMM (None for the first block: layernorm_before then runs as a
        kernel).  Returns (output, statistics of the output rows).  5 launches per block (layernorm_after folded into
        fc1 as well, the default) instead of 7.  ``groups``, ``attn``: as for ``MultiHeadAttention.forward``."""
        att = self.attention.packed()
        mlp = self.packed()
        x = x.contiguous()
        if ln1_stats is None:
            qkv = packing.linear(self.layernorm_before(x), att.wqkv, att.bqkv)
        else:
            pk = self.packed("folded")
            qkv = packing.linear_ln(x, pk.wqkv, pk.bqkv, pk.cqkv, ln1_stats, self.layernorm_before.eps)
        ctx = _attention(qkv, self.num_heads, 1.0 / math.sqrt(self.d_out), groups, attn)
        if _FOLD_LN_MLP:
            pk = self.packed("folded")
            stats2 = torch.empty((x.shape[0] * x.shape[1], self.d_in // packing.STATS_COLS, 2), device=x.device,
                                 dtype=torch.float32)
            res = packing.linear_res_stats(ctx, att.wo, att.bo, x, stats2)
            mid = packing.linear_ln(res, pk.w1, pk.b1, pk.c1, stats2, self.layernorm_after.eps, gelu=True)
        else:
            res = packing.linear(ctx, att.wo, att.bo, residual=x)
            mid = packing.linear(self.layernorm_after(res), mlp.w1, mlp.b1, gelu=True)
        stats = torch.empty((x.shape[0] * x.shape[1], self.d_in // packing.STATS_COLS, 2), device=x.device, dtype=torch.float32)
        out = packing.linear_res_stats(mid, mlp.w2, mlp.b2, res, stats)
        return out, stats


class Encoder(nn.Module):
    """Stack of blocks (reference vit.py:152-170)."""

    def __init__(self, num_layers: int, num_heads: int, hidden_dim: int, d_out: int,
                 mlp_dim: Optional[int] = None):
        super().__init__()
        self.num_layers = num_layers
        self.num_heads = num_heads
        self.hidden_dim = hidden_dim
        self.d_out = d_out
        self.layer = nn.ModuleList(
            Transformer(num_heads=self.num_heads, d_in=self.hidden_dim, d_out=d_out, mlp_dim=mlp_dim)
            for _ in range(self.num_layers)
        )

    def fp8_active(self, x) -> bool:
        return bool(_FUSED and _FP8 and len(self.layer) > 0 and x.numel() > 0 and
                    packing.fp8_supported(x, self.hidden_dim, self.layer[0].mlp_dim))

    def folding_active(self, x) -> bool:
        return bool(_FUSED and _FOLD_LN and not self.fp8_active(x) and len(self.layer) > 0 and x.numel() > 0 and
                    packing.folding_supported(x, self.hidden_dim, self.layer[0].mlp_dim))

    def forward(self, x, ln1_stats: Optional[torch.Tensor] = None, groups=None, hidden: Optional[list] = None,
                attn: Optional[list] = None) -> torch.Tensor:
        """``ln1_stats``: row statistics of x written by the patch-embedding epilogue (see
        ``Embeddings.forward``); without them block 0's layernorm_before runs as a kernel.  ``groups``: x is a
        packed ragged batch (1, M, D) whose attention runs per group of images (``VIT.forward_ragged``).
        ``hidden``: a list that receives x and every block's output (the tensors themselves: each block writes a fresh
        one); ``attn``: a list that receives every block's attention probabilities (B, H, N, N)."""
        if hidden is not None:
            hidden.append(x)
        if self.fp8_active(x):
            for layer in self.layer:
                x = layer.forward_fp8(x, groups, attn)
                if hidden is not None:
                    hidden.append(x)
            return x
        if self.folding_active(x):
            # layernorm_before folded into the QKV GEMM; row statistics of each block's output are
            # produced by its last GEMM's epilogue
            for layer in self.layer:
                x, ln1_stats = layer.forward_folded(x, ln1_stats, groups, attn)
                if hidden is not None:
                    hidden.append(x)
            return x
        for layer in self.layer:
            x = layer(x, groups, attn)
            if hidden is not None:
                hidden.append(x)
        return x


class Embeddings(packing.PackedMixin, nn.Module):
    """Patch projection + CLS token + position embeddings (reference vit.py:173-200)."""

    def __init__(self, patch_size, num_patches, patch_dim, hidden_dim, channels: int = 3, use_mask_token: bool = False):
        super().__init__()
        self.patch_size = patch_size
        self.num_patches = num_patches
        self.patch_dim = patch_dim
        self.hidden_dim = hidden_dim
        self.channels = channels

        self.cls_token = nn.Parameter(torch.zeros((1, 1, hidden_dim)))
        # HF ViTEmbeddings(use_mask_token=True): the embedding of a patch masked by bool_masked_pos
        self.mask_token = nn.Parameter(torch.zeros(1, 1, hidden_dim)) if use_mask_token else None
        self.position_embeddings = nn.Parameter(torch.zeros(1, num_patches + 1, hidden_dim))
        self.projection = Conv2DTriton(
            in_channels=channels,
            out_channels=hidden_dim,
            kernel_size=(self.patch_size, self.patch_size)
        )

    def forward(self, x, stats_out: Optional[torch.Tensor] = None, interpolate_pos_encoding: bool = False,
                bool_masked_pos: Optional[torch.Tensor] = None) -> torch.Tensor:
        """``stats_out`` (optional, fused bf16 path only): (B * N, D/128, 2) fp32 buffer that receives the
        row statistics of the output for the LayerNorm folded into block 0's QKV GEMM.
        ``interpolate_pos_encoding``: (B, C, H, W) at any H, W >= patch size, N = 1 + (H // P) * (W // P), the
        position table resampled to that grid (``interpolate_pos_encoding(H, W)``), like HF ``ViTEmbeddings``.
        ``bool_masked_pos``: bool (B, N - 1), needs ``use_mask_token=True``: a masked patch's embedding is the mask token
        (plus its position embedding), like HF ``ViTEmbeddings``."""
        if bool_masked_pos is not None:
            self.check_mask(bool_masked_pos, x, x.shape[2], x.shape[3], interpolate_pos_encoding)
        if not (_FUSED and x.is_cuda):
            assert stats_out is None
            pos = self.position_embeddings
            if interpolate_pos_encoding:
                H, W = x.shape[2], x.shape[3]
                x = x[:, :, :H // self.patch_size * self.patch_size, :W // self.patch_size * self.patch_size]
                pos = self.interpolate_pos_encoding(H, W)
            tokens = self.projection(x.to(self.projection.weight.dtype)).flatten(2).transpose(1, 2)
            out = torch.empty((x.shape[0], pos.shape[1], self.hidden_dim), device=x.device,
                              dtype=tokens.dtype)
            out[:, 1:, :] = tokens
            packing.finalize_embeddings(self, out, pos, bool_masked_pos)
            return out
        return packing.patch_embed(self, x, stats_out, interpolate=interpolate_pos_encoding, mask=bool_masked_pos)

    def forward_uint8(self, x, image_mean=(0.5, 0.5, 0.5), image_std=(0.5, 0.5, 0.5),
                      rescale_factor: float = 1.0 / 255.0, stats_out: Optional[torch.Tensor] = None,
                      interpolate_pos_encoding: bool = False,
                      bool_masked_pos: Optional[torch.Tensor] = None) -> torch.Tensor:
        """Raw uint8 NHWC pixels (B, H, W, C) -> embeddings: the image processor's rescale and
        normalisation (defaults: HF ``ViTImageProcessor`` of google/vit-base-patch16-224) are folded
        into the patch projection, see ``packing.pack_embeddings_u8``.  ``interpolate_pos_encoding`` and
        ``bool_masked_pos`` as for ``forward``."""
        if bool_masked_pos is not None:
            self.check_mask(bool_masked_pos, x, x.shape[1], x.shape[2], interpolate_pos_encoding)
        return packing.patch_embed_u8(self, x, image_mean, image_std, rescale_factor, stats_out,
                                      interpolate=interpolate_pos_encoding, mask=bool_masked_pos)

    def check_mask(self, bool_masked_pos, x, height: int, width: int, interpolate_pos_encoding: bool) -> None:
        """AssertionError, before anything is launched, unless ``bool_masked_pos`` fits pixels ``x`` of that size."""
        grid = packing.patch_grid(self, height, width)
        packing.check_mask(self, bool_masked_pos, x, grid[0] * grid[1] if interpolate_pos_encoding else self.num_patches)

    def interpolate_pos_encoding(self, height: int, width: int) -> torch.Tensor:
        """(1, 1 + gh * gw, D) position table for a (height, width) input, gh = height // P, gw = width // P:
        HF ``ViTEmbeddings.interpolate_pos_encoding``.  The stored parameter itself at the trained grid; otherwise
        its patch grid resampled bicubically (align_corners=False) by one ``vt_pos_embed_resample`` launch, cached
        per grid for the last few grids (``packing.pos_grid``) with the tables the patch embedding derives from it.
        A new grid's tables are built outside CUDA-graph capture."""
        grid = packing.patch_grid(self, height, width)
        assert grid[0] >= 1 and grid[1] >= 1, f"Image size {(height, width)} is smaller than one {self.patch_size}-pixel patch"
        if grid == packing.native_grid(self):
            return self.position_embeddings
        return packing.pos_grid(self, *grid).pos

    def invalidate_packed(self):
        super().invalidate_packed()
        self.__dict__.pop("_pos_grids", None)

    def _packed_sources(self):
        sources = [self.cls_token, self.position_embeddings, self.projection.weight, self.projection.bias]
        return sources if self.mask_token is None else sources + [self.mask_token]

    def _build_packed(self):
        return packing.pack_embeddings(self)


def _head_on_cls(hidden: torch.Tensor, dense: "LinearWithBias", act: int) -> torch.Tensor:
    """(B, n_out) = act(dense(hidden[:, 0, :])): ONE tensor-core launch (``vt_bgemm``) that reads the CLS
    rows in place through the row stride of its tensor map (no pooling kernel, no copy) and applies bias
    and activation in the epilogue; fp32 models pack the rows into split bf16 pieces first."""
    from .kernels import bgemm as bg
    from .kernels.matmul import _cached
    assert hidden.is_cuda and hidden.dim() == 3 and hidden.stride(2) == 1
    B, _, D = hidden.shape
    w = dense.weight                                       # (in, out)
    n_out = w.shape[1]
    out = torch.empty((B, n_out), device=hidden.device, dtype=hidden.dtype)
    if B == 0:
        return out
    pieces = 1 if hidden.dtype == torch.bfloat16 else bg.split_pieces()
    wp = _cached(w, f"packed{pieces}", lambda p_: bg.pack(p_, p_.data_ptr(), n_out, D, 1, 1,
                                                          (0, 0, p_.stride(1), p_.stride(0)), pieces, pattern=1)[0])
    bias32 = _cached(dense.bias, "f32", lambda b: b.detach().float().contiguous())
    bg.dense_rows(hidden, hidden.data_ptr(), B, D, hidden.stride(0), wp, pieces, n_out, bias32, act, out,
                  out.data_ptr(), n_out)
    return out


class Pooler(nn.Module):
    """HF ``ViTPooler`` (modeling_vit.py:461-474): tanh(dense(CLS hidden state)).  The reference's
    loader already maps ``pooler.dense.{weight,bias}`` (vit/utils.py:63-64) but the reference model has
    no such module; ``VIT(..., add_pooling_layer=True)`` adds it.  On the GPU the dense layer and the tanh
    are one tcgen05 GEMM launch with a tanh epilogue over the CLS rows (``_head_on_cls``); weight is (in, out)."""

    def __init__(self, hidden_dim: int):
        super().__init__()
        self.dense = LinearWithBias(hidden_dim, hidden_dim)

    def forward(self, hidden_states: torch.Tensor) -> torch.Tensor:
        if hidden_states.is_cuda:
            from .kernels import bgemm as bg
            return _head_on_cls(hidden_states, self.dense, bg.ACT_TANH)
        return torch.tanh(self.dense(hidden_states[:, :1, :].contiguous())[:, 0, :])


class DecoderConv(packing.PackedMixin, nn.Module):
    """Parameters of HF ``ViTForMaskedImageModeling.decoder[0]``, the 1x1 ``Conv2d(D, s * s * C)`` in front of the
    PixelShuffle: weight (s * s * C, D, 1, 1), bias (s * s * C,).  ``VIT.masked_image_modeling`` runs it as one GEMM over
    the final hidden states (the weight reshaped to (s * s * C, D) is already K-major)."""

    def __init__(self, hidden_dim: int, out_channels: int):
        super().__init__()
        self.weight = nn.Parameter(torch.zeros(out_channels, hidden_dim, 1, 1))
        self.bias = nn.Parameter(torch.zeros(out_channels))

    def _build_packed(self):
        return SimpleNamespace(w=self.weight.detach().reshape(self.weight.shape[0], -1).contiguous(),
                               b32=self.bias.detach().float().contiguous())


class VITOutput(NamedTuple):
    """What ``VIT.forward`` / ``forward_uint8`` return when ``output_hidden_states`` or ``output_attentions`` is set, like
    HF ``BaseModelOutput``; an unrequested field is None.  ``hidden_states``: num_layers + 1 tensors (B, N, D), the
    embeddings and every block's output before the final LayerNorm.  ``attentions``: num_layers contiguous tensors
    (B, H, N, N) of the model's dtype, softmax(scale * Q K^T) per head."""
    last_hidden_state: torch.Tensor
    hidden_states: Optional[Tuple[torch.Tensor, ...]] = None
    attentions: Optional[Tuple[torch.Tensor, ...]] = None


def _refuse_outputs(what: str, output_hidden_states: bool, output_attentions: bool) -> None:
    assert not (output_hidden_states or output_attentions), \
        f"output_hidden_states / output_attentions are not supported by {what}: call the model itself with them"


class VIT(nn.Module):
    """ViT encoder returning the final-LayerNorm hidden states (B, N, D) — no pooler, like the
    reference (vit.py:203-247) and HF ``ViTModel(add_pooling_layer=False).last_hidden_state``."""

    def __init__(
        self,
        height: int,
        width: int,
        channels: int,
        patch_size: int,
        hidden_dim: int,
        num_heads: int,
        num_layers: int,
        mlp_dim: Optional[int] = None,
        add_pooling_layer: bool = False,
        num_labels: Optional[int] = None,
        use_mask_token: bool = False,
        add_decoder: bool = False,
        encoder_stride: Optional[int] = None,
    ):
        super().__init__()
        assert height == width, "Height and width should be the same"
        assert height % patch_size == 0, "Height should be divisible by the patch size"
        assert width % patch_size == 0, "Width should be divisible by the patch size"

        self.height = height
        self.width = width
        self.channels = channels
        self.patch_size = patch_size
        self.hidden_dim = hidden_dim
        self.num_heads = num_heads
        self.num_layers = num_layers

        assert self.hidden_dim % self.num_heads == 0, f"Hidden dimension should be divisible by number of heads, provided: {self.hidden_dim} {self.num_heads}"

        num_patches = (self.height // self.patch_size) * (self.width // self.patch_size)
        patch_dim = self.patch_size * self.patch_size * self.channels
        d_out = self.hidden_dim // self.num_heads

        self.embeddings = Embeddings(patch_size=self.patch_size, num_patches=num_patches, patch_dim=patch_dim,
                                     hidden_dim=self.hidden_dim, channels=self.channels,
                                     use_mask_token=use_mask_token or add_decoder)
        self.encoder = Encoder(num_layers=self.num_layers, num_heads=self.num_heads, hidden_dim=self.hidden_dim,
                               d_out=d_out, mlp_dim=mlp_dim)
        self.layernorm = LayerNormTriton(dim=self.hidden_dim, eps=1e-12)
        # optional HF pooler (tanh(dense(CLS))): state-dict keys pooler.dense.{weight,bias}
        self.pooler = Pooler(self.hidden_dim) if add_pooling_layer else None
        # optional HF ViTForImageClassification head (Linear on the CLS row of the final hidden states):
        # state-dict keys classifier.{weight,bias}
        self.classifier = LinearWithBias(self.hidden_dim, num_labels) if num_labels else None
        # optional HF ViTForMaskedImageModeling (SimMIM) decoder, Conv2d(D, s^2 C, 1) + PixelShuffle(s) with s =
        # encoder_stride (default: the patch size): state-dict keys decoder.0.{weight,bias}; implies the mask token
        self.encoder_stride = patch_size if encoder_stride is None else encoder_stride
        self.decoder = None
        if add_decoder:
            s = self.encoder_stride
            self.decoder = nn.Sequential(DecoderConv(self.hidden_dim, s * s * self.channels), nn.PixelShuffle(s))

    def invalidate_packed(self) -> None:
        """Drop every derived weight (packed / LayerNorm-folded / uint8-scaled operands of all sub-modules
        and the K-major copies the ``matmul`` entry point keeps).  Needed only after writes that go THROUGH
        ``param.data`` (``p.data.copy_()``, HF-style re-initialisation, EMA): those change neither the
        storage pointer nor the version counter the caches are keyed on; every other kind of update is
        noticed automatically."""
        from .kernels.matmul import clear_derived_cache
        for m in self.modules():
            if isinstance(m, packing.PackedMixin):
                m.invalidate_packed()
            m.__dict__.pop("_u8_pack", None)
        clear_derived_cache()

    @property
    def device(self) -> torch.device:
        return self.layernorm.weight.device

    @property
    def dtype(self) -> torch.dtype:
        return self.layernorm.weight.dtype

    def forward(self, x, interpolate_pos_encoding: bool = False, bool_masked_pos: Optional[torch.Tensor] = None,
                output_hidden_states: bool = False, output_attentions: bool = False):
        """(B, C, H, W) -> final hidden states (B, N, D).  ``interpolate_pos_encoding`` (HF ``ViTModel``'s flag): any
        H, W >= patch size, square or not; N = 1 + (H // P) * (W // P), the position table resampled bicubically to
        that grid (``Embeddings.interpolate_pos_encoding``).  Without it the input must be the model's size.
        ``bool_masked_pos`` (HF ``ViTModel``'s argument, needs ``use_mask_token=True``): bool (B, N - 1) on x's device,
        True = the patch's embedding is replaced by the mask token.  Masked inputs take the gather + GEMM patch
        embedding (``packing.embed_masked``); an all-false mask gives the unmasked result bit for bit.

        ``output_hidden_states`` / ``output_attentions`` (HF ``ViTModel``'s flags): return a ``VITOutput`` instead of the
        tensor, with every layer's hidden states and / or attention probabilities; the final hidden states are the
        same bits as without them.  The hidden states are the tensors the forward computes anyway; on the fused bf16
        path with head dim 64 or 80 each block's probabilities take one ``vt_attn_probs`` launch, elsewhere they are
        the ones the attention materialises.  Not for a list of images."""
        self._check_outputs(x, output_hidden_states, output_attentions)
        if bool_masked_pos is not None:
            assert not isinstance(x, (list, tuple)), "bool_masked_pos is not supported with a list of images"
        if interpolate_pos_encoding:
            assert x.dim() == 4, f"Expected (B, C, H, W) pixels, provided: {tuple(x.shape)}"
            packing.check_any_size(self.embeddings, *x.shape[1:])
            n_tok = 1 + math.prod(packing.patch_grid(self.embeddings, x.shape[2], x.shape[3]))
        else:
            assert x.shape[1:] == (self.channels, self.height, self.width), f"Image size {x.shape[1:]} not matching with the model input size: {self.channels, self.height, self.width}"
            n_tok = None
        if bool_masked_pos is not None:
            self.embeddings.check_mask(bool_masked_pos, x, x.shape[2], x.shape[3], interpolate_pos_encoding)
        stats = self._embed_stats(x, n_tok)
        kw = dict(interpolate_pos_encoding=True) if interpolate_pos_encoding else {}
        if bool_masked_pos is not None:
            kw["bool_masked_pos"] = bool_masked_pos
        x = self.embeddings(x, stats, **kw) if stats is not None else self.embeddings(x, **kw)
        return self._encode(x, stats, output_hidden_states, output_attentions)

    @staticmethod
    def _check_outputs(x, output_hidden_states: bool, output_attentions: bool) -> None:
        if output_hidden_states or output_attentions:
            assert not isinstance(x, (list, tuple)), \
                "output_hidden_states / output_attentions are not supported with a list of images"

    def _encode(self, x: torch.Tensor, stats: Optional[torch.Tensor], output_hidden_states: bool,
                output_attentions: bool):
        """Encoder + final LayerNorm over the embeddings x: the final hidden states, or a ``VITOutput`` when a flag is set."""
        kw = {}
        if output_hidden_states:
            kw["hidden"] = []
        if output_attentions:
            kw["attn"] = []
        x = self.encoder(x, stats, **kw) if stats is not None else self.encoder(x, **kw)
        x = self.layernorm(x)
        if not kw:
            return x
        return VITOutput(x, tuple(kw["hidden"]) if output_hidden_states else None,
                         tuple(kw["attn"]) if output_attentions else None)

    def _embed_stats(self, x: torch.Tensor, n_tok: Optional[int] = None) -> Optional[torch.Tensor]:
        """Buffer for the row statistics of the embeddings when block 0's layernorm_before is folded
        into its QKV GEMM (fused bf16 tensor-core path, hidden size a multiple of 128); None otherwise.
        ``n_tok``: tokens per image (default: the model's own, num_patches + 1)."""
        w = self.embeddings.projection.weight
        batch = x.shape[0]
        if not (x.is_cuda and w.is_cuda and w.dtype == torch.bfloat16 and batch > 0 and self.hidden_dim % 8 == 0
                and x.dtype in (torch.float32, torch.bfloat16, torch.uint8)):
            return None
        probe = torch.empty((1,), device=x.device, dtype=w.dtype)
        if not self.encoder.folding_active(probe):
            return None
        n_tok = self.embeddings.num_patches + 1 if n_tok is None else n_tok
        return torch.empty((batch * n_tok, self.hidden_dim // packing.STATS_COLS, 2), device=x.device,
                           dtype=torch.float32)

    def forward_uint8(self, x, image_mean=(0.5, 0.5, 0.5), image_std=(0.5, 0.5, 0.5),
                      rescale_factor: float = 1.0 / 255.0, interpolate_pos_encoding: bool = False,
                      bool_masked_pos: Optional[torch.Tensor] = None, output_hidden_states: bool = False,
                      output_attentions: bool = False):
        """Forward from RAW uint8 NHWC pixels (B, H, W, C) — the step in front of the reference's
        ``forward``: rescale + normalise (HF ``ViTImageProcessor``) run inside the patch-embedding
        kernel, so the host -> device copy is one byte per pixel value.  ``interpolate_pos_encoding``,
        ``bool_masked_pos``, ``output_hidden_states`` and ``output_attentions`` as for ``forward``."""
        self._check_outputs(x, output_hidden_states, output_attentions)
        if bool_masked_pos is not None:
            assert not isinstance(x, (list, tuple)), "bool_masked_pos is not supported with a list of images"
        if interpolate_pos_encoding:
            assert x.dim() == 4, f"Expected (B, H, W, C) pixels, provided: {tuple(x.shape)}"
            packing.check_any_size(self.embeddings, x.shape[3], x.shape[1], x.shape[2])
            n_tok = 1 + math.prod(packing.patch_grid(self.embeddings, x.shape[1], x.shape[2]))
        else:
            assert tuple(x.shape[1:]) == (self.height, self.width, self.channels), f"Image size {x.shape[1:]} not matching with the model input size: {self.height, self.width, self.channels}"
            n_tok = None
        if bool_masked_pos is not None:
            self.embeddings.check_mask(bool_masked_pos, x, x.shape[1], x.shape[2], interpolate_pos_encoding)
        stats = self._embed_stats(x, n_tok)
        x = self.embeddings.forward_uint8(x, image_mean, image_std, rescale_factor, stats,
                                          interpolate_pos_encoding=interpolate_pos_encoding,
                                          bool_masked_pos=bool_masked_pos)
        return self._encode(x, stats, output_hidden_states, output_attentions)

    def forward_ragged(self, images, image_mean=(0.5, 0.5, 0.5), image_std=(0.5, 0.5, 0.5),
                       rescale_factor: float = 1.0 / 255.0) -> list:
        """Images of different resolutions in one batch: a list of (C, H_i, W_i) float32 / bfloat16 or raw (H_i, W_i, C)
        uint8 tensors (one dtype, the model's channel count, sides of at least one patch) -> the list of final hidden
        states (N_i, D), N_i = 1 + (H_i // P) * (W_i // P), in the caller's order.  Image i gives what
        ``self(images[i][None], interpolate_pos_encoding=True)[0]`` (``forward_uint8`` for uint8, with these image-processor
        constants) gives, bit for bit: each image takes its own patch grid and position table.

        On the fused bf16 path (LayerNorm fold on, only ``layernorm_before`` folded, fold off, FP8) the images' tokens
        are packed into one (sum N_i, D) activation, grouped by token count: one ragged patch gather and one embedding
        GEMM for the list, one launch per dense layer of every block over all rows, one attention launch per distinct
        token count; the returned tensors are views into that buffer.  fp32 models and ``set_fused(False)`` run the list
        image by image through ``forward`` / ``forward_uint8`` (correct, not fast).  Not capturable into a CUDA graph:
        the per-image descriptors are uploaded from the host on every call."""
        hidden, layout = self._ragged_hidden(images, image_mean, image_std, rescale_factor)
        return [hidden[r:r + n] for r, n in zip(layout.row0, layout.tokens)]

    def _ragged_hidden(self, images, image_mean, image_std, rescale_factor) -> tuple:
        """(packed final hidden states (M, D), ``packing.RaggedLayout``) of a ragged batch."""
        grids, u8 = packing.check_ragged(self.embeddings, images)
        assert not torch.cuda.is_current_stream_capturing(), "A ragged batch cannot be captured into a CUDA graph"
        layout = packing.RaggedLayout(grids)
        first = images[0]
        if not (_FUSED and first.is_cuda and self.dtype == torch.bfloat16 and self.hidden_dim % 8 == 0):
            hidden = None
            for i in layout.order:
                if u8:
                    h = self.forward_uint8(images[i][None], image_mean, image_std, rescale_factor,
                                           interpolate_pos_encoding=True)
                else:
                    h = self.forward(images[i][None], interpolate_pos_encoding=True)
                if hidden is None:
                    hidden = torch.empty((layout.rows, h.shape[2]), device=h.device, dtype=h.dtype)
                hidden[layout.row0[i]:layout.row0[i] + layout.tokens[i]].copy_(h[0])
            return hidden, layout
        stats = self._embed_stats(first[None], layout.rows)       # one "image" of M rows
        x = packing.patch_embed_ragged(self.embeddings, images, layout, stats, u8, image_mean, image_std,
                                       rescale_factor)
        x = self.encoder(x, stats, groups=layout.groups)
        x = self.layernorm(x)
        return x[0], layout

    def _ragged_cls(self, images) -> torch.Tensor:
        """(B, D) CLS rows of the final hidden states of a ragged batch, in the caller's order (``vt_gather_rows``)."""
        hidden, layout = self._ragged_hidden(images, (0.5, 0.5, 0.5), (0.5, 0.5, 0.5), 1.0 / 255.0)
        return packing.gather_rows(hidden, layout.row0)

    def _hidden(self, x, interpolate_pos_encoding: bool, bool_masked_pos: Optional[torch.Tensor] = None,
                image_mean=(0.5, 0.5, 0.5), image_std=(0.5, 0.5, 0.5),
                rescale_factor: float = 1.0 / 255.0) -> torch.Tensor:
        """Final hidden states of pixels (B, C, H, W) or raw uint8 (B, H, W, C); a list of images (ragged batch) is
        refused when a mask is given."""
        assert bool_masked_pos is None or not isinstance(x, (list, tuple)), \
            "bool_masked_pos is not supported with a list of images"
        kw = dict(interpolate_pos_encoding=True) if interpolate_pos_encoding else {}
        if bool_masked_pos is not None:
            kw["bool_masked_pos"] = bool_masked_pos
        if x.dtype == torch.uint8:
            return self.forward_uint8(x, image_mean, image_std, rescale_factor, **kw)
        return self.forward(x, **kw)

    def _cls_hidden(self, x, interpolate_pos_encoding: bool, bool_masked_pos) -> torch.Tensor:
        """(B, N, D) final hidden states, or (B, 1, D) CLS rows of a list of images (ragged batch)."""
        if isinstance(x, (list, tuple)):
            assert bool_masked_pos is None, "bool_masked_pos is not supported with a list of images"
            return self._ragged_cls(x)[:, None, :]
        return self._hidden(x, interpolate_pos_encoding, bool_masked_pos)

    def pooler_output(self, x, interpolate_pos_encoding: bool = False,
                      bool_masked_pos: Optional[torch.Tensor] = None, output_hidden_states: bool = False,
                      output_attentions: bool = False) -> torch.Tensor:
        """HF ``ViTModel(...).pooler_output``: tanh(dense(final hidden state of CLS)), (B, D).  ``x`` may also be a list
        of images of different sizes (``forward_ragged``), each with its own patch grid (without a mask)."""
        _refuse_outputs("pooler_output", output_hidden_states, output_attentions)
        assert self.pooler is not None, "Model was built without add_pooling_layer=True"
        return self.pooler(self._cls_hidden(x, interpolate_pos_encoding, bool_masked_pos))

    def logits(self, x, interpolate_pos_encoding: bool = False,
               bool_masked_pos: Optional[torch.Tensor] = None, output_hidden_states: bool = False,
               output_attentions: bool = False) -> torch.Tensor:
        """Class logits (B, num_labels) = classifier(final hidden states[:, 0]) — HF
        ``ViTForImageClassification(...).logits``; needs ``VIT(..., num_labels=...)``.  One tensor-core
        launch over the CLS rows of the final hidden states.  ``x`` may also be a list of images of different sizes
        (``forward_ragged``), each with its own patch grid (without a mask)."""
        _refuse_outputs("logits", output_hidden_states, output_attentions)
        assert self.classifier is not None, "VIT was built without a classifier head (num_labels)"
        hidden = self._cls_hidden(x, interpolate_pos_encoding, bool_masked_pos)
        from .kernels import bgemm as bg
        return _head_on_cls(hidden, self.classifier, bg.ACT_NONE)

    def pooled(self, x, interpolate_pos_encoding: bool = False,
               bool_masked_pos: Optional[torch.Tensor] = None, output_hidden_states: bool = False,
               output_attentions: bool = False) -> torch.Tensor:
        """CLS row of the final hidden states, (B, D): the tensor the data-parallel wrapper gathers.
        uint8 (B, H, W, C) inputs take the fused raw-pixel path.  ``x`` may also be a list of images of different sizes
        (``forward_ragged``), each with its own patch grid (without a mask)."""
        _refuse_outputs("pooled", output_hidden_states, output_attentions)
        if isinstance(x, (list, tuple)):
            assert bool_masked_pos is None, "bool_masked_pos is not supported with a list of images"
            return self._ragged_cls(x)
        hidden = self._hidden(x, interpolate_pos_encoding, bool_masked_pos)
        out = torch.empty((hidden.shape[0], hidden.shape[2]), device=hidden.device, dtype=hidden.dtype)
        _lib.call("vt_pool_cls", hidden.data_ptr(), out.data_ptr(), hidden.shape[0], hidden.shape[2],
                  hidden.stride(0), _lib.dtype_code(hidden), _lib.stream_ptr(hidden))
        return out

    def masked_image_modeling(self, x, bool_masked_pos: Optional[torch.Tensor] = None,
                              interpolate_pos_encoding: bool = False, image_mean=(0.5, 0.5, 0.5),
                              image_std=(0.5, 0.5, 0.5), rescale_factor: float = 1.0 / 255.0,
                              output_hidden_states: bool = False, output_attentions: bool = False) -> tuple:
        """HF ``ViTForMaskedImageModeling`` (SimMIM): (loss or None, reconstruction (B, C, gh * s, gw * s)) like its
        ``MaskedImageModelingOutput``; needs ``VIT(..., add_decoder=True)``, s = ``encoder_stride``.  ``x``: pixels
        (B, C, H, W) or raw uint8 (B, H, W, C) (normalised with these image-processor constants, as ``forward_uint8``).

        The decoder's 1x1 convolution is one GEMM over the final hidden states (CLS rows included), and one
        ``vt_mim_reconstruct`` launch pixel-shuffles its patch rows into the reconstruction in the model's dtype; with
        ``bool_masked_pos`` the same pass computes the masked L1 loss against the (normalised) input pixels, a 0-dim
        fp32 device tensor reduced in a fixed order (no host synchronisation, the same bits on every call).  The loss
        needs s == P and H, W multiples of P; the reconstruction works on any grid (HF only defines square ones)."""
        _refuse_outputs("masked_image_modeling", output_hidden_states, output_attentions)
        assert self.decoder is not None, "VIT was built without the masked image modeling decoder (add_decoder=True)"
        assert not isinstance(x, (list, tuple)), "masked_image_modeling takes a batch tensor, not a list of images"
        u8 = x.dtype == torch.uint8
        H, W = (x.shape[1], x.shape[2]) if u8 else (x.shape[2], x.shape[3])
        s = self.encoder_stride
        P = self.patch_size
        if bool_masked_pos is not None:
            assert s == P, f"The masked image modeling loss needs encoder_stride == patch_size, got {s} and {P}"
            assert H % P == 0 and W % P == 0, f"The masked image modeling loss needs H, W multiples of {P}, got {(H, W)}"
        hidden = self._hidden(x, interpolate_pos_encoding, bool_masked_pos, image_mean, image_std, rescale_factor)
        gh, gw = packing.patch_grid(self.embeddings, H, W)
        pk = self.decoder[0].packed()
        dec = packing.linear(hidden, pk.w, pk.b32)
        if bool_masked_pos is None:
            return packing.mim_reconstruct(dec, gh, gw, s, self.channels)
        norm = self._pixel_norm(image_mean, image_std, x.device) if u8 else None
        pix_code = _lib.VT_U8 if u8 else _lib.dtype_code(x)
        return packing.mim_reconstruct(dec, gh, gw, s, self.channels, x, pix_code, norm, rescale_factor,
                                       bool_masked_pos)

    def _pixel_norm(self, image_mean, image_std, device) -> torch.Tensor:
        """fp32 [2C] device tensor (mean, std) of the image processor for the uint8 loss, built once per constants
        (outside CUDA-graph capture: run the call once before capturing it)."""
        key = (tuple(float(m) for m in image_mean), tuple(float(v) for v in image_std), str(device))
        cache = self.__dict__.setdefault("_pixel_norms", {})
        if key not in cache:
            assert not torch.cuda.is_current_stream_capturing(), \
                "new image-processor constants are uploaded outside CUDA-graph capture: run the call once first"
            assert len(key[0]) == self.channels and len(key[1]) == self.channels
            cache[key] = torch.tensor(key[0] + key[1], dtype=torch.float32, device=device)
        return cache[key]
