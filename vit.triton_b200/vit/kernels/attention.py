"""Fused multi-head attention — host entry point for K3.

New relative to the reference, which runs heads serially through matmul3 / softmax / matmul3
(vit/vit.py:56-74,97-108); the entry point takes the fused-QKV activation the packed QKV GEMM
produces and returns the concatenated context in (B, N, D) layout.
"""
import math
from typing import Optional

import torch

import os

from . import _lib, bgemm as bg


def flash_attention(qkv: torch.Tensor, num_heads: int, scale: Optional[float] = None,
                    out: Optional[torch.Tensor] = None, probs: Optional[list] = None) -> torch.Tensor:
    """qkv: (B, N, 3*D) with columns [Q | K | V], head h at columns h*dh:(h+1)*dh of each third.
    Returns softmax(scale * Q K^T) V per head, concatenated: (B, N, D), written into ``out`` when given (a contiguous
    (B, N, D) tensor of qkv's dtype, e.g. a row range of a larger buffer).  ``probs``: a list that receives the
    attention probabilities softmax(scale * Q K^T), a contiguous (B, H, N, N) tensor of qkv's dtype (HF's
    ``output_attentions``); the context is computed exactly as without it."""
    assert qkv.is_cuda, "Input is not on GPU"
    assert len(qkv.shape) == 3 and qkv.shape[2] % (3 * num_heads) == 0, \
        f"qkv needs to be (B, N, 3*D) with D divisible by num_heads, provided: {qkv.shape}, {num_heads}"
    assert qkv.stride(2) == 1, "qkv last dimension needs to be contiguous"
    B, N, D3 = qkv.shape
    D = D3 // 3
    dh = D // num_heads
    if scale is None:
        scale = 1.0 / math.sqrt(dh)
    if out is None:
        out = torch.empty((B, N, D), device=qkv.device, dtype=qkv.dtype)
    assert out.shape == (B, N, D) and out.dtype == qkv.dtype and out.is_contiguous(), \
        f"out needs to be a contiguous {(B, N, D)} {qkv.dtype} tensor, provided: {tuple(out.shape)} {out.dtype}"
    if out.numel() == 0:
        if probs is not None:
            probs.append(torch.empty((B, num_heads, N, N), device=qkv.device, dtype=qkv.dtype))
        return out
    es = qkv.element_size()
    base = qkv.data_ptr()
    stream = _lib.stream_ptr(qkv)

    if qkv.dtype == torch.bfloat16 and dh in (64, 80) and qkv.stride(1) % 8 == 0 and qkv.stride(0) % 8 == 0 \
            and base % 16 == 0:
        try:
            for b0 in range(0, B, 32768):
                nb = min(32768, B - b0)
                off = b0 * qkv.stride(0) * es
                _lib.call("vt_flash_attn", base + off, base + off + D * es, base + off + 2 * D * es,
                          out[b0:].data_ptr(), nb, num_heads, N, dh, qkv.stride(1), qkv.stride(0), D, N * D,
                          float(scale), stream)
            if probs is not None:
                probs.append(_attention_probs(qkv, num_heads, dh, float(scale)))
            return out
        except _lib.KernelError as exc:
            # a shape outside what the tensor-core kernels implement (e.g. a sequence whose K/V block does
            # not fit shared memory) is refused before anything is launched: the strided path below is exact
            if exc.status != _lib.VT_ERR_UNSUPPORTED:
                raise

    # fp32 / odd-head-dim path: scores, softmax and PV composed over (B, H) batches.  The two contractions
    # run on the tensor cores (vt_bgemm) with q, k, P and v^T packed into K-major bf16 rows — fp32 values
    # split into pieces whose products are accumulated in fp32 (kernels/bgemm.py); the scores are
    # materialised (fp32 is the parity configuration, batch 1).  VT_EXACT_FP32=1: FP32-pipe kernels.
    pm = _composed_probs(qkv, num_heads, dh, float(scale))
    if probs is not None:
        probs.append(pm.view(B, num_heads, N, N))
    code = _lib.dtype_code(qkv)
    if os.environ.get("VT_EXACT_FP32") == "1":
        _lib.call("vt_gemm_strided", pm.data_ptr(), base + 2 * D * es, out.data_ptr(), None, N, dh, N, B,
                  num_heads, _lib.i64x4(num_heads * N * N, N * N, N, 1),
                  _lib.i64x4(qkv.stride(0), dh, qkv.stride(1), 1), _lib.i64x4(N * D, dh, D, 1), 1.0, 0, code,
                  stream)
        return out
    pieces = 1 if qkv.dtype == torch.bfloat16 else bg.split_pieces()
    pp = bg.pack(pm, pm.data_ptr(), N, N, B, num_heads, (num_heads * N * N, N * N, N, 1), pieces, pattern=0)
    # v^T rows: (channel, key) read through swapped strides
    vp = bg.pack(qkv, base + 2 * D * es, dh, N, B, num_heads, (qkv.stride(0), dh, 1, qkv.stride(1)), pieces, pattern=1)
    kp2 = pp.shape[2]
    bg.bgemm(pp.data_ptr(), vp.data_ptr(), out, out.data_ptr(), N, dh, kp2, B, num_heads,
             (num_heads * N * kp2, N * kp2, kp2), (num_heads * dh * kp2, dh * kp2, kp2), (N * D, dh, D))
    return out


def _composed_probs(qkv: torch.Tensor, num_heads: int, dh: int, scale: float) -> torch.Tensor:
    """(B * H, N, N) softmax(scale * Q K^T) of qkv's dtype: the scores by vt_gemm_strided (VT_EXACT_FP32=1) or by
    vt_bgemm over packed q, k rows, then vt_softmax."""
    B, N, D3 = qkv.shape
    D = D3 // 3
    es = qkv.element_size()
    base = qkv.data_ptr()
    stream = _lib.stream_ptr(qkv)
    scores = torch.empty((B * num_heads, N, N), device=qkv.device, dtype=qkv.dtype)
    probs = torch.empty_like(scores)
    code = _lib.dtype_code(qkv)
    if os.environ.get("VT_EXACT_FP32") == "1":
        sq = _lib.i64x4(qkv.stride(0), dh, qkv.stride(1), 1)
        _lib.call("vt_gemm_strided", base, base + D * es, scores.data_ptr(), None, N, N, dh, B, num_heads,
                  sq, _lib.i64x4(qkv.stride(0), dh, 1, qkv.stride(1)),
                  _lib.i64x4(num_heads * N * N, N * N, N, 1), scale, 0, code, stream)
    else:
        pieces = 1 if qkv.dtype == torch.bfloat16 else bg.split_pieces()
        s_head = (qkv.stride(0), dh, qkv.stride(1), 1)                        # (image, head, token, channel)
        qp = bg.pack(qkv, base, N, dh, B, num_heads, s_head, pieces, pattern=0)             # (B*H, N, kq)
        kp = bg.pack(qkv, base + D * es, N, dh, B, num_heads, s_head, pieces, pattern=1)
        kq = qp.shape[2]
        bg.bgemm(qp.data_ptr(), kp.data_ptr(), scores, scores.data_ptr(), N, N, kq, B, num_heads,
                 (num_heads * N * kq, N * kq, kq), (num_heads * N * kq, N * kq, kq), (num_heads * N * N, N * N, N),
                 scale=scale)
    _lib.call("vt_softmax", scores.data_ptr(), probs.data_ptr(), B * num_heads * N, N, N, code, stream)
    return probs


def _attention_probs(qkv: torch.Tensor, num_heads: int, dh: int, scale: float) -> torch.Tensor:
    """(B, H, N, N) bf16 attention probabilities of a bf16 (B, N, 3D) qkv by one vt_attn_probs launch; a shape that
    kernel does not implement takes the composed scores + softmax path."""
    B, N, D3 = qkv.shape
    D = D3 // 3
    es = qkv.element_size()
    probs = torch.empty((B, num_heads, N, N), device=qkv.device, dtype=qkv.dtype)
    try:
        _lib.call("vt_attn_probs", qkv.data_ptr(), qkv.data_ptr() + D * es, probs.data_ptr(), B, num_heads, N, dh,
                  qkv.stride(1), qkv.stride(0), scale, _lib.stream_ptr(qkv))
        return probs
    except _lib.KernelError as exc:
        if exc.status != _lib.VT_ERR_UNSUPPORTED:
            raise
    return _composed_probs(qkv, num_heads, dh, scale).view(B, num_heads, N, N)
