"""Batched tensor-core GEMM (``vt_bgemm``) and operand packing (``vt_pack_bf16``) — host helpers.

Everything that is a dense contraction but not one of the model's four big bf16 layers comes through
here: ``matmul3`` (reference vit/kernels/matmul3.py:111-156), the fp32 model (reference ``matmul``,
vit/kernels/matmul.py:111-156, whose ``tl.dot`` is a TF32 tensor-core product) with its operands split
into bf16 pieces, the composed fp32 attention, the pooler / classifier heads.
"""
import os
from typing import Optional

import torch

from . import _lib

ACT_NONE, ACT_GELU, ACT_TANH, ACT_QUICK_GELU = _lib.VT_ACT_NONE, _lib.VT_ACT_GELU, _lib.VT_ACT_TANH, _lib.VT_ACT_QUICK_GELU
_ACT = {None: ACT_NONE, "": ACT_NONE, "gelu": ACT_GELU, "tanh": ACT_TANH, "quick_gelu": ACT_QUICK_GELU}


def split_pieces() -> int:
    """Pieces an fp32 operand is split into for the tensor cores: 3 (default) = x = hi + lo, three products
    hi*hi + hi*lo + lo*hi (~2^-16 per product, SURVEY.md 7.2); 6 = three-way split with the six products
    of weight >= 2^-16 (VT_FP32_SPLIT=6).  Measured on B200 (tests/test_gpu_kernels.py:
    test_fp32_matmul_split_accuracy, K = 768): 3.2e-5 / 5.3e-5 max-abs for 3 / 6 pieces against 6e-6 on the
    FP32 pipe and ~1e-3 for one TF32 pass — six pieces are NOT more accurate on this hardware, because the
    tensor core adds into its fp32 accumulator with truncation and twice as many K steps lose more than
    the dropped lo*lo products; hence the default."""
    return 6 if os.environ.get("VT_FP32_SPLIT", "3") == "6" else 3


def ceil8(n: int) -> int:
    return (n + 7) // 8 * 8


def pack(src: torch.Tensor, base_ptr: int, rows: int, cols: int, batch_outer: int, batch_inner: int,
         s_src, pieces: int, pattern: int = 0) -> torch.Tensor:
    """(batch_outer * batch_inner, rows, pieces * ceil8(cols)) bf16 K-major rows out of the strided view of
    ``src`` that starts at ``base_ptr`` with element strides ``s_src`` = (outer, inner, row, col)."""
    cpad = ceil8(cols)
    dst = torch.empty((batch_outer * batch_inner, rows, pieces * cpad), device=src.device, dtype=torch.bfloat16)
    _lib.call("vt_pack_bf16", base_ptr, _lib.dtype_code(src), dst.data_ptr(), rows, cols, batch_outer, batch_inner,
              _lib.i64x4(*s_src), _lib.i64x3(batch_inner * rows * pieces * cpad, rows * pieces * cpad, pieces * cpad),
              cpad, pieces, pattern, _lib.stream_ptr(src))
    return dst


def bgemm(a_ptr: int, b_ptr: int, out: torch.Tensor, c_ptr: int, M: int, N: int, K: int, batch_outer: int,
          batch_inner: int, sA, sB, sC, bias32: Optional[torch.Tensor] = None, residual_ptr: Optional[int] = None,
          b_mn: bool = False, scale: float = 1.0, act: int = ACT_NONE) -> None:
    _lib.call("vt_bgemm", a_ptr, b_ptr, c_ptr, _lib.ptr(bias32), residual_ptr, M, N, K, batch_outer, batch_inner,
              _lib.i64x3(*sA), _lib.i64x3(*sB), _lib.i64x3(*sC), 1 if b_mn else 0, float(scale), act,
              _lib.dtype_code(out), _lib.stream_ptr(out))


def pack_weight_nk(w_nk: torch.Tensor, pieces: int) -> torch.Tensor:
    """[N, K] (K-major, fp32 or bf16) weight -> its B-side packed form [N, pieces * ceil8(K)] bf16."""
    N, K = w_nk.shape
    return pack(w_nk, w_nk.data_ptr(), N, K, 1, 1, (0, 0, w_nk.stride(0), w_nk.stride(1)), pieces, pattern=1)[0]


def dense_rows(x: torch.Tensor, x_ptr: int, M: int, K: int, row_stride: int, w_packed: torch.Tensor, pieces: int,
               n_out: int, bias32: Optional[torch.Tensor], act: int, out: torch.Tensor, out_ptr: int, ldc: int,
               residual_ptr: Optional[int] = None) -> None:
    """out[m, :] = act(x[m, :] @ W^T + bias) (+ residual) for M rows of ``x`` that are ``row_stride`` elements
    apart; W comes packed by ``pack_weight_nk`` with the same ``pieces``.  bf16 rows whose stride and length
    the tensor map can address directly (pieces == 1, multiples of 8, 16-byte base) are read in place."""
    cpad = ceil8(K)
    direct = (pieces == 1 and x.dtype == torch.bfloat16 and K % 8 == 0 and row_stride % 8 == 0 and x_ptr % 16 == 0)
    if direct:
        a_ptr, lda = x_ptr, row_stride
    else:
        a = pack(x, x_ptr, M, K, 1, 1, (0, 0, row_stride, 1), pieces, pattern=0)
        a_ptr, lda = a.data_ptr(), pieces * cpad
    kk = pieces * cpad
    bgemm(a_ptr, w_packed.data_ptr(), out, out_ptr, M, n_out, kk, 1, 1, (0, 0, lda), (0, 0, kk), (0, 0, ldc),
          bias32=bias32, residual_ptr=residual_ptr, act=act)
