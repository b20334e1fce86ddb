"""Dense layer matmul — host entry point for K1 (replaces reference vit/kernels/matmul.py:111-156).

Device paths, chosen per call from dtype and alignment (one library, one architecture, all on tcgen05):
  * bf16, K and N multiples of 8, rows of A dense  -> 2-CTA tcgen05/TMEM/TMA GEMM (``vt_gemm_bf16``)
  * fp32                                           -> operands split into bf16 pieces (``vt_pack_bf16``),
                                                      then the batched tcgen05 GEMM with fp32 output
                                                      (``vt_bgemm``): ~2^-16 per product, see kernels/bgemm.py
  * bf16 with odd shapes / strides                 -> one packing pass, then ``vt_bgemm``
VT_EXACT_FP32=1 forces the strided FP32-pipe GEMM (``vt_gemm_strided``) for A/B comparisons.
"""
import os
import weakref
from typing import Optional

import torch

from . import _lib, bgemm as bg

# (id(tensor), tag) -> (weakref, (data_ptr, version), derived tensor).  Only nn.Parameters are cached: a plain
# tensor's storage can be recycled by the allocator under the same pointer, a live Parameter's cannot.
# The key covers in-place updates through the autograd-visible API (version counter) and re-pointing
# (``p.data = other``: data_ptr); writes THROUGH ``p.data`` (``p.data.copy_()``, ``p.data.normal_()``, EMA
# updates) change neither — call ``VIT.invalidate_packed()`` / ``clear_derived_cache()`` after those.
_derived_cache = {}


def clear_derived_cache() -> None:
    """Drop every cached K-major / fp32 copy of a parameter (see the note above)."""
    _derived_cache.clear()


def _cached(param: torch.Tensor, tag: str, make):
    key = (id(param), tag)
    stamp = (param.data_ptr(), param._version)
    hit = _derived_cache.get(key)
    if hit is not None:
        ref, old_stamp, value = hit
        if ref() is param and old_stamp == stamp and value.device == param.device:
            return value
    value = make(param)
    if isinstance(param, torch.nn.Parameter):
        if len(_derived_cache) > 4096:
            _derived_cache.clear()
        _derived_cache[key] = (weakref.ref(param), stamp, value)
    return value


def _k_major(B: torch.Tensor) -> torch.Tensor:
    """(K, N) weight -> [N, K] row-major (K-major operand for the tensor core)."""
    Bt = B.detach().t()
    return Bt if Bt.is_contiguous() else Bt.contiguous()


def _tensor_core_ok(A: torch.Tensor, B: torch.Tensor, N: int, K: int) -> bool:
    if A.dtype != torch.bfloat16 or B.dtype != torch.bfloat16:
        return False
    if (K % 8) or (N % 8) or A.stride(2) != 1 or (A.stride(1) % 8):
        return False
    if A.shape[0] > 1 and A.stride(0) != A.shape[1] * A.stride(1):
        return False
    return A.data_ptr() % 16 == 0


def matmul(A: torch.Tensor, B: torch.Tensor, bias: Optional[torch.Tensor] = None,
           activation: Optional[str] = None) -> torch.Tensor:
    """O[b] = act(A[b] @ B + bias) with fp32 accumulation.

    Args / errors follow the reference's ``matmul_triton`` (matmul.py:124-133): A is (B, T, Cin) with
    any strides, B is (Cin, Cout), bias is (Cout,), activation is None, "gelu" (exact erf) or "quick_gelu"
    (x * sigmoid(1.702 x), CLIP).
    Returns a fresh (B, T, Cout) tensor in A's dtype.
    """
    assert len(A.shape) == 3, "First input matrix needs to have 3 dimensions (B, T, C)"
    assert A.device == B.device and A.is_cuda, "Both matrix should be on GPU"
    assert len(B.shape) == 2 and A.shape[2] == B.shape[0], \
        f"Dimensions are not compatible for matrix multiplication, provided: {A.shape}, {B.shape}"
    if bias is not None:
        assert bias.is_cuda, "Bias is not on GPU"
        assert bias.numel() == B.shape[1], "Bias shape does not match output feature dimension shape"
    if activation:
        assert activation in ["gelu", "quick_gelu"], \
            f"Only the gelu and quick_gelu activations are supported, provided: {activation}"
    act = bg._ACT[activation]

    batch, M, K = A.shape
    N = B.shape[1]
    O = torch.empty((batch, M, N), device=A.device, dtype=A.dtype)
    if O.numel() == 0:
        return O
    stream = _lib.stream_ptr(A)

    if _tensor_core_ok(A, B, N, K):
        Bt = _cached(B, "kmajor", _k_major)
        bias32 = None if bias is None else _cached(bias, "f32", lambda b: b.detach().float().contiguous())
        _lib.call("vt_gemm_bf16", A.data_ptr(), A.stride(1), Bt.data_ptr(), K, O.data_ptr(), N,
                  _lib.VT_BF16, _lib.ptr(bias32), None, 0, batch * M, N, K, act, stream)
        return O

    assert A.dtype == B.dtype, f"Input dtypes need to be same, provided {A.dtype}, {B.dtype}"
    if os.environ.get("VT_EXACT_FP32") == "1":
        if bias is not None and (bias.dtype != A.dtype or not bias.is_contiguous()):
            bias = bias.to(A.dtype).contiguous()
        _lib.call("vt_gemm_strided", A.data_ptr(), B.data_ptr(), O.data_ptr(), _lib.ptr(bias), M, N, K,
                  batch, 1,
                  _lib.i64x4(A.stride(0), 0, A.stride(1), A.stride(2)),
                  _lib.i64x4(0, 0, B.stride(0), B.stride(1)),
                  _lib.i64x4(M * N, 0, N, 1),
                  1.0, act, _lib.dtype_code(A), stream)
        return O

    # tensor cores for everything else: pack A (any strides) and W^T into K-major bf16 rows — fp32 split
    # into pieces whose products are accumulated in fp32 — then the batched tcgen05 GEMM
    pieces = 1 if A.dtype == torch.bfloat16 else bg.split_pieces()
    wp = _cached(B, f"packed{pieces}", lambda w: bg.pack(w, w.data_ptr(), N, K, 1, 1, (0, 0, w.stride(1), w.stride(0)),
                                                        pieces, pattern=1)[0])
    bias32 = None if bias is None else _cached(bias, "f32", lambda b: b.detach().float().contiguous())
    a = bg.pack(A, A.data_ptr(), M, K, batch, 1, (A.stride(0), 0, A.stride(1), A.stride(2)), pieces, pattern=0)
    kk = a.shape[2]
    bg.bgemm(a.data_ptr(), wp.data_ptr(), O, O.data_ptr(), M, N, kk, batch, 1, (M * kk, 0, kk), (0, 0, kk),
             (M * N, 0, N), bias32=bias32, act=act)
    return O
