"""ctypes binding of libvitb200.so (C ABI declared in include/vitb200.h, include/vitb200_resolution.h,
include/vitb200_ragged.h, include/vitb200_mask.h, include/vitb200_attn.h, include/vitb200_preprocess.h,
include/vitb200_tokens.h and include/vitb200_clip.h).

There is deliberately no fallback: if the shared library is missing or a tensor is not on a CUDA
device the entry points raise.  The oracle under /oracle is test infrastructure and is never
imported from here.
"""
import ctypes
import os
from typing import Optional

import torch

_LIB_NAME = "libvitb200.so"
_lib: Optional[ctypes.CDLL] = None

VT_F32 = 0
VT_BF16 = 1
VT_U8 = 2     # raw NHWC pixels (patch embeddings, masked-image-modeling loss)
VT_E4M3 = 3   # FP8 path (vt_gemm_fp8 / vt_layernorm_fp8)
VT_PG_PUT = 1  # vt_pool_cls_allgather modes
VT_PG_GET = 2
# GEMM epilogue activations (VT_ACT_* of include/vitb200_clip.h): vt_bgemm's act, the gelu argument of the other GEMMs
VT_ACT_NONE = 0
VT_ACT_GELU = 1
VT_ACT_TANH = 2
VT_ACT_QUICK_GELU = 3

_c_i32 = ctypes.c_int32
_c_i64 = ctypes.c_int64
_c_f32 = ctypes.c_float
_c_ptr = ctypes.c_void_p
_c_i64p = ctypes.POINTER(ctypes.c_int64)

# name -> argtypes; mirrors include/vitb200.h one to one (tests/test_abi.py checks both directions)
SIGNATURES = {
    "vt_layernorm": [_c_ptr, _c_ptr, _c_ptr, _c_ptr, _c_i64, _c_i32, _c_i64, _c_i64, _c_f32, _c_i32,
                     _c_i32, _c_ptr],
    "vt_add": [_c_ptr, _c_ptr, _c_ptr, _c_i64, _c_i32, _c_ptr],
    "vt_softmax": [_c_ptr, _c_ptr, _c_i64, _c_i32, _c_i64, _c_i32, _c_ptr],
    "vt_gemm_bf16": [_c_ptr, _c_i64, _c_ptr, _c_i64, _c_ptr, _c_i64, _c_i32, _c_ptr, _c_ptr, _c_i64,
                     _c_i32, _c_i32, _c_i32, _c_i32, _c_ptr],
    "vt_gemm_bf16_ln": [_c_ptr, _c_i64, _c_ptr, _c_i64, _c_ptr, _c_i64, _c_ptr, _c_ptr, _c_i64, _c_i32, _c_i32,
                        _c_i32, _c_i32, _c_ptr, _c_ptr, _c_i32, _c_f32, _c_ptr, _c_ptr],
    "vt_gemm_strided": [_c_ptr, _c_ptr, _c_ptr, _c_ptr, _c_i32, _c_i32, _c_i32, _c_i32, _c_i32,
                        _c_i64p, _c_i64p, _c_i64p, _c_f32, _c_i32, _c_i32, _c_ptr],
    "vt_gemm_fp8": [_c_ptr, _c_i64, _c_ptr, _c_i64, _c_ptr, _c_i64, _c_i32, _c_ptr, _c_ptr, _c_ptr, _c_i64, _c_i32,
                    _c_i32, _c_i32, _c_i32, _c_f32, _c_ptr],
    "vt_layernorm_fp8": [_c_ptr, _c_ptr, _c_ptr, _c_ptr, _c_i64, _c_i32, _c_i64, _c_i64, _c_f32, _c_f32, _c_ptr],
    "vt_quantize_rows_fp8": [_c_ptr, _c_i64, _c_ptr, _c_i64, _c_ptr, _c_i32, _c_i32, _c_ptr],
    "vt_bgemm": [_c_ptr, _c_ptr, _c_ptr, _c_ptr, _c_ptr, _c_i32, _c_i32, _c_i32, _c_i32, _c_i32, _c_i64p, _c_i64p,
                 _c_i64p, _c_i32, _c_f32, _c_i32, _c_i32, _c_ptr],
    "vt_pack_bf16": [_c_ptr, _c_i32, _c_ptr, _c_i32, _c_i32, _c_i32, _c_i32, _c_i64p, _c_i64p, _c_i32, _c_i32,
                     _c_i32, _c_ptr],
    "vt_flash_attn": [_c_ptr, _c_ptr, _c_ptr, _c_ptr, _c_i32, _c_i32, _c_i32, _c_i32, _c_i64, _c_i64,
                      _c_i64, _c_i64, _c_f32, _c_ptr],
    "vt_ln_fold": [_c_ptr, _c_i64, _c_ptr, _c_ptr, _c_ptr, _c_ptr, _c_i64, _c_ptr, _c_ptr, _c_i32, _c_i32, _c_i32,
                   _c_ptr],
    "vt_patch_embed_gemm": [_c_ptr, _c_i32, _c_ptr, _c_i64, _c_ptr, _c_ptr, _c_ptr, _c_ptr, _c_ptr, _c_i32, _c_i32,
                            _c_i32, _c_i32, _c_i32, _c_ptr],
    "vt_patching": [_c_ptr, _c_ptr, _c_i32, _c_i32, _c_i32, _c_i32, _c_i32, _c_i32, _c_ptr],
    "vt_embed_finalize": [_c_ptr, _c_ptr, _c_ptr, _c_i32, _c_i32, _c_i32, _c_i32, _c_ptr],
    "vt_conv2d": [_c_ptr, _c_ptr, _c_ptr, _c_ptr, _c_i32, _c_i32, _c_i32, _c_i32, _c_i32, _c_i32,
                  _c_i32, _c_i32, _c_ptr],
    "vt_pool_cls": [_c_ptr, _c_ptr, _c_i32, _c_i32, _c_i64, _c_i32, _c_ptr],
    "vt_pool_cls_allgather": [_c_ptr, _c_i32, _c_i32, _c_i64, _c_i32, _c_ptr, _c_ptr, _c_i32, _c_i32,
                              _c_ptr, _c_ptr, _c_i32, _c_i32, _c_ptr],
}

# name -> argtypes of the any-resolution entry points; mirrors include/vitb200_resolution.h one to one
# (tests/test_abi_resolution.py checks both directions)
RESOLUTION_SIGNATURES = {
    "vt_patch_embed_gemm_hw": [_c_ptr, _c_i32, _c_ptr, _c_i64, _c_ptr, _c_ptr, _c_ptr, _c_ptr, _c_ptr, _c_i32, _c_i32,
                               _c_i32, _c_i32, _c_i32, _c_i32, _c_ptr],
    "vt_pos_embed_resample": [_c_ptr, _c_i32, _c_ptr, _c_i32, _c_i32, _c_i32, _c_i32, _c_ptr],
}

# name -> argtypes of the ragged-batch entry points; mirrors include/vitb200_ragged.h one to one
# (tests/test_abi_ragged.py checks both directions)
RAGGED_SIGNATURES = {
    "vt_patch_embed_ragged_gather": [_c_ptr, _c_i32, _c_i32, _c_i32, _c_i32, _c_ptr, _c_i64, _c_ptr, _c_i32, _c_i64,
                                     _c_ptr],
    "vt_gather_rows": [_c_ptr, _c_i64, _c_ptr, _c_ptr, _c_i64, _c_i32, _c_i32, _c_i32, _c_ptr],
}

# name -> argtypes of the masked-input / masked-image-modeling entry points; mirrors include/vitb200_mask.h one to one
# (tests/test_abi_mask.py checks both directions)
MASK_SIGNATURES = {
    "vt_patch_embed_masked_gather": [_c_ptr, _c_i32, _c_ptr, _c_ptr, _c_ptr, _c_ptr, _c_i64, _c_ptr, _c_i32, _c_i32,
                                     _c_i32, _c_i32, _c_i32, _c_i32, _c_ptr],
    "vt_embed_finalize_masked": [_c_ptr, _c_ptr, _c_ptr, _c_ptr, _c_ptr, _c_i32, _c_i32, _c_i32, _c_i32, _c_ptr],
    "vt_mim_reconstruct": [_c_ptr, _c_ptr, _c_i32, _c_i32, _c_i32, _c_i32, _c_i32, _c_i32, _c_ptr, _c_i32, _c_ptr,
                           _c_f32, _c_ptr, _c_ptr, _c_ptr, _c_ptr],
}

# name -> argtypes of the attention-probabilities entry point; mirrors include/vitb200_attn.h one to one
# (tests/test_abi_attn.py checks both directions)
ATTN_SIGNATURES = {
    "vt_attn_probs": [_c_ptr, _c_ptr, _c_ptr, _c_i32, _c_i32, _c_i32, _c_i32, _c_i64, _c_i64, _c_f32, _c_ptr],
}

# name -> argtypes of the image-processor resize entry points; mirrors include/vitb200_preprocess.h one to one
# (tests/test_abi_preprocess.py checks both directions)
PREPROCESS_SIGNATURES = {
    "vt_resize_u8": [_c_ptr, _c_i32, _c_i32, _c_i32, _c_i32, _c_i64, _c_ptr, _c_i32, _c_ptr, _c_i32, _c_ptr, _c_i32,
                     _c_i32, _c_ptr],
    "vt_resize_u8_list": [_c_ptr, _c_i32, _c_i32, _c_ptr, _c_ptr, _c_i32, _c_i32, _c_ptr],
}

# name -> argtypes of the entry points with a prefix-token count (1 = CLS, 2 = CLS + distillation token); mirrors
# include/vitb200_tokens.h one to one (tests/test_abi_tokens.py checks both directions).  Each is an entry point of
# another table with an int32 prefix in front of the stream.
TOKENS_SIGNATURES = {
    "vt_patch_embed_gemm_hw_prefix": RESOLUTION_SIGNATURES["vt_patch_embed_gemm_hw"][:-1] + [_c_i32, _c_ptr],
    "vt_patch_embed_masked_gather_prefix": MASK_SIGNATURES["vt_patch_embed_masked_gather"][:-1] + [_c_i32, _c_ptr],
    "vt_patch_embed_ragged_gather_prefix": RAGGED_SIGNATURES["vt_patch_embed_ragged_gather"][:-1] + [_c_i32, _c_ptr],
    "vt_pos_embed_resample_prefix": RESOLUTION_SIGNATURES["vt_pos_embed_resample"][:-1] + [_c_i32, _c_ptr],
    "vt_embed_finalize_prefix": SIGNATURES["vt_embed_finalize"][:-1] + [_c_i32, _c_ptr],
    "vt_embed_finalize_masked_prefix": MASK_SIGNATURES["vt_embed_finalize_masked"][:-1] + [_c_i32, _c_ptr],
}

# name -> argtypes of the CLIP entry points; mirrors include/vitb200_clip.h one to one (tests/test_abi_clip.py checks both
# directions)
CLIP_SIGNATURES = {
    "vt_layernorm_stats": [_c_ptr, _c_ptr, _c_ptr, _c_ptr, _c_ptr, _c_i64, _c_i32, _c_i64, _c_i64, _c_f32, _c_ptr],
}


def call_prefix(name: str, prefix: int, *args) -> None:
    """One host path for every prefix-token count: ``name + "_prefix"`` (include/vitb200_tokens.h) with ``prefix`` right
    before the stream (the last of ``args``).  At prefix 1 (CLS only) the call goes to ``name`` itself, the one-line
    wrapper that passes 1: the same kernel and bits, and a ViT model's launches keep the names that launch counts and
    per-kernel timings are keyed on."""
    if prefix == 1:
        call(name, *args)
    else:
        call(name + "_prefix", *args[:-1], prefix, args[-1])


class RaggedImage(ctypes.Structure):
    """``vt_ragged_image`` of include/vitb200_ragged.h: one image of a ragged batch."""
    _fields_ = [("pixels", _c_ptr), ("pos", _c_ptr), ("row0", _c_i64), ("height", _c_i32), ("width", _c_i32),
                ("tokens", _c_i32), ("reserved", _c_i32)]


class ResizeImage(ctypes.Structure):
    """``vt_resize_image`` of include/vitb200_preprocess.h: one image of a resize list."""
    _fields_ = [("pixels", _c_ptr), ("htab", _c_i64), ("vtab", _c_i64), ("height", _c_i32), ("width", _c_i32),
                ("hk", _c_i32), ("vk", _c_i32)]


def lib_path() -> str:
    # VT_LIB selects an alternative build of the same library (A/B measurements of kernel variants)
    override = os.environ.get("VT_LIB")
    if override:
        return override
    return os.path.join(os.path.dirname(os.path.abspath(__file__)), _LIB_NAME)


def load() -> ctypes.CDLL:
    """Load the shared library once; raise (never fall back) when it has not been built."""
    global _lib
    if _lib is not None:
        return _lib
    path = lib_path()
    if not os.path.exists(path):
        raise RuntimeError(
            f"{_LIB_NAME} not found at {path}: build it with `make -C vit.triton_b200` "
            "(or `python -c 'import __graft_entry__ as g; g.build()'`). There is no CPU fallback.")
    lib = ctypes.CDLL(path)
    for name, argtypes in (list(SIGNATURES.items()) + list(RESOLUTION_SIGNATURES.items())
                           + list(RAGGED_SIGNATURES.items()) + list(MASK_SIGNATURES.items())
                           + list(ATTN_SIGNATURES.items()) + list(PREPROCESS_SIGNATURES.items())
                           + list(TOKENS_SIGNATURES.items()) + list(CLIP_SIGNATURES.items())):
        fn = getattr(lib, name)
        fn.argtypes = argtypes
        fn.restype = ctypes.c_int
    lib.vt_version.restype = ctypes.c_int
    lib.vt_status_string.argtypes = [ctypes.c_int]
    lib.vt_status_string.restype = ctypes.c_char_p
    _lib = lib
    return lib


VT_ERR_UNSUPPORTED = -4


class KernelError(RuntimeError):
    def __init__(self, message: str, status: int = 0):
        super().__init__(message)
        self.status = status


def check(rc: int, what: str) -> None:
    if rc != 0:
        msg = load().vt_status_string(rc).decode()
        raise KernelError(f"{what} failed: {msg} (status {rc})", rc)


def dtype_code(t: torch.Tensor) -> int:
    if t.dtype == torch.float32:
        return VT_F32
    if t.dtype == torch.bfloat16:
        return VT_BF16
    raise AssertionError(f"Only float32 and bfloat16 are supported, provided: {t.dtype}")


def stream_ptr(t: torch.Tensor) -> int:
    """Raw cudaStream_t of torch's current stream on the tensor's device."""
    return torch.cuda.current_stream(t.device).cuda_stream


def ptr(t: Optional[torch.Tensor]) -> Optional[int]:
    return None if t is None else t.data_ptr()


def i64x4(a, b, c, d):
    return (ctypes.c_int64 * 4)(a, b, c, d)


def i64x3(a, b, c):
    return (ctypes.c_int64 * 3)(a, b, c)


# Count of kernel launches issued through this module (bench.py reports it as gpu_launches).
launch_count = 0

# Optional profiling hook: event_hook(name, before: bool, args) is called on the launching thread right
# before and right after a kernel is enqueued (bench.py records CUDA events there and reads the shapes
# out of ``args``, the C-ABI argument tuple of the call).
event_hook = None


def call(name: str, *args) -> None:
    global launch_count
    hook = event_hook
    if hook is not None:
        hook(name, True, args)
    rc = getattr(load(), name)(*args)
    if hook is not None:
        hook(name, False, args)
    launch_count += 1
    check(rc, name)
