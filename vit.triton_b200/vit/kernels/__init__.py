"""Kernel entry points with the names the reference exports (vit/kernels/__init__.py:1-7), backed by
hand-written sm_100a CUDA kernels in libvitb200.so.  Importing this package does not load the
library; the first call does, and raises if it is missing (there is no CPU fallback)."""
from .patching import patching
from .matmul import matmul
from .softmax import softmax
from .add import add
from .layernorm import LayerNormTriton, LayerNormB200, layernorm
from .matmul3 import matmul3
from .conv2d import Conv2DTriton, Conv2DB200, conv2d
from .attention import flash_attention
from .resize import resize_uint8

# reference-style aliases (the reference imports e.g. `matmul_triton as matmul`)
matmul_triton = matmul
softmax_triton = softmax
add_triton = add
layernorm_triton = layernorm
conv2d_triton = conv2d
patching_triton = patching
