"""The image processor's resize on the device: PIL ``Image.resize`` (BILINEAR, BICUBIC) of raw uint8 HWC images, byte for
byte (``vt_resize_u8`` / ``vt_resize_u8_list``, csrc/resize_u8.cu, include/vitb200_preprocess.h).

The coefficient tables are PIL's (libImaging/Resample.c, ``precompute_coeffs`` and ``normalize_coeffs_8bpc``), built here
in float64 with its operations in its order, vectorised over output indices.  A table of one axis (in -> out samples) is
int32 [out, 2 + k]: start, count, then k fixed-point weights (units of 2^-22), the first count of them used.  Every table
is validated before it is uploaded: the kernel reads no input sample other than start + j, j < count."""
import functools
from collections import OrderedDict

import numpy as np
import torch

from . import _lib

BILINEAR = 2      # PIL.Image.Resampling codes (transformers' PILImageResampling members compare equal)
BICUBIC = 3
_SUPPORT = {BILINEAR: 1.0, BICUBIC: 2.0}
PRECISION_BITS = 22
TABLES_KEPT = 64  # device tables of batch sizes kept per process (tables read by a captured graph are never freed)

_device_tables = OrderedDict()
_tables_in_graphs = {}


def check_resample(resample) -> int:
    """PIL code -> int; AssertionError unless it is one of the supported filters."""
    assert not isinstance(resample, bool) and resample in _SUPPORT, \
        f"resample must be 2 (PIL BILINEAR) or 3 (PIL BICUBIC), provided: {resample!r}"
    return int(resample)


def _filter(x: np.ndarray, resample: int) -> np.ndarray:
    x = np.abs(x)
    if resample == BILINEAR:
        return np.where(x < 1.0, 1.0 - x, 0.0)
    a = -0.5
    near = ((a + 2.0) * x - (a + 3.0)) * x * x + 1
    far = (((x - 5) * x + 8) * x - 4) * a
    return np.where(x < 1.0, near, np.where(x < 2.0, far, 0.0))


@functools.lru_cache(maxsize=1024)
def _table_cached(in_size: int, out_size: int, resample: int) -> np.ndarray:
    scale = in_size / out_size
    fs = max(scale, 1.0)
    support = _SUPPORT[resample] * fs
    ss = 1.0 / fs
    center = (np.arange(out_size, dtype=np.float64) + 0.5) * scale
    xmin = np.maximum(np.trunc(center - support + 0.5), 0).astype(np.int64)
    count = np.minimum(np.trunc(center + support + 0.5), in_size).astype(np.int64) - xmin
    k = int(count.max())
    taps = np.arange(k, dtype=np.int64)
    w = _filter((taps[None, :] + xmin[:, None] - center[:, None] + 0.5) * ss, resample)
    w = np.where(taps[None, :] < count[:, None], w, 0.0)
    ww = np.zeros(out_size, dtype=np.float64)
    for j in range(k):                       # PIL's sequential sum in tap order (np.sum is pairwise)
        ww = ww + w[:, j]
    w = np.where(ww[:, None] != 0.0, w / np.where(ww == 0.0, 1.0, ww)[:, None], w)
    w = w * (1 << PRECISION_BITS)
    fixed = np.trunc(np.where(w < 0, w - 0.5, w + 0.5))
    table = np.empty((out_size, 2 + k), dtype=np.int32)
    table[:, 0] = xmin
    table[:, 1] = count
    table[:, 2:] = fixed
    validate_table(table, in_size)
    table.flags.writeable = False
    return table


def coeff_table(in_size: int, out_size: int, resample: int = BILINEAR) -> np.ndarray:
    """int32 [out_size, 2 + k] table of one axis, PIL's coefficients for ``resample`` (validated, read-only, cached)."""
    assert in_size >= 1 and out_size >= 1, f"sizes must be at least 1, provided: {in_size} -> {out_size}"
    return _table_cached(int(in_size), int(out_size), check_resample(resample))


def validate_table(table: np.ndarray, in_size: int) -> None:
    """AssertionError unless every entry only reads input samples 0 .. in_size - 1: 0 <= start, 1 <= count <= k,
    start + count <= in_size, and start, start + count nondecreasing (a band of outputs reads one row range)."""
    assert isinstance(table, np.ndarray) and table.dtype == np.int32 and table.ndim == 2 and table.shape[1] >= 3 \
        and table.shape[0] >= 1, "a resize table is an int32 [out, 2 + k] array, k >= 1"
    k = table.shape[1] - 2
    start = table[:, 0].astype(np.int64)
    count = table[:, 1].astype(np.int64)
    assert (start >= 0).all(), "resize table: negative start"
    assert ((count >= 1) & (count <= k)).all(), f"resize table: count outside [1, {k}]"
    assert (start + count <= in_size).all(), f"resize table: taps past the input size {in_size}"
    assert (np.diff(start) >= 0).all() and (np.diff(start + count) >= 0).all(), "resize table: taps not monotone"


def _upload(table: np.ndarray, device) -> torch.Tensor:
    from .. import packing
    return packing._to_device_async(table.tobytes(), device).view(torch.int32).view(table.shape)


def _assert_not_capturing() -> None:
    assert not torch.cuda.is_current_stream_capturing(), \
        "the resize tables of a new input size are uploaded outside CUDA-graph capture: run the call once before capturing"


def _batch_tables(device, H: int, W: int, height: int, width: int, resample: int) -> tuple:
    """(width table, height table) on ``device``, cached per (device, sizes, filter).  Tables read during capture stay
    referenced for the life of the process: a captured graph holds their addresses."""
    key = (str(device), H, W, height, width, resample)
    hit = _device_tables.get(key)
    if hit is None:
        _assert_not_capturing()
        hit = (_upload(coeff_table(W, width, resample), device), _upload(coeff_table(H, height, resample), device))
        _device_tables[key] = hit
        while len(_device_tables) > TABLES_KEPT:
            _device_tables.popitem(last=False)
    else:
        _device_tables.move_to_end(key)
    if torch.cuda.is_current_stream_capturing():
        _tables_in_graphs[key] = hit
    return hit


def check_images(images, channels=None) -> tuple:
    """Host-side checks, before anything is launched: a uint8 (B, H, W, C) tensor or a non-empty list of uint8
    (H_i, W_i, C) tensors on one device, sides >= 1, C in 1..4 (== ``channels`` when given).  Returns (is_list, C)."""
    is_list = isinstance(images, (list, tuple))
    items = list(images) if is_list else [images]
    if is_list:
        assert len(items) > 0, "resize needs at least one image"
    dims = 3 if is_list else 4
    device = None
    C = None
    for i, img in enumerate(items):
        assert isinstance(img, torch.Tensor), f"image {i} is not a tensor: {type(img)}"
        assert img.dtype == torch.uint8, f"resize takes raw uint8 pixels, provided: {img.dtype}"
        assert img.dim() == dims, \
            f"expected {'(H, W, C)' if is_list else '(B, H, W, C)'} uint8 pixels, provided: {tuple(img.shape)}"
        H, W, c = img.shape[-3:]
        assert H >= 1 and W >= 1, f"image {i} has a side < 1: {(H, W)}"
        assert 1 <= c <= 4 and (channels is None or c == channels), \
            f"image {i} has {c} channels, expected {channels if channels is not None else '1 to 4'}"
        assert C is None or c == C, f"all images need one channel count: {C} and {c}"
        C = c
        assert device is None or img.device == device, f"all images need one device: {device} and {img.device}"
        device = img.device
    if not is_list:
        assert items[0].shape[0] >= 1, "resize needs at least one image"
    return is_list, C


def resize_uint8(images, height: int, width: int, resample: int = BILINEAR) -> torch.Tensor:
    """(B, height, width, C) uint8 = ``PIL.Image.resize(img, (width, height), resample)`` of every image, byte for byte
    (HF ``ViTImageProcessorPil.resize``).  ``images``: a CUDA uint8 (B, H, W, C) tensor, or a list of (H_i, W_i, C)
    tensors of any sizes (one device, one C <= 4).  ``resample``: 2 (BILINEAR) or 3 (BICUBIC).

    A batch tensor already of the output size is returned as it is (PIL copies; nothing is launched).  A batch takes
    one ``vt_resize_u8`` launch with tables cached per size, so it can be captured into a CUDA graph once its size has
    been seen.  A list takes one ``vt_resize_u8_list`` launch; its descriptors and the tables of its distinct sizes are
    uploaded in one copy per call, so a list cannot be captured."""
    resample = check_resample(resample)
    assert int(height) >= 1 and int(width) >= 1, f"output size must be at least 1x1, provided: {(height, width)}"
    height, width = int(height), int(width)
    is_list, C = check_images(images)
    if is_list:
        assert not (torch.cuda.is_available() and torch.cuda.is_current_stream_capturing()), \
            "a list of images cannot be resized under CUDA-graph capture: stack them into a batch of one size"
    device = (images[0] if is_list else images).device
    assert device.type == "cuda", f"resize runs on a CUDA device, the images are on {device}"
    if is_list:
        return _resize_list(images, height, width, resample, C, device)
    B, H, W, _ = images.shape
    if (H, W) == (height, width):
        return images
    if images[0].stride() != (W * C, C, 1) or (B > 1 and images.stride(0) < H * W * C):
        images = images.contiguous()
    htab, vtab = _batch_tables(device, H, W, height, width, resample)
    out = torch.empty((B, height, width, C), device=device, dtype=torch.uint8)
    stride = images.stride(0) if B > 1 else H * W * C
    _lib.call("vt_resize_u8", images.data_ptr(), B, H, W, C, stride, htab.data_ptr(), htab.shape[1] - 2,
              vtab.data_ptr(), vtab.shape[1] - 2, out.data_ptr(), height, width, _lib.stream_ptr(out))
    return out


def _resize_list(images, height: int, width: int, resample: int, C: int, device) -> torch.Tensor:
    pixels = [img.contiguous() for img in images]       # referenced until the launch is enqueued
    offsets, chunks, at = {}, [], 0

    def place(in_size: int, out_size: int) -> tuple:
        nonlocal at
        key = (in_size, out_size)
        if key not in offsets:
            t = coeff_table(in_size, out_size, resample)
            offsets[key] = (at, t.shape[1] - 2)
            chunks.append(t.ravel())
            at += t.size
        return offsets[key]

    desc = (_lib.ResizeImage * len(pixels))()
    for i, img in enumerate(pixels):
        H, W = img.shape[0], img.shape[1]
        h_off, hk = place(W, width)
        v_off, vk = place(H, height)
        desc[i] = _lib.ResizeImage(img.data_ptr(), h_off, v_off, H, W, hk, vk)
    head = bytes(desc)                                   # 40 bytes per image: the tables stay 8-byte aligned
    from .. import packing
    buf = packing._to_device_async(head + np.concatenate(chunks).tobytes(), device)
    out = torch.empty((len(pixels), height, width, C), device=device, dtype=torch.uint8)
    _lib.call("vt_resize_u8_list", buf.data_ptr(), len(pixels), C, buf.data_ptr() + len(head), out.data_ptr(),
              height, width, _lib.stream_ptr(out))
    return out
