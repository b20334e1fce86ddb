"""CPU: the image-processor resize — include/vitb200_preprocess.h, the exports of libvitb200.so and the
PREPROCESS_SIGNATURES ctypes table agree in both directions and stay apart from the other headers and tables; argument
rejection without a launch; the host coefficient tables, applied with the kernel's integer rule, equal PIL.Image.resize
byte for byte; the table validator; the host-side refusals of ``resize_uint8`` and ``do_resize`` (no compute calls:
there is no GPU here)."""
import ctypes
import os
import re

import numpy as np
import pytest
import torch
from PIL import Image

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
HEADER = os.path.join(ROOT, "include", "vitb200_preprocess.h")
OTHER_HEADERS = [os.path.join(ROOT, "include", h) for h in
                 ("vitb200.h", "vitb200_resolution.h", "vitb200_ragged.h", "vitb200_mask.h", "vitb200_attn.h")]

_CTYPE = {"int32_t": ctypes.c_int32, "int64_t": ctypes.c_int64, "float": ctypes.c_float}
NAMES = {"vt_resize_u8", "vt_resize_u8_list"}

# (H, W) inputs of tests/test_gpu_resize.py, resized to 224 x 224 there
GPU_SIZES = [(1, 1), (1, 300), (300, 1), (16, 16), (8000, 60), (97, 1201), (375, 500), (223, 225), (224, 100),
             (224, 224), (17, 300), (1000, 37), (4000, 4500)]


def _declarations(path):
    text = re.sub(r"/\*.*?\*/", "", open(path).read(), flags=re.S)
    decls = {}
    for m in re.finditer(r"\b(int|const char\*)\s+(vt_\w+)\s*\(([^)]*)\)\s*;", text):
        args = [a.strip() for a in m.group(3).split(",")] if m.group(3).strip() != "void" else []
        decls[m.group(2)] = args
    return decls


def _lib():
    from vit.kernels import _lib
    if not os.path.exists(_lib.lib_path()):
        import __graft_entry__
        __graft_entry__.build()
    return _lib


def pil_order_resize(img: np.ndarray, htab: np.ndarray, vtab: np.ndarray) -> np.ndarray:
    """(H, W, C) uint8 -> (out_h, out_w, C) with the kernel's integer rule: per pass clamp((2^21 + sum in * w) >> 22),
    width pass first into uint8, except height first for H > 100 W with a shrinking height (PIL 12's Image.resize)."""
    def one_pass(a, table, axis):
        a = np.moveaxis(a, axis, 0).astype(np.int64)
        out = np.empty((table.shape[0],) + a.shape[1:], np.int64)
        for o in range(table.shape[0]):
            s, n = int(table[o, 0]), int(table[o, 1])
            acc = (1 << 21) + np.tensordot(table[o, 2:2 + n].astype(np.int64), a[s:s + n], axes=(0, 0))
            out[o] = np.clip(acc >> 22, 0, 255)
        return np.moveaxis(out, 0, axis).astype(np.uint8)
    H, W = img.shape[:2]
    if H > 100 * W and vtab.shape[0] < H:
        return one_pass(one_pass(img, vtab, 0), htab, 1)
    return one_pass(one_pass(img, htab, 1), vtab, 0)


def _check_against_pil(rng, h, w, oh, ow, resample, channels):
    from vit.kernels.resize import coeff_table
    shape = (h, w, channels) if channels == 3 else (h, w)
    img = rng.integers(0, 256, shape, dtype=np.uint8)
    want = np.asarray(Image.fromarray(img, "RGB" if channels == 3 else "L").resize((ow, oh), resample))
    got = pil_order_resize(img.reshape(h, w, channels), coeff_table(w, ow, resample), coeff_table(h, oh, resample))
    assert np.array_equal(got.reshape(want.shape), want), f"{(h, w)} -> {(oh, ow)}, resample {resample}, C {channels}"


# --------------------------------------------------------------------------------------------------------- ABI
def test_preprocess_header_declares_expected_entry_points():
    assert set(_declarations(HEADER)) == NAMES
    assert '#include "vitb200.h"' in open(HEADER).read()


def test_preprocess_entry_points_are_not_in_the_other_headers():
    for path in OTHER_HEADERS:
        assert not NAMES & set(_declarations(path)), path
        assert not set(_declarations(path)) & set(_declarations(HEADER)), path


def test_library_exports_every_preprocess_symbol_and_ctypes_match():
    mod = _lib()
    lib = mod.load()
    decls = _declarations(HEADER)
    assert set(mod.PREPROCESS_SIGNATURES) == set(decls)
    assert not set(mod.PREPROCESS_SIGNATURES) & (set(mod.SIGNATURES) | set(mod.RESOLUTION_SIGNATURES)
                                                 | set(mod.RAGGED_SIGNATURES) | set(mod.MASK_SIGNATURES)
                                                 | set(mod.ATTN_SIGNATURES))
    for name, argtypes in mod.PREPROCESS_SIGNATURES.items():
        fn = getattr(lib, name)
        assert fn.argtypes == argtypes and fn.restype == ctypes.c_int, f"{name}: not registered by load()"
        args = decls[name]
        assert len(args) == len(argtypes), f"{name}: header has {len(args)} args, ctypes {len(argtypes)}"
        for a, ct in zip(args, argtypes):
            if "*" in a:
                assert ct == ctypes.c_void_p, f"{name}: {a}"
            else:
                assert _CTYPE[a.split()[0]] == ct, f"{name}: {a} vs {ct}"


def test_resize_descriptor_layout():
    mod = _lib()
    assert ctypes.sizeof(mod.ResizeImage) == 40
    assert [f[0] for f in mod.ResizeImage._fields_] == ["pixels", "htab", "vtab", "height", "width", "hk", "vk"]
    text = open(HEADER).read()
    assert re.search(r"const void\* pixels;.*int64_t htab;.*int64_t vtab;.*int32_t height;.*int32_t width;"
                     r".*int32_t hk;.*int32_t vk;", text, flags=re.S)


def test_resize_rejects_bad_arguments_without_a_launch():
    """Argument checks run on the host before anything touches the device (all pointers here are fake)."""
    lib = _lib().load()
    f = 1 << 20
    ok = (f, 2, 10, 12, 3, 360, f, 3, f, 3, f, 224, 224, None)
    bad = [(None, 0), (0, 1), (0, 2), (0, 3), (0, 4), (0, 5), (5, 5), (None, 6), (0, 7), (None, 8), (0, 9),
           (None, 10), (0, 11), (-1, 12), (0, 12)]
    for value, pos in bad:
        args = list(ok)
        args[pos] = value
        assert lib.vt_resize_u8(*args) == -1, (pos, value)
    assert lib.vt_resize_u8(f, 2, 10, 12, 3, 359, f, 3, f, 3, f, 224, 224, None) == -1      # stride < H * W * C
    okl = (f, 4, 3, f, f, 224, 224, None)
    for value, pos in [(None, 0), (0, 1), (-3, 1), (0, 2), (5, 2), (None, 3), (None, 4), (0, 5), (0, 6), (-2, 6)]:
        args = list(okl)
        args[pos] = value
        assert lib.vt_resize_u8_list(*args) == -1, (pos, value)


# ------------------------------------------------------------------------------------------------ tables vs PIL
@pytest.mark.parametrize("resample", [2, 3])
def test_tables_equal_pil_for_every_size_pair_up_to_40(resample):
    rng = np.random.default_rng(resample)
    for n_in in range(1, 41):
        for n_out in range(1, 41):
            channels = 1 if (n_in + n_out) % 2 else 3
            # one axis n_in -> n_out, the other a fixed non-square pair, so both passes are exercised
            _check_against_pil(rng, n_in, 7, n_out, 5, resample, channels)
            _check_against_pil(rng, 6, n_in, 9, n_out, resample, 4 - channels)


@pytest.mark.parametrize("resample", [2, 3])
@pytest.mark.parametrize("channels", [1, 3])
def test_tables_equal_pil_at_model_sizes(resample, channels):
    rng = np.random.default_rng(10 * resample + channels)
    cases = [(h, w, 224, 224) for h, w in GPU_SIZES if h * w <= 2_000_000]
    cases += [(375, 500, 384, 384), (256, 256, 224, 224), (224, 300, 224, 224), (300, 224, 224, 224),  # one axis equal
              (50, 80, 300, 200), (1200, 30, 100, 40), (20000, 3, 224, 224), (6001, 60, 224, 224),
              (6000, 60, 224, 224)]
    for _ in range(6):                                     # random sizes up to 4096 (kept small in area)
        h, w = int(rng.integers(1, 4097)), int(rng.integers(1, 200))
        if rng.integers(2):
            h, w = w, h
        cases.append((h, w, int(rng.integers(1, 400)), int(rng.integers(1, 400))))
    for h, w, oh, ow in cases:
        _check_against_pil(rng, h, w, oh, ow, resample, channels)


# ------------------------------------------------------------------------------------------------ the validator
def test_validator_accepts_every_table_of_the_sweeps():
    from vit.kernels.resize import coeff_table, validate_table
    sizes = [(i, o) for i in range(1, 41) for o in range(1, 41)]
    sizes += [(s, 224) for hw in GPU_SIZES for s in hw] + [(20000, 224), (4096, 1), (1, 4096), (4096, 4095)]
    for resample in (2, 3):
        for n_in, n_out in sizes:
            t = coeff_table(n_in, n_out, resample)
            validate_table(np.array(t), n_in)
            assert t.shape[0] == n_out and not t.flags.writeable


def test_validator_rejects_corrupted_tables():
    from vit.kernels.resize import coeff_table, validate_table
    good = np.array(coeff_table(500, 224, 3))
    k = good.shape[1] - 2

    def corrupt(fn):
        t = good.copy()
        fn(t)
        return t

    bad = [corrupt(lambda t: t.__setitem__((0, 0), -1)),                       # negative start
           corrupt(lambda t: t.__setitem__((5, 1), 0)),                        # no taps
           corrupt(lambda t: t.__setitem__((5, 1), k + 1)),                    # more taps than weights
           corrupt(lambda t: t.__setitem__((223, 0), 500 - int(t[223, 1]) + 1)),  # past the input
           corrupt(lambda t: t.__setitem__((100, 0), int(t[99, 0]) - 1)),      # start going back
           corrupt(lambda t: t.__setitem__((100, 1), int(t[100, 1]) - 3)),     # end going back
           good.astype(np.int64), good[:, :2], good[None], good[:0]]
    for t in bad:
        with pytest.raises(AssertionError):
            validate_table(t, 500)
    validate_table(good, 500)
    with pytest.raises(AssertionError):
        validate_table(good, 499)                                              # the same table for a smaller input


def test_identity_table_gives_the_input_bytes():
    from vit.kernels.resize import coeff_table
    rng = np.random.default_rng(3)
    img = rng.integers(0, 256, (37, 53, 3), dtype=np.uint8)
    for resample in (2, 3):
        assert np.array_equal(pil_order_resize(img, coeff_table(53, 53, resample), coeff_table(37, 37, resample)), img)


# ------------------------------------------------------------------------------------------- host-side refusals
def _tiny(**kw):
    from oracle import hf_oracle
    from vit.vit import VIT
    return VIT(**hf_oracle.vit_kwargs("tiny-b"), **kw)


@pytest.fixture
def no_launch(monkeypatch):
    from vit.kernels import _lib as lib
    calls = []
    monkeypatch.setattr(lib, "call", lambda name, *a: calls.append(name))
    yield calls
    assert calls == []


def test_resample_codes(no_launch):
    from PIL.Image import Resampling
    from transformers.image_utils import PILImageResampling
    from vit.kernels.resize import check_resample
    assert check_resample(2) == 2 and check_resample(3) == 3
    assert check_resample(Resampling.BILINEAR) == 2 and check_resample(PILImageResampling.BICUBIC) == 3
    for bad in (0, 1, 4, 5, True, "bilinear", None, Resampling.LANCZOS):
        with pytest.raises(AssertionError, match=r"2 \(PIL BILINEAR\) or 3 \(PIL BICUBIC\)"):
            check_resample(bad)


def test_resize_uint8_refusals(no_launch, monkeypatch):
    from vit.kernels import resize_uint8
    from vit.kernels import resize as rz
    x = torch.zeros(2, 30, 40, 3, dtype=torch.uint8)
    cases = [((x.float(), 8, 8), "uint8"), (([x[0].float()], 8, 8), "uint8"), (([], 8, 8), "at least one image"),
             ((x[:, :0], 8, 8), "side < 1"), (([x[0], x[1, :, :0]], 8, 8), "side < 1"), ((x[:0], 8, 8), "at least one"),
             ((torch.zeros(2, 3, 4, 5, dtype=torch.uint8), 8, 8), "channels"), ((x[0], 8, 8), r"\(B, H, W, C\)"),
             (([x[0], x[1, ..., :2]], 8, 8), "one channel count"),
             (([x[0], torch.zeros(3, 4, 3, dtype=torch.uint8, device="meta")], 8, 8), "one device"),
             ((x, 0, 8), "at least 1x1"), ((x, 8, 8), "CUDA device"), (([x[0]], 8, 8), "CUDA device")]
    for args, match in cases:
        with pytest.raises(AssertionError, match=match):
            resize_uint8(*args)
    with pytest.raises(AssertionError, match="2 \\(PIL BILINEAR\\)"):
        resize_uint8(x, 8, 8, resample=1)
    monkeypatch.setattr(torch.cuda, "is_available", lambda: True)
    monkeypatch.setattr(torch.cuda, "is_current_stream_capturing", lambda: True)
    with pytest.raises(AssertionError, match="list of images cannot be resized under CUDA-graph capture"):
        resize_uint8([x[0], x[1]], 8, 8)
    with pytest.raises(AssertionError, match="run the call once before capturing"):
        rz._batch_tables(torch.device("cuda", 0), 31, 41, 8, 8, 2)


def test_do_resize_refusals(no_launch):
    model = _tiny(add_pooling_layer=True, num_labels=5)
    x8 = torch.zeros(2, 50, 70, 3, dtype=torch.uint8)
    bad = [(x8.float(), "uint8"), ([x8[0].float()], "uint8"), (x8[..., :1], "channels"), ([], "at least one image"),
           ([x8[0], x8[1, :0]], "side < 1"), ([x8[0], torch.zeros(3, 4, 3, dtype=torch.uint8, device="meta")], "device"),
           (x8, "CUDA device"), ([x8[0], x8[1]], "CUDA device")]
    for inp, match in bad:
        for fn in (model.forward_uint8, model.pooled, model.pooler_output, model.logits):
            with pytest.raises(AssertionError, match=match):
                fn(inp, do_resize=True)
    for fn in (model.forward_uint8, model.pooled, model.pooler_output, model.logits):
        with pytest.raises(AssertionError, match="PIL BILINEAR"):
            fn(x8, do_resize=True, resample=0)
    # already the model's size: nothing to resize, the same tensor goes on (and fails only at the device here)
    native = torch.zeros(2, model.height, model.width, 3, dtype=torch.uint8)
    assert model._resized(native, True, 2) is native
    assert model._resized(x8, False, 2) is x8


def test_do_resize_defaults_leave_signatures_compatible():
    import inspect
    from vit.vit import VIT
    for name in ("forward_uint8", "pooled", "pooler_output", "logits"):
        params = inspect.signature(getattr(VIT, name)).parameters
        assert params["do_resize"].default is False and params["resample"].default == 2
        assert list(params)[-2:] == ["do_resize", "resample"]
