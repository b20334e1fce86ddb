"""The bandwidth-bound row-wise kernels (csrc/rowwise.cu, csrc/fp8_rowwise.cu) at every dispatch branch, element by
element against fp64 references of the same operation on the kernel's own stored inputs.

`launch_layernorm` picks one of ~30 compiled instances from dtype, alignment and the number of 16-byte vectors per
lane (VPL = ceil(dim / EV / 32), EV = 8 bf16 or 4 fp32 elements): the packed bf16 kernel (VPL 1-5), the rows kernel
(bf16 VPL 6, 7, 8, 10, 12, 16; fp32 and fp32 -> bf16 VPL 1-8, 10, 12, 16) and the generic kernel (dim % EV != 0, a
misaligned pointer, a stride that is not a multiple of EV, or a VPL without an instance).  The dims below run each of
them.  Inputs carry NaN in their pad columns (never read), outputs are filled with a NaN sentinel and carry guard
columns and rows that must still hold it afterwards, and row counts are 8k + 3 (a partial last block of 8 warps).
Every `vt_layernorm` launch is made twice back to back: the library flips the row traversal direction on every call,
so the two calls run in opposite directions and must agree bit for bit.

Per-element bound of the LayerNorm output, u = 2^-24, k = ceil(D / 32) + 6 (the longest chain of fp32 adds in a
warp's sum: ceil(D / 32) per lane, 5 shuffle levels, one spare); m, v = exact mean and variance, mean|x| the mean
magnitude of the row:
  * mean: the fp32 sum carries at most k u sum|x|, the division one more u|m|.  With the centred correction of the
    fp32 kernels (mean' = mean + sum(x - mean) / D) the error is that of the centred sum, (k + 1) u sum|x - mean|,
    plus u|m|: both are below e_mu = (k + 3) u (mean|x| + |m|);
  * variance: sum (x_i - mean)^2 / D = v + (m - mean)^2 exactly (the cross term vanishes), the fp32 centring,
    squares and sums add (k + 5) u of it: e_var = e_mu^2 + (k + 5) u (v + e_mu^2);
  * rstd = 1 / sqrtf(var + eps): at most 1 / sqrt(max(v - e_var, 0) + eps) = r_hi, off 1 / sqrt(v + eps) by at most
    r_hi - 1 / sqrt(v + eps) plus 3 roundings (add, sqrt, divide);
  * t = (x - mean) * rstd: |x - m| times the rstd error, plus (e_mu + one rounding of the centring) times r_hi, plus
    one rounding of the product;
  * out = gamma t + beta: |gamma| times the error of t, two roundings of |gamma t| + |beta|, then the output's own
    rounding (one bf16 ulp: half an ulp, the other half for a value that crossed a binade; fp32 output: one more u).
For e4m3 output (vt_layernorm_fp8) the same bound times the scale plus one rounding of the scaling gives an interval
around the fp64 value; the kernel's code must be the nearest e4m3 code of the fp64 value, or its neighbour when the
interval holds a rounding midpoint.

Softmax, p_i = exp(x_i - m), P = sum p: expf(x_i - m) carries the rounding of its argument (u |x_i - m| relative)
and expf's 2 ulps (4u); the sum k u P more plus the elements' own errors, the reciprocal and the product one u
each, then the output's rounding; expf results below the normal range add 2^-146 absolutely.

The rows with planted outliers come from test_gpu_kernels._outlier_rows (massive channels, |mean| / std = 100 and
1000, near-constant, constant and mixed rows).  Rows of one repeated value must give beta exactly.
"""
import math

import pytest
import torch
import torch.nn.functional as F

from test_gpu_kernels import OUTLIER_CASES, _outlier_rows
from test_gpu_persistent import (assert_elementwise, assert_guard, bit_equal, both_directions, dev, sentinel,
                                 ulp_bf16)

pytestmark = pytest.mark.gpu

U = 2.0 ** -24
LN_EPS = 1e-12
E4M3_MAX = 448.0
# values whose fp32 sum of D copies is not D times the value (rows of one repeated value)
CONST_VALUES = (100.7, -3.3, 0.1, 3333.3)


@pytest.fixture(autouse=True)
def _seed():
    torch.manual_seed(0)


def _lib():
    from vit.kernels import _lib
    return _lib


def _code(dtype):
    lib = _lib()
    return {torch.float32: lib.VT_F32, torch.bfloat16: lib.VT_BF16}[dtype]


def _stream():
    return torch.cuda.current_stream().cuda_stream


def _free():
    torch.cuda.synchronize()
    torch.cuda.empty_cache()


def padded(values, stride, offset=0):
    """A NaN-filled flat buffer holding `values` (rows, cols) at row stride `stride`, starting `offset` elements in;
    returns (buffer, the (rows, cols) view)."""
    rows, cols = values.shape
    buf = torch.full((offset + rows * stride + 8,), float("nan"), device=dev(), dtype=values.dtype)
    view = buf[offset:offset + rows * stride].view(rows, stride)[:, :cols]
    view.copy_(values)
    return buf, view


# ------------------------------------------------------------------------------------------------ LayerNorm
def ln_rows(rows, dim, dtype, seed):
    """rows x dim inputs: every outlier case of _outlier_rows (16 rows each), one row per CONST_VALUES value, the
    rest ordinary rows (randn * 2 + 0.5), stored in `dtype`."""
    g = torch.Generator().manual_seed(seed)
    parts = [_outlier_rows(case, 16, dim) for case in OUTLIER_CASES]
    parts.append(torch.tensor(CONST_VALUES, dtype=torch.float32)[:, None].expand(-1, dim))
    x = torch.cat(parts)
    assert x.shape[0] < rows
    x = torch.cat([x, torch.randn(rows - x.shape[0], dim, generator=g) * 2 + 0.5])
    return x.to(dev(), dtype)


def ln_params(dim, dtype, seed):
    g = torch.Generator().manual_seed(seed + 1)
    gamma = (1 + 0.2 * torch.randn(dim, generator=g)).to(dev(), dtype)
    beta = (0.2 * torch.randn(dim, generator=g)).to(dev(), dtype)
    return gamma, beta


def ln_ref_and_bound(x, gamma, beta, out_dtype=None, scale=1.0):
    """fp64 LayerNorm of the stored inputs (times scale) and the per-element bound of the module docstring (without
    the output rounding when out_dtype is None)."""
    x64, g64, b64 = x.double(), gamma.double(), beta.double()
    D = x.shape[1]
    k = math.ceil(D / 32) + 6
    m = x64.mean(1, keepdim=True)
    v = ((x64 - m) ** 2).mean(1, keepdim=True)
    ref = F.layer_norm(x64, (D,), g64, b64, LN_EPS)
    e_mu = (k + 3) * U * (x64.abs().mean(1, keepdim=True) + m.abs())
    e_var = e_mu ** 2 + (k + 5) * U * (v + e_mu ** 2)
    r_hi = 1.0 / ((v - e_var).clamp_min(0) + LN_EPS).sqrt()
    d_r = (r_hi - 1.0 / (v + LN_EPS).sqrt()) + 3 * U * r_hi
    dx = (x64 - m).abs()
    t_max = (dx + e_mu) * r_hi
    e_t = dx * d_r + (e_mu + U * (dx + e_mu)) * r_hi + U * t_max
    ga = g64.abs()
    err = ga * e_t + 2 * U * (ga * t_max + b64.abs())
    ref, err = ref * scale, err * scale + U * scale * (ref.abs() + err)
    if out_dtype == torch.bfloat16:
        err = err + ulp_bf16(ref.abs() + err)
    elif out_dtype == torch.float32:
        err = err + U * (ref.abs() + err)
    return ref, err


def constant_rows(x):
    """Indices of the rows that hold one repeated value."""
    return ((x == x[:, :1]).all(dim=1)).nonzero().flatten()


def run_layernorm(x, gamma, beta, out_dtype, in_stride=None, out_stride=None, x_offset=0):
    """vt_layernorm over x (rows, dim) stored at in_stride (NaN pad) and x_offset elements into its buffer, into
    sentinel-filled outputs at out_stride with a guard row: twice, in opposite directions, bit-identical; checked
    element by element against fp64 and for guards.  Returns the (rows, dim) result."""
    lib = _lib()
    rows, dim = x.shape
    in_stride = in_stride or dim
    out_stride = out_stride or dim
    _, xv = padded(x, in_stride, x_offset)
    n_out = (rows + 1) * out_stride

    def make():
        return (sentinel((n_out,), out_dtype),)

    def launch(out):
        lib.call("vt_layernorm", xv.data_ptr(), gamma.data_ptr(), beta.data_ptr(), out.data_ptr(), rows, dim,
                 in_stride, out_stride, LN_EPS, _code(x.dtype), _code(out_dtype), _stream())

    def view(out):
        return out[:rows * out_stride].view(rows, out_stride)[:, :dim]

    def check_fn(outs):
        out = outs[0]
        region = torch.zeros(n_out, dtype=torch.bool, device=dev())
        region[:rows * out_stride].view(rows, out_stride)[:, :dim] = True
        assert_guard(out, region, "layernorm output")
        ref, bound = ln_ref_and_bound(x, gamma, beta, out_dtype)
        assert_elementwise(view(out), ref, bound, what=f"layernorm {x.dtype}->{out_dtype} dim {dim}")

    first = both_directions(make, launch, check_fn)
    return view(first[0])


def assert_constant_rows_give_beta(x, gamma, beta, got):
    rows = constant_rows(x)
    assert rows.numel() > 0
    want = beta.to(got.dtype).expand(rows.numel(), -1)
    bad = ~(got[rows] == want)
    assert not bad.any(), (f"{int(bad.any(dim=1).sum())} of {rows.numel()} constant rows are not beta: row "
                           f"{int(rows[bad.any(dim=1)][0])} value {x[rows[bad.any(dim=1)][0], 0].item()}, worst "
                           f"|out - beta| {(got[rows].double() - want.double()).abs().max().item():.3g}")


ROWS = 8 * 24 + 3
# packed bf16 kernel: VPL 1-5; rows kernel: VPL 6, 7, 8, 10, 12, 16; VPL 9 (2304) has no instance: generic kernel
BF16_DIMS = [136, 512, 768, 1000, 1280, 1536, 1664, 2048, 2560, 3072, 4096, 2304]
# fp32 rows kernel: VPL 1-8, 10, 12, 16; VPL 9 (1152) and 33 (4100) take the generic kernel
F32_DIMS = [100, 256, 384, 500, 640, 768, 896, 1024, 1280, 1536, 2048, 1152, 4100]


@pytest.mark.parametrize("dim", BF16_DIMS)
def test_layernorm_bf16_every_instance(dim):
    x = ln_rows(ROWS, dim, torch.bfloat16, dim)
    gamma, beta = ln_params(dim, torch.bfloat16, dim)
    got = run_layernorm(x, gamma, beta, torch.bfloat16, in_stride=dim + 24, out_stride=dim + 16)
    assert_constant_rows_give_beta(x, gamma, beta, got)


@pytest.mark.parametrize("dim", F32_DIMS)
@pytest.mark.parametrize("out_dtype", [torch.float32, torch.bfloat16])
def test_layernorm_f32_every_instance(dim, out_dtype):
    x = ln_rows(ROWS, dim, torch.float32, dim)
    gamma, beta = ln_params(dim, torch.float32, dim)
    run_layernorm(x, gamma, beta, out_dtype, in_stride=dim + 12, out_stride=dim + 8)


@pytest.mark.parametrize("dim", [768, 1000, 1152, 2048, 4100])
@pytest.mark.parametrize("out_dtype", [torch.float32, torch.bfloat16])
def test_layernorm_f32_constant_rows_give_beta(dim, out_dtype):
    """A row of one repeated value has variance 0: LayerNorm gives beta.  sum / D of fp32 values is not exact, so
    the mean needs the centred correction; without it x - mean is a rounding residue that rstd = 1 / sqrt(eps)
    blows up to ~gamma."""
    x = ln_rows(ROWS, dim, torch.float32, dim)
    gamma, beta = ln_params(dim, torch.float32, dim)
    got = run_layernorm(x, gamma, beta, out_dtype, in_stride=dim + 12, out_stride=dim + 8)
    assert_constant_rows_give_beta(x, gamma, beta, got)


@pytest.mark.parametrize("route", ["dim", "pointer", "in_stride", "out_stride"])
@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16])
def test_layernorm_generic_routes(route, dtype):
    """The generic kernel through each way into it: dim % EV != 0, an input pointer one element past 16-byte
    alignment, an input or output row stride that is not a multiple of EV."""
    dim = {"dim": 770 if dtype == torch.bfloat16 else 766}.get(route, 768)
    x = ln_rows(8 * 19 + 3, dim, dtype, 7)
    gamma, beta = ln_params(dim, dtype, 7)
    kw = dict(in_stride=dim + 8, out_stride=dim + 8)
    if route == "pointer":
        kw["x_offset"] = 1
    elif route == "in_stride":
        kw["in_stride"] = dim + 3
    elif route == "out_stride":
        kw["out_stride"] = dim + 5
    got = run_layernorm(x, gamma, beta, dtype, **kw)
    if dtype == torch.bfloat16:
        assert_constant_rows_give_beta(x, gamma, beta, got)


def test_layernorm_c2_final_shape():
    """The final LayerNorm of the default forward at C2: 256 images x 197 tokens, D = 768, bf16."""
    x = (torch.randn(50432, 768, device=dev()) * 1.5 + 0.3).bfloat16()
    x[::97] = _outlier_rows("massive_channels", x[::97].shape[0], 768).to(dev()).bfloat16()
    gamma, beta = ln_params(768, torch.bfloat16, 768)
    run_layernorm(x, gamma, beta, torch.bfloat16)


def test_layernorm_over_2_31_elements():
    """One bf16 call over more than 2^31 elements (2^31 / 768 + 1024 rows): its last 1024 rows equal a call on just
    those rows bit for bit and match fp64; both directions agree."""
    lib = _lib()
    D, tail = 768, 1024
    rows = (2 ** 31 + D - 1) // D + tail
    x = torch.empty(rows, D, device=dev(), dtype=torch.bfloat16)
    for r0 in range(0, rows, 1 << 18):
        x[r0:r0 + (1 << 18)] = (torch.randn(min(1 << 18, rows - r0), D, device=dev()) * 2 + 0.5).bfloat16()
    x[-tail:-tail + 96] = torch.cat([_outlier_rows(c, 16, D) for c in OUTLIER_CASES]).to(dev()).bfloat16()
    gamma, beta = ln_params(D, torch.bfloat16, 3)
    outs = []
    for _ in range(2):      # back to back: opposite directions
        outs.append(torch.empty(rows, D, device=dev(), dtype=torch.bfloat16))
    for out in outs:
        lib.call("vt_layernorm", x.data_ptr(), gamma.data_ptr(), beta.data_ptr(), out.data_ptr(), rows, D, D, D,
                 LN_EPS, lib.VT_BF16, lib.VT_BF16, _stream())
    torch.cuda.synchronize()
    assert bit_equal(outs[0], outs[1]), "output depends on the traversal direction"
    del outs[1]
    big_tail = outs[0][-tail:].clone()
    del outs
    _free()
    own = run_layernorm(x[-tail:].contiguous(), gamma, beta, torch.bfloat16)
    assert bit_equal(big_tail, own), "the last rows of the large call differ from a call of their own"
    ref, bound = ln_ref_and_bound(x[-tail:], gamma, beta, torch.bfloat16)
    assert_elementwise(big_tail, ref, bound, what="layernorm tail rows")
    del x
    _free()


# ------------------------------------------------------------------------------------------------ FP8 LayerNorm
def e4m3_codes(v):
    """Nearest e4m3 codes (as decoded fp64) of fp64 values, saturating at +-448 like cvt.rn.satfinite."""
    return v.clamp(-E4M3_MAX, E4M3_MAX).float().to(torch.float8_e4m3fn).double()


def run_layernorm_fp8(x, gamma, beta, scale, in_stride, out_stride):
    """vt_layernorm_fp8 into a sentinel-filled buffer with guard bytes past dim and a guard row; returns the decoded
    (rows, dim) codes after checking guards and codes against fp64."""
    lib = _lib()
    rows, dim = x.shape
    _, xv = padded(x, in_stride)
    out = sentinel(((rows + 1) * out_stride,), torch.uint8)
    lib.call("vt_layernorm_fp8", xv.data_ptr(), gamma.data_ptr(), beta.data_ptr(), out.data_ptr(), rows, dim,
             in_stride, out_stride, LN_EPS, float(scale), _stream())
    torch.cuda.synchronize()
    region = torch.zeros_like(out, dtype=torch.bool)
    region[:rows * out_stride].view(rows, out_stride)[:, :dim] = True
    assert_guard(out, region, "e4m3 layernorm output")
    got = out[:rows * out_stride].view(rows, out_stride)[:, :dim].contiguous().view(torch.float8_e4m3fn).double()
    ref, err = ln_ref_and_bound(x, gamma, beta, None, scale)
    err = err + 2.0 ** -30 * ref.abs()       # the fp64 -> fp32 step of the reference cast
    want, lo, hi = e4m3_codes(ref), e4m3_codes(ref - err), e4m3_codes(ref + err)
    ok = (got >= lo) & (got <= hi)
    bad = ~ok
    if bad.any():
        r, c = bad.nonzero()[0].tolist()
        raise AssertionError(f"e4m3 layernorm dim {dim}: {int(bad.sum())} codes are neither the nearest code of the "
                             f"fp64 value nor its neighbour across a midpoint inside the fp32 error; first ({r}, {c}): "
                             f"got {got[r, c].item()}, fp64 {ref[r, c].item()} (nearest {want[r, c].item()}, "
                             f"error {err[r, c].item():.3g})")
    return got, ref


# VPL 1-8 (1664: VPL 7)
@pytest.mark.parametrize("dim", [136, 264, 768, 1024, 1280, 1536, 1664, 2048])
def test_layernorm_fp8_every_vpl(dim):
    x = ln_rows(ROWS, dim, torch.bfloat16, dim)
    gamma, beta = ln_params(dim, torch.bfloat16, dim)
    run_layernorm_fp8(x, gamma, beta, 16.0, in_stride=dim + 16, out_stride=dim + 24)


def _block_with_layernorm(dim, gamma, beta):
    from vit.vit import Transformer
    block = Transformer(num_heads=dim // 64, d_in=dim, d_out=64).to(dev(), torch.bfloat16)
    with torch.no_grad():
        block.layernorm_before.weight.copy_(gamma)
        block.layernorm_before.bias.copy_(beta)
    return block


@pytest.mark.parametrize("dim", [1024, 1280])
def test_layernorm_fp8_does_not_saturate_at_the_pack_scale(dim):
    """One-hot rows (|y| = sqrt(D - 1) on the channel of the largest |gamma|) and massive-channel rows, quantised at
    the activation scale the FP8 pack divides out of the QKV layer: no element may reach e4m3's saturation, so every
    code is the nearest code of LN(x) * scale and none is +-448."""
    from vit import packing
    g = torch.Generator().manual_seed(dim)      # the oracle's LayerNorm init
    gamma = (1 + 0.02 * torch.randn(dim, generator=g)).to(dev(), torch.bfloat16)
    beta = (0.02 * torch.randn(dim, generator=g)).to(dev(), torch.bfloat16)
    block = _block_with_layernorm(dim, gamma, beta)
    q8 = block.packed("fp8")
    _, s_w = packing.quantize_weight_fp8(block.attention.packed().wqkv)
    scales = (s_w / q8.cqkv).unique()
    assert scales.numel() == 1
    scale = float(scales[0])
    c = int(gamma.float().abs().argmax())
    one_hot = torch.zeros(16, dim)
    one_hot[:, c] = torch.logspace(-3, 3, 16)
    one_hot[8:, c] *= -1
    x = torch.cat([one_hot, _outlier_rows("massive_channels", 32, dim)]).to(dev(), torch.bfloat16)
    x = torch.cat([x, (torch.randn(ROWS - x.shape[0], dim, device=dev()) * 2).bfloat16()])
    ref = ln_ref_and_bound(x, gamma, beta, None, scale)[0]
    assert ref.abs().max().item() < E4M3_MAX, (f"scale {scale}: |LN(x)| * scale reaches {ref.abs().max().item():.1f}, "
                                               f"e4m3 saturates at 448")
    got, ref = run_layernorm_fp8(x, gamma, beta, scale, in_stride=dim, out_stride=dim + 8)
    assert not ((got.abs() == E4M3_MAX) & (ref.abs() < E4M3_MAX)).any()


def test_layernorm_fp8_rejects_dim_above_2048():
    """dim > 2048 (VPL > 8) has no instance: VT_ERR_UNSUPPORTED, and nothing is written."""
    lib = _lib()
    rows, dim = 11, 2056
    x = torch.randn(rows, dim, device=dev()).bfloat16()
    gamma, beta = ln_params(dim, torch.bfloat16, 1)
    out = sentinel((rows * dim,), torch.uint8)
    rc = lib.load().vt_layernorm_fp8(x.data_ptr(), gamma.data_ptr(), beta.data_ptr(), out.data_ptr(), rows, dim, dim,
                                     dim, LN_EPS, 16.0, _stream())
    torch.cuda.synchronize()
    assert rc == lib.VT_ERR_UNSUPPORTED
    assert_guard(out, torch.zeros_like(out, dtype=torch.bool), "rejected e4m3 layernorm")


# ------------------------------------------------------------------------------------------------ weight quantisation
def quantize_restatement(w):
    """The kernel's arithmetic in torch, on the CPU: s = amax / 448 in fp32 (1 when that is not a normal float),
    inv = 1 / s, w * inv in fp32, clamp +-448, round to nearest even e4m3."""
    wf = w.float().cpu()
    amax = wf.abs().amax(dim=1)
    s = amax / 448.0
    s = torch.where(s >= 2.0 ** -126, s, torch.ones_like(s))
    inv = 1.0 / s
    q = (wf * inv[:, None]).clamp(-E4M3_MAX, E4M3_MAX).to(torch.float8_e4m3fn)
    return q.view(torch.uint8), s


def run_quantize(w, ldw, ldo):
    lib = _lib()
    N, K = w.shape
    _, wv = padded(w, ldw)
    out = sentinel(((N + 1) * ldo,), torch.uint8)
    scales = sentinel((N + 3,), torch.float32)
    lib.call("vt_quantize_rows_fp8", wv.data_ptr(), ldw, out.data_ptr(), ldo, scales.data_ptr(), N, K, _stream())
    torch.cuda.synchronize()
    region = torch.zeros_like(out, dtype=torch.bool)
    region[:N * ldo].view(N, ldo)[:, :K] = True
    assert_guard(out, region, "e4m3 weights")
    sreg = torch.zeros_like(scales, dtype=torch.bool)
    sreg[:N] = True
    assert_guard(scales, sreg, "weight scales")
    return out[:N * ldo].view(N, ldo)[:, :K].cpu(), scales[:N].cpu()


def _rounds_above_448(n):
    """bf16 values a whose fp32 a * (1 / (a / 448)) is above 448 (the clamp / satfinite path)."""
    a = (torch.rand(1 << 16) * 8 + 0.01).bfloat16().float()
    v = a * (1.0 / (a / 448.0))
    found = a[v > 448.0]
    assert found.numel() >= n
    return found[:n]


def test_quantize_rows_fp8_bit_exact():
    """Scales and codes bit for bit against the restatement: N % 8 != 0, K % 128 != 0, NaN between K and ldw, guard
    bytes between K and ldo, an all-zero row, rows whose max element rounds above 448."""
    N, K = 203, 772
    w = torch.randn(N, K) * torch.logspace(-4, 2, N)[:, None]
    w[5] = 0.0
    big = _rounds_above_448(4)
    for i, a in enumerate(big):
        w[17 + i] = torch.randn(K).clamp(-1, 1) * a * 0.9
        w[17 + i, 3 + i] = a * (-1) ** i
    w = w.bfloat16()
    codes, scales = run_quantize(w.to(dev()), K + 12, K + 8)
    want_codes, want_scales = quantize_restatement(w)
    assert torch.equal(scales.view(torch.int32), want_scales.view(torch.int32)), "scales differ"
    diff = codes != want_codes
    assert not diff.any(), f"{int(diff.sum())} codes differ, first at {diff.nonzero()[0].tolist()}"
    assert (codes[5] == 0).all() and scales[5].item() == 1.0
    dec = codes.view(torch.float8_e4m3fn).float()
    assert (dec[17:21].abs().amax(dim=1) == E4M3_MAX).all()
    assert torch.isfinite(dec).all()


def test_quantize_rows_fp8_near_zero_row():
    """A row whose amax / 448 is subnormal has no finite reciprocal: it takes scale 1 and quantises to zero codes,
    no NaN; the other rows are unaffected."""
    N, K = 11, 260
    w = torch.randn(N, K)
    w[3] = 0.0
    w[3, :3] = torch.tensor([1e-37, 0.0, -3e-38])
    w[7] = 0.0
    w[7, 100] = 2e-36
    w = w.bfloat16()
    codes, scales = run_quantize(w.to(dev()), K, K + 4)
    want_codes, want_scales = quantize_restatement(w)
    dec = codes.view(torch.float8_e4m3fn).float()
    assert torch.isfinite(dec).all(), f"{int((~torch.isfinite(dec)).sum())} NaN codes"
    assert scales[3].item() == 1.0 and scales[7].item() == 1.0 and (dec[3] == 0).all() and (dec[7] == 0).all()
    assert torch.equal(scales.view(torch.int32), want_scales.view(torch.int32))
    assert torch.equal(codes, want_codes)


# ------------------------------------------------------------------------------------------------ softmax
def softmax_rows(rows, cols, dtype, seed):
    g = torch.Generator().manual_seed(seed)
    hi = 80.0 if dtype == torch.float32 else 20.0
    x = torch.randn(rows, cols, generator=g) * 3
    x[0] = torch.linspace(-hi, hi, cols)                      # logits over the full range
    x[1] = torch.rand(cols, generator=g) * 2 * hi - hi
    x[2] = 1.7                                                # one repeated value
    x[3, 1::3] = float("-inf")                                # -inf entries (never a whole row)
    x[4, 1:] = float("-inf")
    x[5] = x[5] * 10 - 40
    return x.to(dev(), dtype)


def softmax_ref_and_bound(x, out_dtype):
    x64 = x.double()
    cols = x.shape[1]
    k = math.ceil(cols / 32) + 5
    m = x64.amax(1, keepdim=True)
    d = (x64 - m).nan_to_num(neginf=0.0).abs()
    ref = torch.softmax(x64, dim=1)
    delta = U * d + 4 * U
    rho = (ref * delta).sum(1, keepdim=True) + k * U * (1 + delta.amax(1, keepdim=True))
    err = ref * (delta + rho + 3 * U) * (1 + 1e-3) + 2.0 ** -146
    if out_dtype == torch.bfloat16:
        err = err + ulp_bf16(ref + err)
    return ref, err


def run_softmax(x, in_stride):
    lib = _lib()
    rows, cols = x.shape
    _, xv = padded(x, in_stride)
    out = sentinel(((rows + 1) * cols,), x.dtype)
    lib.call("vt_softmax", xv.data_ptr(), out.data_ptr(), rows, cols, in_stride, _code(x.dtype), _stream())
    torch.cuda.synchronize()
    region = torch.zeros_like(out, dtype=torch.bool)
    region[:rows * cols] = True
    assert_guard(out, region, "softmax output")
    return out[:rows * cols].view(rows, cols)


@pytest.mark.parametrize("cols", [1, 31, 32, 33, 197, 577, 1025, 4097])
@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16])
def test_softmax_against_fp64(cols, dtype):
    x = softmax_rows(8 * 5 + 3, cols, dtype, cols)
    got = run_softmax(x, cols + 7)
    ref, bound = softmax_ref_and_bound(x, dtype)
    assert_elementwise(got, ref, bound, what=f"softmax {dtype} cols {cols}")
    assert (got[2] == got[2][0]).all(), "a row of one repeated value must come out uniform"


def test_softmax_over_2_31_elements():
    """One bf16 call over more than 2^31 elements (2^31 / 1025 + 1024 rows of 1025: fp32 output_attentions of 256
    images at 512^2 reaches 3.2e9 per layer): the last 1024 rows equal a call of their own bit for bit and match
    fp64."""
    lib = _lib()
    C, tail = 1025, 1024
    rows = (2 ** 31 + C - 1) // C + tail
    x = torch.empty(rows, C, device=dev(), dtype=torch.bfloat16)
    for r0 in range(0, rows, 1 << 18):
        x[r0:r0 + (1 << 18)] = (torch.randn(min(1 << 18, rows - r0), C, device=dev()) * 4).bfloat16()
    x[-tail:-tail + 6] = softmax_rows(6, C, torch.bfloat16, 5)
    out = torch.empty(rows, C, device=dev(), dtype=torch.bfloat16)
    lib.call("vt_softmax", x.data_ptr(), out.data_ptr(), rows, C, C, lib.VT_BF16, _stream())
    torch.cuda.synchronize()
    big_tail = out[-tail:].clone()
    del out
    _free()
    own = run_softmax(x[-tail:].contiguous(), C)
    assert bit_equal(big_tail, own), "the last rows of the large call differ from a call of their own"
    ref, bound = softmax_ref_and_bound(x[-tail:], torch.bfloat16)
    assert_elementwise(big_tail, ref, bound, what="softmax tail rows")
    del x
    _free()


# ------------------------------------------------------------------------------------------------ add, pool, gather
@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16])
@pytest.mark.parametrize("n", [1, 7, 4099, 3 * 2 ** 22 + 5])
@pytest.mark.parametrize("offsets", [(0, 0, 0), (1, 0, 0), (0, 1, 0), (0, 0, 1), "inplace"])
def test_add_bit_exact(dtype, n, offsets):
    """vt_add == torch a + b bit for bit: 16-byte vectors (four in flight, then the remainder loop) with a scalar
    tail, the scalar kernel when a, b or out is one element off alignment, and out = a in place."""
    lib = _lib()
    inplace = offsets == "inplace"
    oa, ob, oo = (0, 0, 0) if inplace else offsets
    a_buf = torch.randn(n + 2, device=dev()).to(dtype)
    b_buf = torch.randn(n + 2, device=dev()).to(dtype)
    a, b = a_buf[oa:oa + n], b_buf[ob:ob + n]
    want = a + b
    if inplace:
        out_buf, out = a_buf, a
    else:
        out_buf = sentinel((n + 2,), dtype)
        out = out_buf[oo:oo + n]
    lib.call("vt_add", a.data_ptr(), b.data_ptr(), out.data_ptr(), n, _code(dtype), _stream())
    torch.cuda.synchronize()
    assert bit_equal(out, want), f"{int((_bits_of(out) != _bits_of(want)).sum())} elements differ"
    if not inplace:
        region = torch.zeros(n + 2, dtype=torch.bool, device=dev())
        region[oo:oo + n] = True
        assert_guard(out_buf, region, "add output")


def _bits_of(t):
    return t.view(torch.int32 if t.dtype == torch.float32 else torch.int16)


@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16])
def test_pool_cls_bit_exact(dtype):
    """vt_pool_cls: out[b] = x[b, 0, :] with a batch stride larger than N * D; a guard row after the output."""
    lib = _lib()
    B, N, D = 37, 197, 768
    stride = N * D + 40
    x = torch.randn(B * stride, device=dev()).to(dtype)
    out = sentinel(((B + 1) * D,), dtype)
    lib.call("vt_pool_cls", x.data_ptr(), out.data_ptr(), B, D, stride, _code(dtype), _stream())
    torch.cuda.synchronize()
    want = x.view(B, stride)[:, :D]
    assert bit_equal(out[:B * D].view(B, D), want)
    region = torch.zeros_like(out, dtype=torch.bool)
    region[:B * D] = True
    assert_guard(out, region, "pool output")


@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16])
def test_gather_rows_bit_exact(dtype):
    """vt_gather_rows with repeated and descending indices into rows of stride ldo > cols (guards between), and
    rows = 0 returning 0 without writing."""
    lib = _lib()
    M, ldx, cols, ldo = 1000, 800, 777, 792
    x = torch.randn(M, ldx, device=dev()).to(dtype)
    idx = torch.tensor([999, 998, 500, 500, 3, 0, 0, 999, 42] + list(range(900, 700, -7)), device=dev())
    rows = idx.numel()
    out = sentinel(((rows + 1) * ldo,), dtype)
    lib.call("vt_gather_rows", x.data_ptr(), ldx, idx.data_ptr(), out.data_ptr(), ldo, rows, cols, _code(dtype),
             _stream())
    torch.cuda.synchronize()
    assert bit_equal(out[:rows * ldo].view(rows, ldo)[:, :cols], x[idx, :cols])
    region = torch.zeros_like(out, dtype=torch.bool)
    region[:rows * ldo].view(rows, ldo)[:, :cols] = True
    assert_guard(out, region, "gather output")
    empty = sentinel((ldo,), dtype)
    rc = lib.load().vt_gather_rows(x.data_ptr(), ldx, idx.data_ptr(), empty.data_ptr(), ldo, 0, cols, _code(dtype),
                                   _stream())
    torch.cuda.synchronize()
    assert rc == 0
    assert_guard(empty, torch.zeros_like(empty, dtype=torch.bool), "gather of zero rows")
