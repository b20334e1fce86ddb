"""The persistent kernels past their first work item: the 2-CTA GEMM (csrc/gemm2_sm100.cu, also the token-mode patch
embedding) and the attention kernels (csrc/attn5_sm100.cu) at sizes where every group / CTA walks many tiles, in both
traversal directions, under restricted grids, element by element against fp64 references of the same operation on
the kernel's own operands.

Why these cases.  A GEMM group takes supertiles g, g + groups, ... and an attention CTA takes (image, head) pairs
blockIdx.x, + grid, ...; the TMEM accumulator double buffer, the operand-ring and staging phases, the epilogue's
one-tile-ahead prefetch of bias / column sums / LayerNorm row statistics and the pacing all start to matter from a
group's second tile on.  `vt_debug_set_sm_partition` caps the grid so a few groups (down to one) walk every tile at
small sizes; the production sizes (C2: 256 images of 197 tokens) give ~8-32 supertiles per group at full grid.

Every launch goes through `both_directions`: two consecutive library calls, which walk the row tiles (images) in
opposite orders (api.cu flips the direction on every hot-path call), into separate sentinel-filled buffers that must
come out bit-identical.  Outputs carry guard columns / rows / images that must still hold the sentinel afterwards.

Per-element bound of a bf16 GEMM output (derived here, used by every GEMM case):
  * one rounding of the output: 1 bf16 ulp of the reference value (1 e4m3 ulp for e4m3 output) -- round-to-nearest
    is half an ulp; the other half covers a pre-rounding value that crossed into the next binade;
  * the fp32 accumulation: the tensor core adds into its fp32 accumulator with truncation (DESIGN.md section 4), so
    one ulp (2^-23 relative) per add, K adds, each at most sum_k |a_k b_k|:  K * 2^-23 * (|A| . |B|)_ij;
  * the fp32 epilogue (bias, column scale, residual, LayerNorm fold): EPI_OPS * 2^-23 times the sum of the
    magnitudes of the terms it combines, and for the LayerNorm fold a relative error RSTD_REL on rstd (fp32 merge of
    up to ten (sum, M2) partials and rsqrtf: some 20 fp32 ulps; 2^-18 is 32 ulps);
  * GELU: the error of its input times max |gelu'| (1.13) plus the approximation error of gelu_erf_poly_x2,
    5.6e-7 absolute with an exact exp2 (csrc/common.cuh), plus ex2.approx's relative error (2^-22) on a term of at
    most 0.17 (0.5|x| erfc(|x|/sqrt 2)), 4e-8: GELU_ABS = 1e-6 leaves 4e-7 for the evaluation order.
"""
import contextlib
import ctypes
import math

import pytest
import torch

pytestmark = pytest.mark.gpu

EPS32 = 2.0 ** -23
EPI_OPS = 4
RSTD_REL = 2.0 ** -18
GELU_SLOPE = 1.13
GELU_ABS = 1e-6
LN_EPS = 1e-12

BF16_SENTINEL = 0x7FC0        # bf16 quiet NaN
E4M3_SENTINEL = 0x7F          # e4m3fn NaN
F32_SENTINEL = 0x7FC00000     # fp32 quiet NaN


@pytest.fixture(autouse=True)
def _seed():
    torch.manual_seed(0)


def dev():
    return torch.device("cuda:0")


def _lib():
    from vit.kernels import _lib
    return _lib


@contextlib.contextmanager
def sm_partition(gemm_groups, attn_ctas):
    """Cap the 2-CTA GEMM at `gemm_groups` groups of four CTAs and attn5 at `attn_ctas` CTAs (0 = all SMs); the cap is
    read at launch time.  Always back to (0, 0) on the way out, also when the body fails."""
    fn = _lib().load().vt_debug_set_sm_partition
    fn.argtypes = [ctypes.c_int, ctypes.c_int]
    fn.restype = None
    fn(gemm_groups, attn_ctas)
    try:
        yield
    finally:
        fn(0, 0)


# ------------------------------------------------------------------------------------------------ buffers and checks
def _bits(t):
    """The raw bits of a buffer, as integers of the same width."""
    return t.view({torch.bfloat16: torch.int16, torch.uint8: torch.uint8, torch.float32: torch.int32}[t.dtype])


def sentinel(shape, dtype):
    bits = {torch.bfloat16: BF16_SENTINEL, torch.uint8: E4M3_SENTINEL, torch.float32: F32_SENTINEL}[dtype]
    return _bits(torch.empty(shape, device=dev(), dtype=dtype)).fill_(bits).view(dtype)


def assert_guard(buf, region, what):
    """Everything of `buf` outside buf[region] must still be the sentinel."""
    sent = _bits(sentinel((1,), buf.dtype))[0]
    bits = _bits(buf).clone()
    bits[region] = sent
    touched = int((bits != sent).sum())
    assert touched == 0, f"{what}: {touched} elements written outside the logical result"


def bit_equal(a, b):
    return torch.equal(_bits(a), _bits(b))


def both_directions(make_outputs, launch, check=None):
    """Two calls of the same entry point, back to back with no other library call in between: the library flips its
    traversal direction on every call, so one runs with each.  `make_outputs()` returns a tuple of fresh
    sentinel-filled buffers (an in-place residual is copied into each); both are made before the first call.  The
    first result goes to `check` (the reference comparison), then the two must agree bit for bit; when they do not,
    the second one is checked too, so the report locates the wrong tiles of whichever direction is wrong.  Returns
    the first result."""
    first, second = make_outputs(), make_outputs()
    launch(*first)
    launch(*second)
    torch.cuda.synchronize()
    same = [bit_equal(a, b) for a, b in zip(first, second)]
    if check is not None:
        check(first)
        if not all(same):
            check(second)
    for i, s in enumerate(same):
        assert s, f"output {i} depends on the traversal direction"
    return first


def assert_elementwise(got, ref64, bound64, tile=256, what="output"):
    """|got - ref| <= bound for every element of the 2-D logical result (a NaN anywhere fails).  On failure: how many
    elements, the worst one with its 256 x 256 tile, and how many distinct tiles fail -- a scheduling bug (whole
    tiles) reads differently from an arithmetic one (scattered elements)."""
    got64 = got.double()
    err = (got64 - ref64).abs()
    bad = ~(err <= bound64)
    n_bad = int(bad.sum())
    if n_bad == 0:
        return
    ratio = torch.where(bad, torch.nan_to_num(err / bound64, nan=float("inf"), posinf=float("inf")), 0.0)
    r, c = divmod(int(ratio.argmax()), got.shape[1])
    rows, cols = bad.nonzero(as_tuple=True)
    n_cb = (got.shape[1] + tile - 1) // tile
    tiles = torch.unique((rows // tile) * n_cb + cols // tile).numel()
    raise AssertionError(
        f"{what}: {n_bad} of {bad.numel()} elements outside the bound; worst ({r}, {c}) in tile (row block "
        f"{r // tile}, column block {c // tile}): got {got64[r, c].item()}, want {ref64[r, c].item()}, bound "
        f"{bound64[r, c].item():.3g}; {tiles} distinct {tile}x{tile} tiles fail")


def ulp(v, mant_bits, min_exp):
    """Spacing of the format (mant_bits explicit mantissa bits, smallest normal exponent min_exp) at |v|."""
    _, e = torch.frexp(v)
    return torch.exp2(((e - 1).clamp_min(min_exp) - mant_bits).to(v.dtype))


def ulp_bf16(v):
    return ulp(v, 7, -126)


def ulp_e4m3(v):
    return ulp(v, 3, -6)


def ref_products(A, B, chunk=8192):
    """(A . B^T, |A| . |B|^T) in fp64 on the GPU, in row chunks; A [M, K], B [N, K] hold the kernel's operands."""
    Bd = B.double()
    Ba = Bd.abs()
    acc = torch.empty((A.shape[0], B.shape[0]), device=dev(), dtype=torch.float64)
    absacc = torch.empty_like(acc)
    for m0 in range(0, A.shape[0], chunk):
        a = A[m0:m0 + chunk].double()
        acc[m0:m0 + chunk] = a @ Bd.t()
        absacc[m0:m0 + chunk] = a.abs() @ Ba.t()
    return acc, absacc


def gelu64(x):
    return 0.5 * x * (1.0 + torch.erf(x * (1.0 / math.sqrt(2.0))))


def stats_ref_and_bound(r, e):
    """Per-128-column (sum, M2 about the group mean) of the fp32 pre-rounding values the epilogue sees, whose fp64
    reference is r (rows, N) with per-element bound e, and the bound on each of them:
      sum: sum_i e_i from the values, plus the fp32 sums the kernel forms -- x - pivot (pivot = the group's first
        value), two chains of 64 adds, their sum, + 128 * pivot: at most 70 ulps of sum_i |x_i - pivot|, and one of
        the total;
      M2:  the values' error moves M2 by at most 2 sqrt(M2) ||e|| + ||e||^2 (centring is a projection); the kernel's
        Q = sum (x - pivot)^2 carries 70 ulps of Q and M2 = Q - S^2 / 128 the error of S through 2|S| dS / 128,
        plus one rounding of the result."""
    rows, n = r.shape
    r = r.view(rows, n // 128, 128)
    e = e.view(rows, n // 128, 128)
    d = (r - r[..., :1]).abs() + e + e[..., :1]
    s = r.sum(-1)
    m2 = ((r - r.mean(-1, keepdim=True)) ** 2).sum(-1)
    e_s = e.sum(-1) + 70 * EPS32 * d.sum(-1) + EPS32 * s.abs()
    en = e.norm(dim=-1)
    d_sh = d.sum(-1)
    e_sh = 70 * EPS32 * d_sh
    e_m2 = 2 * m2.sqrt() * en + en ** 2 + 70 * EPS32 * (d ** 2).sum(-1) + (2 * d_sh * e_sh + e_sh ** 2) / 128 + \
        EPS32 * m2
    return torch.stack([s, m2], -1), torch.stack([e_s, e_m2], -1)


def assert_stats(got, r, e, what="row statistics"):
    """got (rows, N/128, 2) fp32 against stats_ref_and_bound(r, e)."""
    ref, bound = stats_ref_and_bound(r, e)
    rows = got.shape[0]
    assert_elementwise(got.reshape(rows, -1), ref.reshape(rows, -1), bound.reshape(rows, -1), what=what)


def group_stats64(x):
    """(M, K) -> (M, K/128, 2) fp64 (sum, M2 about the group's own mean): the rowstats layout of vt_gemm_bf16_ln."""
    M, K = x.shape
    xc = x.double().view(M, K // 128, 128)
    return torch.stack([xc.sum(-1), ((xc - xc.mean(-1, keepdim=True)) ** 2).sum(-1)], dim=2)


# ------------------------------------------------------------------------------------------------ 2-CTA GEMM
class GemmCase:
    """One launch of vt_gemm_bf16_ln (bf16 operands) or vt_gemm_fp8 (e4m3 operands) with its operands, its
    sentinel-filled outputs and its fp64 reference.  Flags: gelu, res (residual), inplace (the residual aliases the
    output), stats (row statistics out), lnf ("colsum" | "zero": LayerNorm folded into the epilogue), out8 (e4m3
    output, FP8 only); lda > K pads A and Bt with NaN columns the kernel must never read."""

    def __init__(self, M, K, N, fp8=False, gelu=False, res=False, inplace=False, stats=False, lnf=None, out8=False,
                 lda=None):
        from vit import packing
        self.M, self.K, self.N = M, K, N
        self.fp8, self.gelu, self.res, self.inplace, self.stats, self.lnf, self.out8 = \
            fp8, gelu, res or inplace or stats, inplace, stats, lnf, out8
        self.lda = lda or K
        self.ldo = N + 64
        self.bias = (0.5 * torch.randn(N, device=dev())).contiguous()
        self.rowstats = self.colsum = None
        self.out_scale = 8.0
        if fp8:
            a = (16.0 * torch.randn(M, K, device=dev())).to(torch.float8_e4m3fn)
            w = (torch.randn(N, K, device=dev()) / math.sqrt(K))
            scale = w.abs().amax(dim=1) / 448.0
            b = (w / scale[:, None]).to(torch.float8_e4m3fn)
            self.colscale = (scale / 16.0).contiguous()
            self.A = self._pad(a.view(torch.uint8))
            self.B = self._pad(b.view(torch.uint8))
        else:
            a = 2.0 * torch.randn(M, K, device=dev()) + (0.7 if lnf else 0.0)
            w = (torch.randn(N, K, device=dev()) / math.sqrt(K)).bfloat16()
            if lnf:
                ln = torch.nn.LayerNorm(K).to(dev())
                with torch.no_grad():
                    ln.weight.copy_(1 + 0.2 * torch.randn(K, device=dev()))
                    ln.bias.copy_(0.2 * torch.randn(K, device=dev()))
                # the pack kernel's folded operands: W' (gamma in, zero-sum rows or not), b', colsum
                w, self.bias, self.colsum = packing.fold_layernorm(w.contiguous(), self.bias, ln,
                                                                   zero_sum=lnf == "zero")
                self.st64 = group_stats64(a.bfloat16())
                self.rowstats = self.st64.float().contiguous()
            self.A = self._pad(a.bfloat16())
            self.B = self._pad(w)
        self.residual = torch.randn(M, N, device=dev()).bfloat16() if self.res else None

    def _pad(self, t):
        """[rows, K] -> [rows, lda] with NaN in the padding columns."""
        if self.lda == self.K:
            return t.contiguous()
        out = sentinel((t.shape[0], self.lda), t.dtype)
        out[:, :self.K] = t
        return out

    def outputs(self):
        out = sentinel((self.M + 64, self.ldo), torch.uint8 if self.out8 else torch.bfloat16)
        if self.inplace:
            out[:self.M, :self.N] = self.residual
        if not self.stats:
            return (out,)
        return out, sentinel((self.M + 64, self.N // 128, 2), torch.float32)

    def launch(self, out, stats=None):
        L = _lib()
        res_ptr, ldr = L.ptr(self.residual), self.N
        if self.inplace:
            res_ptr, ldr = out.data_ptr(), self.ldo
        stream = L.stream_ptr(out)
        if self.fp8:
            L.call("vt_gemm_fp8", self.A.data_ptr(), self.lda, self.B.data_ptr(), self.lda, out.data_ptr(), self.ldo,
                   L.VT_E4M3 if self.out8 else L.VT_BF16, self.bias.data_ptr(), self.colscale.data_ptr(), res_ptr,
                   ldr, self.M, self.N, self.K, int(self.gelu), self.out_scale, stream)
        else:
            L.call("vt_gemm_bf16_ln", self.A.data_ptr(), self.lda, self.B.data_ptr(), self.lda, out.data_ptr(),
                   self.ldo, self.bias.data_ptr(), res_ptr, ldr, self.M, self.N, self.K, int(self.gelu),
                   L.ptr(self.rowstats), L.ptr(self.colsum), self.K if self.lnf else 0, LN_EPS, L.ptr(stats), stream)

    def run(self, checked=False):
        return both_directions(self.outputs, self.launch, self.check if checked else None)

    def operand(self, t):
        t = t[:, :self.K]
        return t.view(torch.float8_e4m3fn) if self.fp8 else t

    def check(self, outs):
        """Every element of the output (and of the row statistics) within the bound of the module docstring, and
        nothing written outside the logical result."""
        M, N, K = self.M, self.N, self.K
        acc, absacc = ref_products(self.operand(self.A), self.operand(self.B))
        bias = self.bias.double()[None]
        if self.fp8:
            cs = self.colscale.double()[None]
            pre = acc * cs + bias
            e = EPS32 * K * absacc * cs + EPI_OPS * EPS32 * ((acc * cs).abs() + bias.abs())
        elif self.lnf:
            mean = self.st64[..., 0].sum(-1, keepdim=True) / K
            var = (self.st64[..., 1].sum(-1) + 128 * ((self.st64[..., 0] / 128 - mean) ** 2).sum(-1)) / K
            rstd = (var[:, None] + LN_EPS).rsqrt()
            terms = [rstd * acc, bias]
            if self.lnf == "colsum":
                terms.append(-rstd * mean * self.colsum.double()[None])
            pre = sum(terms)
            mag = sum(t.abs() for t in terms)
            e = EPS32 * K * rstd * absacc + RSTD_REL * (mag - bias.abs()) + EPI_OPS * EPS32 * mag
        else:
            pre = acc + bias
            e = EPS32 * K * absacc + EPI_OPS * EPS32 * (acc.abs() + bias.abs())
        del acc, absacc
        if self.res:
            r = self.residual.double()
            e = e + EPI_OPS * EPS32 * (pre.abs() + r.abs())
            pre = pre + r
        if self.stats:
            assert_stats(outs[1][:M], pre, e)
            assert_guard(outs[1], (slice(0, M),), "row statistics")
        want = pre
        if self.gelu:
            want = gelu64(pre)
            e = GELU_SLOPE * e + GELU_ABS
        out = outs[0]
        if self.out8:
            s = self.out_scale
            want = (want * s).clamp(-448.0, 448.0)
            got = out[:M, :N].view(torch.float8_e4m3fn)
            assert_elementwise(got, want, ulp_e4m3(want) + s * e, what="e4m3 output")
        else:
            assert_elementwise(out[:M, :N], want, ulp_bf16(want) + e)
        assert_guard(out, (slice(0, M), slice(0, N)), "output")

    def check_grid_independent(self, outs, groups):
        """Under each cap of the grid the result is bit-identical to the full-grid one: which group computes a tile
        must not change a bit of it."""
        for g in groups:
            with sm_partition(g, 0):
                again = self.run()
            for a, b in zip(outs, again):
                assert bit_equal(a, b), f"{g} GEMM groups give a different result from the full grid"


C2_ROWS = 256 * 197
PRODUCTION = {
    # ViT-B/16 at C2 (256 images): the bf16 path with the LayerNorm fold (zero-sum weights, as packed)
    "qkv": dict(M=C2_ROWS, K=768, N=2304, lnf="zero"),
    "out_proj": dict(M=C2_ROWS, K=768, N=768, res=True, stats=True),     # 5 stages; 197 x 3 tiles: ghost tile
    "fc1": dict(M=C2_ROWS, K=768, N=3072, lnf="zero", gelu=True),
    "fc2": dict(M=C2_ROWS, K=3072, N=768, res=True, stats=True),         # 6 stages with a residual
    # the VT_FP8 path (its out-projection stays bf16)
    "fp8_qkv": dict(M=C2_ROWS, K=768, N=2304, fp8=True),
    "fp8_fc1": dict(M=C2_ROWS, K=768, N=3072, fp8=True, gelu=True, out8=True),
    "fp8_fc2": dict(M=C2_ROWS, K=3072, N=768, fp8=True, res=True),
    # ViT-H: ln_parts = 10, the most row-statistics registers of the fast path
    "vith_qkv": dict(M=64 * 257, K=1280, N=1280, lnf="colsum"),
}


@pytest.mark.parametrize("name", list(PRODUCTION))
def test_gemm_production_size_many_tiles_per_group(name):
    """Full grid at production size: ~8-32 supertiles per group, both launch forms (clusters of four and pairs)."""
    case = GemmCase(**PRODUCTION[name])
    outs = case.run(checked=True)
    case.check_grid_independent(outs, (7,))


SMALL_M = 197 * 24          # 19 row blocks (odd): the last row block pairs column blocks, a ghost where N / 256 is odd
RESTRICTED = {
    "plain": dict(K=768, N=2304),
    "gelu": dict(K=768, N=3072, gelu=True),
    "res": dict(K=768, N=768, res=True),
    "res_in_place": dict(K=768, N=768, inplace=True),
    "res_stats": dict(K=768, N=768, stats=True),
    "res_stats_deep": dict(K=3072, N=768, stats=True),
    "lnf_colsum": dict(K=768, N=2304, lnf="colsum"),
    "lnf_zero_sum": dict(K=768, N=2304, lnf="zero"),
    "lnf_zero_sum_gelu": dict(K=768, N=3072, lnf="zero", gelu=True),
    "fp8_plain": dict(K=768, N=2304, fp8=True),
    "fp8_gelu": dict(K=768, N=3072, fp8=True, gelu=True),
    "fp8_res": dict(K=3072, N=768, fp8=True, res=True),
    "fp8_e4m3_out": dict(K=768, N=3072, fp8=True, gelu=True, out8=True),
    "ragged_k_nan_padding": dict(K=744, N=768, lda=768),
    "ragged_k_nan_padding_res_stats": dict(K=744, N=768, lda=768, stats=True),
}


@pytest.mark.parametrize("name", list(RESTRICTED))
def test_gemm_restricted_grid_walks_every_tile(name):
    """M = 4728 under 1, 2, 3 and 7 groups: with one group, four CTAs walk all 29 / 86 / 114 supertiles.  Every
    epilogue of the bf16 kernel, both stage configurations, the FP8 forms, and K % 64 != 0."""
    case = GemmCase(M=SMALL_M, **RESTRICTED[name])
    outs = case.run(checked=True)
    case.check_grid_independent(outs, (1, 2, 3, 7))


# ------------------------------------------------------------------------------------------------ token-mode patch embedding
@pytest.mark.parametrize("B,groups", [(256, (7,)), (257, (7,)), (37, (1,))])
def test_patch_embed_token_mode_many_tiles(B, groups):
    """vt_patch_embed_gemm at 224^2, P = 16, D = 768 with row statistics: C2 (224 row blocks, ~9 supertiles per
    group), 257 images (225 row blocks: a ghost tail) and 37 images on one group.  Reference: conv2d as a GEMM on the
    same bf16 patches in fp64 + bias + the bf16 position table; every 4-image slice equals a 4-image call bit for bit."""
    L = _lib()
    S, P, C, D = 224, 16, 3, 768
    n = (S // P) ** 2
    T, K = n + 1, C * P * P
    x = torch.randn(B, C, S, S, device=dev()).bfloat16()
    w = (0.03 * torch.randn(D, K, device=dev())).bfloat16()
    bias = (0.1 * torch.randn(D, device=dev())).contiguous()
    posb = torch.randn(T, D, device=dev()).bfloat16()

    def outputs(nb):
        return lambda: (sentinel((nb + 1, T, D), torch.bfloat16), sentinel((nb * T + 64, D // 128, 2), torch.float32))

    def launch(b0, nb):
        def go(out, stats):
            work = torch.empty((nb, (T + 31) // 32 * 32, K), device=dev(), dtype=torch.bfloat16)
            L.call("vt_patch_embed_gemm", x[b0:].data_ptr(), L.VT_BF16, w.data_ptr(), K, bias.data_ptr(),
                   posb.data_ptr(), out.data_ptr(), stats.data_ptr(), work.data_ptr(), nb, C, S, P, D,
                   L.stream_ptr(x))
        return go

    patches = x.unfold(2, P, P).unfold(3, P, P).permute(0, 2, 3, 1, 4, 5).reshape(B, n, K)
    A = torch.cat([torch.zeros(B, 1, K, device=dev(), dtype=torch.bfloat16), patches], 1).reshape(B * T, K)
    acc, absacc = ref_products(A, w)
    pos = posb.double().repeat(B, 1)
    pre = acc + bias.double()[None] + pos
    e = EPS32 * K * absacc + EPI_OPS * EPS32 * (acc.abs() + bias.double().abs()[None] + pos.abs())
    del acc, absacc

    def check(outs):
        out, stats = outs
        assert_elementwise(out[:B].reshape(B * T, D), pre, ulp_bf16(pre) + e)
        assert_guard(out, (slice(0, B),), "output")
        assert_stats(stats[:B * T], pre, e)
        assert_guard(stats, (slice(0, B * T),), "row statistics")

    out, stats = both_directions(outputs(B), launch(0, B), check)
    for g in groups:
        with sm_partition(g, 0):
            again = both_directions(outputs(B), launch(0, B))
        assert bit_equal(again[0], out) and bit_equal(again[1], stats), f"{g} groups differ from the full grid"
    for b0 in range(0, B, 4):
        nb = min(4, B - b0)
        sub_out, sub_stats = outputs(nb)()
        launch(b0, nb)(sub_out, sub_stats)
        assert bit_equal(sub_out[:nb], out[b0:b0 + nb]), f"images {b0}..{b0 + nb - 1}: slice differs from a call"
        assert bit_equal(sub_stats[:nb * T], stats[b0 * T:(b0 + nb) * T]), f"images {b0}..: statistics differ"


# ------------------------------------------------------------------------------------------------ attention
def _attn_launch(qkv, B, H, N, dh, pad):
    """vt_flash_attn on the fused [B, N, 3 * H * dh] buffer into a [B + 1, N, H * dh + pad] output (row stride with
    guard columns, one guard image)."""
    L = _lib()
    D = H * dh
    es = qkv.element_size()

    def go(out):
        base = qkv.data_ptr()
        L.call("vt_flash_attn", base, base + D * es, base + 2 * D * es, out.data_ptr(), B, H, N, dh, 3 * D, N * 3 * D,
               D + pad, N * (D + pad), 1.0 / math.sqrt(dh), L.stream_ptr(qkv))
    return go


def _attn_check(qkv, out, B, H, N, dh, chunk=16):
    """Each (image, head) on its own against an fp64 softmax reference: relative Frobenius error <= 1e-2 and every
    element within 2e-2, so one wrong item cannot hide in a global norm."""
    D = H * dh
    worst_rel, worst_abs = (0.0, None), (0.0, None)
    for b0 in range(0, B, chunk):
        q, k, v = qkv[b0:b0 + chunk].double().view(-1, N, 3, H, dh).permute(2, 0, 3, 1, 4)
        o = torch.softmax(q @ k.transpose(-1, -2) / math.sqrt(dh), -1) @ v            # (b, H, N, dh)
        got = out[b0:b0 + chunk, :, :D].double().reshape(-1, N, H, dh).transpose(1, 2)
        assert not torch.isnan(got).any(), f"images {b0}..: NaN (unwritten) output"
        rel = (got - o).flatten(2).norm(dim=-1) / o.flatten(2).norm(dim=-1).clamp_min(1e-30)
        mx = (got - o).abs().flatten(2).amax(-1)
        i = int(rel.argmax())
        if rel.flatten()[i] > worst_rel[0]:
            worst_rel = (rel.flatten()[i].item(), (b0 + i // H, i % H))
        i = int(mx.argmax())
        if mx.flatten()[i] > worst_abs[0]:
            worst_abs = (mx.flatten()[i].item(), (b0 + i // H, i % H))
    assert worst_rel[0] <= 1e-2, f"(image, head) {worst_rel[1]}: relative error {worst_rel[0]:.3g}"
    assert worst_abs[0] <= 2e-2, f"(image, head) {worst_abs[1]}: element error {worst_abs[0]:.3g}"


def _attn_run(qkv, B, H, N, dh, checked=False, pad=64):
    D = H * dh

    def check(outs):
        _attn_check(qkv, outs[0], B, H, N, dh)
        assert_guard(outs[0], (slice(0, B), slice(None), slice(0, D)), "attention output")

    out, = both_directions(lambda: (sentinel((B + 1, N, D + pad), torch.bfloat16),),
                           _attn_launch(qkv, B, H, N, dh, pad), check if checked else None)
    return out


def _attn_sub_batch(qkv, full, H, N, dh, lo, nb, pad=64):
    sub = sentinel((nb + 1, N, H * dh + pad), torch.bfloat16)
    _attn_launch(qkv[lo:lo + nb], nb, H, N, dh, pad)(sub)
    assert bit_equal(sub[:nb], full[lo:lo + nb]), f"images {lo}..{lo + nb - 1}: sub-batch call differs"


@pytest.mark.parametrize("B,H,N,dh,caps", [
    (256, 12, 197, 64, ()),              # attn5 at C2: 3072 pairs, ~21 per CTA
    (16, 12, 197, 64, (1, 3, 7)),        # two query tiles per pair, 192 pairs on 1 / 3 / 7 CTAs
    (16, 12, 100, 64, (1, 3, 7)),        # one query tile per pair
    (32, 12, 577, 64, ()),               # attn5mb (no CTA cap): several KV blocks, online softmax
    (64, 16, 257, 80, ()),               # attn5mb, ViT-H heads
])
def test_attention_many_items_per_cta(B, H, N, dh, caps):
    qkv = torch.randn(B, N, 3 * H * dh, device=dev()).bfloat16()
    out = _attn_run(qkv, B, H, N, dh, checked=True)
    for a in caps:
        with sm_partition(0, a):
            again = _attn_run(qkv, B, H, N, dh)
        assert bit_equal(again, out), f"attention on {a} CTAs differs from the full grid"
    for lo in sorted({0, B // 2 - 1, B - 3}):
        _attn_sub_batch(qkv, out, H, N, dh, lo, 3)
