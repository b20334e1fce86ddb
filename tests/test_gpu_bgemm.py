"""The batched tensor-core GEMM (csrc/bgemm_sm100.cu, `vt_bgemm`), its operand packing (csrc/pack_split.cu,
`vt_pack_bf16`) and the fp32-output GEMM (csrc/gemm_sm100.cu, `vt_gemm_bf16` with fp32 output) past their first tile,
element by element against fp64 references, plus the host paths built on them (fp32 `matmul`, `matmul3`, the composed
attention, the pooler and classifier heads).

Why these cases.  Both kernels are persistent: grid = min(tiles, SMs) and CTA b takes tiles b, b + grid, ...  The TMEM
accumulator's second buffer, the second phase of its empty barrier, an operand ring whose phase carries from one tile
into the next and the epilogue's decode of any tile but blockIdx.x only run once a CTA has a second tile.  Every
multi-tile case asserts tiles >= 2 * SMs (read from the device), so every CTA runs at least two.  Tiles are 128 x 128
(K-major B) or 128 x 64 (MN-major B) for vt_bgemm, 128 x 256 (N > 128) or 128 x 128 for the fp32-output GEMM.

Buffers.  Operands live inside NaN-filled storage: rows longer than K (NaN columns past K) and batch blocks longer than
the matrix (NaN rows between batches), so a finite, correct result shows the kernel's TMA reads stop at the matrix and
zero-fill the rest.  Outputs live inside NaN-filled buffers with row strides > N and batch strides > M * ldc; nothing
outside the logical result may change, in particular rows >= M of a batch must not land in the next one.  Some cases
offset C (and the residual) by one element, which takes the epilogue's scalar store path.  Schedule independence:
batches (first, middle, last) or a 128-aligned block of rows are recomputed by calls of their own, where every tile is
a CTA's first, and must equal their slice of the many-tile call bit for bit.

Per-element bound, |got - ref| <= bound, ref in fp64 on the kernel's own operands (bf16 operands) or on the fp32
inputs (split operands):
  * one rounding of the output: 1 ulp of the reference value in the output format (bf16 or fp32);
  * the fp32 accumulation: the tensor core adds into its fp32 accumulator with truncation (DESIGN.md section 4),
    at most one ulp (2^-23 relative) of the running sum per add, K' adds:  K' * 2^-23 * (|A| . |B|), K' the packed K
    (pieces * cpad for split operands, whose piece products add up to at most PIECE_MASS = 1 + 2^-7 times |a||b|);
  * the split of fp32 operands (vt_pack_bf16): hi = bf16(x) is within 2^-9 |x|, lo = bf16(x - hi) leaves
    |x - hi - lo| <= 2^-18 |x|.  Three pieces keep hi.hi + hi.lo + lo.hi and drop lo.lo (<= 2^-18 |a||b|) and the
    residue of lo on either side (<= 2^-18 |a||b| each): SPLIT3 = 3 * 2^-18 (x 1.03 for the second-order terms).  Six
    pieces split once more (x3 = bf16(x - hi - lo), residue <= 2^-27 |x|) and keep every product of weight >= 2^-18;
    they drop a2.a3, a3.a2, a3.a3 and the two residues: SPLIT6 = 5 * 2^-27;
  * the fp32 epilogue (scale, bias, residual): EPI_OPS * 2^-23 times the magnitudes of the terms it combines;
  * GELU (erff): the error of its input times max |gelu'| = 1.13, plus its own evaluation: 0.5 x (1 + erff(x/sqrt 2))
    with erff within 2 ulps (2^-23 absolute), the argument's rounding (erf' <= 1.13: 0.4 |x| 2^-23), the add and the
    product's rounding: 2^-23 (|x| + 0.2 x^2 + |gelu|), doubled for the evaluation order;
  * tanh (tanhf): input error times 1 plus 2 ulps of the result, 2^-22 |tanh|.
The composed attention carries the score error through the softmax: with per-score bounds Es (the GEMM bound above
plus the scores' output rounding), the exact softmax moves by |dp_j| <= p_j |ds_j| + p_j sum_l p_l |ds_l|, so
  sum_j |dp_j| |v_j| <= (P o Es) |V| + rowsum(P o Es) (P |V|),
the softmax's own fp32 evaluation (expf within 2 ulps, the max subtraction, an N-term sum, one division and product)
adds SOFTMAX_REL = 2^-23 (N + 8 + 2 max |s - m|) of each p, bf16 probabilities one ulp of each p (ulp(P) |V|), and the
P.V GEMM its own K' and split terms on P |V| (x 1.01 for the perturbed P).
"""
import math

import pytest
import torch

pytestmark = pytest.mark.gpu

EPS32 = 2.0 ** -23
EPI_OPS = 4
PIECE_MASS = 1.0 + 2.0 ** -7
SPLIT = {1: 0.0, 3: 3.0 * 1.03 * 2.0 ** -18, 6: 5.0 * 2.0 ** -27}
GELU_SLOPE = 1.13

ACT_NONE, ACT_GELU, ACT_TANH = 0, 1, 2

BF16_SENTINEL = 0x7FC0        # bf16 quiet NaN
F32_SENTINEL = 0x7FC00000     # fp32 quiet NaN


@pytest.fixture(autouse=True)
def _seed():
    torch.manual_seed(0)


def dev():
    return torch.device("cuda:0")


def _lib():
    from vit.kernels import _lib
    return _lib


def sms():
    return torch.cuda.get_device_properties(0).multi_processor_count


def assert_many_tiles(tiles):
    assert tiles >= 2 * sms(), f"{tiles} tiles do not give every one of the {sms()} SMs a second tile"


def bgemm_tiles(M, N, batches, b_mn):
    return -(-M // 128) * -(-N // (64 if b_mn else 128)) * batches


def ceil8(n):
    return (n + 7) // 8 * 8


# ------------------------------------------------------------------------------------------------ buffers and checks
def _bits(t):
    return t.view({torch.bfloat16: torch.int16, torch.float32: torch.int32}[t.dtype])


def sentinel(shape, dtype):
    bits = {torch.bfloat16: BF16_SENTINEL, torch.float32: F32_SENTINEL}[dtype]
    return _bits(torch.empty(shape, device=dev(), dtype=dtype)).fill_(bits).view(dtype)


def bit_equal(a, b):
    return torch.equal(_bits(a), _bits(b))


def assert_guard(buf, region, what):
    """Everything of `buf` outside `region(buf)` (a view of it) must still be the sentinel."""
    sent = _bits(sentinel((1,), buf.dtype))[0]
    bits = _bits(buf).clone()
    region(bits).fill_(sent)
    touched = int((bits != sent).sum())
    assert touched == 0, f"{what}: {touched} elements written outside the logical result"


def assert_elementwise(got, ref64, bound64, tile=(128, 128), what="output"):
    """|got - ref| <= bound for every element of the (batch, rows, cols) result (a NaN anywhere fails).  On failure:
    how many elements, the worst one with its kernel tile, and how many distinct tiles fail -- a scheduling bug
    (whole tiles) reads differently from an arithmetic one (scattered elements)."""
    got64 = got.double()
    if got64.dim() == 2:
        got64, ref64, bound64 = got64[None], ref64[None], bound64[None]
    ref64, bound64 = ref64.expand_as(got64), bound64.expand_as(got64)
    err = (got64 - ref64).abs()
    bad = ~(err <= bound64)
    n_bad = int(bad.sum())
    if n_bad == 0:
        return
    ratio = torch.where(bad, torch.nan_to_num(err / bound64, nan=float("inf"), posinf=float("inf")), 0.0)
    Z, R, C = got64.shape
    i = int(ratio.argmax())
    z, r, c = i // (R * C), (i // C) % R, i % C
    zs, rows, cols = bad.nonzero(as_tuple=True)
    n_cb = -(-C // tile[1])
    n_rb = -(-R // tile[0])
    tiles = torch.unique((zs * n_rb + rows // tile[0]) * n_cb + cols // tile[1]).numel()
    raise AssertionError(
        f"{what}: {n_bad} of {bad.numel()} elements outside the bound; worst (batch {z}, row {r}, column {c}) in "
        f"tile (row block {r // tile[0]}, column block {c // tile[1]}): got {got64[z, r, c].item()}, want "
        f"{ref64[z, r, c].item()}, bound {bound64[z, r, c].item():.3g}; {tiles} distinct {tile[0]}x{tile[1]} tiles "
        f"fail")


def ulp(v, mant_bits, min_exp):
    """Spacing of the format (mant_bits explicit mantissa bits, smallest normal exponent min_exp) at |v|."""
    _, e = torch.frexp(v)
    return torch.exp2(((e - 1).clamp_min(min_exp) - mant_bits).to(v.dtype))


def ulp_out(v, dtype):
    return ulp(v, 7, -126) if dtype == torch.bfloat16 else ulp(v, 23, -126)


def gelu64(x):
    return 0.5 * x * (1.0 + torch.erf(x * (1.0 / math.sqrt(2.0))))


def act_ref_and_bound(act, pre, e):
    """act(pre) in fp64 and the bound of the fp32 epilogue's act(pre + err), |err| <= e."""
    if act == ACT_GELU:
        g = gelu64(pre)
        return g, GELU_SLOPE * e + 2 * EPS32 * (pre.abs() + 0.2 * pre * pre + g.abs())
    if act == ACT_TANH:
        t = torch.tanh(pre)
        return t, e + 2 * EPS32 * t.abs()
    return pre, e


def products(A, B):
    """(A . B^T, |A| . |B|^T) in fp64, batched with broadcasting; A [..., M, K], B [..., N, K]."""
    A, B = A.double(), B.double()
    return A @ B.transpose(-1, -2), A.abs() @ B.abs().transpose(-1, -2)


# ------------------------------------------------------------------------------------------------ vt_bgemm direct
class BgemmCase:
    """One vt_bgemm launch on bf16 operands inside NaN-padded storage.  a_bcast / b_bcast: "inner" or "outer" gives
    the operand a batch stride of 0 on that level, "both" shares one matrix with all batches; res: None, "sep" or
    "inplace" (residual == C); ctx: C in the attention-context layout (Bo, M, Bi * N); scalar: C and the residual
    start one element past a 16-byte boundary, so the epilogue stores element by element."""

    GAP = 3           # NaN rows between operand batches
    CGAP = 2          # unwritten rows between output batches

    def __init__(self, M, N, K, Bo=1, Bi=1, b_mn=False, out=torch.bfloat16, act=ACT_NONE, bias=True, scale=1.0,
                 res=None, a_bcast=None, b_bcast=None, ctx=False, scalar=False):
        self.M, self.N, self.K, self.Bo, self.Bi = M, N, K, Bo, Bi
        self.b_mn, self.out, self.act, self.scale, self.res = b_mn, out, act, scale, res
        self.ctx, self.scalar = ctx, scalar
        self.tiles = bgemm_tiles(M, N, Bo * Bi, b_mn)
        self.A, self.sA = self._operand(M, K, a_bcast, 1.0)
        if b_mn:
            self.B, self.sB = self._operand(K, N, b_bcast, 1.0 / math.sqrt(K))
        else:
            self.B, self.sB = self._operand(N, K, b_bcast, 1.0 / math.sqrt(K))
        self.bias = (0.5 * torch.randn(N, device=dev())).contiguous() if bias else None
        if ctx:
            self.ldc = ceil8(Bi * N) + 8
            self.sC = ((M + self.CGAP) * self.ldc, N, self.ldc)
        else:
            self.ldc = ceil8(N) + 8
            self.sC = (Bi * (M + self.CGAP) * self.ldc, (M + self.CGAP) * self.ldc, self.ldc)
        self.c_off = 1 if scalar else 0
        self.c_numel = self.c_off + (Bo + 1) * self.sC[0] + 64      # one guard image past the last batch
        self.residual = torch.randn(Bo, Bi, M, N, device=dev()).to(out) if res else None

    def _operand(self, rows, cols, bcast, gain):
        """[bo, bi, rows + GAP, ld] bf16 with the matrix in [..., :rows, :cols] and NaN elsewhere; the element
        strides the kernel gets, 0 on a broadcast level."""
        bo = 1 if bcast in ("outer", "both") else self.Bo
        bi = 1 if bcast in ("inner", "both") else self.Bi
        ld = ceil8(cols) + 8
        buf = sentinel((bo, bi, rows + self.GAP, ld), torch.bfloat16)
        buf[:, :, :rows, :cols] = (gain * torch.randn(bo, bi, rows, cols, device=dev())).bfloat16()
        s = (0 if bcast in ("outer", "both") else buf.stride(0), 0 if bcast in ("inner", "both") else buf.stride(1),
             ld)
        return buf, s

    def view(self, flat):
        """The logical (Bo, Bi, M, N) result inside a flat C buffer."""
        return flat.as_strided((self.Bo, self.Bi, self.M, self.N), (self.sC[0], self.sC[1], self.ldc, 1),
                               flat.storage_offset() + self.c_off)

    def output(self):
        flat = sentinel((self.c_numel,), self.out)
        if self.res == "inplace":
            self.view(flat).copy_(self.residual)
        return flat

    def launch(self, flat, zo=0, zi=0, bo=None, bi=None, m0=0, rows=None):
        """Batches [zo, zo + bo) x [zi, zi + bi) and rows [m0, m0 + rows) as one call (default: everything)."""
        L = _lib()
        es = flat.element_size()
        bo, bi, rows = bo or self.Bo, bi or self.Bi, rows or self.M
        a = self.A.data_ptr() + 2 * (zo * self.sA[0] + zi * self.sA[1] + m0 * self.sA[2])
        b = self.B.data_ptr() + 2 * (zo * self.sB[0] + zi * self.sB[1])
        c_el = self.c_off + zo * self.sC[0] + zi * self.sC[1] + m0 * self.ldc
        c = flat.data_ptr() + es * c_el
        r = None
        if self.res == "inplace":
            r = c
        elif self.res == "sep":
            rflat = sentinel((self.c_numel,), self.out)
            self.view(rflat).copy_(self.residual)
            self._rflat = rflat                       # alive until the kernel is done (synchronised by the caller)
            r = rflat.data_ptr() + es * c_el
        L.call("vt_bgemm", a, b, c, L.ptr(self.bias), r, rows, self.N, self.K, bo, bi, L.i64x3(*self.sA),
               L.i64x3(*self.sB), L.i64x3(*self.sC), int(self.b_mn), self.scale, self.act,
               L.VT_F32 if self.out == torch.float32 else L.VT_BF16, L.stream_ptr(flat))

    def run(self):
        flat = self.output()
        self.launch(flat)
        torch.cuda.synchronize()
        return flat

    def logical_operands(self):
        A = self.A[:, :, :self.M, :self.K]
        B = self.B[:, :, :self.K, :self.N].transpose(-1, -2) if self.b_mn else self.B[:, :, :self.N, :self.K]
        return A, B

    def check(self, flat):
        A, B = self.logical_operands()
        acc, absacc = products(A, B)
        s = self.scale
        pre = s * acc
        e = abs(s) * self.K * EPS32 * absacc + EPI_OPS * EPS32 * pre.abs()
        if self.bias is not None:
            bias = self.bias.double()
            e = e + EPI_OPS * EPS32 * bias.abs()
            pre = pre + bias
        want, e = act_ref_and_bound(self.act, pre, e)
        if self.res:
            r = self.residual.double()
            e = e + EPI_OPS * EPS32 * (want.abs() + r.abs())
            want = want + r
        want = want.expand(self.Bo, self.Bi, self.M, self.N)
        bound = ulp_out(want, self.out) + e
        got = self.view(flat)
        Z = self.Bo * self.Bi
        assert_elementwise(got.reshape(Z, self.M, self.N), want.reshape(Z, self.M, self.N),
                           bound.expand_as(want).reshape(Z, self.M, self.N), tile=(128, 64 if self.b_mn else 128))
        assert_guard(flat, self.view, "output")

    def check_batches_alone(self, flat, batches):
        """Each listed (zo, zi) batch as a one-batch call equals its slice of the full call bit for bit."""
        for zo, zi in batches:
            sub = self.output()
            self.launch(sub, zo, zi, 1, 1)
            torch.cuda.synchronize()
            assert bit_equal(self.view(sub)[zo, zi], self.view(flat)[zo, zi]), \
                f"batch ({zo}, {zi}) computed alone differs from its slice of the full call"

    def check_rows_alone(self, flat, m0, rows):
        """Rows [m0, m0 + rows) of batch (0, 0), a 128-aligned block with its own A pointer, as one call."""
        assert m0 % 128 == 0 and rows % 128 == 0 and bgemm_tiles(rows, self.N, 1, self.b_mn) <= sms()
        sub = self.output()
        self.launch(sub, 0, 0, 1, 1, m0, rows)
        torch.cuda.synchronize()
        assert bit_equal(self.view(sub)[0, 0, m0:m0 + rows], self.view(flat)[0, 0, m0:m0 + rows]), \
            f"rows {m0}..{m0 + rows - 1} computed alone differ from their slice of the full call"


MANY_TILES = {
    # ragged M / N / K: 64 batches of 197 x 330 x 520 (384 K-major / 768 MN-major tiles), GELU, residual alongside
    "ragged": dict(M=197, N=330, K=520, Bo=64, scale=0.25, act=ACT_GELU, res="sep"),
    # ragged, fp32 output, tanh, residual in place, no bias
    "ragged_f32_tanh_in_place": dict(M=197, N=330, K=520, Bo=64, out=torch.float32, scale=0.5, act=ACT_TANH,
                                     bias=False, res="inplace"),
    # 96 batches of 197 x 200 x 136: N % 32 != 0 tail chunks, scalar stores (C and residual one element off)
    "tails_scalar_store": dict(M=197, N=200, K=136, Bo=96, scale=0.125, res="inplace", scalar=True),
    # weight shared by all batches (batch strides 0) with a large M: the fp32 model's fc1 (bf16 operands here)
    "shared_weight": dict(M=1576, N=3072, K=768, Bo=2, b_bcast="both", out=torch.float32, act=ACT_GELU),
    # (outer, inner) batches into the attention-context layout (Bo, M, Bi * N): P . V of 32 images x 12 heads
    "two_level_context": dict(M=197, N=64, K=197, Bo=32, Bi=12, ctx=True, bias=False, scale=1.0),
    "two_level_context_f32_res": dict(M=197, N=64, K=197, Bo=32, Bi=12, ctx=True, out=torch.float32, res="sep",
                                      scale=-0.75),
    # 4096 batches of 8 x 8 x 8: one k-block per tile, the ring and the TMEM buffer change on every tile
    "one_k_block": dict(M=8, N=8, K=8, Bo=64, Bi=64, res="inplace", scalar=True, out=torch.float32, scale=2.0),
    # a long K' (the fp32 fc2 split: 3 x 3072) with 2+ tiles per CTA, fp32 output, residual alongside
    "long_k": dict(M=3152, N=1536, K=9216, out=torch.float32, res="sep", b_bcast="both"),
}


@pytest.mark.parametrize("b_mn", [False, True], ids=["kmajor_bn128", "mnmajor_bn64"])
@pytest.mark.parametrize("name", list(MANY_TILES))
def test_bgemm_many_tiles_per_cta(name, b_mn):
    """vt_bgemm with K-major (BN = 128, 4 stages) and MN-major (BN = 64, 6 stages) B at >= 2 tiles per CTA: every
    element against fp64, guards, and the first / a middle / the last batch (or a 128-row block of a large M) as a
    call of its own, bit-equal to its slice."""
    case = BgemmCase(b_mn=b_mn, **MANY_TILES[name])
    assert_many_tiles(case.tiles)
    flat = case.run()
    case.check(flat)
    Z = case.Bo * case.Bi
    if Z > 1:
        case.check_batches_alone(flat, [divmod(z, case.Bi) for z in sorted({0, Z // 2 + 1, Z - 1}) if z < Z])
    if case.M >= 1024:
        case.check_rows_alone(flat, 512, 512 if case.N <= 1536 else 256)


@pytest.mark.parametrize("b_mn", [False, True], ids=["kmajor", "mnmajor"])
@pytest.mark.parametrize("operand,level", [("a", "inner"), ("a", "outer"), ("b", "inner"), ("b", "outer")])
def test_bgemm_one_level_broadcast(operand, level, b_mn):
    """A batch stride of 0 on one level broadcasts the operand along that level only (torch broadcasting of a size-1
    batch dimension); the other level keeps its own matrices."""
    kw = {f"{operand}_bcast": level}
    case = BgemmCase(M=130, N=72, K=96, Bo=3, Bi=5, b_mn=b_mn, scale=0.5, res="sep", **kw)
    flat = case.run()
    case.check(flat)
    case.check_batches_alone(flat, [(2, 4), (1, 3)])


# ------------------------------------------------------------------------------------------------ vt_pack_bf16
PACK_ROWS, PACK_COLS, PACK_BO, PACK_BI = 197, 1100, 2, 3     # 6 x 197 x 1104 = 1,304,928 > 148 * 32 * 256


def pack_restated(x, pieces, pattern):
    """hi = bf16(x), lo = bf16(x - hi), lo2 = bf16((x - hi) - lo), differences in fp32, torch's RNE conversion."""
    x = x.float()
    hi = x.bfloat16()
    r1 = x - hi.float()
    lo = r1.bfloat16()
    lo2 = (r1 - lo.float()).bfloat16()
    if pieces == 1:
        return [hi]
    if pieces == 3:
        return [hi, hi, lo] if pattern == 0 else [hi, lo, hi]
    return [hi, hi, lo, hi, lo, lo2] if pattern == 0 else [hi, lo, hi, lo2, lo, hi]


@pytest.mark.parametrize("transposed", [False, True], ids=["rows", "transposed"])
@pytest.mark.parametrize("src_dtype", [torch.float32, torch.bfloat16], ids=["f32", "bf16"])
@pytest.mark.parametrize("pieces", [1, 3, 6])
def test_pack_bf16_bit_exact_over_several_grid_passes(pieces, src_dtype, transposed):
    """Every packed element bit for bit against the torch restatement, over more elements than one grid-stride pass
    covers; zero columns C..cpad-1 in every piece; a gap after each destination row must keep its sentinel."""
    L = _lib()
    R, C, Bo, Bi = PACK_ROWS, PACK_COLS, PACK_BO, PACK_BI
    cpad = ceil8(C)
    assert Bo * Bi * R * cpad > 148 * 32 * 256
    mag = torch.logspace(-6, 6, C, device=dev())
    x = (torch.randn(Bo, Bi, R, C, device=dev()) * mag).to(src_dtype)
    if transposed:                     # the source is stored [.., C, R] and read through swapped strides
        store = x.transpose(2, 3).contiguous()
        s_src = (store.stride(0), store.stride(1), 1, R)
    else:
        store = x
        s_src = (x.stride(0), x.stride(1), x.stride(2), 1)
    ldd = pieces * cpad + 8
    for pattern in ((0,) if pieces == 1 else (0, 1)):
        dst = sentinel((Bo, Bi, R + 1, ldd), torch.bfloat16)
        s_dst = (dst.stride(0), dst.stride(1), ldd)
        L.call("vt_pack_bf16", store.data_ptr(), L.dtype_code(store), dst.data_ptr(), R, C, Bo, Bi, L.i64x4(*s_src),
               L.i64x3(*s_dst), cpad, pieces, pattern, L.stream_ptr(store))
        torch.cuda.synchronize()
        want = torch.zeros(Bo, Bi, R, pieces, cpad, device=dev(), dtype=torch.bfloat16)
        for i, piece in enumerate(pack_restated(x, pieces, pattern)):
            want[..., i, :C] = piece
        got = dst[:, :, :R, :pieces * cpad].reshape(Bo, Bi, R, pieces, cpad)
        diff = _bits(got) != _bits(want)
        if diff.any():
            idx = diff.nonzero()[0].tolist()
            raise AssertionError(f"pattern {pattern}: {int(diff.sum())} elements differ, first at (batch {idx[:2]}, "
                                 f"row {idx[2]}, piece {idx[3]}, column {idx[4]}): got {got[tuple(idx)].item()}, "
                                 f"want {want[tuple(idx)].item()}")
        assert_guard(dst, lambda t: t[:, :, :R, :pieces * cpad], f"pattern {pattern}: destination")


# ------------------------------------------------------------------------------------------------ host paths
@pytest.mark.parametrize("pieces", [3, 6])
def test_fp32_matmul_split_many_tiles(pieces, monkeypatch):
    """fp32 `matmul` (8, 197, 768) . (768, 3072) + bias + GELU: split operands, 8 batches x 2 x 24 = 384 tiles."""
    from vit.kernels import matmul
    monkeypatch.setenv("VT_FP32_SPLIT", str(pieces))
    Bn, M, K, N = 8, 197, 768, 3072
    assert_many_tiles(bgemm_tiles(M, N, Bn, False))
    a = torch.randn(Bn, M, K, device=dev())
    w = torch.randn(K, N, device=dev()) / math.sqrt(K)
    bias = torch.randn(N, device=dev())
    got = matmul(a, w, bias, "gelu")
    acc, absacc = products(a, w.t())
    kk = pieces * ceil8(K)
    e = (kk * EPS32 * PIECE_MASS + SPLIT[pieces]) * absacc + EPI_OPS * EPS32 * (acc.abs() + bias.double().abs())
    want, e = act_ref_and_bound(ACT_GELU, acc + bias.double(), e)
    assert_elementwise(got, want, ulp_out(want, torch.float32) + e)


MATMUL3 = {
    # name: (dtype, A shape, B shape, B consumed MN-major in place)
    "f32_split": (torch.float32, (192, 197, 64), (192, 64, 197), False),
    "bf16_in_place_mn_major": (torch.bfloat16, (160, 197, 96), (160, 96, 136), True),
    "bf16_packed_197_keys": (torch.bfloat16, (192, 197, 64), (192, 64, 197), False),
}


@pytest.mark.parametrize("name", list(MATMUL3))
def test_matmul3_many_tiles(name):
    from vit.kernels import bgemm as bg, matmul3
    dtype, sa, sb, b_mn = MATMUL3[name]
    Bn, M, K = sa
    N = sb[2]
    assert_many_tiles(bgemm_tiles(M, N, Bn, b_mn))
    a = torch.randn(*sa, device=dev()).to(dtype)
    b = torch.randn(*sb, device=dev()).to(dtype)
    s = 1 / math.sqrt(K)
    got = matmul3(a, b, apply_scaling=True, scale_factor=s)
    pieces = 1 if dtype == torch.bfloat16 else bg.split_pieces()
    kk = pieces * ceil8(K)
    acc, absacc = products(a, b.transpose(1, 2))
    want = s * acc
    e = s * (kk * EPS32 * PIECE_MASS + SPLIT[pieces]) * absacc + EPI_OPS * EPS32 * want.abs()
    assert_elementwise(got, want, ulp_out(want, dtype) + e, tile=(128, 64 if b_mn else 128))


@pytest.mark.parametrize("dtype,dh", [(torch.float32, 64), (torch.float32, 80), (torch.bfloat16, 48)])
def test_composed_attention_many_tiles(dtype, dh):
    """flash_attention on its composed path (fp32, or a head dim the fused kernels do not take): 16 images x 12 heads
    of 197 tokens, 768 score tiles and 384 P.V tiles.  Every element of every (image, head) within the bound of the
    module docstring; the report counts the (image, head) pairs that fail."""
    from vit.kernels import bgemm as bg, flash_attention
    B, H, N = 16, 12, 197
    D = H * dh
    assert_many_tiles(min(bgemm_tiles(N, N, B * H, False), bgemm_tiles(N, dh, B * H, False)))
    qkv = torch.randn(B, N, 3 * D, device=dev()).to(dtype)
    got = flash_attention(qkv, H)
    pieces = 1 if dtype == torch.bfloat16 else bg.split_pieces()
    scale = 1.0 / math.sqrt(dh)
    q, k, v = qkv.double().view(B, N, 3, H, dh).permute(2, 0, 3, 1, 4)        # (B, H, N, dh)
    s = scale * (q @ k.transpose(-1, -2))
    es = scale * (pieces * ceil8(dh) * EPS32 * PIECE_MASS + SPLIT[pieces]) * (q.abs() @ k.abs().transpose(-1, -2)) \
        + EPI_OPS * EPS32 * s.abs() + ulp_out(s, dtype)
    p = torch.softmax(s, -1)
    va = v.abs()
    pva = p @ va
    spread = (s - s.amax(-1, keepdim=True)).abs().amax(-1, keepdim=True)
    smx = EPS32 * (N + 8 + 2 * spread)
    pes = p * es
    kk = pieces * ceil8(N)
    bound = 1.01 * (pes @ va + pes.sum(-1, keepdim=True) * pva) + smx * pva \
        + 1.01 * (kk * EPS32 * PIECE_MASS + SPLIT[pieces]) * pva
    if dtype == torch.bfloat16:
        bound = bound + ulp_out(p, dtype) @ va
    want = p @ v
    bound = bound + ulp_out(want, dtype)
    got = got.view(B, N, H, dh).transpose(1, 2)
    assert_elementwise(got.reshape(-1, dh), want.reshape(-1, dh), bound.reshape(-1, dh), tile=(N, dh),
                       what="attention output (tiles = (image, head) pairs)")


@pytest.mark.parametrize("dtype", [torch.bfloat16, torch.float32], ids=["bf16", "f32"])
@pytest.mark.parametrize("head", ["pooler", "classifier"])
def test_heads_on_cls_rows_many_tiles(head, dtype):
    """Pooler (tanh) and classifier head through `_head_on_cls` on hidden states (8192, 5, 768) whose non-CLS rows
    are NaN: the CLS rows are read in place through the row stride (bf16) or packed from it (fp32), 384 / 512
    tiles."""
    from vit.kernels import bgemm as bg
    from vit.vit import LinearWithBias, Pooler, _head_on_cls
    Bn, T, D = 8192, 5, 768
    n_out = D if head == "pooler" else 1000
    assert_many_tiles(bgemm_tiles(Bn, n_out, 1, False))
    hidden = sentinel((Bn, T, D), dtype)
    hidden[:, 0] = torch.randn(Bn, D, device=dev()).to(dtype)
    dense = Pooler(D).dense if head == "pooler" else LinearWithBias(D, n_out)
    with torch.no_grad():
        dense.weight.copy_(torch.randn(D, n_out) / math.sqrt(D))
        dense.bias.copy_(0.5 * torch.randn(n_out))
    dense = dense.to(dev(), dtype)
    act = ACT_TANH if head == "pooler" else ACT_NONE
    got = _head_on_cls(hidden, dense, act)
    pieces = 1 if dtype == torch.bfloat16 else bg.split_pieces()
    acc, absacc = products(hidden[:, 0], dense.weight.t())
    bias = dense.bias.double()
    e = (pieces * D * EPS32 * PIECE_MASS + SPLIT[pieces]) * absacc + EPI_OPS * EPS32 * (acc.abs() + bias.abs())
    want, e = act_ref_and_bound(act, acc + bias, e)
    assert_elementwise(got, want, ulp_out(want, dtype) + e)


# ------------------------------------------------------------------------------------------------ vt_gemm_bf16, fp32 out
GEMM_F32 = {
    "bias_gelu": dict(N=768, gelu=True),                     # BN = 256: 394 x 3 = 1182 tiles
    "bias_residual": dict(N=768, res="sep"),
    "residual_in_place_bn128": dict(N=128, res="inplace"),   # BN = 128: 394 tiles
    "tail_n136_in_place": dict(N=136, res="inplace"),        # BN = 256, one partial column tile per row block
    "tail_n136_gelu": dict(N=136, gelu=True, bias=False),
}


@pytest.mark.parametrize("name", list(GEMM_F32))
def test_gemm_bf16_f32_out_many_tiles(name):
    """vt_gemm_bf16 with fp32 output (csrc/gemm_sm100.cu) at M = 50432 (256 images x 197 tokens), K = 768, every
    element against fp64; guard rows and columns; a 128-aligned block of rows as its own call equals its slice."""
    L = _lib()
    kw = GEMM_F32[name]
    M, K, N = 256 * 197, 768, kw["N"]
    gelu, res = kw.get("gelu", False), kw.get("res")
    bn = 256 if N > 128 else 128
    tiles = -(-M // 128) * -(-N // bn)
    assert_many_tiles(tiles)
    A = torch.randn(M, K, device=dev()).bfloat16()
    W = (torch.randn(N, K, device=dev()) / math.sqrt(K)).bfloat16()
    bias = (0.5 * torch.randn(N, device=dev())) if kw.get("bias", True) else None
    residual = torch.randn(M, N, device=dev()) if res else None
    ldo = N + 64

    def output():
        out = sentinel((M + 64, ldo), torch.float32)
        if res == "inplace":
            out[:M, :N] = residual
        return out

    def launch(out, m0=0, rows=M):
        r_ptr, ldr = None, 0
        if res == "inplace":
            r_ptr, ldr = out.data_ptr() + 4 * m0 * ldo, ldo
        elif res == "sep":
            r_ptr, ldr = residual.data_ptr() + 4 * m0 * N, N
        L.call("vt_gemm_bf16", A.data_ptr() + 2 * m0 * K, K, W.data_ptr(), K, out.data_ptr() + 4 * m0 * ldo, ldo,
               L.VT_F32, L.ptr(bias), r_ptr, ldr, rows, N, K, int(gelu), L.stream_ptr(A))

    out = output()
    launch(out)
    torch.cuda.synchronize()
    acc, absacc = products(A, W)
    e = K * EPS32 * absacc + EPI_OPS * EPS32 * acc.abs()
    pre = acc
    if bias is not None:
        pre = pre + bias.double()
        e = e + EPI_OPS * EPS32 * bias.double().abs()
    want, e = act_ref_and_bound(ACT_GELU if gelu else ACT_NONE, pre, e)
    del acc, absacc
    if res:
        r = residual.double()
        e = e + EPI_OPS * EPS32 * (want.abs() + r.abs())
        want = want + r
    assert_elementwise(out[:M, :N], want, ulp_out(want, torch.float32) + e, tile=(128, bn))
    assert_guard(out, lambda t: t[:M, :N], "output")

    m0, rows = 128 * 200, 128 * (sms() // -(-N // bn))
    sub = output()
    launch(sub, m0, rows)
    torch.cuda.synchronize()
    assert bit_equal(sub[m0:m0 + rows, :N], out[m0:m0 + rows, :N]), \
        f"rows {m0}..{m0 + rows - 1} computed alone differ from their slice of the full call"
