"""GPU: the fused attention kernels of vt_flash_attn (csrc/attn5_sm100.cu) element by element.

attn5 (head dim 64, N <= 208) takes, per (image, head) item, either the bounded-logit path (no row max; the last
VT_ATTN5_POLY = 2 pairs of every 16 score columns through ex2_poly_x2 on the FMA pipe) or the exact two-pass path;
vt_debug_set_attn_bound(1) / (0) lets the kernel choose / forces the exact path.  attn5mb (head dim 64 with N > 208,
every head dim 80) runs an online softmax over KV blocks of bkv keys, the last one shorter.

Every launch goes through `both_directions` (both traversal orders, bit-equal).  Q, K and V are three separate
allocations with row stride H * dh + 24 and GAP rows between images, a whole image after the last one; the padding,
the gap rows and that image are NaN, so a read outside the tensor maps' extents (0 * NaN = NaN in the P V MMA) shows
up in the output.  The output has the same layout filled with a NaN sentinel, which must survive outside [B, N, H * dh].

A. Exact dyadic inputs.  scale = 0.08664339780807495 makes fp32(scale * 1.4426950408889634f), the launchers'
scale_log2, exactly 2^-3.  Q = 2 A and K = 4 Bm with A holding two entries +-1 per row in the first dh - 1 columns (a
coinciding pair gives +-2) and a 1 in the last, Bm entries in {-2, ..., 2} in the first dh - 1 columns and 0 in the
last, except key 0, which is 4 e_(dh-1): every score q.k = 8 (A . Bm) is an integer below 2^12, exact in fp32 whatever
the accumulation order, and every exponent argument is an integer a = A . Bm in [-4, 4] (bounded path, m = 0) or in
[-8, 0] (exact paths), with the row maximum 4 on key 0.  ex2.approx (2^-22) and ex2_poly_x2 (2^n * 0.99992818) are then within 2^-13 of 2^a, so P
rounded to bf16 is exactly 2^a.  V holds integers in [-8, 8].  The sums the tensor core forms are then exact in fp32:
  * exact paths: P in [2^-8, 1], N <= 2305 < 2^12 keys: row sums below 2^12 and P V sums below 2^15, both multiples
    of 2^-8, i.e. at most 20 and 23 significant bits;
  * bounded path: P in [2^-4, 2^4], N <= 208: row sums below 2^12 and P V sums below 2^15 in multiples of 2^-4.
So the only inexact steps are rcp.approx.ftz of the row sum (1 ulp), the fp32 product with it and the bf16 rounding.
In attn5mb the rescale factor alpha = ex2.approx(m_run - m_new) is kept exact by the row maximum in block 0: from
block 1 on m_new = m_run and alpha = ex2.approx(0) = 1, so the online sums are the plain sums.  With q the fp64
quotient, every output must be within 1 bf16 ulp of q and equal bf16_rn(q) unless q lies within 2^-22 |q| of a bf16
rounding midpoint (fewer than 1 % of the elements may be excused so).

B. Every probability read out through V.  Head h reads keys [h dh, h dh + dh) through V = identity on that window
(zero elsewhere), all heads with the same Q and K: output column c of head h is P^[i, h dh + c] / S^[i].

C. Random inputs.  In log2 units a_ij = c q_i.k_j with c = scale log2(e), A_ij = c sum_d |q_id k_jd|, u = 2^-24.
The kernel's exponent argument is off by e_ij <= dh 2^-23 A_ij (fp32 accumulation with truncation) + u (|a_ij| +
|m_i|) (the fma with the row max) + 2^-23 |a_ij| (scale_log2 rounded to fp32), so P_j before rounding has the relative
error ln2 e_ij + EXP_ERR (ex2.approx 2^-22, ex2_poly_x2 POLY_REL + 2^-23); rounding P to bf16 adds 2^-8:
  eps_i = 2^-8 + EXP_ERR + ln2 max_j e_ij.
The output is sum_j P^_j v_j / sum_j P^_j with P^_j = Z w_j (1 + eta_j), |eta_j| <= eps_i, hence
  |o - o_ref| <= 2 eps_i / (1 - eps_i) sum_j w_j |v_j|
plus the fp32 sums of S^ and of P V (N adds each, 2^-23 relative), rcp.approx and the product (8 2^-23), in attn5mb
the rescale of every block (4 2^-23 each), all relative to sum_j w_j |v_j|, plus one bf16 ulp of o_ref for the final
rounding (half an ulp, the other half for a value that crossed a binade) and N 2^-100 max|v| for exponentials that
flush to zero.  Per element:
  |o - o_ref| <= ulp_bf16(o_ref) + (2 eps_i / (1 - eps_i) + (2N + 4 nblk + 8) 2^-23) sum_j w_ij |v_jc| + N 2^-100 max|v|.
The worst-case bound is dominated by the bf16 rounding of P and cannot see a bias of 1e-3 on a quarter of the
columns, so the bounded path is also checked for one: the mean relative error of the probabilities in the polynomial
columns (key % 16 >= 12) and in the others must agree within POLY_REL plus six standard errors.
"""
import contextlib
import ctypes
import math

import pytest
import torch

from test_gpu_persistent import assert_guard, bit_equal, both_directions, dev, sentinel, sm_partition, ulp_bf16

pytestmark = pytest.mark.gpu

LOG2E = 1.4426950408889634
LN2 = math.log(2.0)
U = 2.0 ** -24
POLY_REL = 7.52e-5                          # ex2_poly_x2 on [-0.5, 0.5], restated in test_abi_attn.py
EXP_ERR = POLY_REL + 2.0 ** -23             # >= 2^-22 of ex2.approx
BF16_P = 2.0 ** -8                          # relative rounding error of P in bf16
DYADIC_SCALE = 0.08664339780807495
PADC = 24                                   # padding columns of every row
GAP = 3                                     # NaN rows between two images
NAN = float("nan")

ATTN5_N = [1, 2, 15, 16, 17, 31, 32, 33, 64, 100, 127, 128, 129, 192, 197, 198, 207, 208]
ATTN5MB_64_N = [209, 224, 257, 416, 417, 577, 625, 1025, 1370, 2305]
ATTN5MB_80_N = [1, 17, 128, 129, 197, 208, 209, 257, 577, 1025]
HEADS = (1, 3, 12, 16)


def _shapes():
    """(dh, N, B, H): H cycles through 1, 3, 12, 16; two shapes have more than 2 * 148 items, so CTAs walk several."""
    out = []
    for i, (dh, N) in enumerate([(64, n) for n in ATTN5_N] + [(64, n) for n in ATTN5MB_64_N] +
                                [(80, n) for n in ATTN5MB_80_N]):
        H = HEADS[i % 4]
        B = 3 if N <= 257 else (2 if N <= 625 else 1)
        if H >= 12 and N > 577:
            H = 3
        out.append((dh, N, B, H))
    out[ATTN5_N.index(197)] = (64, 197, 16, 12)                                    # attn5: 384 items, 2 per pair
    out[len(ATTN5_N) + len(ATTN5MB_64_N) + ATTN5MB_80_N.index(257)] = (80, 257, 12, 16)   # attn5mb: 576 items
    return out


SHAPES = _shapes()


def _id(s):
    dh, N, B, H = s
    return f"dh{dh}-N{N}-B{B}-H{H}"


def _lib():
    from vit.kernels import _lib
    return _lib


def is_attn5(dh, N):
    return dh == 64 and N <= 208


def blocks(N, dh):
    """(blocks per item, keys per block, keys of the last block) as the launchers choose them."""
    if is_attn5(dh, N):
        return 1, (N + 15) // 16 * 16, N
    nblk = -(-N // 208)
    bkv = (-(-N // nblk) + 15) // 16 * 16
    return nblk, bkv, N - (nblk - 1) * bkv


def items(dh, N, B, H):
    return B * H * -(-N // 128)


@contextlib.contextmanager
def attn_bound(mode):
    """vt_debug_set_attn_bound: 1 = items whose logits are bounded skip the row max (the default), 0 = every item
    takes the exact two-pass path; back to -1 (the environment's default) on the way out."""
    fn = _lib().load().vt_debug_set_attn_bound
    fn.argtypes = [ctypes.c_int]
    fn.restype = None
    fn(mode)
    try:
        yield
    finally:
        fn(-1)


def paths(dh, N):
    return (1, 0) if is_attn5(dh, N) else (1,)


# ---------------------------------------------------------------------------------------------------- launches
def operand(x):
    """(B, N, H, dh) values exact in bf16 -> a separate NaN-filled (B + 1, N + GAP, H dh + PADC) bf16 allocation
    holding them in [:B, :N, :H dh]."""
    B, N, H, dh = x.shape
    buf = torch.full((B + 1, N + GAP, H * dh + PADC), NAN, dtype=torch.bfloat16, device=dev())
    buf[:B, :N, :H * dh] = x.reshape(B, N, H * dh).to(torch.bfloat16)
    return buf


def flash(ops, scale, B=None, lo=0):
    """vt_flash_attn over images lo .. lo + B of the operand buffers `ops` = (q, k, v, H, dh), both directions, into
    sentinel buffers of the same layout; checks the guards.  Returns the output as (B, H, N, dh)."""
    L = _lib()
    q, k, v, H, dh = ops
    Bq, Ng, rs = q.shape
    B = Bq - 1 - lo if B is None else B
    N = Ng - GAP
    bs = Ng * rs
    off = lo * bs * 2

    def go(out):
        rc = L.load().vt_flash_attn(q.data_ptr() + off, k.data_ptr() + off, v.data_ptr() + off, out.data_ptr(), B, H,
                                    N, dh, rs, bs, rs, bs, scale, L.stream_ptr(q))
        assert rc == 0, f"vt_flash_attn returned {rc}"

    out, = both_directions(lambda: (sentinel((B + 1, Ng, rs), torch.bfloat16),), go)
    assert_guard(out, (slice(0, B), slice(0, N), slice(0, H * dh)), "attention output")
    return out[:B, :N, :H * dh].reshape(B, N, H, dh).permute(0, 2, 1, 3)


def operands(q, k, v):
    """(q, k, v, H, dh): three operand buffers of (B, N, H, dh) tensors."""
    return tuple(operand(t) for t in (q, k, v)) + (q.shape[2], q.shape[3])


def as_bhnd(x):
    """(B, N, H, dh) -> (B, H, N, dh) fp64 on the device."""
    return x.to(dev()).double().permute(0, 2, 1, 3)


def bf16_exact(x):
    return x.to(torch.bfloat16).double()


# ---------------------------------------------------------------------------------------------------- references
def reference(q, k, v, scale, nblk):
    """fp64 softmax(scale q k^T) v on the kernel's own bf16 operands ((B, H, N, dh) fp64) and the per-element bound of
    the module docstring.  Returns (o_ref, bound, w) with w the fp64 probabilities (B, H, N, N)."""
    B, H, N, dh = q.shape
    c = scale * LOG2E
    a = c * (q @ k.transpose(-1, -2))
    A = c * (q.abs() @ k.abs().transpose(-1, -2))
    m = a.amax(-1, keepdim=True)
    w = torch.exp2(a - m)
    w = w / w.sum(-1, keepdim=True)
    arg = dh * 2.0 ** -23 * A + U * (a.abs() + m.abs()) + 2.0 ** -23 * a.abs()
    eps = BF16_P + EXP_ERR + LN2 * arg.amax(-1, keepdim=True)
    o = w @ v
    T = w @ v.abs()
    rel = 2 * eps / (1 - eps) + (2 * N + 4 * nblk + 8) * 2.0 ** -23
    bound = ulp_bf16(o) + rel * T + N * 2.0 ** -100 * v.abs().amax()
    return o, bound, w


def assert_within(got, ref, bound, what):
    """|got - ref| <= bound for every element of (B, H, N, C) results; on failure the worst element as
    (image, head, row, column) and the number of (image, head) pairs that fail."""
    got = got.double()
    err = (got - ref).abs()
    bad = ~(err <= bound)
    n_bad = int(bad.sum())
    if n_bad == 0:
        return
    ratio = torch.where(bad, torch.nan_to_num(err / bound, nan=float("inf"), posinf=float("inf")), 0.0)
    idx = torch.unravel_index(ratio.argmax(), ratio.shape)
    b, h, i, j = (int(t) for t in idx)
    pairs = int(bad.flatten(2).any(-1).sum())
    raise AssertionError(
        f"{what}: {n_bad} of {bad.numel()} elements outside the bound in {pairs} of {bad.shape[0] * bad.shape[1]} "
        f"(image, head) pairs; worst (image {b}, head {h}, row {i}, column {j}): got {got[b, h, i, j].item()!r}, "
        f"want {ref[b, h, i, j].item()!r}, bound {bound[b, h, i, j].item():.3g}")


def rn_bf16(x):
    """Round fp64 to the nearest bf16 value, ties to even, without a double rounding through fp32."""
    ulp = ulp_bf16(x)
    return torch.round(x / ulp) * ulp


def assert_rounded_quotient(got, qv, slack, what):
    """got (bf16) within 1 bf16 ulp of the fp64 quotient qv, and equal to bf16_rn(qv) wherever qv is farther than
    `slack` from a bf16 rounding midpoint.  Returns the share of elements excused."""
    got = got.double()
    ulp = ulp_bf16(qv)
    assert_within(got, qv, ulp, f"{what}: more than one bf16 ulp from the exact quotient")
    t = qv / ulp
    dmid = (t - torch.floor(t) - 0.5).abs() * ulp
    strict = dmid > slack
    bad = strict & (got != rn_bf16(qv))
    if bool(bad.any()):
        b, h, i, j = (int(t) for t in bad.nonzero()[0])
        raise AssertionError(f"{what}: {int(bad.sum())} elements not the rounded quotient, first (image {b}, head {h}, "
                             f"row {i}, column {j}): got {got[b, h, i, j].item()!r}, quotient {qv[b, h, i, j].item()!r}")
    return 1.0 - strict.double().mean().item()


# ---------------------------------------------------------------------------------------------------- inputs
def dyadic_qkv(B, N, H, dh, seed):
    """(q, k, v, a): Q = 2 A, K = 4 Bm, V integers in [-8, 8] as (B, N, H, dh) float
    tensors, and the integer logits a = A Bm^T (log2 units) as (B, H, N, N) fp64 on the device."""
    g = torch.Generator().manual_seed(seed)
    Ai = torch.zeros(B, N, H, dh)
    Ai[..., dh - 1] = 1.0
    idx = torch.randint(dh - 1, (B, N, H, 2), generator=g)
    sgn = (torch.randint(2, (B, N, H, 2), generator=g) * 2 - 1).float()
    Ai.scatter_add_(3, idx, sgn)
    Bm = torch.randint(-2, 3, (B, N, H, dh), generator=g).float()
    Bm *= (torch.rand((B, N, H, dh), generator=g) < 0.3).float()
    Bm[..., dh - 1] = 0.0
    Bm[:, 0] = 0.0
    Bm[:, 0, :, dh - 1] = 4.0           # key 0: logit 4 in every row, the row maximum
    v = torch.randint(-8, 9, (B, N, H, dh), generator=g).float()
    a = as_bhnd(Ai) @ as_bhnd(Bm).transpose(-1, -2)
    return 2 * Ai, 4 * Bm, v, a


def window_v(B, N, H, dh):
    """V of head h: the identity on keys [h dh, h dh + dh), zero elsewhere."""
    v = torch.zeros(B, N, H, dh)
    for h in range(H):
        for c in range(dh):
            if h * dh + c < N:
                v[:, h * dh + c, h, c] = 1.0
    return v


def random_qkv(B, N, H, dh, seed, gain=1.0):
    g = torch.Generator().manual_seed(seed)
    return tuple(bf16_exact(gain * torch.randn((B, N, H, dh), generator=g)).float() for _ in range(3))


def dyadic_quotient(a, v):
    """The exact quotient sum_j 2^a_ij v_jc / sum_j 2^a_ij in fp64."""
    w = torch.exp2(a - a.amax(-1, keepdim=True))
    return (w @ v) / w.sum(-1, keepdim=True)


def dyadic_slack(qv):
    """rcp.approx.ftz (1 fp32 ulp) and the fp32 product: 2^-23 + 2^-24 < 2^-22 relative."""
    return 2.0 ** -22 * qv.abs()


def test_dyadic_scale_is_an_exact_power_of_two():
    s = torch.tensor(DYADIC_SCALE, dtype=torch.float32)
    assert (s * torch.tensor(LOG2E, dtype=torch.float32)).item() == 0.125


def test_block_table():
    """The KV blocks of attn5mb at every tested N (printed), and the shapes the cases are chosen for."""
    for dh, N, B, H in SHAPES:
        if not is_attn5(dh, N):
            nblk, bkv, last = blocks(N, dh)
            print(f"dh {dh} N {N:5d}: {nblk:2d} blocks, {nblk - 1:2d} x {bkv} keys + {last}; "
                  f"{items(dh, N, B, H)} items (B {B}, H {H})")
    assert blocks(209, 64) == (2, 112, 97) and blocks(416, 64) == (2, 208, 208)
    assert blocks(577, 64) == (3, 208, 161) and blocks(2305, 64) == (12, 208, 17)
    assert {blocks(N, 64)[0] for N in ATTN5MB_64_N} == {2, 3, 4, 5, 7, 12}
    assert sum(items(*s) > 2 * 148 for s in SHAPES) >= 2


# ---------------------------------------------------------------------------------------------------- A: dyadic
@pytest.mark.parametrize("shape", SHAPES, ids=_id)
def test_dyadic_inputs_give_the_rounded_quotient(shape):
    dh, N, B, H = shape
    q, k, v, a = dyadic_qkv(B, N, H, dh, seed=N * 31 + dh + H)
    assert a.abs().max() <= 4
    ops = operands(q, k, v)
    assert (a[..., 0] == 4).all() and a.amax(-1).eq(4).all()
    qv = dyadic_quotient(a, as_bhnd(v))
    for mode in paths(dh, N):
        with attn_bound(mode):
            got = flash(ops, DYADIC_SCALE)
        excused = assert_rounded_quotient(got, qv, dyadic_slack(qv), f"{_id(shape)} bound mode {mode}")
        assert excused < 0.01, f"{excused:.3%} of the elements lie next to a rounding midpoint"


# ---------------------------------------------------------------------------------------------------- C: random
@pytest.mark.parametrize("shape", SHAPES, ids=_id)
def test_random_inputs_within_the_derived_bound(shape):
    dh, N, B, H = shape
    q, k, v = random_qkv(B, N, H, dh, seed=N * 17 + dh + H)
    ops = operands(q, k, v)
    scale = 1.0 / math.sqrt(dh)
    nblk = blocks(N, dh)[0]
    ref, bound, _ = reference(as_bhnd(q), as_bhnd(k), as_bhnd(v), scale, nblk)
    first = None
    for mode in paths(dh, N):
        with attn_bound(mode):
            got = flash(ops, scale)
        assert_within(got, ref, bound, f"{_id(shape)} bound mode {mode}")
        first = got if first is None else first
    if is_attn5(dh, N):
        for cap in (1, 3, 7):
            with sm_partition(0, cap):
                again = flash(ops, scale)
            assert bit_equal(again, first), f"attn5 on {cap} CTAs differs from the full grid"
    if B >= 2:
        sub = flash(ops, scale, B=B - 1, lo=1)
        assert bit_equal(sub, first[1:]), "a sub-batch call differs from its slice of the batch"


# ---------------------------------------------------------------------------------------------------- B: through V
B_SHAPES = [(64, 2), (64, 17), (64, 100), (64, 197), (64, 208), (64, 257), (64, 577), (64, 2305), (80, 17),
            (80, 197), (80, 577)]


@pytest.mark.parametrize("dh,N", B_SHAPES)
def test_every_probability_read_out_through_v(dh, N):
    """Dyadic Q, K: every probability is the rounded quotient 2^a_ij / sum_j 2^a_ij; columns past the last key are 0."""
    H = -(-N // dh)
    B = 2
    q, k, _, a = dyadic_qkv(B, N, 1, dh, seed=N + 5 * dh)
    q, k = q.expand(B, N, H, dh).contiguous(), k.expand(B, N, H, dh).contiguous()
    v = window_v(B, N, H, dh)
    ops = operands(q, k, v)
    w = torch.exp2(a - a.amax(-1, keepdim=True))
    pv = w / w.sum(-1, keepdim=True)
    for mode in paths(dh, N):
        with attn_bound(mode):
            got = flash(ops, DYADIC_SCALE)
        probs = got.permute(0, 2, 1, 3).reshape(B, N, H * dh)[:, :, :N]         # (B, row, key)
        assert (got.permute(0, 2, 1, 3).reshape(B, N, H * dh)[:, :, N:] == 0).all(), "a column past the last key"
        want = pv[:, 0]
        excused = assert_rounded_quotient(probs[:, None], want[:, None], dyadic_slack(want)[:, None],
                                          f"dh {dh} N {N} bound mode {mode}: probabilities")
        assert excused < 0.01


def _attn_probs(q, k, scale):
    """vt_attn_probs on a fused (B, N, 3D) buffer built from (B, N, H, dh) q, k: (B, H, N, N) bf16."""
    L = _lib()
    B, N, H, dh = q.shape
    D = H * dh
    qkv = torch.zeros(B, N, 3 * D, dtype=torch.bfloat16, device=dev())
    qkv[:, :, :D] = q.reshape(B, N, D).to(qkv)
    qkv[:, :, D:2 * D] = k.reshape(B, N, D).to(qkv)
    out = torch.empty(B, H, N, N, dtype=torch.bfloat16, device=dev())
    L.call("vt_attn_probs", qkv.data_ptr(), qkv.data_ptr() + 2 * D, out.data_ptr(), B, H, N, dh, 3 * D, 3 * D * N,
           scale, L.stream_ptr(qkv))
    torch.cuda.synchronize()
    return out


def _probs_bound(q, k, scale, N, nblk):
    """fp64 probabilities (B, 1, N, N) and the bound on P^_ij / S^_i rounded to bf16: 2^-8 for P^_ij, 2^-8 for the
    weighted mean of the roundings inside S^, 2 E_i for the arguments, exponentials and sums, one bf16 ulp for the
    output rounding (crossing a binade included) and 2^-126 for exponentials that flush to zero."""
    qd, kd = as_bhnd(q[:, :, :1]), as_bhnd(k[:, :, :1])
    dh = qd.shape[-1]
    c = scale * LOG2E
    a = c * (qd @ kd.transpose(-1, -2))
    A = c * (qd.abs() @ kd.abs().transpose(-1, -2))
    m = a.amax(-1, keepdim=True)
    ref = torch.softmax(a * LN2, dim=-1)
    arg = dh * 2.0 ** -23 * A + U * (a.abs() + m.abs()) + 2.0 ** -23 * a.abs()
    E = LN2 * arg.amax(-1, keepdim=True) + EXP_ERR + (2 * N + 4 * nblk + 8) * 2.0 ** -23
    return ref, (2 * BF16_P + 2 * E) * ref + ulp_bf16(ref) + 2.0 ** -126


def _attn_probs_bound(q, k, scale, N):
    """The bound of vt_attn_probs (test_gpu_outputs.py)."""
    qd, kd = as_bhnd(q[:, :, :1]), as_bhnd(k[:, :, :1])
    dh = qd.shape[-1]
    c = scale / LN2
    a = c * (qd @ kd.transpose(-1, -2))
    A = c * (qd.abs() @ kd.abs().transpose(-1, -2))
    m = a.amax(-1, keepdim=True)
    ref = torch.softmax(a * LN2, dim=-1)
    arg = 2 * dh * U * A + U * (a.abs() + m.abs())
    E = 2 * LN2 * arg.amax(-1, keepdim=True) + 2.0 ** -20 + (N + 4) * 2 * U
    return ulp_bf16(ref) + 2 * E * ref + 2.0 ** -126


@pytest.mark.parametrize("dh,N", B_SHAPES)
def test_random_probabilities_read_out_through_v(dh, N):
    """Random Q, K: every probability against the fp64 softmax; each row sums to 1 within the summed bound (a padded
    key counted in S^ fails this at small N); the same Q, K through vt_attn_probs agree within both bounds.  On the
    bounded path, the polynomial columns carry no bias beyond the polynomial's own error."""
    H = -(-N // dh)
    B = 4 if N <= 257 else 2
    g = torch.Generator().manual_seed(N * 3 + dh)
    q1 = bf16_exact(torch.randn((B, N, 1, dh), generator=g)).float()
    k1 = bf16_exact(torch.randn((B, N, 1, dh), generator=g)).float()
    q, k = q1.expand(B, N, H, dh).contiguous(), k1.expand(B, N, H, dh).contiguous()
    ops = operands(q, k, window_v(B, N, H, dh))
    scale = 1.0 / math.sqrt(dh)
    nblk = blocks(N, dh)[0]
    ref, bound = _probs_bound(q, k, scale, N, nblk)
    ref, bound = ref[:, 0], bound[:, 0]
    other = _attn_probs(q, k, scale)[:, 0].double()
    assert_within(other[:, None], ref[:, None], _attn_probs_bound(q, k, scale, N), "vt_attn_probs")
    for mode in paths(dh, N):
        with attn_bound(mode):
            got = flash(ops, scale)
        rows = got.permute(0, 2, 1, 3).reshape(B, N, H * dh)
        assert (rows[:, :, N:] == 0).all(), "a column past the last key"
        probs = rows[:, :, :N].double()
        what = f"dh {dh} N {N} bound mode {mode}"
        assert_within(probs[:, None], ref[:, None], bound[:, None], what)
        dev_sum = (probs.sum(-1) - 1).abs()
        assert (dev_sum <= bound.sum(-1)).all(), f"{what}: a row sum off by {dev_sum.max().item():.3e}"
        assert_within(probs[:, None], other[:, None], (bound + _attn_probs_bound(q, k, scale, N)[:, 0])[:, None],
                      f"{what}: against vt_attn_probs")
        if mode == 1 and is_attn5(dh, N) and N >= 16:
            ok = ref > 2.0 ** -60
            rel = torch.where(ok, probs / ref - 1, 0.0)
            poly = (torch.arange(N, device=dev()) % 16 >= 12).expand_as(rel) & ok
            mufu = ~poly & ok
            mp, mm = rel[poly].mean().item(), rel[mufu].mean().item()
            se = math.sqrt(rel[poly].var().item() / int(poly.sum()) + rel[mufu].var().item() / int(mufu.sum()))
            print(f"{what}: mean relative error {mp:.3e} (polynomial columns) vs {mm:.3e}, standard error {se:.1e}")
            assert abs(mp - mm) <= POLY_REL + 6 * se, f"{what}: the polynomial columns are biased by {mp - mm:.3e}"


# ---------------------------------------------------------------------------------------------------- F: hostile rows
@pytest.mark.parametrize("dh,N", [(64, 577), (64, 2305), (80, 577), (80, 209)])
@pytest.mark.parametrize("where", ["last", "first"])
def test_row_maximum_far_in_one_block(dh, N, where):
    """Every row's maximum sits on one key of the last (or the first) KV block, 150 log2 units above the rest:
    alpha = 2^-150 flushes the earlier blocks to zero (or the later blocks' exponentials do)."""
    B, H = 2, 3
    q, k, v = random_qkv(B, N, H, dh, seed=N + dh)
    j = N - 1 if where == "last" else 0
    scale = 1.0 / math.sqrt(dh)
    q[:, :, :, 0] = 4.0
    k[:, :, :, 0] = 0.0
    k[:, j, :, 0] = bf16_exact(torch.tensor(150.0 / (4 * scale * LOG2E))).item() + 32
    ops = operands(q, k, v)
    ref, bound, _ = reference(as_bhnd(q), as_bhnd(k), as_bhnd(v), scale, blocks(N, dh)[0])
    got = flash(ops, scale)
    assert_within(got, ref, bound, f"maximum in the {where} block")


@pytest.mark.parametrize("dh,N", [(64, 197), (64, 17), (64, 577), (80, 257)])
@pytest.mark.parametrize("vgain", [1.0, 1e4, 1e-4])
def test_equal_keys_and_extreme_values(dh, N, vgain):
    """Head 0: every key of an image equal (uniform rows); head 1: random; head 2: all-zero Q.  V scaled to ~1e4 or
    ~1e-4."""
    B, H = 2, 3
    q, k, v = random_qkv(B, N, H, dh, seed=N * 7 + dh)
    k[:, :, 0] = k[:, :1, 0]
    q[:, :, 2] = 0.0
    v = bf16_exact(v * vgain).float()
    ops = operands(q, k, v)
    scale = 1.0 / math.sqrt(dh)
    ref, bound, _ = reference(as_bhnd(q), as_bhnd(k), as_bhnd(v), scale, blocks(N, dh)[0])
    for mode in paths(dh, N):
        with attn_bound(mode):
            got = flash(ops, scale)
        assert_within(got, ref, bound, f"V gain {vgain} bound mode {mode}")


@pytest.mark.parametrize("N", [197, 64, 17])
def test_items_around_the_bounded_path_threshold(N):
    """One launch, one head per ratio rho of the Cauchy-Schwarz bound (as the kernel admits it, margin included) to
    kLogitBound5: Q and K rows are +-r u along one direction u, so the logits reach +-64 rho / 1.1; rho < 1 takes the
    bounded path with logits near +-58, rho > 1 the exact path, and rho = 2.8 puts logits at +-163, past the range in
    which ex2_poly_x2's exponent add is valid."""
    rhos = [0.5, 0.9, 0.97, 0.99, 1.01, 1.05, 1.5, 2.0, 2.8]
    B, H, dh = 3, len(rhos), 64
    scale = 0.125
    g = torch.Generator().manual_seed(N)
    q = torch.zeros(B, N, H, dh)
    k = torch.zeros(B, N, H, dh)
    for h, rho in enumerate(rhos):
        L = 64 * rho / 1.1                         # the largest logit: c r^2 with |u| = 1
        r = math.sqrt(L / (scale * LOG2E))
        rq = r * (0.5 + 0.5 * torch.rand((B, N), generator=g))
        rq[:, 0] = r
        sq = torch.randint(2, (B, N), generator=g) * 2 - 1
        sk = torch.randint(2, (B, N), generator=g) * 2 - 1
        q[:, :, h, :] = (sq * rq)[..., None] / 8
        rk = r * (0.9 + 0.1 * torch.rand((B, N), generator=g))
        rk[:, 0] = r
        k[:, :, h, :] = (sk * rk)[..., None] / 8
    q, k = bf16_exact(q).float(), bf16_exact(k).float()
    v = random_qkv(B, N, H, dh, seed=N + 1)[2]
    ops = operands(q, k, v)
    ref, bound, _ = reference(as_bhnd(q), as_bhnd(k), as_bhnd(v), scale, 1)
    for mode in (1, 0):
        with attn_bound(mode):
            got = flash(ops, scale)
        for h, rho in enumerate(rhos):
            assert_within(got[:, h:h + 1], ref[:, h:h + 1], bound[:, h:h + 1], f"rho {rho} bound mode {mode}")


# ---------------------------------------------------------------------------------------------------- E, G, H: host
def test_flash_attention_writes_only_its_rows():
    from vit.kernels import flash_attention
    B, N, H, dh = 5, 197, 3, 64
    D = H * dh
    qkv = torch.randn(B, N, 3 * D, device=dev()).bfloat16()
    buf = sentinel((B + 4, N, D), torch.bfloat16)
    flash_attention(qkv, H, out=buf[2:2 + B])
    torch.cuda.synchronize()
    assert_guard(buf, slice(2, 2 + B), "flash_attention(out=...)")
    q, k, v = (as_bhnd(t.reshape(B, N, H, dh)) for t in qkv.split(D, dim=2))
    ref, bound, _ = reference(q, k, v, 1 / 8, 1)
    assert_within(buf[2:2 + B].reshape(B, N, H, dh).permute(0, 2, 1, 3), ref, bound, "flash_attention(out=...)")


def test_flash_attention_crosses_the_host_chunk_boundary():
    """32769 images: flash_attention launches the kernel on 32768 images and then on one."""
    from vit.kernels import flash_attention
    B, N, H, dh = 32769, 2, 1, 64
    g = torch.Generator().manual_seed(2)
    qkv = torch.randn((B, N, 3 * dh), generator=g).bfloat16().to(dev())
    got = flash_attention(qkv, H)
    torch.cuda.synchronize()
    q, k, v = (as_bhnd(t.reshape(B, N, H, dh)) for t in qkv.split(dh, dim=2))
    ref, bound, _ = reference(q, k, v, 1 / 8, 1)
    assert_within(got.reshape(B, N, H, dh).permute(0, 2, 1, 3), ref, bound, "32769 images")


@pytest.mark.parametrize("N,dh", [(197, 64), (577, 64), (197, 80)])
def test_flash_attention_negative_scale(N, dh):
    """scale = -0.125 on Q, K with entries 8 {-1, 0, 1}: the logits span hundreds of log2 units, so an exponential
    taken against the scaled maximum of the raw scores (the minimum of the logits) overflows.  vt_flash_attn refuses
    the scale and flash_attention takes the composed path; its scores, multiples of 8 below 2^9, are exact in bf16,
    so the error is the composed path's own: bf16 probabilities (2^-8 relative each, the softmax's fp32 exponentials
    and normalisation 2^-20), an fp32 P V sum (N 2^-23) and the bf16 output rounding."""
    from vit.kernels import _lib, flash_attention
    B, H = 2, 2
    D = H * dh
    g = torch.Generator().manual_seed(N + dh)
    qk = 8.0 * torch.randint(-1, 2, (B, N, 2 * D), generator=g).float()
    v = torch.randn((B, N, D), generator=g)
    qkv = torch.cat([qk, v], dim=2).bfloat16().to(dev())
    got = flash_attention(qkv, H, scale=-0.125)
    torch.cuda.synchronize()
    q, k, vv = (as_bhnd(t.reshape(B, N, H, dh)) for t in qkv.split(D, dim=2))
    s = -0.125 * (q @ k.transpose(-1, -2))
    assert (s.abs() <= 512).all() and (torch.remainder(s, 8) == 0).all()
    w = torch.softmax(s, dim=-1)
    ref = w @ vv
    bound = ulp_bf16(ref) + (2 * BF16_P + 2.0 ** -20 + (N + 8) * 2.0 ** -23) * (w @ vv.abs())
    got = got.reshape(B, N, H, dh).permute(0, 2, 1, 3)
    assert torch.isfinite(got.float()).all(), "non-finite output"
    assert_within(got, ref, bound, "scale -0.125")
    out = sentinel((B, N, D), torch.bfloat16)
    base = qkv.data_ptr()
    rc = _lib.load().vt_flash_attn(base, base + 2 * D, base + 4 * D, out.data_ptr(), B, H, N, dh, 3 * D, 3 * D * N, D,
                                   D * N, -0.125, _lib.stream_ptr(qkv))
    torch.cuda.synchronize()
    assert rc == _lib.VT_ERR_UNSUPPORTED, f"vt_flash_attn took scale -0.125 (returned {rc})"
    assert_guard(out, slice(0, 0), "a refused call")
