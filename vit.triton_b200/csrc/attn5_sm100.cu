// K3 (main variant for head dim 64, single KV block): persistent fused attention forward on
// tcgen05 with TWO de-phased softmax groups over a double-buffered score tile.
//
//   ctx[b, i, h*64:(h+1)*64] = softmax_j( scale * q[b,i,h] . k[b,j,h] ) @ v[b,j,h]      (bf16, N <= 208)
//
// Replaces the reference's per-head matmul3 -> softmax -> matmul3 -> slice-assign chain
// (vit/vit.py:60-72,101-108) for all heads at once; the score matrix never leaves the SM.
//
// What the earlier variants taught (profiles/README.md): the exponentials need ~1750 cycles of MUFU
// per 128 x 208 tile and SM sub-partition, but a tile costs ~3800 cycles when the same warps walk
// "row max -> exchange -> exp -> P ready -> (MMA round trip) -> read O -> store" in lock-step
// (attn4), and ~3900 when two slots alias S, P and O in TMEM and so serialise their MMAs (attn3).
// Here the two groups run the SAME lean per-item code as attn4 but on alternate items, half a period
// apart, each on its own score buffer; all non-MUFU phases and the tensor-core round trips of one
// group (wait for O, read + store it, wait for the next scores, row max) fall into the other
// group's exp pass:
//
//   TMEM (512 columns)   S0 [0, 208)   S1 [208, 416)   O [416, 480)   row sums [480, 496)
//   item v uses S[v & 1] and belongs to group v & 1; P (bf16x2) overwrites the thread's own consumed
//   scores; O and the row sums (second N = 16 MMA against a tile of ones) are shared by both groups:
//   PV_v is issued only after group (v-1) & 1 has read O_{v-1}, half a period earlier.
//
//   A CTA walks (image, head) PAIRS; the query tiles of a pair are consecutive items (nqt = 1 or 2, one per group)
//   and share ONE K and ONE V stage (stage = pair & 1): half the operand traffic, and a stage is requested three
//   item periods before the MMA issuer needs it.
//
//   warps 0-7 / 8-15  softmax group 0 / 1: warp = 8 * group + 4 * column_half + row_quarter.  Per item:
//                     logit bound (max |q|^2, max |k|^2 from the operand tiles, while Q K^T runs) | wait S |
//                     [row max + exchange, only when the bound fails] | exp -> P | arrive P-ready — and straight on
//                     to the group's next item.  They never touch O.
//   warp 16           TMA producer (decodes the items into a shared-memory ring, allocates TMEM)
//   warp 17           MMA issuer: per item v: wait P_v, V_v, O_{v-1} read | PV_v (+ row sums) |
//                     S_{v+2} = Q K^T into S[v & 1]
//   warps 18-21       epilogue (one per TMEM lane quarter), all items in order: wait O_v | read O + row
//                     sum | release O | scale by 1 / sum, bf16, SWIZZLE_128B staging | TMA store.
//                     Round 1 had the softmax warps do this: per group and item the chain was wait-S 360 /
//                     row max 810 / exchange 140 / exp 2670 / wait-O 1000 / O read 170 / store 620 cycles,
//                     i.e. 1790 cycles in which a group's MUFU-bound exp pass could not start (two groups
//                     = 2885 cycles per item against 1664 of MUFU work); with the O path on its own warps
//                     a group's period is wait-S + max + exp and the kernel runs against the MUFU pipe.
//
// Sequences longer than 208 keys and head dim 80 run attn5mb_fwd_kernel below (online softmax over KV blocks).
#include <cstdlib>

#include "attn_softmax.cuh"
#include "common.cuh"
#include "tensormap.h"

namespace vt {

namespace {

constexpr int kDH5 = 64;
constexpr int kQTile5 = 128;
constexpr int kThreads5 = (16 + 2) * 32;               // 576: multi-block kernel (O accumulated by the softmax warps)
constexpr int kThreads5s = (16 + 2 + 4) * 32;          // 704: single-block kernel (+ 4 epilogue warps)
constexpr int kQBytes5 = kQTile5 * kDH5 * 2;           // 16 KB
constexpr int kMaxN5 = 208;
constexpr int kSCols5 = 208;                           // columns per score buffer
constexpr int kOCol5 = 2 * kSCols5;                    // 416: O (64 columns) then the row sums (16 columns)
constexpr int kLCol5 = kOCol5 + kDH5;                  // 480
constexpr int kStageBytes5 = 32 * 64 * 2;              // per epilogue warp: 32 rows x 64 bf16 (SWIZZLE_128B)
constexpr int kOnesBytes5 = 16 * 16 * 2;
constexpr int kOnesBytes5s = 16 * 128;                 // single-block kernel: 16 K rows x 128 B of ones (see the PV MMAs)
constexpr int kRing5 = 8;
constexpr int kSmemLimit5 = 232448;
// -DVT_ATTN5_EXP_TURNS=1: the two softmax groups take strict turns on the MUFU pipe (experiment, measured no
// faster: 73.9 vs 74.3 us per launch at C2 — an exp pass run ALONE by one group's 8 warps takes 2700 cycles,
// as long as the other group's P -> PV -> S round trip + row-max pass that it would hide)
#ifndef VT_ATTN5_EXP_TURNS
#define VT_ATTN5_EXP_TURNS 0
#endif
constexpr bool kExpTurns5 = VT_ATTN5_EXP_TURNS != 0;

struct Attn5Params {
  int N, H, B;
  int nqt;            // query tiles per (image, head)
  int bkv;            // key rows loaded per item (N rounded up to 16)
  long long total_items;
  int reverse;        // walk the images from the last to the first (L2 reuse, see api.cu)
  int no_bound;       // 1: every item takes the exact two-pass softmax (VT_ATTN_NO_BOUND=1, A/B and tests)
  float scale_log2;
  long long* dbg;     // cycle counters, developer build only (make EXTRA=-DVT_ATTN5_DBG, tools/attn_dbg.py)
};

enum { C_QFULL = 0, C_QEMPTY = 2, C_KFULL = 4, C_KEMPTY = 6, C_VFULL = 8, C_VEMPTY = 10, C_SFULL = 12,
       C_PFULL = 14, C_OFULL = 16, C_OREAD = 18, C_PHALF = 19, C_XTOK = 21, C_NBARS = 23 };
// C_XTOK + g: the exp pass of group g's next item may start (the other group has finished the exp pass of the
// item before it): the two groups take turns on the MUFU pipe, see the softmax warps of attn5_fwd_kernel.
// C_PHALF (experiment, -DVT_ATTN5_SPLIT): the first (up to) four 16-column groups of every softmax
// warp's P are in TMEM — the MMA issuer starts O = P V on those keys while the second part of the exp
// pass is still running.  Measured SLOWER (79.6 vs 75.0 us per launch at C2): the mid-pass
// tcgen05.wait::st + fence + arrive costs the exp pass more than the shorter wait for O gives back.
[[maybe_unused]] constexpr int kSplitGroups5 = 4;

__device__ __noinline__ void mbar_wait_slow5(uint32_t bar, uint32_t parity) { mbar_wait(bar, parity); }
__device__ __forceinline__ void mbar_wait_lean5(uint32_t bar, uint32_t parity) {
  if (!mbar_try_wait(bar, parity)) mbar_wait_slow5(bar, parity);
}

// Row max over NG (1..7) groups of 16 score columns starting at TMEM address a.  Only the first nv
// of the 16 * NG columns are real keys; nj - N < 16, so at most the LAST group is partly masked.
// Groups are loaded in pairs, the next pair is in flight while the current one is folded.  (One
// 64-column load + the rest was measured much slower: 94 vs 76 us per launch at C2.)
template <int NG>
__device__ __forceinline__ float max_groups5(uint32_t a, int nv) {
  constexpr int kPairs = (NG + 1) / 2;
  float m0 = -INFINITY, m1 = -INFINITY;
  uint32_t r[kPairs][2][16];
  auto load_pair = [&](int pr) {
    tmem_ld_32x16(a + 32 * pr, r[pr][0]);
    if (2 * pr + 1 < NG) tmem_ld_32x16(a + 32 * pr + 16, r[pr][1]);
  };
  load_pair(0);
#pragma unroll
  for (int pr = 0; pr < kPairs; ++pr) {
    tmem_ld_wait();
    if (pr + 1 < kPairs) load_pair(pr + 1);
#pragma unroll
    for (int h = 0; h < 2; ++h) {
      const int g = 2 * pr + h;
      if (g < NG) {
        if (g < NG - 1 || nv >= 16 * NG) {     // warp-uniform
#pragma unroll
          for (int i = 0; i < 16; i += 4) {
            m0 = fmax3(m0, __uint_as_float(r[pr][h][i]), __uint_as_float(r[pr][h][i + 1]));
            m1 = fmax3(m1, __uint_as_float(r[pr][h][i + 2]), __uint_as_float(r[pr][h][i + 3]));
          }
        } else {
#pragma unroll
          for (int i = 0; i < 16; ++i)
            if (16 * g + i < nv) m0 = fmaxf(m0, __uint_as_float(r[pr][h][i]));
        }
      }
    }
  }
  return fmaxf(m0, m1);
}

// exp2 of two BOUNDED arguments (|x| <= 64: the bounded-logit path) on the FMA pipe instead of the MUFU:
// x = n + f with n = rint(x) read out of the mantissa of x + 1.5 * 2^23, 2^f by a degree-3 polynomial on
// [-0.5, 0.5] (max relative error 7.52e-5, far below the bf16 rounding of P; valid for -126 < x < 128,
// tests/test_abi_attn.py), 2^n added into the exponent field.
// Six packed-fp32 instructions + two integer ones per pair against two MUFU slots (16 cycles of the
// quarter-rate pipe): VT_ATTN5_POLY pairs of every eight take this route.
__device__ __forceinline__ float2 ex2_poly_x2(float2 x) {
  const float2 magic = make_float2(12582912.0f, 12582912.0f);
  const float2 xf = __fadd2_rn(x, magic);
  const float2 n = __fadd2_rn(xf, make_float2(-12582912.0f, -12582912.0f));
  const float2 f = __ffma2_rn(n, make_float2(-1.0f, -1.0f), x);
  float2 p = __ffma2_rn(f, make_float2(0.055170852690935135f, 0.055170852690935135f),
                        make_float2(0.2426093965768814f, 0.2426093965768814f));
  p = __ffma2_rn(p, f, make_float2(0.6932609677314758f, 0.6932609677314758f));
  p = __ffma2_rn(p, f, make_float2(0.9999281764030457f, 0.9999281764030457f));
  return make_float2(__uint_as_float(__float_as_uint(p.x) + (__float_as_uint(xf.x) << 23)),
                     __uint_as_float(__float_as_uint(p.y) + (__float_as_uint(xf.y) << 23)));
}
// Measured at C2 / C4 in isolation (us per launch, two A/B rounds on one box): 0 pairs 70.9 / 49.1, 2 pairs 69.8 / 48.4,
// 3 pairs 69.0 / 47.8, 4 pairs 70.7 / 48.7 (the FMA side becomes the longer one) — and INSIDE the power-capped C2
// forward, where the SM clock is 1.2 instead of 1.9 GHz and the kernel is bound by instruction issue rather than by HBM
// latency (ms per forward over 100 graph replays, three rounds on one box): 1 pair 8.622, 2 pairs 8.588 - 8.628,
// 3 pairs 8.664, 4 pairs 8.708, 5 pairs 8.775; 0 pairs 9.020 against 8.940 for 3 pairs on another box.  Two it is.
#ifndef VT_ATTN5_POLY
#define VT_ATTN5_POLY 2
#endif

// one group: p = exp2(s * scale - m) -> bf16x2 -> TMEM columns dst .. dst + 7
template <bool MASKED, bool BOUNDED = false>
__device__ __forceinline__ void exp_group5(const uint32_t (&r)[16], uint32_t dst, int nv_in_group, float scale_log2,
                                           float m) {
  uint32_t pk[8];
  const float2 sc2 = make_float2(scale_log2, scale_log2), nm2 = make_float2(-m, -m);
#pragma unroll
  for (int i = 0; i < 16; i += 2) {
    // one FFMA2 (sm_100 f32x2) for the two arguments
    const float2 a2 = __ffma2_rn(make_float2(__uint_as_float(r[i]), __uint_as_float(r[i + 1])), sc2, nm2);
    float p0, p1;
    if (BOUNDED && VT_ATTN5_POLY > 0 && (8 - (i >> 1)) <= VT_ATTN5_POLY) {   // the last VT_ATTN5_POLY pairs of the group
      const float2 pp = ex2_poly_x2(a2);
      p0 = pp.x;
      p1 = pp.y;
    } else {
      p0 = ex2_approx(a2.x);
      p1 = ex2_approx(a2.y);
    }
    if (MASKED) {
      if (i >= nv_in_group) p0 = 0.f;
      if (i + 1 >= nv_in_group) p1 = 0.f;
    }
    pk[i >> 1] = pack_bf16x2(p0, p1);
  }
  tmem_st_32x8(dst, pk);
}

// p = exp2(s * scale - m) over the same NG groups; P (bf16x2) of group g overwrites TMEM columns
// a + 8g .. a + 8g + 7 (scores this thread has already consumed).  Groups are loaded in pairs, the
// next pair is in flight during the math of the current one.
template <int NG, bool BOUNDED = false>
__device__ __forceinline__ void exp_groups5(uint32_t a, int nv, float scale_log2, float m, uint32_t half_bar,
                                            int lane) {
  constexpr int kPairs = (NG + 1) / 2;
  uint32_t r[kPairs][2][16];
  auto load_pair = [&](int pr) {
    tmem_ld_32x16(a + 32 * pr, r[pr][0]);
    if (2 * pr + 1 < NG) tmem_ld_32x16(a + 32 * pr + 16, r[pr][1]);
  };
  load_pair(0);
#pragma unroll
  for (int pr = 0; pr < kPairs; ++pr) {
    tmem_ld_wait();
    if (pr + 1 < kPairs) load_pair(pr + 1);
#pragma unroll
    for (int h = 0; h < 2; ++h) {
      const int g = 2 * pr + h;
      if (g < NG) {
        if (g < NG - 1 || nv >= 16 * NG)
          exp_group5<false, BOUNDED>(r[pr][h], a + 8 * g, 16, scale_log2, m);
        else
          exp_group5<true, BOUNDED>(r[pr][h], a + 8 * g, nv - 16 * (NG - 1), scale_log2, m);
      }
    }
#ifdef VT_ATTN5_SPLIT
    if (pr == (kPairs >= 2 ? 1 : 0)) {   // min(NG, kSplitGroups5) groups of P are written: hand them over
      tmem_st_wait();
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive(half_bar);
    }
#endif
  }
  tmem_st_wait();
}

// |row|^2 of one 64-element bf16 row (128 B) of a SWIZZLE_128B tile, packed bf16x2 FMAs on four chains (the
// result only feeds a bound with a 10 % margin).  Chunk order is rotated by the row's swizzle phase so that
// the 32 lanes of a warp (32 consecutive rows) spread over all banks.
__device__ __forceinline__ float row_sumsq_bf16x64(uint32_t row_addr, int sw) {
  uint32_t acc[4] = {0u, 0u, 0u, 0u};
#pragma unroll
  for (int j = 0; j < 8; ++j) {
    uint32_t x[4];
    asm volatile("ld.shared.v4.u32 {%0, %1, %2, %3}, [%4];"
                 : "=r"(x[0]), "=r"(x[1]), "=r"(x[2]), "=r"(x[3])
                 : "r"(row_addr + (static_cast<uint32_t>(j ^ sw) << 4)));
#pragma unroll
    for (int i = 0; i < 4; ++i) asm("fma.rn.bf16x2 %0, %1, %1, %0;" : "+r"(acc[i]) : "r"(x[i]));
  }
  float t = 0.f;
#pragma unroll
  for (int i = 0; i < 4; ++i) t += bf16_lo(acc[i]) + bf16_hi(acc[i]);
  return t;
}

// Logits bounded by Cauchy-Schwarz: |scale_log2 * q.k| <= kLogitBound5 for every (query, key) of the item means
// exp2 needs no shift (softmax is shift-invariant; fp32 / bf16 hold 2^+-64 with room for the row sum and P.V),
// so the row-max pass and the exchange between the two column halves are skipped (see the softmax warps).
constexpr float kLogitBound5 = 64.0f;
constexpr float kBoundMargin5 = 1.21f;     // (1.1)^2 on the squared norms: bf16 accumulation of the sums of squares

__global__ void __launch_bounds__(kThreads5s, 1)
attn5_fwd_kernel(const __grid_constant__ CUtensorMap tma_q, const __grid_constant__ CUtensorMap tma_k,
                 const __grid_constant__ CUtensorMap tma_v, const __grid_constant__ CUtensorMap tma_o,
                 const Attn5Params p) {
  extern __shared__ uint8_t smem_raw[];
  const uint32_t smem_base = (smem_u32(smem_raw) + 1023u) & ~1023u;
  uint8_t* smem_gen = smem_raw + (smem_base - smem_u32(smem_raw));

  const int kv_bytes = p.bkv * kDH5 * 2;
  // [Q0][Q1][K0][K1][V0][V1][staging 4 x 4 KB][ones][barriers][tmem slot][item ring][row max exchange]
  const uint32_t q_smem = smem_base;
  const uint32_t k_smem = q_smem + 2 * kQBytes5;
  const uint32_t v_smem = k_smem + 2 * kv_bytes;
  const int stage_off = 2 * kQBytes5 + 4 * kv_bytes;
  const uint32_t stage_smem = smem_base + stage_off;
  const int ones_off = stage_off + 4 * kStageBytes5;
  const uint32_t ones_smem = smem_base + ones_off;
  const int bar_off = ones_off + kOnesBytes5s;
  const uint32_t bar_base = smem_base + bar_off;
  const uint32_t tmem_slot = bar_base + 8u * C_NBARS;
  const int slot_off = bar_off + 8 * C_NBARS;
  volatile uint32_t* tmem_slot_gen = reinterpret_cast<volatile uint32_t*>(smem_gen + slot_off);
  int4* ring = reinterpret_cast<int4*>(smem_gen + slot_off + 8);                 // [kRing5] (16-byte aligned)
  float* xm = reinterpret_cast<float*>(smem_gen + slot_off + 8 + 16 * kRing5);   // [2 groups][2 halves][128]
  uint32_t* nrm = reinterpret_cast<uint32_t*>(xm + 2 * 2 * kQTile5);             // [2 groups][2 items][q | k][8 warps]
  auto bar = [&](int i) { return bar_base + 8u * i; };

  const int warp_idx = threadIdx.x >> 5;
  const int lane = threadIdx.x & 31;

  if (warp_idx == 17 && lane == 0) {
    for (int i = 0; i < C_NBARS; ++i)
      mbar_init(bar(i), (i == C_PFULL || i == C_PFULL + 1 || i == C_PHALF || i == C_PHALF + 1 || i == C_XTOK ||
                         i == C_XTOK + 1)       ? 8
                        : (i == C_QEMPTY || i == C_QEMPTY + 1)
                            ? 9     // tcgen05.commit of Q K^T + the 8 softmax warps of the group (norm reads)
                        : (i == C_KEMPTY || i == C_KEMPTY + 1) ? 9 * p.nqt     // the same from every item of the pair
                        : (i == C_VEMPTY || i == C_VEMPTY + 1) ? p.nqt         // tcgen05.commit of P V of every item
                        : (i == C_OREAD) ? 4
                                         : 1);
    fence_barrier_init();
    tma_prefetch_desc(&tma_q);
    tma_prefetch_desc(&tma_k);
    tma_prefetch_desc(&tma_v);
    tma_prefetch_desc(&tma_o);
  }
  if (warp_idx == 0) {   // the tile of ones behind the row sums (read through the async proxy)
#pragma unroll
    for (int i = 0; i < kOnesBytes5s / 16 / 32; ++i)
      reinterpret_cast<uint4*>(smem_gen + ones_off)[lane + 32 * i] =
          make_uint4(0x3F803F80u, 0x3F803F80u, 0x3F803F80u, 0x3F803F80u);
    fence_proxy_async_smem();
  }
  if (warp_idx == 16) {
    tmem_alloc<512>(tmem_slot);
    tmem_relinquish();
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot_gen;
  pdl_wait();                 // (VT_PDL) the QKV GEMM's output is read from here on
  pdl_launch_dependents();

  // Work list of this CTA: (image, head) pairs blockIdx.x, blockIdx.x + grid, ...; a pair is nqt (1 or 2) items,
  // its query tiles, which follow each other in the item sequence and SHARE one K and one V tile: item `it`
  // uses Q buffer / score buffer / softmax group it & 1 and K/V stage (it >> kv_shift) & 1.  (Round 2 first loaded
  // K and V per item: twice the operand traffic, and with two stages per operand the in-order producer could
  // request an item's K only ~1.3 item periods ahead — the MMA issuer waited 500 cycles per item for Q/K and
  // 190 for V.  A shared stage is requested three periods ahead.)
  const long long total_pairs = p.total_items / p.nqt;
  const long long first_pair = blockIdx.x;
  const long long pair_step = gridDim.x;
  const int n_pairs = (total_pairs > first_pair)
                          ? static_cast<int>((total_pairs - first_pair + pair_step - 1) / pair_step)
                          : 0;
  const int kv_shift = p.nqt == 2 ? 1 : 0;
  const int n_items = n_pairs << kv_shift;
  const int nj = (p.N + 15) & ~15;     // score columns (MMA N)
  const int n16 = nj >> 4;             // 16-column groups: half 0 takes the first (n16 + 1) / 2
  const int ng0 = (n16 + 1) >> 1;

  if (warp_idx == 16) {
    // ------------------------------------------------------------------ TMA producer
    for (int it = 0; it < n_items; ++it) {
      const int kvi = it >> kv_shift;                       // K/V stage use counter = local pair index
      const int qt = it & (p.nqt - 1);
      const unsigned bh = static_cast<unsigned>(first_pair + static_cast<long long>(kvi) * pair_step);
      const int head = static_cast<int>(bh % static_cast<unsigned>(p.H));
      int img = static_cast<int>(bh / static_cast<unsigned>(p.H));
      if (p.reverse) img = p.B - 1 - img;
      const int b = it & 1;
      const uint32_t ph = (static_cast<uint32_t>(it) >> 1) & 1u;
      const int s = kvi & 1;
      const uint32_t kph = (static_cast<uint32_t>(kvi) >> 1) & 1u;
      mbar_wait(bar(C_QEMPTY + b), ph ^ 1u);
      if (elect_one_sync()) {
        // item coordinates for the softmax warps: visible to them through the barrier chain
        // C_QFULL -> (MMA issuer) -> C_SFULL; the ring is deeper than the producer can run ahead
        ring[it & (kRing5 - 1)] = make_int4(img, head, qt, 0);
        mbar_arrive_expect_tx(bar(C_QFULL + b), kQBytes5);
        tma_load_3d(&tma_q, bar(C_QFULL + b), q_smem + b * kQBytes5, head * kDH5, qt * kQTile5, img, kEvictFirst);
      }
      __syncwarp();
      if (qt == 0) {              // first item of the pair: its K tile
        mbar_wait(bar(C_KEMPTY + s), kph ^ 1u);
        if (elect_one_sync()) {
          mbar_arrive_expect_tx(bar(C_KFULL + s), kv_bytes);
          tma_load_3d(&tma_k, bar(C_KFULL + s), k_smem + s * kv_bytes, head * kDH5, 0, img, kEvictFirst);
        }
        __syncwarp();
      }
      if (qt == p.nqt - 1) {      // last item of the pair: its V tile (behind the pair's query tiles)
        mbar_wait(bar(C_VEMPTY + s), kph ^ 1u);
        if (elect_one_sync()) {
          mbar_arrive_expect_tx(bar(C_VFULL + s), kv_bytes);
          tma_load_3d(&tma_v, bar(C_VFULL + s), v_smem + s * kv_bytes, head * kDH5, 0, img, kEvictFirst);
        }
        __syncwarp();
      }
    }
  } else if (warp_idx == 17) {
    // ------------------------------------------------------------------ MMA issuer
    // S_v = Q K^T into score buffer v & 1 (free: PV_{v-2}, issued earlier by this thread, is the last
    // reader of that buffer and tcgen05.mma executes in issue order).
#ifdef VT_ATTN5_DBG
    unsigned macc[6] = {0, 0, 0, 0, 0, 0};
    unsigned mt = static_cast<unsigned>(clock());
#define VT_MTICK(i) { const unsigned t_ = static_cast<unsigned>(clock()); macc[i] += t_ - mt; mt = t_; }
#else
#define VT_MTICK(i)
#endif
    auto issue_scores = [&](int v) {
      const int b = v & 1;
      const uint32_t ph = (static_cast<uint32_t>(v) >> 1) & 1u;
      const int kvi = v >> kv_shift;
      const int s = kvi & 1;
      VT_MTICK(3)
      mbar_wait(bar(C_QFULL + b), ph);
      mbar_wait(bar(C_KFULL + s), (static_cast<uint32_t>(kvi) >> 1) & 1u);
      VT_MTICK(4)
      tc_fence_after();
      if (elect_one_sync()) {
        const uint32_t idesc = make_idesc_bf16(kQTile5, nj, 0, 0);
        const uint64_t qd = make_desc_kmajor_sw128(q_smem + b * kQBytes5);
        const uint64_t kd = make_desc_kmajor_sw128(k_smem + s * kv_bytes);
#pragma unroll
        for (int k = 0; k < kDH5 / 16; ++k)
          umma_ss(tmem_base + b * kSCols5, qd + 2 * k, kd + 2 * k, idesc, k != 0 ? 1u : 0u);
        umma_commit(bar(C_SFULL + b));
        umma_commit(bar(C_KEMPTY + s));     // one of the nqt commits + 8 nqt norm-read arrivals that free the stage
        umma_commit(bar(C_QEMPTY + b));
      }
      __syncwarp();
    };
    if (n_items > 0) issue_scores(0);
    if (n_items > 1) issue_scores(1);
#ifdef VT_ATTN5_DBG
    for (int i = 0; i < 6; ++i) macc[i] = 0;
    mt = static_cast<unsigned>(clock());
#endif
    for (int v = 0; v < n_items; ++v) {
      const int b = v & 1;
      const uint32_t ph = (static_cast<uint32_t>(v) >> 1) & 1u;
      const int kvi = v >> kv_shift;
      const int vs = kvi & 1;                  // V stage of the item's pair
      // ---- O_v = P_v V_v and the row sums P_v 1
      mbar_wait(bar(C_VFULL + vs), (static_cast<uint32_t>(kvi) >> 1) & 1u);
      VT_MTICK(0)
      if (v > 0) mbar_wait(bar(C_OREAD), static_cast<uint32_t>(v - 1) & 1u);   // O columns free
      VT_MTICK(1)
      // ONE MMA per 16 keys, N = 80: the B operand is MN-major with two 64-element groups, the V tile and —
      // one leading-byte-offset further — a tile of ones whose first 16 columns give the row sums, which
      // land in the 16 TMEM columns right behind O.  (Round 1 issued a second N = 16 MMA per step; the
      // issuer spent 1489 cycles per item on 26 + 4 MMAs, ~50 each whatever their N, and the P -> PV -> S
      // round trip is on each softmax group's critical path.)  The ones tile is 16 K rows x 128 B; every
      // element is 1, so its swizzle is moot, and the per-step descriptor re-bases LBO onto it.
      const uint32_t idesc = make_idesc_bf16(kQTile5, kDH5 + 16, 0, 1);
      const uint32_t v_tile = v_smem + vs * kv_bytes;
      const uint32_t s_tmem = tmem_base + b * kSCols5;
      // 16 keys: 8 packed P columns, 2048 B of V.  P of group k lives at the start of its owner's
      // columns: half 0 owns groups [0, ng0)
      auto pv_step = [&](int k, uint32_t acc) {
        const uint32_t a_tmem = s_tmem + (k < ng0 ? 8 * k : 16 * ng0 + 8 * (k - ng0));
        const uint32_t v_k = v_tile + 2048u * k;
        umma_ts(tmem_base + kOCol5, a_tmem, make_desc_mnmajor_sw128(v_k, ones_smem - v_k), idesc, acc);
      };
#ifdef VT_ATTN5_SPLIT
      // first part: the (up to) four leading groups of each column half, ready half-way through the exp pass
      const int na0 = ng0 < kSplitGroups5 ? ng0 : kSplitGroups5;
      const int na1 = (n16 - ng0) < kSplitGroups5 ? (n16 - ng0) : kSplitGroups5;
      mbar_wait(bar(C_PHALF + b), ph);
      tc_fence_after();
      if (elect_one_sync()) {
        for (int k = 0; k < na0; ++k) pv_step(k, k != 0 ? 1u : 0u);
        for (int k = ng0; k < ng0 + na1; ++k) pv_step(k, 1u);
      }
      __syncwarp();
      mbar_wait(bar(C_PFULL + b), ph);
      VT_MTICK(2)
      tc_fence_after();
      if (elect_one_sync()) {
        for (int k = na0; k < ng0; ++k) pv_step(k, 1u);
        for (int k = ng0 + na1; k < n16; ++k) pv_step(k, 1u);
        umma_commit(bar(C_OFULL + b));
        umma_commit(bar(C_VEMPTY + vs));
      }
      __syncwarp();
#else
      mbar_wait(bar(C_PFULL + b), ph);
      VT_MTICK(2)
      tc_fence_after();
      if (elect_one_sync()) {
        for (int k = 0; k < n16; ++k) pv_step(k, k != 0 ? 1u : 0u);
        umma_commit(bar(C_OFULL + b));
        umma_commit(bar(C_VEMPTY + vs));
      }
      __syncwarp();
#endif
      if (v + 2 < n_items) issue_scores(v + 2);
      VT_MTICK(5)
    }
#ifdef VT_ATTN5_DBG
    if (p.dbg != nullptr && lane == 0) {
      long long* d = p.dbg + (2LL * gridDim.x + blockIdx.x) * 8;
      for (int i = 0; i < 6; ++i) d[i] = macc[i];
    }
#endif
#undef VT_MTICK
  } else if (warp_idx >= 18) {
    // ------------------------------------------------------------------ epilogue warps (O path)
    const int rq = warp_idx & 3;             // TMEM lane quarter this warp may read
    const int ew = warp_idx - 18;            // staging tile
    const uint32_t t_lane = tmem_base + (static_cast<uint32_t>(rq * 32) << 16);
    const uint32_t stage_addr = stage_smem + ew * kStageBytes5;
    uint8_t* stage_row = smem_gen + stage_off + ew * kStageBytes5 + lane * 128;
    const int sw = lane & 7;                 // SWIZZLE_128B phase of this thread's staging row
    for (int v = 0; v < n_items; ++v) {
      const int b = v & 1;
      const uint32_t ph = (static_cast<uint32_t>(v) >> 1) & 1u;
      // the previous store out of my staging tile has long been read: check now, off the critical path
      if (lane == 0) tma_store_wait_read<0>();
      mbar_wait_lean5(bar(C_OFULL + b), ph);
      tc_fence_after();
      const int4 desc = ring[v & (kRing5 - 1)];   // (image, head, query tile)
      const bool live = desc.z * kQTile5 + rq * 32 < p.N;      // warp-uniform
      uint32_t pk[32];                            // my row's 64 output columns as bf16 pairs
      if (live) {
        uint32_t rl[8];
        tmem_ld_32x8(t_lane + kLCol5, rl);        // every one of the 16 sum columns holds the row sum
        uint32_t r[32];
        tmem_ld_32x32(t_lane + kOCol5, r);
        tmem_ld_wait();
        float inv;
        asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(inv) : "f"(__uint_as_float(rl[0])));
        const float2 inv2 = make_float2(inv, inv);
#pragma unroll
        for (int i = 0; i < 32; i += 2) {
          const float2 o = __fmul2_rn(make_float2(__uint_as_float(r[i]), __uint_as_float(r[i + 1])), inv2);
          pk[i >> 1] = pack_bf16x2(o.x, o.y);
        }
        tmem_ld_32x32(t_lane + kOCol5 + 32, r);
        tmem_ld_wait();
#pragma unroll
        for (int i = 0; i < 32; i += 2) {
          const float2 o = __fmul2_rn(make_float2(__uint_as_float(r[i]), __uint_as_float(r[i + 1])), inv2);
          pk[16 + (i >> 1)] = pack_bf16x2(o.x, o.y);
        }
      }
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive(bar(C_OREAD));   // O and the row sums are in registers: PV of the next item may go
      if (!live) continue;
      // stage this warp's [32 rows x 64 columns] as a SWIZZLE_128B tile and TMA-store it (the staging tile
      // is free: lane 0 waited for the previous store above, the __syncwarp ordered that before these writes)
#pragma unroll
      for (int jj = 0; jj < 8; ++jj)
        *reinterpret_cast<uint4*>(stage_row + ((jj ^ sw) << 4)) =
            make_uint4(pk[4 * jj], pk[4 * jj + 1], pk[4 * jj + 2], pk[4 * jj + 3]);
      fence_proxy_async_smem();
      __syncwarp();
      if (lane == 0) {
        asm volatile("cp.async.bulk.tensor.3d.global.shared::cta.bulk_group [%0, {%2, %3, %4}], [%1];"
                     :
                     : "l"(reinterpret_cast<uint64_t>(&tma_o)), "r"(stage_addr), "r"(desc.y * kDH5),
                       "r"(desc.z * kQTile5 + rq * 32), "r"(desc.x)
                     : "memory");
        tma_store_commit();
      }
    }
    if (lane == 0) tma_store_wait<0>();
  } else {
    // ------------------------------------------------------------------ softmax warps
    const int g = warp_idx >> 3;             // group = score buffer = item parity
    const int half = (warp_idx >> 2) & 1;    // column half
    const int rq = warp_idx & 3;             // row quarter = TMEM lane group
    const int row_in_tile = rq * 32 + lane;
    const uint32_t t_lane = tmem_base + (static_cast<uint32_t>(rq * 32) << 16);
    const int bar_id = 1 + g * 4 + rq;       // named barrier of the two warps sharing these rows
    float* x_mine = xm + (g * 2 + half) * kQTile5 + row_in_tile;
    const float* x_other = xm + (g * 2 + (half ^ 1)) * kQTile5 + row_in_tile;
    // my columns: 16-column groups [g0, g0 + ng)
    const int ng = half ? (n16 - ng0) : ng0;
    const int c0 = half ? 16 * ng0 : 0;
    const int nvr = p.N - c0;                // valid columns counted from my first
    const uint32_t t_mine = t_lane + g * kSCols5 + c0;

#ifdef VT_ATTN5_DBG
    const bool dbg_on = p.dbg != nullptr;
    unsigned dacc[7] = {0, 0, 0, 0, 0, 0, 0};
    const unsigned dt0 = static_cast<unsigned>(clock());
    unsigned tc = 0;
#define VT_TICK5(i) if (dbg_on) { const unsigned t_ = static_cast<unsigned>(clock()); dacc[i] += t_ - tc; tc = t_; }
#define VT_TICK5_START() if (dbg_on) tc = static_cast<unsigned>(clock());
#else
#define VT_TICK5(i)
#define VT_TICK5_START()
#endif
    // Logit bound (see kLogitBound5): thread tg of the group squares key row tg and (tg >= 128) query row tg - 128
    const int tg = threadIdx.x & 255;
    const int wg = warp_idx & 7;
    const int grp_bar = 9 + g;               // named barrier of the group's 256 threads
    const uint32_t q_row = q_smem + g * kQBytes5 + (tg & 127) * 128;
    const float bound_c = p.scale_log2 * p.scale_log2 * kBoundMargin5;
    uint32_t ph = 0;
    for (int v = g; v < n_items; v += 2, ph ^= 1u) {
      VT_TICK5_START()
      // ---- while Q K^T of this item runs: max |q|^2 and max |k|^2 over the item's rows, out of the operand tiles.
      // The tiles are released to the producer by the MMA's commit AND these eight warps (barrier counts 9).
      bool fast;
      {
        const int kvi = v >> kv_shift;
        const int ks = kvi & 1;
        mbar_wait_lean5(bar(C_KFULL + ks), (static_cast<uint32_t>(kvi) >> 1) & 1u);
        mbar_wait_lean5(bar(C_QFULL + g), ph);
        float k2 = 0.f, q2 = 0.f;
        if (tg < p.bkv) k2 = row_sumsq_bf16x64(k_smem + ks * kv_bytes + tg * 128, tg & 7);
        if (tg >= 128) q2 = row_sumsq_bf16x64(q_row, tg & 7);
        // non-negative floats order like their bit patterns; a NaN (sign clear) sorts above every number
        const uint32_t k2m = __reduce_max_sync(0xffffffffu, __float_as_uint(k2) & 0x7fffffffu);
        const uint32_t q2m = __reduce_max_sync(0xffffffffu, __float_as_uint(q2) & 0x7fffffffu);
        uint32_t* slot = nrm + ((g * 2 + ((v >> 1) & 1)) << 4);     // double-buffered per item of the group
        if (lane == 0) {
          slot[wg] = q2m;
          slot[8 + wg] = k2m;
          mbar_arrive(bar(C_KEMPTY + ks));
          mbar_arrive(bar(C_QEMPTY + g));
        }
        named_bar_sync(grp_bar, 256);
        const uint4 qa = *reinterpret_cast<const uint4*>(slot), qb = *reinterpret_cast<const uint4*>(slot + 4);
        const uint4 ka = *reinterpret_cast<const uint4*>(slot + 8), kb = *reinterpret_cast<const uint4*>(slot + 12);
        const uint32_t qmx = max(max(max(qa.x, qa.y), max(qa.z, qa.w)), max(max(qb.x, qb.y), max(qb.z, qb.w)));
        const uint32_t kmx = max(max(max(ka.x, ka.y), max(ka.z, ka.w)), max(max(kb.x, kb.y), max(kb.z, kb.w)));
        // (a NaN or an infinity fails the comparison: such items take the exact two-pass path)
        fast = !p.no_bound && (__uint_as_float(qmx) * __uint_as_float(kmx) * bound_c <= kLogitBound5 * kLogitBound5);
      }
      VT_TICK5(5)
      mbar_wait_lean5(bar(C_SFULL + g), ph);
      VT_TICK5(0)
      tc_fence_after();
      const int4 desc = ring[v & (kRing5 - 1)];   // (image, head, query tile)
      // warp-uniform: all 32 query rows of this warp lie beyond the sequence (N = 197: the last row
      // quarter of every second tile).  Such a warp keeps the barrier protocol and skips the work;
      // its P rows stay undefined (MMA rows are independent, the rows are never stored).
      const bool live = desc.z * kQTile5 + rq * 32 < p.N;
      if (live) {
        float m = 0.f;
        if (!fast) {   // group-uniform
          // pass 1: row max over my columns, exchanged with the other half of the row
          float mx = -INFINITY;
          switch (ng) {   // warp-uniform
            case 7: mx = max_groups5<7>(t_mine, nvr); break;
            case 6: mx = max_groups5<6>(t_mine, nvr); break;
            case 5: mx = max_groups5<5>(t_mine, nvr); break;
            case 4: mx = max_groups5<4>(t_mine, nvr); break;
            case 3: mx = max_groups5<3>(t_mine, nvr); break;
            case 2: mx = max_groups5<2>(t_mine, nvr); break;
            case 1: mx = max_groups5<1>(t_mine, nvr); break;
            default: break;
          }
          *x_mine = mx;
          VT_TICK5(1)
          named_bar_sync(bar_id, 64);
          m = fmaxf(mx, *x_other) * p.scale_log2;
          VT_TICK5(2)
        }
        // (experiment, off by default) the groups take turns on the MUFU pipe: item v's exp pass starts when
        // item v - 1's (the other group's) is over
        if (kExpTurns5 && v > 0) mbar_wait_lean5(bar(C_XTOK + g), static_cast<uint32_t>((v - 1) >> 1) & 1u);
        VT_TICK5(4)
        // pass 2: exponentials; P overwrites my own consumed scores
        if (VT_ATTN5_POLY > 0 && fast) {   // bounded arguments: part of the exponentials on the FMA pipe
          switch (ng) {
            case 7: exp_groups5<7, true>(t_mine, nvr, p.scale_log2, m, bar(C_PHALF + g), lane); break;
            case 6: exp_groups5<6, true>(t_mine, nvr, p.scale_log2, m, bar(C_PHALF + g), lane); break;
            case 5: exp_groups5<5, true>(t_mine, nvr, p.scale_log2, m, bar(C_PHALF + g), lane); break;
            case 4: exp_groups5<4, true>(t_mine, nvr, p.scale_log2, m, bar(C_PHALF + g), lane); break;
            case 3: exp_groups5<3, true>(t_mine, nvr, p.scale_log2, m, bar(C_PHALF + g), lane); break;
            case 2: exp_groups5<2, true>(t_mine, nvr, p.scale_log2, m, bar(C_PHALF + g), lane); break;
            case 1: exp_groups5<1, true>(t_mine, nvr, p.scale_log2, m, bar(C_PHALF + g), lane); break;
            default: break;
          }
        } else
        switch (ng) {
          case 7: exp_groups5<7>(t_mine, nvr, p.scale_log2, m, bar(C_PHALF + g), lane); break;
          case 6: exp_groups5<6>(t_mine, nvr, p.scale_log2, m, bar(C_PHALF + g), lane); break;
          case 5: exp_groups5<5>(t_mine, nvr, p.scale_log2, m, bar(C_PHALF + g), lane); break;
          case 4: exp_groups5<4>(t_mine, nvr, p.scale_log2, m, bar(C_PHALF + g), lane); break;
          case 3: exp_groups5<3>(t_mine, nvr, p.scale_log2, m, bar(C_PHALF + g), lane); break;
          case 2: exp_groups5<2>(t_mine, nvr, p.scale_log2, m, bar(C_PHALF + g), lane); break;
          case 1: exp_groups5<1>(t_mine, nvr, p.scale_log2, m, bar(C_PHALF + g), lane); break;
          default: break;
        }
        // the exchange slot is rewritten in this group's next item: both readers are past it (each reads
        // before it arrives on the named barrier of the next item)
      } else if (kExpTurns5 && v > 0) {
        mbar_wait_lean5(bar(C_XTOK + g), static_cast<uint32_t>((v - 1) >> 1) & 1u);   // keep the phase protocol
      }
      if (kExpTurns5) {   // hand the MUFU to the other group (item v + 1)
        __syncwarp();
        if (lane == 0) mbar_arrive(bar(C_XTOK + (g ^ 1)));
      }
      tc_fence_before();
      __syncwarp();
#ifdef VT_ATTN5_SPLIT
      if (lane == 0 && (!live || ng == 0)) mbar_arrive(bar(C_PHALF + g));   // warps that skipped the exp pass
#endif
      if (lane == 0) mbar_arrive(bar(C_PFULL + g));
      VT_TICK5(3)
    }
#ifdef VT_ATTN5_DBG
    if (dbg_on && (warp_idx & 7) == 0 && lane == 0) {
      long long* d = p.dbg + (2LL * blockIdx.x + g) * 8;
      for (int i = 0; i < 7; ++i) d[i] = dacc[i];
      d[7] = static_cast<unsigned>(clock()) - dt0;
    }
#endif
#undef VT_TICK5
#undef VT_TICK5_START
  }

  tc_fence_before();
  __syncthreads();
  if (warp_idx == 16) {
    tc_fence_after();
    tmem_dealloc<512>(tmem_base);
  }
}

// ------------------------------------------------------------------------------------------------
// Multi-block variant (N > 208: ViT-B/16 @ 384 has 577 tokens = 3 KV blocks of 208/208/161): the same
// two de-phased groups, group g owns the items of parity g and walks ALL KV blocks of an item on its
// own score buffer with the online-softmax recurrence (running max, rescale factor alpha, output
// accumulator of 32 columns per thread in registers).  A "unit" is one KV block of one item; the
// MMA issuer and the producer alternate between the two groups' unit streams.
// ------------------------------------------------------------------------------------------------
struct Attn5MbParams {
  int N, H, B;
  int nqt;
  int bkv, nblk;      // key rows per block (multiple of 16, <= 208), blocks per item (>= 2)
  long long total_items;
  int reverse;
  float scale_log2;
};

// Non-pipelined forms for the multi-block kernel: the 33 accumulator registers that stay live
// across the passes leave room for one pair of groups (32 registers) in flight, not two.
template <int NG>
__device__ __forceinline__ float max_groups5_np(uint32_t a, int nv) {
  float m0 = -INFINITY, m1 = -INFINITY;
#pragma unroll
  for (int pr = 0; pr < (NG + 1) / 2; ++pr) {
    uint32_t r[2][16];
    tmem_ld_32x16(a + 32 * pr, r[0]);
    if (2 * pr + 1 < NG) tmem_ld_32x16(a + 32 * pr + 16, r[1]);
    tmem_ld_wait();
#pragma unroll
    for (int h = 0; h < 2; ++h) {
      const int g = 2 * pr + h;
      if (g < NG) {
        if (g < NG - 1 || nv >= 16 * NG) {
#pragma unroll
          for (int i = 0; i < 16; i += 4) {
            m0 = fmax3(m0, __uint_as_float(r[h][i]), __uint_as_float(r[h][i + 1]));
            m1 = fmax3(m1, __uint_as_float(r[h][i + 2]), __uint_as_float(r[h][i + 3]));
          }
        } else {
#pragma unroll
          for (int i = 0; i < 16; ++i)
            if (16 * g + i < nv) m0 = fmaxf(m0, __uint_as_float(r[h][i]));
        }
      }
    }
  }
  return fmaxf(m0, m1);
}

template <int NG>
__device__ __forceinline__ void exp_groups5_np(uint32_t a, int nv, float scale_log2, float m) {
#pragma unroll
  for (int pr = 0; pr < (NG + 1) / 2; ++pr) {
    uint32_t r[2][16];
    tmem_ld_32x16(a + 32 * pr, r[0]);
    if (2 * pr + 1 < NG) tmem_ld_32x16(a + 32 * pr + 16, r[1]);
    tmem_ld_wait();
#pragma unroll
    for (int h = 0; h < 2; ++h) {
      const int g = 2 * pr + h;
      if (g < NG) {
        if (g < NG - 1 || nv >= 16 * NG)
          exp_group5<false>(r[h], a + 8 * g, 16, scale_log2, m);
        else
          exp_group5<true>(r[h], a + 8 * g, nv - 16 * (NG - 1), scale_log2, m);
      }
    }
  }
  tmem_st_wait();
}

// Head dim 80 (ViT-H): 160-byte rows do not fit the 128-byte swizzle, so every Q/K/V tile is a
// 64-column SWIZZLE_128B part plus a 16-column SWIZZLE_32B part ("tail"); Q K^T gets a fifth K step on
// the tails, P V a second N = 16 MMA per K step into output columns [64, 80), and the row sums move
// to TMEM columns [496, 512): O [416, 496) + sums fill the 512 columns exactly.
template <int DH>
__global__ void __launch_bounds__(kThreads5, 1)
attn5mb_fwd_kernel(const __grid_constant__ CUtensorMap tma_q, const __grid_constant__ CUtensorMap tma_k,
                   const __grid_constant__ CUtensorMap tma_v, const __grid_constant__ CUtensorMap tma_o,
                   const __grid_constant__ CUtensorMap tma_qt, const __grid_constant__ CUtensorMap tma_kt,
                   const __grid_constant__ CUtensorMap tma_vt, const Attn5MbParams p) {
  static_assert(DH == 64 || DH == 80, "head dim 64 or 80");
  constexpr int kDT = DH - kDH5;                  // 0 or 16: columns of the SWIZZLE_32B tail
  constexpr int kHalfCols = DH / 2;               // output columns per softmax thread
  constexpr int kStage = 32 * kHalfCols * 2;      // staging bytes per warp
  constexpr int kLCol = kOCol5 + DH;              // row sums
  constexpr int kQTailBytes = kQTile5 * kDT * 2;
  extern __shared__ uint8_t smem_raw[];
  const uint32_t smem_base = (smem_u32(smem_raw) + 1023u) & ~1023u;
  uint8_t* smem_gen = smem_raw + (smem_base - smem_u32(smem_raw));

  const int kv_bytes = p.bkv * kDH5 * 2;          // SWIZZLE_128B part of one K or V block
  const int kv_tail = p.bkv * kDT * 2;            // SWIZZLE_32B part
  // [Q x2][K x2][V x2][Q tails x2][K tails x2][V tails x2][staging][ones][barriers]...; buffers indexed by GROUP
  const uint32_t q_smem = smem_base;
  const uint32_t k_smem = q_smem + 2 * kQBytes5;
  const uint32_t v_smem = k_smem + 2 * kv_bytes;
  const uint32_t qt_smem = v_smem + 2 * kv_bytes;
  const uint32_t kt_smem = qt_smem + 2 * kQTailBytes;
  const uint32_t vt_smem = kt_smem + 2 * kv_tail;
  const int stage_off = 2 * kQBytes5 + 4 * kv_bytes + 2 * kQTailBytes + 4 * kv_tail;
  const uint32_t stage_smem = smem_base + stage_off;
  const int ones_off = stage_off + 16 * kStage;
  const uint32_t ones_smem = smem_base + ones_off;
  constexpr int kOnesB = (DH == kDH5) ? kOnesBytes5s : kOnesBytes5;   // dh 64: the 16 x 128 B tile behind the N = 80 PV MMA
  const int bar_off = ones_off + kOnesB;
  const uint32_t bar_base = smem_base + bar_off;
  const uint32_t tmem_slot = bar_base + 8u * C_NBARS;
  const int slot_off = bar_off + 8 * C_NBARS;
  volatile uint32_t* tmem_slot_gen = reinterpret_cast<volatile uint32_t*>(smem_gen + slot_off);
  int4* ring = reinterpret_cast<int4*>(smem_gen + slot_off + 8);
  float* xm = reinterpret_cast<float*>(smem_gen + slot_off + 8 + 16 * kRing5);
  auto bar = [&](int i) { return bar_base + 8u * i; };

  const int warp_idx = threadIdx.x >> 5;
  const int lane = threadIdx.x & 31;

  if (warp_idx == 17 && lane == 0) {
    for (int i = 0; i < C_NBARS; ++i)
      mbar_init(bar(i), (i == C_PFULL || i == C_PFULL + 1 || i == C_OREAD || i == C_PHALF || i == C_PHALF + 1) ? 8 : 1);
    fence_barrier_init();
    tma_prefetch_desc(&tma_q);
    tma_prefetch_desc(&tma_k);
    tma_prefetch_desc(&tma_v);
    tma_prefetch_desc(&tma_o);
    if (kDT) {
      tma_prefetch_desc(&tma_qt);
      tma_prefetch_desc(&tma_kt);
      tma_prefetch_desc(&tma_vt);
    }
  }
  if (warp_idx == 0) {
#pragma unroll
    for (int i = 0; i < kOnesB / 16 / 32; ++i)
      reinterpret_cast<uint4*>(smem_gen + ones_off)[lane + 32 * i] =
          make_uint4(0x3F803F80u, 0x3F803F80u, 0x3F803F80u, 0x3F803F80u);
    fence_proxy_async_smem();
  }
  if (warp_idx == 16) {
    tmem_alloc<512>(tmem_slot);
    tmem_relinquish();
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot_gen;
  pdl_wait();
  pdl_launch_dependents();

  const long long first_item = blockIdx.x;
  const long long item_step = gridDim.x;
  const int n_items = (p.total_items > first_item)
                          ? static_cast<int>((p.total_items - first_item + item_step - 1) / item_step)
                          : 0;
  const int nblk = p.nblk;
  const int bkv = p.bkv;
  // items of group g: g, g + 2, ...; its unit stream has n_items_g * nblk entries
  const int units0 = ((n_items + 1) >> 1) * nblk;
  const int units1 = (n_items >> 1) * nblk;
  // the two block shapes: blocks 0 .. nblk-2 have bkv keys, the last one the rest
  const int nv_last = p.N - (nblk - 1) * bkv;
  const int nj_full = bkv;
  const int nj_last = (nv_last + 15) & ~15;

  if (warp_idx == 16) {
    // ------------------------------------------------------------------ TMA producer
    // pairs of items (one per group), their blocks interleaved so neither group waits for the other
    for (int it0 = 0; it0 < n_items; it0 += 2) {
      int img[2], head[2];
#pragma unroll
      for (int g = 0; g < 2; ++g) {
        const int it = it0 + g;
        if (it >= n_items) continue;
        const unsigned item = static_cast<unsigned>(first_item + static_cast<long long>(it) * item_step);
        const int qt = static_cast<int>(item % static_cast<unsigned>(p.nqt));
        const unsigned bh = item / static_cast<unsigned>(p.nqt);
        head[g] = static_cast<int>(bh % static_cast<unsigned>(p.H));
        img[g] = static_cast<int>(bh / static_cast<unsigned>(p.H));
        if (p.reverse) img[g] = p.B - 1 - img[g];
        const uint32_t ph = (static_cast<uint32_t>(it0) >> 1) & 1u;   // group-local item index = it0 / 2
        mbar_wait(bar(C_QEMPTY + g), ph ^ 1u);
        if (elect_one_sync()) {
          ring[it & (kRing5 - 1)] = make_int4(img[g], head[g], qt, 0);
          mbar_arrive_expect_tx(bar(C_QFULL + g), kQBytes5 + kQTailBytes);
          tma_load_3d(&tma_q, bar(C_QFULL + g), q_smem + g * kQBytes5, head[g] * DH, qt * kQTile5, img[g], kEvictFirst);
          if (kDT)
            tma_load_3d(&tma_qt, bar(C_QFULL + g), qt_smem + g * kQTailBytes, head[g] * DH + kDH5, qt * kQTile5, img[g],
                        kEvictFirst);
        }
        __syncwarp();
      }
      for (int j = 0; j < nblk; ++j) {
        const uint32_t ph = static_cast<uint32_t>((it0 >> 1) * nblk + j) & 1u;   // group-local unit index
#pragma unroll
        for (int g = 0; g < 2; ++g) {
          if (it0 + g >= n_items) continue;
          mbar_wait(bar(C_KEMPTY + g), ph ^ 1u);
          if (elect_one_sync()) {
            mbar_arrive_expect_tx(bar(C_KFULL + g), kv_bytes + kv_tail);
            tma_load_3d(&tma_k, bar(C_KFULL + g), k_smem + g * kv_bytes, head[g] * DH, j * bkv, img[g], kEvictNormal);
            if (kDT)
              tma_load_3d(&tma_kt, bar(C_KFULL + g), kt_smem + g * kv_tail, head[g] * DH + kDH5, j * bkv, img[g], kEvictNormal);
          }
          __syncwarp();
          mbar_wait(bar(C_VEMPTY + g), ph ^ 1u);
          if (elect_one_sync()) {
            mbar_arrive_expect_tx(bar(C_VFULL + g), kv_bytes + kv_tail);
            tma_load_3d(&tma_v, bar(C_VFULL + g), v_smem + g * kv_bytes, head[g] * DH, j * bkv, img[g], kEvictNormal);
            if (kDT)
              tma_load_3d(&tma_vt, bar(C_VFULL + g), vt_smem + g * kv_tail, head[g] * DH + kDH5, j * bkv, img[g], kEvictNormal);
          }
          __syncwarp();
        }
      }
    }
  } else if (warp_idx == 17) {
    // ------------------------------------------------------------------ MMA issuer
    // S of group g's unit lu into score buffer g (free: the PV of the group's previous unit, issued
    // earlier by this thread, is the last reader and tcgen05.mma executes in issue order).
    auto issue_scores = [&](int g, int lu) {
      const int li = lu / nblk;            // group-local item index
      const int j = lu - li * nblk;
      const int nj = (j == nblk - 1) ? nj_last : nj_full;
      if (j == 0) mbar_wait(bar(C_QFULL + g), static_cast<uint32_t>(li) & 1u);
      mbar_wait(bar(C_KFULL + g), static_cast<uint32_t>(lu) & 1u);
      tc_fence_after();
      if (elect_one_sync()) {
        const uint32_t idesc = make_idesc_bf16(kQTile5, nj, 0, 0);
        const uint64_t qd = make_desc_kmajor_sw128(q_smem + g * kQBytes5);
        const uint64_t kd = make_desc_kmajor_sw128(k_smem + g * kv_bytes);
#pragma unroll
        for (int k = 0; k < kDH5 / 16; ++k)
          umma_ss(tmem_base + g * kSCols5, qd + 2 * k, kd + 2 * k, idesc, k != 0 ? 1u : 0u);
        if (kDT)   // fifth K step on the 16-column SWIZZLE_32B tiles (rows of 32 B, 8-row atoms of 256 B)
          umma_ss(tmem_base + g * kSCols5, make_smem_desc(qt_smem + g * kQTailBytes, 0, 256, 6),
                  make_smem_desc(kt_smem + g * kv_tail, 0, 256, 6), idesc, 1u);
        umma_commit(bar(C_SFULL + g));
        umma_commit(bar(C_KEMPTY + g));
        if (j == nblk - 1) umma_commit(bar(C_QEMPTY + g));
      }
      __syncwarp();
    };
    int lu[2] = {0, 0};
    const int units[2] = {units0, units1};
    if (units0 > 0) issue_scores(0, 0);
    if (units1 > 0) issue_scores(1, 0);
    int issued = 0;
    int g = 0;
    while (lu[0] < units0 || lu[1] < units1) {
      if (lu[g] >= units[g]) g ^= 1;
      const int u = lu[g];
      const uint32_t ph = static_cast<uint32_t>(u) & 1u;
      const int j = u % nblk;
      const int nj = (j == nblk - 1) ? nj_last : nj_full;
      const int n16 = nj >> 4;
      const int ng0 = (n16 + 1) >> 1;
      mbar_wait(bar(C_VFULL + g), ph);
      if (issued > 0) mbar_wait(bar(C_OREAD), static_cast<uint32_t>(issued - 1) & 1u);   // O columns free
      mbar_wait(bar(C_PFULL + g), ph);
      tc_fence_after();
      if (elect_one_sync()) {
        const uint32_t idesc = make_idesc_bf16(kQTile5, kDH5, 0, 1);
        const uint32_t idesc_l = make_idesc_bf16(kQTile5, 16, 0, 1);
        const uint64_t vd = make_desc_mnmajor_sw128(v_smem + g * kv_bytes, 1024);
        const uint64_t od = make_smem_desc(ones_smem, 256, 256, 6);
        const uint64_t vtd = make_smem_desc(vt_smem + g * kv_tail, 256, 256, 6);   // MN-major, SWIZZLE_32B
        const uint32_t s_tmem = tmem_base + g * kSCols5;
        for (int k = 0; k < n16; ++k) {   // 16 keys: 2048 B of the main V tile, 512 B of the tail tile
          const uint32_t a_tmem = s_tmem + (k < ng0 ? 8 * k : 16 * ng0 + 8 * (k - ng0));
          if (kDT == 0) {
            // head dim 64: ONE N = 80 MMA per 16 keys — V plus, one re-based leading-byte-offset away, a tile of
            // ones whose first 16 columns give the row sums right behind O (as in attn5_fwd_kernel: the tensor pipe
            // spends ~50 cycles on an MMA this small whatever its N); 244 -> 237 us per launch at 577 tokens
            const uint32_t v_k = v_smem + g * kv_bytes + 2048u * k;
            umma_ts(tmem_base + kOCol5, a_tmem, make_desc_mnmajor_sw128(v_k, ones_smem - v_k),
                    make_idesc_bf16(kQTile5, kDH5 + 16, 0, 1), k != 0 ? 1u : 0u);
          } else {
            umma_ts(tmem_base + kOCol5, a_tmem, vd + 128 * k, idesc, k != 0 ? 1u : 0u);
            umma_ts(tmem_base + kOCol5 + kDH5, a_tmem, vtd + 32 * k, idesc_l, k != 0 ? 1u : 0u);
            umma_ts(tmem_base + kLCol, a_tmem, od, idesc_l, k != 0 ? 1u : 0u);
          }
        }
        umma_commit(bar(C_OFULL + g));
        umma_commit(bar(C_VEMPTY + g));
      }
      __syncwarp();
      ++issued;
      if (++lu[g] < units[g]) issue_scores(g, lu[g]);
      g ^= 1;
    }
  } else {
    // ------------------------------------------------------------------ softmax warps
    const int g = warp_idx >> 3;
    const int half = (warp_idx >> 2) & 1;
    const int rq = warp_idx & 3;
    const int row_in_tile = rq * 32 + lane;
    const uint32_t t_lane = tmem_base + (static_cast<uint32_t>(rq * 32) << 16);
    // [32 rows x 64 B] SWIZZLE_64B (dh 64) or [32 rows x 80 B] unswizzled (dh 80)
    const uint32_t stage_addr = stage_smem + warp_idx * kStage;
    uint8_t* stage_row = smem_gen + stage_off + warp_idx * kStage + lane * (kHalfCols * 2);
    const int sw = (kDT == 0) ? ((lane >> 1) & 3) : 0;
    const int bar_id = 1 + g * 4 + rq;
    float* x_mine = xm + (g * 2 + half) * kQTile5 + row_in_tile;
    const float* x_other = xm + (g * 2 + (half ^ 1)) * kQTile5 + row_in_tile;
    // my columns in the two block shapes
    const int n16_full = nj_full >> 4, n16_last = nj_last >> 4;
    const int ng0_full = (n16_full + 1) >> 1, ng0_last = (n16_last + 1) >> 1;
    const int ng_full = half ? (n16_full - ng0_full) : ng0_full;
    const int ng_last = half ? (n16_last - ng0_last) : ng0_last;
    const int c0_full = half ? 16 * ng0_full : 0, c0_last = half ? 16 * ng0_last : 0;
    const int units = g ? units1 : units0;

    int4 desc = make_int4(0, 0, 0, 0);
    bool live = false;
    float m_run = -INFINITY, l_acc = 0.f;
    float o_acc[kHalfCols];
    int j = 0, li = 0;
    for (int lu = 0; lu < units; ++lu) {
      const uint32_t ph = static_cast<uint32_t>(lu) & 1u;
      const bool last_blk = (j == nblk - 1);
      const int ng = last_blk ? ng_last : ng_full;
      const int c0 = last_blk ? c0_last : c0_full;
      const int nvr = (last_blk ? nv_last : nj_full) - c0;
      const uint32_t t_mine = t_lane + g * kSCols5 + c0;

      mbar_wait_lean5(bar(C_SFULL + g), ph);
      tc_fence_after();
      if (j == 0) {
        desc = ring[(2 * li + g) & (kRing5 - 1)];
        live = desc.z * kQTile5 + rq * 32 < p.N;
        m_run = -INFINITY;
      }
      float alpha = 0.f;
      if (live) {
        float mx = -INFINITY;
        switch (ng) {   // warp-uniform
          case 7: mx = max_groups5_np<7>(t_mine, nvr); break;
          case 6: mx = max_groups5_np<6>(t_mine, nvr); break;
          case 5: mx = max_groups5_np<5>(t_mine, nvr); break;
          case 4: mx = max_groups5_np<4>(t_mine, nvr); break;
          case 3: mx = max_groups5_np<3>(t_mine, nvr); break;
          case 2: mx = max_groups5_np<2>(t_mine, nvr); break;
          case 1: mx = max_groups5_np<1>(t_mine, nvr); break;
          default: break;
        }
        *x_mine = mx;
        named_bar_sync(bar_id, 64);
        const float m_new = fmaxf(m_run, fmaxf(mx, *x_other) * p.scale_log2);
        alpha = ex2_approx(m_run - m_new);   // first block: exp2(-inf) = 0
        m_run = m_new;
        switch (ng) {
          case 7: exp_groups5_np<7>(t_mine, nvr, p.scale_log2, m_new); break;
          case 6: exp_groups5_np<6>(t_mine, nvr, p.scale_log2, m_new); break;
          case 5: exp_groups5_np<5>(t_mine, nvr, p.scale_log2, m_new); break;
          case 4: exp_groups5_np<4>(t_mine, nvr, p.scale_log2, m_new); break;
          case 3: exp_groups5_np<3>(t_mine, nvr, p.scale_log2, m_new); break;
          case 2: exp_groups5_np<2>(t_mine, nvr, p.scale_log2, m_new); break;
          case 1: exp_groups5_np<1>(t_mine, nvr, p.scale_log2, m_new); break;
          default: break;
        }
        // the exchange slot is rewritten in the next unit: both readers are past it (they arrive on the
        // named barrier of the next unit only after this unit's read)
      }
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive(bar(C_PFULL + g));

      if (last_blk && lane == 0) tma_store_wait_read<0>();
      mbar_wait_lean5(bar(C_OFULL + g), ph);
      tc_fence_after();
      if (live) {
        uint32_t r[32];
        uint32_t r8[8];
        uint32_t rl[8];
        tmem_ld_32x32(t_lane + kOCol5 + half * kHalfCols, r);          // my DH / 2 contiguous output columns
        if (kDT) tmem_ld_32x8(t_lane + kOCol5 + half * kHalfCols + 32, r8);
        tmem_ld_32x8(t_lane + kLCol, rl);
        tmem_ld_wait();
        if (j == 0) {
#pragma unroll
          for (int i = 0; i < 32; ++i) o_acc[i] = __uint_as_float(r[i]);
          if (kDT) {
#pragma unroll
            for (int i = 0; i < 8; ++i) o_acc[32 + i] = __uint_as_float(r8[i]);
          }
          l_acc = __uint_as_float(rl[0]);
        } else {
          const float2 al2 = make_float2(alpha, alpha);
#pragma unroll
          for (int i = 0; i < 32; i += 2) {
            const float2 o = __ffma2_rn(make_float2(o_acc[i], o_acc[i + 1]), al2,
                                        make_float2(__uint_as_float(r[i]), __uint_as_float(r[i + 1])));
            o_acc[i] = o.x;
            o_acc[i + 1] = o.y;
          }
          if (kDT) {
#pragma unroll
            for (int i = 0; i < 8; i += 2) {
              const float2 o = __ffma2_rn(make_float2(o_acc[32 + i], o_acc[33 + i]), al2,
                                          make_float2(__uint_as_float(r8[i]), __uint_as_float(r8[i + 1])));
              o_acc[32 + i] = o.x;
              o_acc[33 + i] = o.y;
            }
          }
          l_acc = fmaf(l_acc, alpha, __uint_as_float(rl[0]));
        }
      }
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive(bar(C_OREAD));
      if (live && last_blk) {
        float inv;
        asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(inv) : "f"(l_acc));
        const float2 inv2 = make_float2(inv, inv);
        auto scaled = [&](int i) {
          const float2 o = __fmul2_rn(make_float2(o_acc[i], o_acc[i + 1]), inv2);
          return pack_bf16x2(o.x, o.y);
        };
#pragma unroll
        for (int jj = 0; jj < kHalfCols / 8; ++jj) {
          uint4 o4;
          o4.x = scaled(8 * jj + 0);
          o4.y = scaled(8 * jj + 2);
          o4.z = scaled(8 * jj + 4);
          o4.w = scaled(8 * jj + 6);
          *reinterpret_cast<uint4*>(stage_row + ((jj ^ sw) << 4)) = o4;
        }
        fence_proxy_async_smem();
        __syncwarp();
        if (lane == 0) {
          asm volatile("cp.async.bulk.tensor.3d.global.shared::cta.bulk_group [%0, {%2, %3, %4}], [%1];"
                       :
                       : "l"(reinterpret_cast<uint64_t>(&tma_o)), "r"(stage_addr),
                         "r"(desc.y * DH + half * kHalfCols), "r"(desc.z * kQTile5 + rq * 32), "r"(desc.x)
                       : "memory");
          tma_store_commit();
        }
      }
      if (++j == nblk) { j = 0; ++li; }
    }
    if (lane == 0) tma_store_wait<0>();
  }

  tc_fence_before();
  __syncthreads();
  if (warp_idx == 16) {
    tc_fence_after();
    tmem_dealloc<512>(tmem_base);
  }
}

long long* g_attn5_dbg = nullptr;
int g_attn5_max_ctas = 0;   // > 0: at most this many CTAs per attention launch (SM partitioning, see api.cu)
int g_attn5_bound = -1;     // -1: VT_ATTN_NO_BOUND decides; 0 / 1: forced off / on (developer hook)

}  // namespace

void attn5_set_debug_buffer(void* ptr) { g_attn5_dbg = static_cast<long long*>(ptr); }
void attn5_set_bound(int mode) { g_attn5_bound = mode; }
void attn5_set_max_ctas(int n) { g_attn5_max_ctas = n; }

int attn5_fwd_tcgen05(const void* q, const void* k, const void* v, void* out, int B, int H, int N,
                      int dh, long long qkv_row_stride, long long qkv_batch_stride,
                      long long out_row_stride, long long out_batch_stride, float scale, int reverse,
                      cudaStream_t stream) {
  if (!q || !k || !v || !out || B <= 0 || H <= 0 || N <= 0) return VT_ERR_ARG;
  if (dh != kDH5 || N > kMaxN5) return VT_ERR_UNSUPPORTED;
  // the row max is taken over the raw scores and then scaled: the maximum of the scaled logits only for scale > 0
  if (!(scale > 0.f) || !(scale < INFINITY)) return VT_ERR_UNSUPPORTED;
  if ((qkv_row_stride % 8) || (qkv_batch_stride % 8) || (out_row_stride % 8) || (out_batch_stride % 8))
    return VT_ERR_ALIGN;
  if ((reinterpret_cast<uintptr_t>(q) | reinterpret_cast<uintptr_t>(k) | reinterpret_cast<uintptr_t>(v) |
       reinterpret_cast<uintptr_t>(out)) & 15)
    return VT_ERR_ALIGN;

  Attn5Params p;
  p.N = N;
  p.H = H;
  p.B = B;
  p.nqt = (N + kQTile5 - 1) / kQTile5;
  p.bkv = (N + 15) & ~15;
  p.total_items = static_cast<long long>(B) * H * p.nqt;
  if (p.total_items >= (1LL << 31)) return VT_ERR_UNSUPPORTED;
  p.scale_log2 = scale * 1.4426950408889634f;
  p.reverse = reverse;
  static const int no_bound = [] { const char* e = getenv("VT_ATTN_NO_BOUND"); return (e && e[0] == '1') ? 1 : 0; }();
  p.no_bound = g_attn5_bound >= 0 ? (g_attn5_bound == 0) : no_bound;
  p.dbg = g_attn5_dbg;
  const int smem = 1024 + 2 * kQBytes5 + 4 * p.bkv * kDH5 * 2 + 4 * kStageBytes5 + kOnesBytes5s + 8 * C_NBARS + 8 +
                   16 * kRing5 + 2 * 2 * kQTile5 * 4 + 2 * 2 * 16 * 4;
  if (smem > kSmemLimit5) return VT_ERR_UNSUPPORTED;

  const uint64_t cols = static_cast<uint64_t>(H) * dh;
  CUtensorMap tq, tk, tv, to;
  int rc = make_tmap_bf16_3d(&tq, q, cols, N, B, qkv_row_stride, qkv_batch_stride, kDH5, kQTile5, TMAP_SW_128);
  if (rc) return rc;
  rc = make_tmap_bf16_3d(&tk, k, cols, N, B, qkv_row_stride, qkv_batch_stride, kDH5, p.bkv, TMAP_SW_128);
  if (rc) return rc;
  rc = make_tmap_bf16_3d(&tv, v, cols, N, B, qkv_row_stride, qkv_batch_stride, kDH5, p.bkv, TMAP_SW_128);
  if (rc) return rc;
  rc = make_tmap_bf16_3d(&to, out, cols, N, B, out_row_stride, out_batch_stride, kDH5, 32, TMAP_SW_128);
  if (rc) return rc;

  static int granted[kMaxDevices] = {0};
  if (const int rc_attr = ensure_dynamic_smem(attn5_fwd_kernel, smem, granted)) return rc_attr;
  int dev = 0, sms = 148;
  cudaGetDevice(&dev);
  cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
  const long long pairs = static_cast<long long>(B) * H;     // a CTA walks whole (image, head) pairs
  if (g_attn5_max_ctas > 0 && g_attn5_max_ctas < sms) sms = g_attn5_max_ctas;
  const long long grid = pairs < sms ? pairs : sms;
  return static_cast<int>(launch_maybe_pdl(attn5_fwd_kernel, dim3(static_cast<unsigned>(grid)), dim3(kThreads5s), smem, stream,
                                           tq, tk, tv, to, p));
}

// Head dim 64 with N > 208 (several KV blocks per item, online softmax) and head dim 80 with any N:
// the two-group kernel with per-group unit streams.
template <int DH>
static int launch_attn5mb(const void* q, const void* k, const void* v, void* out, int B, int H, int N,
                          long long qkv_row_stride, long long qkv_batch_stride, long long out_row_stride,
                          long long out_batch_stride, const Attn5MbParams& p, cudaStream_t stream) {
  constexpr int kDT = DH - kDH5;
  constexpr int kStage = 32 * (DH / 2) * 2;
  const int smem = 1024 + 2 * kQTile5 * DH * 2 + 4 * p.bkv * DH * 2 + 16 * kStage + (DH == kDH5 ? kOnesBytes5s : kOnesBytes5) +
                   8 * C_NBARS + 8 +
                   16 * kRing5 + 2 * 2 * kQTile5 * 4;
  if (smem > kSmemLimit5) return VT_ERR_UNSUPPORTED;
  const uint64_t cols = static_cast<uint64_t>(H) * DH;
  CUtensorMap tq, tk, tv, to, tqt, tkt, tvt;
  int rc = make_tmap_bf16_3d(&tq, q, cols, N, B, qkv_row_stride, qkv_batch_stride, kDH5, kQTile5, TMAP_SW_128);
  if (rc) return rc;
  rc = make_tmap_bf16_3d(&tk, k, cols, N, B, qkv_row_stride, qkv_batch_stride, kDH5, p.bkv, TMAP_SW_128);
  if (rc) return rc;
  rc = make_tmap_bf16_3d(&tv, v, cols, N, B, qkv_row_stride, qkv_batch_stride, kDH5, p.bkv, TMAP_SW_128);
  if (rc) return rc;
  if (kDT) {
    rc = make_tmap_bf16_3d(&tqt, q, cols, N, B, qkv_row_stride, qkv_batch_stride, 16, kQTile5, TMAP_SW_32);
    if (rc) return rc;
    rc = make_tmap_bf16_3d(&tkt, k, cols, N, B, qkv_row_stride, qkv_batch_stride, 16, p.bkv, TMAP_SW_32);
    if (rc) return rc;
    rc = make_tmap_bf16_3d(&tvt, v, cols, N, B, qkv_row_stride, qkv_batch_stride, 16, p.bkv, TMAP_SW_32);
    if (rc) return rc;
    rc = make_tmap_bf16_3d(&to, out, cols, N, B, out_row_stride, out_batch_stride, DH / 2, 32, TMAP_SW_NONE);
  } else {
    tqt = tq; tkt = tk; tvt = tv;   // unused
    rc = make_tmap_bf16_3d(&to, out, cols, N, B, out_row_stride, out_batch_stride, 32, 32, TMAP_SW_64);
  }
  if (rc) return rc;

  auto kern = attn5mb_fwd_kernel<DH>;
  static int granted[kMaxDevices] = {0};
  if (const int rc_attr = ensure_dynamic_smem(kern, smem, granted)) return rc_attr;
  int dev = 0, sms = 148;
  cudaGetDevice(&dev);
  cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
  const long long grid = p.total_items < sms ? p.total_items : sms;
  return static_cast<int>(launch_maybe_pdl(kern, dim3(static_cast<unsigned>(grid)), dim3(kThreads5), smem, stream, tq, tk, tv, to,
                                           tqt, tkt, tvt, p));
}

int attn5mb_fwd_tcgen05(const void* q, const void* k, const void* v, void* out, int B, int H, int N,
                        int dh, long long qkv_row_stride, long long qkv_batch_stride,
                        long long out_row_stride, long long out_batch_stride, float scale, int reverse,
                        cudaStream_t stream) {
  if (!q || !k || !v || !out || B <= 0 || H <= 0 || N <= 0) return VT_ERR_ARG;
  if (dh != 64 && dh != 80) return VT_ERR_UNSUPPORTED;
  if (!(scale > 0.f) || !(scale < INFINITY)) return VT_ERR_UNSUPPORTED;   // as attn5_fwd_tcgen05
  if ((qkv_row_stride % 8) || (qkv_batch_stride % 8) || (out_row_stride % 8) || (out_batch_stride % 8))
    return VT_ERR_ALIGN;
  if ((reinterpret_cast<uintptr_t>(q) | reinterpret_cast<uintptr_t>(k) | reinterpret_cast<uintptr_t>(v) |
       reinterpret_cast<uintptr_t>(out)) & 15)
    return VT_ERR_ALIGN;

  Attn5MbParams p;
  p.N = N;
  p.H = H;
  p.B = B;
  p.nqt = (N + kQTile5 - 1) / kQTile5;
  p.nblk = (N + kMaxN5 - 1) / kMaxN5;
  const int bkv = (N + p.nblk - 1) / p.nblk;
  p.bkv = (bkv + 15) & ~15;
  if ((p.nblk - 1) * p.bkv >= N) return VT_ERR_UNSUPPORTED;   // the last block must hold at least one key
  p.total_items = static_cast<long long>(B) * H * p.nqt;
  if (p.total_items * p.nblk >= (1LL << 31)) return VT_ERR_UNSUPPORTED;
  p.scale_log2 = scale * 1.4426950408889634f;
  p.reverse = reverse;
  if (dh == 64)
    return launch_attn5mb<64>(q, k, v, out, B, H, N, qkv_row_stride, qkv_batch_stride, out_row_stride,
                              out_batch_stride, p, stream);
  return launch_attn5mb<80>(q, k, v, out, B, H, N, qkv_row_stride, qkv_batch_stride, out_row_stride,
                            out_batch_stride, p, stream);
}

}  // namespace vt
