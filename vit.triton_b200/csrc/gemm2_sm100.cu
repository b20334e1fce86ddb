// K1 (main variant): persistent 2-CTA bf16 GEMM — tcgen05.mma.cta_group::2 on a CTA pair.
//
//   out[M,N] = epilogue( A[M,K] . Bt[N,K]^T + bias[N] ) (+ residual[M,N]),  bf16 in / bf16 out
//
// Same contract as gemm_sm100.cu (which stays as the fp32-output / fallback variant); this one is
// what the bf16 model runs.  Reference ops replaced: matmul_kernel (vit/kernels/matmul.py:40-108)
// with its bias / GELU epilogue, and add_kernel (vit/vit.py:140,147) via the residual epilogue.
//
// Launch: regular clusters of two, PREFERRED clusters of four (two pairs on two tiles that share an operand, which is
// then loaded in halves and TMA-multicast to the other pair: see the kernel), programmatic stream serialisation.
// A pair of CTAs (one TPC) owns a 256 x 256 output tile: CTA r holds rows [128r, 128r+128)
// of the tile in its TMEM (128 lanes x 256 fp32 columns, double buffered = all 512 columns) and
// loads A rows [128r, +128) and Bt rows [128r, +128) of every 64-wide K block, so each SM pulls
// 32 KB per K block from L2 instead of 48 KB for the same number of MACs.  Only the leader CTA
// issues MMAs (M=256, N=256, K=16); both CTAs' TMA loads complete on the leader's mbarrier.
//
// Epilogue: 8 warps per CTA; warp (q, g) owns TMEM lanes 32q..32q+31 and columns 128g..128g+127
// (16 warps x 64 columns measured no faster).  Per 64-column chunk: tcgen05.ld -> +bias (lane-owned,
// broadcast with shuffles) -> (LayerNorm fold: x rstd of the row) -> (+residual from smem) -> (GELU) ->
// bf16 -> SWIZZLE_128B staging buffer -> TMA store.  The residual chunk is TMA-LOADED into the same
// staging buffer before the accumulator is ready, so neither residual reads nor output writes go
// through per-thread global accesses (the v1 row-per-thread stores made the epilogue the bottleneck:
// profiles/r01_*).  The chunks of the eight warps are PACED over the tile (see the epilogue) because
// simultaneous store bursts collide with the operand stream on the SM's L2 port; per-tile operands
// (bias, row statistics of the folded LayerNorm) are prefetched one tile ahead because with 224 KB of
// shared memory configured there is no L1 and every global load is an L2 round trip.
#include <cstdlib>

#include "common.cuh"
#include "tensormap.h"

namespace vt {

namespace {

constexpr int BM = 128;          // rows per CTA (pair tile = 256)
constexpr int BN = 256;          // tile columns
constexpr int BNH = 128;         // Bt rows loaded per CTA
constexpr int BK = 64;
#ifndef VT_EPI_WARPS
#define VT_EPI_WARPS 8
#endif
constexpr int kEpiWarps = VT_EPI_WARPS;            // 4 lane quarters x (2 | 4) column groups
constexpr int kColGroups = kEpiWarps / 4;
constexpr int kColsPerWarp = BN / kColGroups;       // 64
constexpr int kThreads = 128 + kEpiWarps * 32;
constexpr int kABytes = BM * BK * 2;
constexpr int kBBytes = BNH * BK * 2;
constexpr int kStageBytes = kABytes + kBBytes;          // 32 KB
constexpr int kChunkCols = 64;
constexpr int kStagingBytes = 32 * kChunkCols * 2;      // 4 KB: 32 rows x 64 bf16
constexpr int kChunks = kColsPerWarp / kChunkCols;          // chunks per warp

// Shared-memory split between operand stages and epilogue staging (227 KB in all):
//   5 stages + one staging buffer per chunk (no reuse inside a tile)   -> short-K residual launches
//   6 stages + ONE staging buffer per epilogue warp (reused per chunk)  -> everything else
// Five 32 KB stages cover ~3000 cycles of operand latency under load and the MMA issuer still waits
// for operands 40 % of the time; the sixth stage shortens a QKV tile from 7313 to 6837 cycles and an
// fc2 tile from 27073 to 26197.  Serialising the two chunks of a warp on one staging buffer used to
// cost the GELU and LayerNorm-fold epilogues more than that; with the paced epilogue (the chunks are
// spread over the tile anyway) only the K = 768 residual epilogue still prefers two buffers
// (66.2k vs 70.9k cycles per out-proj launch).
template <int kStagesT, int kStageBufsT>
struct G2Cfg {
  static constexpr int kStages = kStagesT;
  static constexpr int kStageBufs = kStageBufsT;
  static constexpr int kEpiBytes = kEpiWarps * kStageBufs * kStagingBytes;
  static constexpr int kNumBars = 2 * kStages + 4 + kChunks * kEpiWarps;
  static constexpr int kSmemBytes = 1024 + kStages * kStageBytes + kEpiBytes + 8 * kNumBars + 16;
  static_assert(kSmemBytes <= 232448, "over the 227 KB shared-memory limit");
};
using G2Deep = G2Cfg<6, 1>;
using G2Wide = G2Cfg<5, 2>;
constexpr uint32_t kPeerMask = 0xFEFFFFFFu;             // clears the CTA-rank bit of a cluster smem address

// EPI_NOCS (with EPI_LNF): the folded weights have zero-sum rows (packing._fold_layernorm_zero_sum), so the
// mean term is already inside the accumulator and the epilogue needs no column sums.
enum : int { EPI_GELU = 1, EPI_RES = 2, EPI_LNF = 4, EPI_STATS = 8, EPI_NOCS = 16, EPI_CSCALE = 32, EPI_QGELU = 64 };
// EPI_QGELU: quick GELU x * sigmoid(1.702 x) (CLIP) where EPI_GELU applies exact GELU; the two never combine.
// EPI_CSCALE (FP8 operands): out = acc * colscale_n + bias_n — the per-output-channel dequantisation scale of the
// e4m3 weights times the activation scale (Gemm2Params::colsum carries it).
// PREC: 0 = bf16 operands, bf16 output (kind::f16); 1 = e4m3 operands, bf16 output; 2 = e4m3 operands, e4m3 output
// (kind::f8f6f4: 128 K elements per 128-byte swizzle row, K = 32 per MMA, twice the MACs per operand byte).

struct Gemm2Params {
  int M, N, K;
  int num_m_tiles, num_n_tiles;   // in units of the 256 x 256 pair tile
  int reverse;                    // walk the row tiles from the last to the first (L2 reuse, see api.cu)
  const float* bias;
  // LayerNorm folded into the epilogue (EPI_LNF): out = rstd_m * acc + (-rstd_m * mean_m) * colsum_n + bias_n
  // with (sum, M2) of the A row given as ln_parts = ln_dim / 128 partial pairs (M2 about the group mean)
  // rowstats[(m*ln_parts + i)*2 .. +1]
  const float* rowstats;
  const float* colsum;
  float ln_inv_dim, ln_eps;
  int ln_parts;
  // EPI_STATS: write (sum, M2 = sum of squares about the group mean) of every 128-column group (one
  // epilogue warp's share of a tile) of every output row to stats_out[(m * (N/128) + group) * 2 .. +1]:
  // no atomics, so results are bit-reproducible
  float* stats_out;
  long long* dbg;   // optional per-CTA cycle counters (vt_debug_set_buffer); null in production
  // Epilogue pacing (see the epilogue): cycles between the start slots of the tile's store bursts,
  // 0 = off; pace_q = additional stagger between the four lane-quarter warps of a slot
  int pace, pace_q;
  float out_scale;   // PREC 2: multiplier applied before the e4m3 cast of the output
  // Token mode (patch embedding, EPI_RES): the M rows are images of tok_pad rows each (tok_pad % 32 == 0, so a
  // 32-row epilogue tile never straddles two images), of which the first `tokens` are real.  The output map is
  // 3-D (column, token, image: TMA clips the padding rows), the "residual" map is the [tokens, N] position table
  // addressed by token, and row statistics go to row image * tokens + token.  0 = off.
  int tok_pad, tokens;
};

__device__ __forceinline__ uint32_t cluster_ctarank() {
  uint32_t r;
  asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(r));
  return r;
}
__device__ __forceinline__ void cluster_sync_all() {
  asm volatile("barrier.cluster.arrive.release.aligned;\n\tbarrier.cluster.wait.acquire.aligned;" ::: "memory");
}

template <int kCols>
__device__ __forceinline__ void tmem_alloc_2cta(uint32_t smem_dst) {
  asm volatile("tcgen05.alloc.cta_group::2.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_dst),
               "n"(kCols)
               : "memory");
}
__device__ __forceinline__ void tmem_relinquish_2cta() {
  asm volatile("tcgen05.relinquish_alloc_permit.cta_group::2.sync.aligned;" ::: "memory");
}
template <int kCols>
__device__ __forceinline__ void tmem_dealloc_2cta(uint32_t taddr) {
  asm volatile("tcgen05.dealloc.cta_group::2.sync.aligned.b32 %0, %1;" ::"r"(taddr), "n"(kCols)
               : "memory");
}

// TMA load whose completion bytes are credited to the mbarrier at the same offset in the LEADER CTA.
__device__ __forceinline__ void tma_load_2d_2cta(const CUtensorMap* m, uint32_t bar, uint32_t dst,
                                                 int c0, int c1, uint64_t hint) {
  asm volatile(
      "cp.async.bulk.tensor.2d.cta_group::2.shared::cluster.global.mbarrier::complete_tx::bytes"
      ".L2::cache_hint [%0], [%1, {%3, %4}], [%2], %5;"
      :
      : "r"(dst), "l"(reinterpret_cast<uint64_t>(m)), "r"(bar & kPeerMask), "r"(c0), "r"(c1),
        "l"(hint)
      : "memory");
}

// The same, multicast: the box lands at the same offset in every CTA of `mask` and each destination's bytes are
// credited to the leader barrier of the DESTINATION's pair (checked with tools/mcast_bench.cu, mode 8).
__device__ __forceinline__ void tma_load_2d_2cta_mc(const CUtensorMap* m, uint32_t bar, uint32_t dst,
                                                    int c0, int c1, uint16_t mask, uint64_t hint) {
  asm volatile(
      "cp.async.bulk.tensor.2d.cta_group::2.shared::cluster.global.mbarrier::complete_tx::bytes"
      ".multicast::cluster.L2::cache_hint [%0], [%1, {%3, %4}], [%2], %5, %6;"
      :
      : "r"(dst), "l"(reinterpret_cast<uint64_t>(m)), "r"(bar & kPeerMask), "r"(c0), "r"(c1), "h"(mask),
        "l"(hint)
      : "memory");
}
__device__ __forceinline__ uint32_t cluster_nctarank() {
  uint32_t r;
  asm volatile("mov.u32 %0, %%cluster_nctarank;" : "=r"(r));
  return r;
}

__device__ __forceinline__ void umma_ss_2cta(uint32_t d_tmem, uint64_t a_desc, uint64_t b_desc,
                                             uint32_t idesc, uint32_t accumulate) {
  asm volatile(
      "{\n\t"
      ".reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::2.kind::f16 [%0], %1, %2, %3, p;\n\t"
      "}\n"
      :
      : "r"(d_tmem), "l"(a_desc), "l"(b_desc), "r"(idesc), "r"(accumulate)
      : "memory");
}

__device__ __forceinline__ void umma_ss_2cta_f8(uint32_t d_tmem, uint64_t a_desc, uint64_t b_desc,
                                                uint32_t idesc, uint32_t accumulate) {
  asm volatile(
      "{\n\t"
      ".reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::2.kind::f8f6f4 [%0], %1, %2, %3, p;\n\t"
      "}\n"
      :
      : "r"(d_tmem), "l"(a_desc), "l"(b_desc), "r"(idesc), "r"(accumulate)
      : "memory");
}

// Instruction descriptor for kind::f8f6f4 with e4m3 x e4m3 -> f32 (A / B format fields 0 = E4M3), K-major operands.
__host__ __device__ constexpr uint32_t make_idesc_e4m3(int m, int n) {
  return (1u << 4) | (static_cast<uint32_t>(n >> 3) << 17) | (static_cast<uint32_t>(m >> 4) << 24);
}

// four floats -> four e4m3 bytes (saturating), lowest address first
__device__ __forceinline__ uint32_t pack_e4m3x4(float a, float b, float c, float d) {
  uint16_t lo, hi;
  asm("cvt.rn.satfinite.e4m3x2.f32 %0, %1, %2;" : "=h"(lo) : "f"(b), "f"(a));
  asm("cvt.rn.satfinite.e4m3x2.f32 %0, %1, %2;" : "=h"(hi) : "f"(d), "f"(c));
  return static_cast<uint32_t>(lo) | (static_cast<uint32_t>(hi) << 16);
}

// Arrive (once all prior MMAs of this thread completed) on the barrier at this offset in BOTH CTAs.
__device__ __forceinline__ void umma_commit_2cta(uint32_t bar, uint16_t mask) {
  asm volatile(
      "tcgen05.commit.cta_group::2.mbarrier::arrive::one.shared::cluster.multicast::cluster.b64 "
      "[%0], %1;"
      :
      : "r"(bar), "h"(mask)
      : "memory");
}

// Arrive on the barrier at this offset in the leader CTA (works from either CTA of the pair).
__device__ __forceinline__ void mbar_arrive_leader(uint32_t bar) {
  asm volatile("mbarrier.arrive.shared::cluster.b64 _, [%0];" ::"r"(bar & kPeerMask) : "memory");
}

#ifdef VT_GELU_AS   // A/B switch: the two-MUFU Abramowitz-Stegun form
__device__ __forceinline__ float2 gelu_epi2(float2 x) { return gelu_erf_bf16_x2(x); }
#else
__device__ __forceinline__ float2 gelu_epi2(float2 x) { return gelu_erf_poly_x2(x); }
#endif

template <int EPI, typename Cfg, int PREC = 0>
__global__ void __launch_bounds__(kThreads, 1)     // cluster dimensions come with the launch: 2, preferred 4
gemm2_bf16_kernel(const __grid_constant__ CUtensorMap tma_a, const __grid_constant__ CUtensorMap tma_b,
                  const __grid_constant__ CUtensorMap tma_out,
                  const __grid_constant__ CUtensorMap tma_res, const __grid_constant__ CUtensorMap tma_a64,
                  const __grid_constant__ CUtensorMap tma_b64, const Gemm2Params p) {
  constexpr int kStages = Cfg::kStages;
  constexpr int kStageBufs = Cfg::kStageBufs;
  constexpr int kEpiBytes = Cfg::kEpiBytes;
  constexpr int kNumBars = Cfg::kNumBars;
  constexpr bool kFp8In = PREC != 0;
  constexpr bool kFp8Out = PREC == 2;
  constexpr int kBKE = kFp8In ? 2 * BK : BK;       // K ELEMENTS per 128-byte operand row
  static_assert(!kFp8Out || (kStageBufs == 1 && !(EPI & (EPI_RES | EPI_STATS | EPI_LNF))), "e4m3 output: plain / GELU epilogue");
  static_assert(!(EPI & EPI_CSCALE) || !(EPI & EPI_LNF), "column scales and the LayerNorm fold do not combine");
  extern __shared__ uint8_t smem_raw[];
  const uint32_t smem_base = (smem_u32(smem_raw) + 1023u) & ~1023u;
  uint8_t* smem_gen = smem_raw + (smem_base - smem_u32(smem_raw));

  const uint32_t tiles_addr = smem_base;
  const uint32_t epi_addr = smem_base + kStages * kStageBytes;
  const uint32_t bar_addr = epi_addr + kEpiBytes;
  auto full_bar = [&](int s) { return bar_addr + 8u * s; };
  auto empty_bar = [&](int s) { return bar_addr + 8u * (kStages + s); };
  auto tfull_bar = [&](int s) { return bar_addr + 8u * (2 * kStages + s); };
  auto tempty_bar = [&](int s) { return bar_addr + 8u * (2 * kStages + 2 + s); };
  auto res_bar = [&](int w, int c) { return bar_addr + 8u * (2 * kStages + 4 + kChunks * w + c); };
  const uint32_t tmem_slot = bar_addr + 8u * kNumBars;
  volatile uint32_t* tmem_slot_gen = reinterpret_cast<volatile uint32_t*>(
      smem_gen + kStages * kStageBytes + kEpiBytes + 8 * kNumBars);

  // Warp roles.  The warp scheduler favours the highest warp id among eligible warps, so the
  // single-thread MMA issuer and the TMA producer sit ABOVE the epilogue warps: with the issuer at
  // warp 1 the GELU epilogue starved it of issue slots (tensor pipe idle 30 % of the fc1 GEMM).
  constexpr int kWarpTmem = kEpiWarps;          // TMEM alloc / dealloc
  constexpr int kWarpProducer = kEpiWarps + 2;
  constexpr int kWarpMma = kEpiWarps + 3;
  const int warp_idx = threadIdx.x >> 5;
  const int lane = threadIdx.x & 31;
  // An aligned GROUP of four CTAs = two CTA pairs works through a list of SUPERTILES: two 256 x 256 tiles that share
  // one operand (the same column block on two adjacent row blocks: B is shared; or, for the last row block of an odd
  // count, two adjacent column blocks: A is shared).  The device launches a group either as ONE cluster of four (the
  // preferred size, 132 of a B200's 148 SMs) — then each pair loads its private operand as before and only HALF of the
  // shared one, multicast to the CTA of the same rank in the other pair, a quarter less operand traffic out of L2 — or
  // as two regular clusters of two, which load everything themselves: the same work list and the same results.
  const uint32_t cta_rank = cluster_ctarank();        // 0..1 or 0..3
  const bool quad = cluster_nctarank() == 4;
  const uint32_t half = cta_rank & 1u;                // CTA within its pair: rows [128 half, +128) of the pair tile
  const int pair = static_cast<int>((blockIdx.x >> 1) & 1u);   // pair within the group (= cta_rank >> 1 in a cluster of four)
  const bool is_leader = (half == 0);
  const uint16_t pair_mask = static_cast<uint16_t>(3u << (cta_rank & 2u));          // both CTAs of my pair
  const uint16_t cluster_mask = quad ? static_cast<uint16_t>(0xF) : static_cast<uint16_t>(3);
  const uint16_t share_mask = static_cast<uint16_t>((1u << half) | (1u << (half + 2)));   // my rank in both pairs

  if (warp_idx == kWarpProducer && lane == 0) {
    tma_prefetch_desc(&tma_a);
    tma_prefetch_desc(&tma_b);
    tma_prefetch_desc(&tma_out);
    if (EPI & EPI_RES) tma_prefetch_desc(&tma_res);
  }
  if (warp_idx == kWarpMma && lane == 0) {
    for (int s = 0; s < kStages; ++s) {
      mbar_init(full_bar(s), 1);      // leader's producer arrive.expect_tx (covers both CTAs' bytes)
      mbar_init(empty_bar(s), quad ? 2 : 1);     // multicast tcgen05.commit of every pair that reads what I load
    }
    for (int s = 0; s < 2; ++s) {
      mbar_init(tfull_bar(s), 1);                 // multicast tcgen05.commit
      mbar_init(tempty_bar(s), 2 * kEpiWarps);    // epilogue warps of BOTH CTAs (leader's copy is used)
    }
    for (int w = 0; w < kEpiWarps; ++w)
      for (int c = 0; c < kChunks; ++c) mbar_init(res_bar(w, c), 1);
    fence_barrier_init();
  }
  if (warp_idx == kWarpTmem) {
    tmem_alloc_2cta<512>(tmem_slot);
    tmem_relinquish_2cta();
  }
  tc_fence_before();
  cluster_sync_all();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot_gen;
  // everything above touched only this CTA's own state: from here on the predecessor's output is read
  pdl_wait();
  pdl_launch_dependents();

  // supertiles: [0, main_st) = (row-block pair mp, column block n), n fastest; then the last row block of an odd
  // count, column blocks in pairs (the second tile of the last one may lie right of the matrix: a ghost that loads
  // zeros and stores nothing)
  const int main_st = (p.num_m_tiles >> 1) * p.num_n_tiles;
  const int num_tiles = main_st + ((p.num_m_tiles & 1) ? ((p.num_n_tiles + 1) >> 1) : 0);   // supertiles
  // (row block, column block, shared operand: 0 = B, 1 = A) of MY pair's tile of supertile t
  auto decode_tile = [&](int t, int& m_blk, int& n_blk) -> int {
    int m_lin, share;
    if (t < main_st) {
      const int mp = t / p.num_n_tiles;
      n_blk = t - mp * p.num_n_tiles;
      m_lin = 2 * mp + pair;
      share = 0;
    } else {
      m_lin = p.num_m_tiles - 1;
      n_blk = 2 * (t - main_st) + pair;
      share = 1;
    }
    m_blk = p.reverse ? p.num_m_tiles - 1 - m_lin : m_lin;
    return share;
  };
  const int num_kb = (p.K + kBKE - 1) / kBKE;
  long long dbg_acc[8] = {0, 0, 0, 0, 0, 0, 0, 0};
  const long long dbg_t0 = p.dbg ? clock64() : 0;
  unsigned long long dbg_ns0 = 0;
  if (p.dbg) asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(dbg_ns0));
  const int first_tile = static_cast<int>(blockIdx.x >> 2);
  const int tile_step = static_cast<int>(gridDim.x >> 2);

  if (warp_idx == kWarpProducer) {
    // ------------------------------------------------------------------ TMA producer (both CTAs)
    // The loop is executed by the whole warp (warp-uniform control flow keeps addresses and
    // coordinates in uniform registers); one elected lane issues the TMA instructions.
    int s = 0;
    uint32_t phase = 0;
    for (int t = first_tile; t < num_tiles; t += tile_step) {
      int m_blk, n_blk;
      const int share = decode_tile(t, m_blk, n_blk);
      const int a_row = m_blk * (2 * BM) + static_cast<int>(half) * BM;
      const int b_row = n_blk * BN + static_cast<int>(half) * BNH;
      for (int kb = 0; kb < num_kb; ++kb) {
        long long w0 = 0;
        if (p.dbg) w0 = clock64();
        mbar_wait(empty_bar(s), phase ^ 1u);
        if (p.dbg) dbg_acc[4] += clock64() - w0;
        const uint32_t a_dst = tiles_addr + s * kStageBytes;
        const uint32_t b_dst = a_dst + kABytes;
        if (elect_one_sync()) {
          if (is_leader) mbar_arrive_expect_tx(full_bar(s), 2 * kStageBytes);
          if (!quad) {
            tma_load_2d_2cta(&tma_a, full_bar(s), a_dst, kb * kBKE, a_row, kEvictNormal);
            tma_load_2d_2cta(&tma_b, full_bar(s), b_dst, kb * kBKE, b_row, kEvictLast);
          } else if (share == 0) {
            // rows [64 pair, +64) of the shared 128-row B box, into my smem and that of my rank in the other pair
            tma_load_2d_2cta(&tma_a, full_bar(s), a_dst, kb * kBKE, a_row, kEvictNormal);
            tma_load_2d_2cta_mc(&tma_b64, full_bar(s), b_dst + pair * (kBBytes / 2), kb * kBKE, b_row + pair * (BNH / 2),
                                share_mask, kEvictLast);
          } else {
            tma_load_2d_2cta_mc(&tma_a64, full_bar(s), a_dst + pair * (kABytes / 2), kb * kBKE, a_row + pair * (BM / 2),
                                share_mask, kEvictNormal);
            tma_load_2d_2cta(&tma_b, full_bar(s), b_dst, kb * kBKE, b_row, kEvictLast);
          }
        }
        __syncwarp();
        if (++s == kStages) { s = 0; phase ^= 1u; }
      }
    }
  } else if (warp_idx == kWarpMma) {
    // ------------------------------------------------------------------ MMA issuer (leader only)
    // Warp-uniform loop, one elected lane issues.  (Issuing from inside an `if (lane == 0)` region
    // made the compiler wrap every UTCHMMA in an ELECT / R2UR.BROADCAST loop — ~19 instructions
    // per MMA — and the GELU epilogue then starved the issuer: tensor pipe 56 % instead of 80 %.)
    if (is_leader) {
      constexpr uint32_t idesc = kFp8In ? make_idesc_e4m3(2 * BM, BN) : make_idesc_bf16(2 * BM, BN, 0, 0);
      int s = 0;
      uint32_t phase = 0;
      int as = 0;
      uint32_t aphase = 0;
      for (int t = first_tile; t < num_tiles; t += tile_step) {
        long long w0 = 0;
        if (p.dbg) w0 = clock64();
        mbar_wait(tempty_bar(as), aphase ^ 1u);
        if (p.dbg) dbg_acc[3] += clock64() - w0;
        tc_fence_after();
        const uint32_t d_tmem = tmem_base + as * BN;
        for (int kb = 0; kb < num_kb; ++kb) {
          if (p.dbg) w0 = clock64();
          mbar_wait(full_bar(s), phase);
          if (p.dbg) dbg_acc[2] += clock64() - w0;
          tc_fence_after();
          const uint32_t a_src = tiles_addr + s * kStageBytes;
          const uint32_t b_src = a_src + kABytes;
          if (elect_one_sync()) {
            const uint64_t adesc = make_desc_kmajor_sw128(a_src);
            const uint64_t bdesc = make_desc_kmajor_sw128(b_src);
#pragma unroll
            for (int k = 0; k < BK / 16; ++k) {
              // advancing K by 16 bf16 (32 e4m3) = 32 bytes = 2 units of the 16-byte start-address field
              if (kFp8In) umma_ss_2cta_f8(d_tmem, adesc + 2 * k, bdesc + 2 * k, idesc, (kb | k) != 0 ? 1u : 0u);
              else umma_ss_2cta(d_tmem, adesc + 2 * k, bdesc + 2 * k, idesc, (kb | k) != 0 ? 1u : 0u);
            }
            umma_commit_2cta(empty_bar(s), cluster_mask);
          }
          __syncwarp();
          if (++s == kStages) { s = 0; phase ^= 1u; }
        }
        if (elect_one_sync()) umma_commit_2cta(tfull_bar(as), pair_mask);
        __syncwarp();
        if (++as == 2) { as = 0; aphase ^= 1u; }
      }
    }
  } else if (warp_idx < kEpiWarps) {
    // ------------------------------------------------------------------ epilogue (both CTAs)
    const int ew = warp_idx;
    const int q = warp_idx & 3;
    const int cgrp = ew >> 2;   // column group
    uint32_t stage_buf[kChunks];
    uint8_t* stage_gen[kChunks];
#pragma unroll
    for (int c = 0; c < kChunks; ++c) {
      stage_buf[c] = epi_addr + (kStageBufs * ew + (c % kStageBufs)) * kStagingBytes;
      stage_gen[c] = smem_gen + kStages * kStageBytes + (kStageBufs * ew + (c % kStageBufs)) * kStagingBytes;
    }
    const int sw = lane & 7;   // swizzle phase of this thread's staging row
    int as = 0;
    uint32_t aphase = 0;
    uint32_t rphase = 0;

    // Per-column and per-row epilogue operands.  With 224 KB of the SM's 228 KB configured as shared
    // memory there is practically no L1: every __ldg is an L2 round trip (~700 cycles under load),
    // and loading the bias of each 32-column step at the step cost the plain epilogue 3300 cycles per
    // tile, four fifths of it latency (tools/gemm_dbg.py).  So: lane l keeps the bias (and the folded
    // LayerNorm's column sums) of columns 4l..4l+3 of this warp's 128 — ONE coalesced 16-byte load per
    // tile — and the steps broadcast them with shuffles; those loads and the row statistics of the
    // NEXT tile are issued before the current tile's staging buffers drain.
    static_assert(kColsPerWarp == 128, "lane-owned bias layout: 32 lanes x 4 columns");
    constexpr int kRsRegs = 5;                     // row statistics prefetched as up to 5 float4 (K <= 1280)
    const bool rs_fast = (EPI & EPI_LNF) && (p.ln_parts % 2 == 0) && (p.ln_parts <= 2 * kRsRegs) &&
                         (reinterpret_cast<uintptr_t>(p.rowstats) & 15) == 0;
    float4 b4n = make_float4(0.f, 0.f, 0.f, 0.f), c4n = make_float4(0.f, 0.f, 0.f, 0.f);
    float4 rsn[kRsRegs];
#pragma unroll
    for (int i = 0; i < kRsRegs; ++i) rsn[i] = make_float4(0.f, 0.f, 0.f, 0.f);
    auto tile_origin = [&](int t, int& row0, int& col0) {
      int m_blk, n_blk;
      decode_tile(t, m_blk, n_blk);
      row0 = m_blk * (2 * BM) + static_cast<int>(half) * BM + q * 32;
      col0 = n_blk * BN + cgrp * kColsPerWarp;
    };
    auto prefetch_operands = [&](int t) {
      int row0, col0;
      tile_origin(t, row0, col0);
      const int cb = col0 + 4 * lane;
      const bool in = cb + 3 < p.N;              // N % 8 == 0: groups of 4 are all in or all out
      b4n = (p.bias != nullptr && in) ? __ldg(reinterpret_cast<const float4*>(p.bias + cb))
                                      : make_float4(0.f, 0.f, 0.f, 0.f);
      if (EPI & EPI_CSCALE)
        c4n = in ? __ldg(reinterpret_cast<const float4*>(p.colsum + cb)) : make_float4(0.f, 0.f, 0.f, 0.f);
      if (EPI & EPI_LNF) {
        if (!(EPI & EPI_NOCS))
          c4n = in ? __ldg(reinterpret_cast<const float4*>(p.colsum + cb)) : make_float4(0.f, 0.f, 0.f, 0.f);
        const int row = row0 + lane;
        if (rs_fast && row < p.M) {
          const float4* parts =
              reinterpret_cast<const float4*>(p.rowstats + static_cast<long long>(row) * p.ln_parts * 2);
#pragma unroll
          for (int i = 0; i < kRsRegs; ++i)
            if (2 * i < p.ln_parts) rsn[i] = __ldg(parts + i);
        }
      }
    };
    if (first_tile < num_tiles) prefetch_operands(first_tile);

    for (int t = first_tile; t < num_tiles; t += tile_step) {
      int row0, col0;
      tile_origin(t, row0, col0);
      const float4 b4 = b4n, c4 = c4n;
      // token mode: (image, first token) of this warp's 32 rows; res_row = row coordinate of the residual map
      int img = 0, tok0 = row0;
      if ((EPI & EPI_RES) && p.tok_pad > 0) {
        img = row0 / p.tok_pad;
        tok0 = row0 - img * p.tok_pad;
      }

      if (EPI & EPI_RES) {
        if (lane == 0) {
#pragma unroll
          for (int c = 0; c < kStageBufs; ++c) {
            mbar_arrive_expect_tx(res_bar(ew, c), kStagingBytes);
            tma_load_2d(&tma_res, res_bar(ew, c), stage_buf[c], col0 + c * kChunkCols, tok0,
                        p.tok_pad > 0 ? kEvictNormal : kEvictFirst);
          }
        }
      }

      float ln_a = 1.f, ln_b = 0.f;
      if (EPI & EPI_LNF) {
        // Row statistics arrive as per-128-column (sum, M2) partials, M2 = sum of squares about the
        // group's OWN mean; they are merged the Chan / Welford way (sum of the M2 plus 128 * squared
        // distance of every group mean from the row mean), so the variance is a sum of non-negative
        // centred terms like the reference's two-pass form (vit/kernels/layernorm.py:51-85) and never a
        // difference of two large numbers (rows with |mean| >> std, massive-activation channels).
        const int row = row0 + lane;
        if (row < p.M) {
          float sx = 0.f, m2 = 0.f;
          if (rs_fast) {                            // fixed order: deterministic
#pragma unroll
            for (int i = 0; i < kRsRegs; ++i)
              if (2 * i < p.ln_parts) sx += rsn[i].x + rsn[i].z;
            const float mean_f = sx * p.ln_inv_dim;
#pragma unroll
            for (int i = 0; i < kRsRegs; ++i) {
              if (2 * i < p.ln_parts) {
                const float d0 = fmaf(rsn[i].x, 1.0f / 128.0f, -mean_f);
                const float d1 = fmaf(rsn[i].z, 1.0f / 128.0f, -mean_f);
                m2 += rsn[i].y + rsn[i].w;
                m2 = fmaf(128.0f * d0, d0, m2);
                m2 = fmaf(128.0f * d1, d1, m2);
              }
            }
          } else {
            const float2* parts =
                reinterpret_cast<const float2*>(p.rowstats) + static_cast<long long>(row) * p.ln_parts;
            for (int i = 0; i < p.ln_parts; ++i) sx += __ldg(parts + i).x;
            const float mean_s = sx * p.ln_inv_dim;
            for (int i = 0; i < p.ln_parts; ++i) {
              const float2 st = __ldg(parts + i);
              const float d = fmaf(st.x, 1.0f / 128.0f, -mean_s);
              m2 += st.y;
              m2 = fmaf(128.0f * d, d, m2);
            }
          }
          const float mean = sx * p.ln_inv_dim;
          const float var = m2 * p.ln_inv_dim;
          // var == 0 exactly: every element equals the mean, LN(x) = beta whatever rstd is (the reference
          // multiplies rstd by x - mean = 0); rstd = 1/sqrt(eps) would only amplify the rounding residue
          // of the zero-sum weight rows
          ln_a = var > 0.f ? rsqrtf(var + p.ln_eps) : 0.f;
          ln_b = -ln_a * mean;
        }
      }

      long long w0 = 0;
      if (p.dbg) w0 = clock64();
      // Pacing.  All eight warps would otherwise read their accumulator quarter and push their chunk
      // through the TMA at the same moment, twice per tile: the 32 KB store bursts collide with the
      // operand loads on the SM's L2 port (which the mainloop alone already fills) and every tile loses
      // 300-600 cycles (tools/gemm_dbg.py: a SLOWER epilogue made the same GEMM faster).  When the
      // accumulator was not ready yet (the epilogue is ahead of the mainloop) chunk c of column group g
      // therefore starts no earlier than slot (2c + g) after the accumulator arrived; a warp that
      // found the accumulator waiting is behind and does not pace.
      const bool ahead = !mbar_test_wait(tfull_bar(as), aphase);
      if (ahead) mbar_wait(tfull_bar(as), aphase);
      if (p.dbg) { const long long w1 = clock64(); dbg_acc[0] += w1 - w0; w0 = w1; }
      tc_fence_after();
      // (the CTA's last tile has no mainloop left to protect: pacing it would only lengthen the tail)
      const bool paced = ahead && p.pace > 0 && (t + tile_step < num_tiles);
      const long long pace_t0 = paced ? clock64() + q * p.pace_q : 0;
      const uint32_t t_addr = tmem_base + (static_cast<uint32_t>(q * 32) << 16) + as * BN + cgrp * kColsPerWarp;

      // EPI_STATS: sums of (x - pivot) and (x - pivot)^2 over this warp's 128 columns of the row, even / odd
      // columns apart; the pivot is the row's first value in the group, so the squares stay of the order of
      // the spread inside the group and M2 = Q - S^2 / 128 loses nothing to cancellation
      float2 st_sum2 = make_float2(0.f, 0.f), st_sq2 = make_float2(0.f, 0.f), st_npiv2 = make_float2(0.f, 0.f);
#pragma unroll
      for (int c = 0; c < kChunks; ++c) {
        const int col = col0 + c * kChunkCols;
        const bool live = col < p.N;   // warp-uniform: chunk not entirely right of the matrix
        if (!kFp8Out && kStageBufs < kChunks && c >= kStageBufs) {
          // the staging buffer is shared with an earlier chunk of this tile: its store must have read it
          if (lane == 0) {
            tma_store_wait_read<0>();
            if (EPI & EPI_RES) {
              mbar_arrive_expect_tx(res_bar(ew, c), kStagingBytes);
              tma_load_2d(&tma_res, res_bar(ew, c), stage_buf[c], col, tok0, p.tok_pad > 0 ? kEvictNormal : kEvictFirst);
            }
          }
          __syncwarp();
        }
        if (EPI & EPI_RES) mbar_wait(res_bar(ew, c), rphase);
        if (paced) {
          const long long until = pace_t0 + static_cast<long long>(2 * c + cgrp) * p.pace;
          while (clock64() < until) __nanosleep(32);
        }
        uint8_t* rowp = stage_gen[c] + lane * 128;
#pragma unroll
        for (int hh = 0; hh < 2; ++hh) {
          uint32_t r[32];
          tmem_ld_32x32(t_addr + c * kChunkCols + hh * 32, r);
          // bias (and folded-LayerNorm term) of these 32 columns, broadcast from the owning lanes
          // while the TMEM load is in flight
          float4 bv[8];
          float4 cv[(EPI & EPI_CSCALE) ? 8 : 1];
#pragma unroll
          for (int g = 0; g < 8; ++g) {
            const int src = 16 * c + 8 * hh + g;
            bv[g].x = __shfl_sync(0xffffffffu, b4.x, src);
            bv[g].y = __shfl_sync(0xffffffffu, b4.y, src);
            bv[g].z = __shfl_sync(0xffffffffu, b4.z, src);
            bv[g].w = __shfl_sync(0xffffffffu, b4.w, src);
            if (EPI & EPI_CSCALE) {
              cv[g].x = __shfl_sync(0xffffffffu, c4.x, src);
              cv[g].y = __shfl_sync(0xffffffffu, c4.y, src);
              cv[g].z = __shfl_sync(0xffffffffu, c4.z, src);
              cv[g].w = __shfl_sync(0xffffffffu, c4.w, src);
            }
            if ((EPI & EPI_LNF) && !(EPI & EPI_NOCS)) {
              float4 cs;
              cs.x = __shfl_sync(0xffffffffu, c4.x, src);
              cs.y = __shfl_sync(0xffffffffu, c4.y, src);
              cs.z = __shfl_sync(0xffffffffu, c4.z, src);
              cs.w = __shfl_sync(0xffffffffu, c4.w, src);
              const float2 lb = make_float2(ln_b, ln_b);
              const float2 lo = __ffma2_rn(lb, make_float2(cs.x, cs.y), make_float2(bv[g].x, bv[g].y));
              const float2 hi = __ffma2_rn(lb, make_float2(cs.z, cs.w), make_float2(bv[g].z, bv[g].w));
              bv[g] = make_float4(lo.x, lo.y, hi.x, hi.y);
            }
          }
          tmem_ld_wait();
          if (c == kChunks - 1 && hh == 1) {
            // accumulator fully read: hand the TMEM stage back to the MMA issuer before the math
            tc_fence_before();
            __syncwarp();
            if (lane == 0) mbar_arrive_leader(tempty_bar(as));
          }
          if (!live) continue;
#pragma unroll
          for (int jj = 0; jj < 4; ++jj) {
            const int j = hh * 4 + jj;           // 16-byte group within the 128-byte staging row
            // eight accumulator columns as four packed fp32 pairs: every add / FMA below is one FFMA2
            // (sm_100 f32x2) instead of two scalar instructions — the epilogues are bound by instruction
            // issue (fc1 + GELU: 174 -> 162 us per launch at C2)
            float2 v[4];
#pragma unroll
            for (int q = 0; q < 4; ++q)
              v[q] = make_float2(__uint_as_float(r[8 * jj + 2 * q]), __uint_as_float(r[8 * jj + 2 * q + 1]));
            {
              const float4 b0 = bv[2 * jj], b1 = bv[2 * jj + 1];
              const float2 bp[4] = {make_float2(b0.x, b0.y), make_float2(b0.z, b0.w), make_float2(b1.x, b1.y),
                                    make_float2(b1.z, b1.w)};
              if (EPI & EPI_CSCALE) {
                const float4 c0 = cv[2 * jj], c1 = cv[2 * jj + 1];
                const float2 cp[4] = {make_float2(c0.x, c0.y), make_float2(c0.z, c0.w), make_float2(c1.x, c1.y),
                                      make_float2(c1.z, c1.w)};
#pragma unroll
                for (int q = 0; q < 4; ++q) v[q] = __ffma2_rn(v[q], cp[q], bp[q]);
              } else if (EPI & EPI_LNF) {
                const float2 a2 = make_float2(ln_a, ln_a);
#pragma unroll
                for (int q = 0; q < 4; ++q) v[q] = __ffma2_rn(v[q], a2, bp[q]);
              } else {
#pragma unroll
                for (int q = 0; q < 4; ++q) v[q] = __fadd2_rn(v[q], bp[q]);
              }
            }
            uint4* slot = reinterpret_cast<uint4*>(rowp + ((j ^ sw) << 4));
            if (EPI & EPI_RES) {
              const uint4 r4 = *slot;
              v[0] = __fadd2_rn(v[0], make_float2(bf16_lo(r4.x), bf16_hi(r4.x)));
              v[1] = __fadd2_rn(v[1], make_float2(bf16_lo(r4.y), bf16_hi(r4.y)));
              v[2] = __fadd2_rn(v[2], make_float2(bf16_lo(r4.z), bf16_hi(r4.z)));
              v[3] = __fadd2_rn(v[3], make_float2(bf16_lo(r4.w), bf16_hi(r4.w)));
            }
            if (EPI & EPI_GELU) {
#pragma unroll
              for (int q = 0; q < 4; ++q) v[q] = gelu_epi2(v[q]);
            }
            if (EPI & EPI_QGELU) {
#pragma unroll
              for (int q = 0; q < 4; ++q) v[q] = quick_gelu_bf16_x2(v[q]);
            }
            if (EPI & EPI_STATS) {
              if (c == 0 && hh == 0 && jj == 0) st_npiv2 = make_float2(-v[0].x, -v[0].x);
#pragma unroll
              for (int q = 0; q < 4; ++q) {
                const float2 d = __fadd2_rn(v[q], st_npiv2);
                st_sum2 = __fadd2_rn(st_sum2, d);
                st_sq2 = __ffma2_rn(d, d, st_sq2);
              }
            }
            if (kFp8Out) {
              // e4m3 output: the warp's 128 columns are ONE 128-byte staging row (32 rows x 128 B, SWIZZLE_128B);
              // these eight columns are half of the 16-byte group (c * 4 + hh * 2 + jj / 2)
              const float2 os = make_float2(p.out_scale, p.out_scale);
#pragma unroll
              for (int q = 0; q < 4; ++q) v[q] = __fmul2_rn(v[q], os);
              uint2 o2;
              o2.x = pack_e4m3x4(v[0].x, v[0].y, v[1].x, v[1].y);
              o2.y = pack_e4m3x4(v[2].x, v[2].y, v[3].x, v[3].y);
              uint8_t* row8 = stage_gen[0] + lane * 128;
              *reinterpret_cast<uint2*>(row8 + (((c * 4 + hh * 2 + (jj >> 1)) ^ sw) << 4) + ((jj & 1) << 3)) = o2;
            } else {
              uint4 o4;
              o4.x = pack_bf16x2(v[0].x, v[0].y);
              o4.y = pack_bf16x2(v[1].x, v[1].y);
              o4.z = pack_bf16x2(v[2].x, v[2].y);
              o4.w = pack_bf16x2(v[3].x, v[3].y);
              *slot = o4;
            }
          }
        }
        if ((EPI & EPI_STATS) && c == kChunks - 1) {
          long long row = row0 + lane;
          bool row_ok = row < p.M;
          if (p.tok_pad > 0) {
            row_ok = row_ok && (tok0 + lane < p.tokens);   // rows past the last image exist in the last tile
            row = static_cast<long long>(img) * p.tokens + tok0 + lane;
          }
          if (col0 < p.N && row_ok) {             // N % 128 == 0: a warp's two chunks are both in or both out
            float2* dst = reinterpret_cast<float2*>(p.stats_out) + row * (p.N >> 7) + (col0 >> 7);
            const float s_sh = st_sum2.x + st_sum2.y, q_sh = st_sq2.x + st_sq2.y;
            *dst = make_float2(fmaf(-128.0f, st_npiv2.x, s_sh), fmaxf(fmaf(-s_sh * (1.0f / 128.0f), s_sh, q_sh), 0.f));
          }
        }
        if (kFp8Out) {
          if (c == kChunks - 1 && col0 < p.N) {     // one store of the warp's 128 e4m3 columns (N % 128 == 0, host)
            fence_proxy_async_smem();
            __syncwarp();
            if (lane == 0) {
              tma_store_2d(&tma_out, stage_buf[0], col0, row0);
              tma_store_commit();
            }
          }
        } else if (live) {
          fence_proxy_async_smem();
          __syncwarp();
          if (lane == 0) {
            if ((EPI & EPI_RES) && p.tok_pad > 0) tma_store_3d(&tma_out, stage_buf[c], col, tok0, img);
            else tma_store_2d(&tma_out, stage_buf[c], col, row0);
            tma_store_commit();
          }
        }
      }
      if (p.dbg) { const long long w1 = clock64(); dbg_acc[1] += w1 - w0; w0 = w1; }
      if (t + tile_step < num_tiles) prefetch_operands(t + tile_step);
      // staging buffers must be drained (read by the TMA engine) before the next tile reuses them
      if (lane == 0) tma_store_wait_read<0>();
      __syncwarp();
      if (p.dbg) dbg_acc[6] += clock64() - w0;
      rphase ^= 1u;
      if (++as == 2) { as = 0; aphase ^= 1u; }
    }
    if (lane == 0) tma_store_wait<0>();
  }

  if (p.dbg && lane == 0 && (warp_idx == kWarpProducer || warp_idx == kWarpMma || warp_idx == 0)) {
    long long* d = p.dbg + static_cast<long long>(blockIdx.x) * 8;
    if (warp_idx == 0) {
      d[0] = dbg_acc[0]; d[1] = dbg_acc[1]; d[6] = dbg_acc[6]; d[5] = clock64() - dbg_t0;
      unsigned long long ns1;
      asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(ns1));
      d[7] = static_cast<long long>(ns1 - dbg_ns0);      // wall time of the same interval: d[5] / d[7] = the real SM clock
      d[6] = static_cast<long long>(dbg_ns0);            // absolute start (replaces the store-drain counter): launch skew / gaps
    }
    if (warp_idx == kWarpMma) { d[2] = dbg_acc[2]; d[3] = dbg_acc[3]; }
    if (warp_idx == kWarpProducer) { d[4] = dbg_acc[4]; }
  }
  tc_fence_before();
  cluster_sync_all();
  if (warp_idx == kWarpTmem) {
    tc_fence_after();
    tmem_dealloc_2cta<512>(tmem_base);
  }
}

long long* g_dbg_buffer = nullptr;
int g_max_groups2 = 0;      // > 0: at most this many groups of four CTAs per GEMM launch (SM partitioning, see api.cu)

int g_num_sms2 = 0;
int num_sms2() {
  if (g_num_sms2 == 0) {
    int dev = 0;
    cudaGetDevice(&dev);
    cudaDeviceGetAttribute(&g_num_sms2, cudaDevAttrMultiProcessorCount, dev);
    if (g_num_sms2 <= 0) g_num_sms2 = 148;
  }
  return g_num_sms2;
}

template <int EPI, typename Cfg, int PREC = 0>
int launch2(const CUtensorMap& ta, const CUtensorMap& tb, const CUtensorMap& to,
            const CUtensorMap& tr, const CUtensorMap& ta64, const CUtensorMap& tb64, const Gemm2Params& p,
            cudaStream_t stream) {
  auto kern = gemm2_bf16_kernel<EPI, Cfg, PREC>;
  static int granted[kMaxDevices] = {0};
  if (const int rc_attr = ensure_dynamic_smem(kern, Cfg::kSmemBytes, granted)) return rc_attr;
  const int supertiles = (p.num_m_tiles >> 1) * p.num_n_tiles + ((p.num_m_tiles & 1) ? ((p.num_n_tiles + 1) >> 1) : 0);
  int groups = num_sms2() / 4;
  if (g_max_groups2 > 0 && g_max_groups2 < groups) groups = g_max_groups2;
  if (supertiles < groups) groups = supertiles;
  // regular clusters of 2 (one tcgen05 CTA pair), preferred clusters of 4 (two pairs that share an operand by TMA
  // multicast; VT_GEMM_QUAD=0: pairs only), programmatic dependent launch
  static const bool quad = [] { const char* e = getenv("VT_GEMM_QUAD"); return !(e && e[0] == '0'); }();
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = dim3(4 * groups);
  cfg.blockDim = dim3(kThreads);
  cfg.dynamicSmemBytes = Cfg::kSmemBytes;
  cfg.stream = stream;
  cudaLaunchAttribute attr[3];
  int na = 0;
  attr[na].id = cudaLaunchAttributeClusterDimension;
  attr[na].val.clusterDim.x = 2; attr[na].val.clusterDim.y = 1; attr[na].val.clusterDim.z = 1;
  ++na;
  if (quad) {
    attr[na].id = cudaLaunchAttributePreferredClusterDimension;
    attr[na].val.preferredClusterDim.x = 4; attr[na].val.preferredClusterDim.y = 1; attr[na].val.preferredClusterDim.z = 1;
    ++na;
  }
  if (pdl_enabled()) {
    attr[na].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    attr[na].val.programmaticStreamSerializationAllowed = 1;
    ++na;
  }
  cfg.attrs = attr;
  cfg.numAttrs = na;
  return static_cast<int>(cudaLaunchKernelEx(&cfg, kern, ta, tb, to, tr, ta64, tb64, p));
}

}  // namespace

void gemm2_set_debug_buffer(void* ptr) { g_dbg_buffer = static_cast<long long*>(ptr); }
void gemm2_set_max_groups(int n) { g_max_groups2 = n; }

// bf16 in / bf16 out 2-CTA GEMM.  Same argument meaning as gemm_bf16_tcgen05 (out dtype fixed), plus
// the optional LayerNorm fold (rowstats [+ colsum]: the A operand is the un-normalised activation and
// the weights carry gamma; without colsum their rows must sum to zero) and the optional output row statistics for the next fold.
int gemm2_bf16_tcgen05(const void* A, long long lda, const void* Bt, long long ldb, void* out,
                       long long ldo, const float* bias, const void* residual, long long ldr, int M,
                       int N, int K, int gelu, const float* rowstats, const float* colsum, int ln_dim,
                       float ln_eps, float* stats_out, int reverse, cudaStream_t stream) {
  if (!A || !Bt || !out || M <= 0 || N <= 0 || K <= 0 || !gemm_act_ok(gelu)) return VT_ERR_ARG;
  if (gelu && residual) return VT_ERR_UNSUPPORTED;
  if (colsum && !rowstats) return VT_ERR_ARG;
  if (rowstats && (residual || stats_out || ln_dim <= 0)) return VT_ERR_UNSUPPORTED;
  if (stats_out && (!residual || (N % 128))) return VT_ERR_UNSUPPORTED;
  if (rowstats && (ln_dim % 128)) return VT_ERR_UNSUPPORTED;
  if ((K % 8) || (lda % 8) || (ldb % 8) || (N % 8) || (ldo % 8) || (residual && (ldr % 8)))
    return VT_ERR_ALIGN;
  if ((reinterpret_cast<uintptr_t>(A) | reinterpret_cast<uintptr_t>(Bt) |
       reinterpret_cast<uintptr_t>(out) | reinterpret_cast<uintptr_t>(residual) |
       reinterpret_cast<uintptr_t>(bias) | reinterpret_cast<uintptr_t>(colsum)) & 15)
    return VT_ERR_ALIGN;
  if ((reinterpret_cast<uintptr_t>(rowstats) | reinterpret_cast<uintptr_t>(stats_out)) & 7)
    return VT_ERR_ALIGN;

  CUtensorMap ta, tb, to, tr, ta64, tb64;
  int rc = make_tmap_bf16_2d(&ta, A, K, M, lda, BK, BM, TMAP_SW_128);
  if (rc) return rc;
  rc = make_tmap_bf16_2d(&tb, Bt, K, N, ldb, BK, BNH, TMAP_SW_128);
  if (rc) return rc;
  rc = make_tmap_bf16_2d(&ta64, A, K, M, lda, BK, BM / 2, TMAP_SW_128);     // half boxes of the shared operand
  if (rc) return rc;
  rc = make_tmap_bf16_2d(&tb64, Bt, K, N, ldb, BK, BNH / 2, TMAP_SW_128);
  if (rc) return rc;
  rc = make_tmap_bf16_2d(&to, out, N, M, ldo, kChunkCols, 32, TMAP_SW_128);
  if (rc) return rc;
  if (residual) {
    rc = make_tmap_bf16_2d(&tr, residual, N, M, ldr, kChunkCols, 32, TMAP_SW_128);
    if (rc) return rc;
  } else {
    tr = to;
  }

  Gemm2Params p;
  p.M = M; p.N = N; p.K = K;
  p.num_m_tiles = (M + 2 * BM - 1) / (2 * BM);
  p.num_n_tiles = (N + BN - 1) / BN;
  p.reverse = reverse;
  p.bias = bias;
  p.rowstats = rowstats;
  p.colsum = colsum;
  p.ln_inv_dim = ln_dim > 0 ? 1.0f / static_cast<float>(ln_dim) : 0.f;
  p.ln_eps = ln_eps;
  p.ln_parts = ln_dim / 128;
  p.stats_out = stats_out;
  p.dbg = g_dbg_buffer;
  p.out_scale = 1.f;
  p.tok_pad = 0;
  p.tokens = 0;
  // Slot spacing: 21 % of the ideal tile time (K blocks x 4 MMAs x 128 cycles), at most that of a
  // K = 768 tile (1290 cycles: a K = 3072 tile gains nothing from wider slots), plus 5 % between the
  // four lane-quarter warps of a slot.  Measured (tools/gemm_dbg.py, cycles per launch at C2):
  // plain QKV 174.0k -> 157.9k, folded QKV 174.1k -> 159.3k, fc1 + GELU 230.7k -> 214.4k,
  // out-proj + residual 71.6k -> 67.0k, fc2 212.3k -> 206.5k.  VT_GEMM_PACE / VT_GEMM_PACE_Q (permille)
  // override; 0 switches pacing off.
  static const int pace_pm = [] { const char* e = getenv("VT_GEMM_PACE"); return e ? atoi(e) : 210; }();
  static const int pace_q_pm = [] { const char* e = getenv("VT_GEMM_PACE_Q"); return e ? atoi(e) : 50; }();
  long long ideal = static_cast<long long>((K + BK - 1) / BK) * 512;
  if (ideal > 6144) ideal = 6144;
  p.pace = static_cast<int>(ideal * pace_pm / 1000);
  p.pace_q = static_cast<int>(ideal * pace_q_pm / 1000);
  // Shared-memory split per epilogue (see G2Cfg): only the short-K residual epilogue (out-proj: its
  // residual chunks are TMA-prefetched into the staging buffers) keeps two staging buffers per warp;
  // everything else takes the sixth operand stage — with the paced epilogue and the prefetched
  // operands that now also holds for GELU (215.7k -> 209.4k cycles per fc1 launch) and the LayerNorm
  // fold (7947 -> 7050 cycles per tile).  VT_GEMM_STAGES=5|6 forces one for every launch,
  // VT_LNF_STAGES=5|6 for the LayerNorm-fold launches only, VT_GELU_STAGES=5|6 for the GELU and quick-GELU launches.
  static const int forced = [] {
    const char* e = getenv("VT_GEMM_STAGES");
    return (e && (e[0] == '5' || e[0] == '6')) ? (e[0] - '0') : 0;
  }();
  static const int forced_lnf = [] {
    const char* e = getenv("VT_LNF_STAGES");
    return (e && (e[0] == '5' || e[0] == '6')) ? (e[0] - '0') : 0;
  }();
  const bool epilogue_heavy = residual && K < 2048;
  bool deep = forced ? (forced == 6) : !epilogue_heavy;
  if (rowstats && forced_lnf) deep = (forced_lnf == 6);
  static const int forced_gelu = [] {
    const char* e = getenv("VT_GELU_STAGES");
    return (e && (e[0] == '5' || e[0] == '6')) ? (e[0] - '0') : 0;
  }();
  if (gelu && forced_gelu) deep = (forced_gelu == 6);
#define VT_G2_LAUNCH(E) (deep ? launch2<E, G2Deep>(ta, tb, to, tr, ta64, tb64, p, stream) : launch2<E, G2Wide>(ta, tb, to, tr, ta64, tb64, p, stream))
  const bool quick = gelu == kActQuickGelu;
  if (rowstats && !colsum) {
    if (!gelu) return VT_G2_LAUNCH(EPI_LNF | EPI_NOCS);
    return quick ? VT_G2_LAUNCH(EPI_LNF | EPI_NOCS | EPI_QGELU) : VT_G2_LAUNCH(EPI_LNF | EPI_NOCS | EPI_GELU);
  }
  if (rowstats) {
    if (!gelu) return VT_G2_LAUNCH(EPI_LNF);
    return quick ? VT_G2_LAUNCH(EPI_LNF | EPI_QGELU) : VT_G2_LAUNCH(EPI_LNF | EPI_GELU);
  }
  if (gelu) return quick ? VT_G2_LAUNCH(EPI_QGELU) : VT_G2_LAUNCH(EPI_GELU);
  if (residual) return stats_out ? VT_G2_LAUNCH(EPI_RES | EPI_STATS) : VT_G2_LAUNCH(EPI_RES);
  return VT_G2_LAUNCH(0);
#undef VT_G2_LAUNCH
}

// K2b: the patch-embedding GEMM in token mode.  A = gathered patch rows [B * tok_pad, K] (patch_gather.cu: row 0 of
// every image and the rows >= tokens are zero), W = conv weight [D, K] K-major, bias = conv bias (fp32),
// posb = bf16 [tokens, D] position table with row 0 = cls + pos[0] - bias:
//   out[b, t, :] = A[b, t, :] . W^T + bias + posb[t, :]        (t < tokens; + row statistics for the LayerNorm fold)
int gemm2_patch_tokens(const void* A, long long lda, const void* W, long long ldw, void* out, const float* bias,
                       const void* posb, float* stats_out, int B, int tok_pad, int tokens, int D, int K, int reverse,
                       cudaStream_t stream) {
  if (!A || !W || !out || !bias || !posb || B <= 0 || tokens <= 0 || D <= 0 || K <= 0) return VT_ERR_ARG;
  if ((tok_pad % 32) || tok_pad < tokens) return VT_ERR_ARG;
  if ((K % 8) || (lda % 8) || (ldw % 8) || (D % 8)) return VT_ERR_ALIGN;
  if (stats_out && (D % 128)) return VT_ERR_UNSUPPORTED;
  if ((reinterpret_cast<uintptr_t>(A) | reinterpret_cast<uintptr_t>(W) | reinterpret_cast<uintptr_t>(out) |
       reinterpret_cast<uintptr_t>(posb) | reinterpret_cast<uintptr_t>(bias)) & 15)
    return VT_ERR_ALIGN;
  if (reinterpret_cast<uintptr_t>(stats_out) & 7) return VT_ERR_ALIGN;
  const long long M = static_cast<long long>(B) * tok_pad;
  if (M >= (1LL << 31)) return VT_ERR_UNSUPPORTED;

  CUtensorMap ta, tb, to, tr, ta64, tb64;
  int rc = make_tmap_bf16_2d(&ta, A, K, M, lda, BK, BM, TMAP_SW_128);
  if (rc) return rc;
  rc = make_tmap_bf16_2d(&tb, W, K, D, ldw, BK, BNH, TMAP_SW_128);
  if (rc) return rc;
  rc = make_tmap_bf16_2d(&ta64, A, K, M, lda, BK, BM / 2, TMAP_SW_128);
  if (rc) return rc;
  rc = make_tmap_bf16_2d(&tb64, W, K, D, ldw, BK, BNH / 2, TMAP_SW_128);
  if (rc) return rc;
  rc = make_tmap_bf16_3d(&to, out, D, tokens, B, D, static_cast<uint64_t>(tokens) * D, kChunkCols, 32, TMAP_SW_128);
  if (rc) return rc;
  rc = make_tmap_bf16_2d(&tr, posb, D, tokens, D, kChunkCols, 32, TMAP_SW_128);
  if (rc) return rc;

  Gemm2Params p;
  p.M = static_cast<int>(M); p.N = D; p.K = K;
  p.num_m_tiles = static_cast<int>((M + 2 * BM - 1) / (2 * BM));
  p.num_n_tiles = (D + BN - 1) / BN;
  p.reverse = reverse;
  p.bias = bias;
  p.rowstats = nullptr;
  p.colsum = nullptr;
  p.ln_inv_dim = 0.f;
  p.ln_eps = 0.f;
  p.ln_parts = 0;
  p.stats_out = stats_out;
  p.dbg = g_dbg_buffer;
  p.out_scale = 1.f;
  p.tok_pad = tok_pad;
  p.tokens = tokens;
  long long ideal = static_cast<long long>((K + BK - 1) / BK) * 512;
  if (ideal > 6144) ideal = 6144;
  p.pace = static_cast<int>(ideal * 210 / 1000);
  p.pace_q = static_cast<int>(ideal * 50 / 1000);
  return stats_out ? launch2<EPI_RES | EPI_STATS, G2Wide>(ta, tb, to, tr, ta64, tb64, p, stream)
                   : launch2<EPI_RES, G2Wide>(ta, tb, to, tr, ta64, tb64, p, stream);
}

// FP8 form (behind vt_gemm_fp8 / VT_FP8=1, off the bf16 headline metric): A [M,K] and Bt [N,K] are e4m3 bytes
// (row strides in bytes, multiples of 16), accumulated in fp32 by tcgen05.mma kind::f8f6f4;
//   out = act(acc * colscale[n] + bias[n]) (+ residual)      colscale = weight scale of channel n x activation scale
// out is bf16 [M,N] or, with out_e4m3, e4m3(out * out_scale) (N % 128 == 0, no residual).
int gemm2_fp8_tcgen05(const void* A, long long lda, const void* Bt, long long ldb, void* out, long long ldo,
                      int out_e4m3, const float* bias, const float* colscale, const void* residual, long long ldr,
                      int M, int N, int K, int gelu, float out_scale, int reverse, cudaStream_t stream) {
  if (!A || !Bt || !out || !colscale || M <= 0 || N <= 0 || K <= 0 || !gemm_act_ok(gelu)) return VT_ERR_ARG;
  if (gelu && residual) return VT_ERR_UNSUPPORTED;
  if (out_e4m3 && (residual || (N % 128))) return VT_ERR_UNSUPPORTED;
  if ((K % 16) || (lda % 16) || (ldb % 16) || (N % 8) || (ldo % (out_e4m3 ? 16 : 8)) || (residual && (ldr % 8)))
    return VT_ERR_ALIGN;
  if ((reinterpret_cast<uintptr_t>(A) | reinterpret_cast<uintptr_t>(Bt) | reinterpret_cast<uintptr_t>(out) |
       reinterpret_cast<uintptr_t>(residual) | reinterpret_cast<uintptr_t>(bias) |
       reinterpret_cast<uintptr_t>(colscale)) & 15)
    return VT_ERR_ALIGN;

  CUtensorMap ta, tb, to, tr, ta64, tb64;
  int rc = make_tmap_u8_2d(&ta, A, K, M, lda, 2 * BK, BM, TMAP_SW_128);
  if (rc) return rc;
  rc = make_tmap_u8_2d(&tb, Bt, K, N, ldb, 2 * BK, BNH, TMAP_SW_128);
  if (rc) return rc;
  rc = make_tmap_u8_2d(&ta64, A, K, M, lda, 2 * BK, BM / 2, TMAP_SW_128);
  if (rc) return rc;
  rc = make_tmap_u8_2d(&tb64, Bt, K, N, ldb, 2 * BK, BNH / 2, TMAP_SW_128);
  if (rc) return rc;
  if (out_e4m3) rc = make_tmap_u8_2d(&to, out, N, M, ldo, 128, 32, TMAP_SW_128);
  else rc = make_tmap_bf16_2d(&to, out, N, M, ldo, kChunkCols, 32, TMAP_SW_128);
  if (rc) return rc;
  if (residual) {
    rc = make_tmap_bf16_2d(&tr, residual, N, M, ldr, kChunkCols, 32, TMAP_SW_128);
    if (rc) return rc;
  } else {
    tr = to;
  }

  Gemm2Params p;
  p.M = M; p.N = N; p.K = K;
  p.num_m_tiles = (M + 2 * BM - 1) / (2 * BM);
  p.num_n_tiles = (N + BN - 1) / BN;
  p.reverse = reverse;
  p.bias = bias;
  p.rowstats = nullptr;
  p.colsum = colscale;
  p.ln_inv_dim = 0.f;
  p.ln_eps = 0.f;
  p.ln_parts = 0;
  p.stats_out = nullptr;
  p.dbg = g_dbg_buffer;
  p.out_scale = out_scale;
  p.tok_pad = 0;
  p.tokens = 0;
  long long ideal = static_cast<long long>((K + 2 * BK - 1) / (2 * BK)) * 512;
  if (ideal > 6144) ideal = 6144;
  p.pace = static_cast<int>(ideal * 210 / 1000);
  p.pace_q = static_cast<int>(ideal * 50 / 1000);
  const bool quick = gelu == kActQuickGelu;
  if (out_e4m3) {
    if (quick) return launch2<EPI_CSCALE | EPI_QGELU, G2Deep, 2>(ta, tb, to, tr, ta64, tb64, p, stream);
    return gelu ? launch2<EPI_CSCALE | EPI_GELU, G2Deep, 2>(ta, tb, to, tr, ta64, tb64, p, stream)
                : launch2<EPI_CSCALE, G2Deep, 2>(ta, tb, to, tr, ta64, tb64, p, stream);
  }
  if (residual) return launch2<EPI_CSCALE | EPI_RES, G2Deep, 1>(ta, tb, to, tr, ta64, tb64, p, stream);
  if (quick) return launch2<EPI_CSCALE | EPI_QGELU, G2Deep, 1>(ta, tb, to, tr, ta64, tb64, p, stream);
  if (gelu) return launch2<EPI_CSCALE | EPI_GELU, G2Deep, 1>(ta, tb, to, tr, ta64, tb64, p, stream);
  return launch2<EPI_CSCALE, G2Deep, 1>(ta, tb, to, tr, ta64, tb64, p, stream);
}

}  // namespace vt
