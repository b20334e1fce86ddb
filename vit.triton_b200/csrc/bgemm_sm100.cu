// Batched general GEMM on tcgen05 (vt_bgemm): every contraction of the host API that is NOT one of the
// model's four big bf16 dense layers (those run the 2-CTA kernel, gemm2_sm100.cu) —
//
//   C[z] = act( scale * A[z] . B[z] + bias ) (+ residual[z]),   z = (outer, inner) batch index
//
//   * matmul3 (reference vit/kernels/matmul3.py:111-156: O[b] = s * A[b] . B[b], a tl.dot kernel) — B may be
//     given as [K, N] row-major exactly like the reference passes it (MN-major UMMA operand, no transpose
//     copy) or as [N, K] (K-major);
//   * the fp32 model (BASELINE configs[0]): fp32 operands are split into bf16 pieces by pack_split.cu
//     (a = a_hi + a_lo, three products a_hi b_hi + a_hi b_lo + a_lo b_hi laid side by side along K' = 3K),
//     so this kernel sees a bf16 GEMM with fp32 output: ~2^-16 relative per product, 4.7e-5 on the final
//     hidden states against 3.1e-3 for one TF32 pass (SURVEY.md 7.2) — the reference's own tl.dot
//     (matmul.py:92) is TF32;
//   * the pooler / classifier heads: A = the CLS rows of the final hidden states read in place through
//     the row stride of the tensor map, tanh epilogue (HF ViTPooler, modeling_vit.py:461-474; the reference
//     maps pooler.dense in vit/utils.py:63-64).
//
// Structure: persistent, one CTA per SM, 384 threads: warp 0 TMA producer, warp 1 MMA issuer (one elected
// lane, M = 128, N = BN, K = 16), warp 2 TMEM allocator, warps 4-11 epilogue (tcgen05.ld -> scale / bias /
// activation / residual -> fp32 | bf16 global stores).  Operands arrive through 4-D tensor maps
// (k, row, inner batch, outer batch), so batches need no pointer arrays and a tile never crosses a batch:
// rows and K columns beyond the matrix are zero-filled by TMA.  Tile = 128 x 128 (K-major B) or 128 x 64
// (MN-major B: one 64-element SWIZZLE_128B group per K row, the configuration the attention kernel uses
// for V), 4 / 6 smem stages of 64 K elements, double-buffered TMEM accumulator.
#include "common.cuh"
#include "tensormap.h"

namespace vt {

namespace {

constexpr int GB_BM = 128;
constexpr int GB_BK = 64;
constexpr int GB_EPI_WARPS = 8;
constexpr int GB_THREADS = 128 + GB_EPI_WARPS * 32;

enum : int { ACT_NONE = kActNone, ACT_GELU = kActGelu, ACT_TANH = kActTanh, ACT_QUICK_GELU = kActQuickGelu };

struct BgemmParams {
  int M, N, K;
  int num_m_tiles, num_n_tiles;
  int batch_inner, batch_total;
  int a_inner, a_outer;          // operand has its own data per inner / outer batch (else that coordinate is 0)
  int b_inner, b_outer;
  void* C;
  long long sCo, sCi, ldc;       // element strides of C: outer batch, inner batch, row (column stride 1)
  const void* residual;          // same dtype and strides as C, nullable
  const float* bias;             // [N] fp32, nullable
  float scale;
  int act;
  int out_f32;
  int vec_ok;                    // C (and residual) rows are 16-byte aligned: vector stores allowed
};

__device__ __forceinline__ void tma_load_4d(const CUtensorMap* m, uint32_t bar, uint32_t dst, int c0, int c1,
                                            int c2, int c3, uint64_t hint) {
  asm volatile(
      "cp.async.bulk.tensor.4d.shared::cluster.global.mbarrier::complete_tx::bytes.L2::cache_hint"
      " [%0], [%1, {%3, %4, %5, %6}], [%2], %7;"
      :
      : "r"(dst), "l"(reinterpret_cast<uint64_t>(m)), "r"(bar), "r"(c0), "r"(c1), "r"(c2), "r"(c3), "l"(hint)
      : "memory");
}

template <int BN, bool B_MN>
struct BgCfg {
  static constexpr int kABytes = GB_BM * GB_BK * 2;
  static constexpr int kBBytes = BN * GB_BK * 2;
  static constexpr int kStageBytes = kABytes + kBBytes;
  static constexpr int kStages = (BN >= 128) ? 4 : 6;
  static constexpr int kTmemCols = 2 * BN;
  static constexpr int kSmemBytes = 1024 + kStages * kStageBytes + 256;
};

template <int BN, bool B_MN>
__global__ void __launch_bounds__(GB_THREADS, 1)
bgemm_tcgen05_kernel(const __grid_constant__ CUtensorMap tma_a, const __grid_constant__ CUtensorMap tma_b,
                     const BgemmParams p) {
  using Cfg = BgCfg<BN, B_MN>;
  constexpr int kStages = Cfg::kStages;
  static_assert(!B_MN || BN == 64, "MN-major B: one 64-element swizzle group per K row");

  extern __shared__ uint8_t smem_raw[];
  const uint32_t smem_base = (smem_u32(smem_raw) + 1023u) & ~1023u;
  uint8_t* smem_gen = smem_raw + (smem_base - smem_u32(smem_raw));
  const uint32_t tiles_addr = smem_base;
  const uint32_t bar_addr = smem_base + kStages * Cfg::kStageBytes;
  auto full_bar = [&](int s) { return bar_addr + 8u * s; };
  auto empty_bar = [&](int s) { return bar_addr + 8u * (kStages + s); };
  auto tfull_bar = [&](int s) { return bar_addr + 8u * (2 * kStages + s); };
  auto tempty_bar = [&](int s) { return bar_addr + 8u * (2 * kStages + 2 + s); };
  const uint32_t tmem_slot = bar_addr + 8u * (2 * kStages + 4);
  volatile uint32_t* tmem_slot_gen =
      reinterpret_cast<volatile uint32_t*>(smem_gen + kStages * Cfg::kStageBytes + 8 * (2 * kStages + 4));

  const int warp_idx = threadIdx.x >> 5;
  const int lane = threadIdx.x & 31;

  if (warp_idx == 0 && lane == 0) {
    tma_prefetch_desc(&tma_a);
    tma_prefetch_desc(&tma_b);
  }
  if (warp_idx == 1 && lane == 0) {
    for (int s = 0; s < kStages; ++s) {
      mbar_init(full_bar(s), 1);
      mbar_init(empty_bar(s), 1);
    }
    for (int s = 0; s < 2; ++s) {
      mbar_init(tfull_bar(s), 1);
      mbar_init(tempty_bar(s), GB_EPI_WARPS);
    }
    fence_barrier_init();
  }
  if (warp_idx == 2) {
    tmem_alloc<Cfg::kTmemCols>(tmem_slot);
    tmem_relinquish();
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot_gen;

  const int tiles_per_batch = p.num_m_tiles * p.num_n_tiles;
  const long long num_tiles = static_cast<long long>(tiles_per_batch) * p.batch_total;
  const int num_kb = (p.K + GB_BK - 1) / GB_BK;

  // tile t -> (batch z, m block, n block): n fastest, so the CTAs of a wave share A rows through L2
  auto decode = [&](long long t, int& z, int& m_blk, int& n_blk) {
    z = static_cast<int>(t / tiles_per_batch);
    const int r = static_cast<int>(t - static_cast<long long>(z) * tiles_per_batch);
    m_blk = r / p.num_n_tiles;
    n_blk = r - m_blk * p.num_n_tiles;
  };

  if (warp_idx == 0) {
    // ------------------------------------------------------------------ TMA producer
    int s = 0;
    uint32_t phase = 0;
    for (long long t = blockIdx.x; t < num_tiles; t += gridDim.x) {
      int z, m_blk, n_blk;
      decode(t, z, m_blk, n_blk);
      const int zo = z / p.batch_inner, zi = z - zo * p.batch_inner;
      const int azi = p.a_inner ? zi : 0, azo = p.a_outer ? zo : 0;
      const int bzi = p.b_inner ? zi : 0, bzo = p.b_outer ? zo : 0;
      for (int kb = 0; kb < num_kb; ++kb) {
        mbar_wait(empty_bar(s), phase ^ 1u);
        if (elect_one_sync()) {
          const uint32_t a_dst = tiles_addr + s * Cfg::kStageBytes;
          const uint32_t b_dst = a_dst + Cfg::kABytes;
          mbar_arrive_expect_tx(full_bar(s), Cfg::kStageBytes);
          tma_load_4d(&tma_a, full_bar(s), a_dst, kb * GB_BK, m_blk * GB_BM, azi, azo, kEvictNormal);
          if (B_MN)   // B is [K, N] with N contiguous: box = 64 n x 64 k
            tma_load_4d(&tma_b, full_bar(s), b_dst, n_blk * BN, kb * GB_BK, bzi, bzo, kEvictNormal);
          else        // B is [N, K] with K contiguous: box = 64 k x BN n
            tma_load_4d(&tma_b, full_bar(s), b_dst, kb * GB_BK, n_blk * BN, bzi, bzo, kEvictNormal);
        }
        __syncwarp();
        if (++s == kStages) { s = 0; phase ^= 1u; }
      }
    }
  } else if (warp_idx == 1) {
    // ------------------------------------------------------------------ MMA issuer
    constexpr uint32_t idesc = make_idesc_bf16(GB_BM, BN, 0, B_MN ? 1 : 0);
    int s = 0;
    uint32_t phase = 0;
    int as = 0;
    uint32_t aphase = 0;
    for (long long t = blockIdx.x; t < num_tiles; t += gridDim.x) {
      mbar_wait(tempty_bar(as), aphase ^ 1u);
      tc_fence_after();
      const uint32_t d_tmem = tmem_base + as * BN;
      for (int kb = 0; kb < num_kb; ++kb) {
        mbar_wait(full_bar(s), phase);
        tc_fence_after();
        if (elect_one_sync()) {
          const uint32_t a_src = tiles_addr + s * Cfg::kStageBytes;
          const uint32_t b_src = a_src + Cfg::kABytes;
          const uint64_t adesc = make_desc_kmajor_sw128(a_src);
          // K-major: 16 K elements = 32 bytes along the row (+2 in 16-byte units); MN-major: 16 K rows of
          // 128 bytes = two 8-row swizzle atoms (+128 units)
          const uint64_t bdesc = B_MN ? make_desc_mnmajor_sw128(b_src, 1024) : make_desc_kmajor_sw128(b_src);
#pragma unroll
          for (int k = 0; k < GB_BK / 16; ++k)
            umma_ss(d_tmem, adesc + 2 * k, bdesc + (B_MN ? 128 : 2) * k, idesc, (kb | k) != 0 ? 1u : 0u);
          umma_commit(empty_bar(s));
        }
        __syncwarp();
        if (++s == kStages) { s = 0; phase ^= 1u; }
      }
      if (elect_one_sync()) umma_commit(tfull_bar(as));
      __syncwarp();
      if (++as == 2) { as = 0; aphase ^= 1u; }
    }
  } else if (warp_idx >= 4) {
    // ------------------------------------------------------------------ epilogue
    const int q = warp_idx & 3;            // TMEM lane quarter this warp may read
    const int half = (warp_idx - 4) >> 2;  // which half of the BN columns
    constexpr int kColsPerWarp = BN / 2;
    int as = 0;
    uint32_t aphase = 0;
    for (long long t = blockIdx.x; t < num_tiles; t += gridDim.x) {
      int z, m_blk, n_blk;
      decode(t, z, m_blk, n_blk);
      const int zo = z / p.batch_inner, zi = z - zo * p.batch_inner;
      const int row = m_blk * GB_BM + q * 32 + lane;
      const long long c_off = zo * p.sCo + zi * p.sCi + static_cast<long long>(row) * p.ldc;
      mbar_wait(tfull_bar(as), aphase);
      tc_fence_after();
#pragma unroll 1
      for (int c = 0; c < kColsPerWarp / 32; ++c) {
        const int col_in_tile = half * kColsPerWarp + c * 32;
        const int col = n_blk * BN + col_in_tile;
        uint32_t r[32];
        tmem_ld_32x32(tmem_base + (static_cast<uint32_t>(q * 32) << 16) + as * BN + col_in_tile, r);
        tmem_ld_wait();
        if (col >= p.N || row >= p.M) continue;
        float v[32];
#pragma unroll
        for (int i = 0; i < 32; ++i) {
          float x = __uint_as_float(r[i]) * p.scale;
          if (p.bias != nullptr && col + i < p.N) x += __ldg(p.bias + col + i);
          v[i] = x;
        }
        if (p.act == ACT_GELU) {
#pragma unroll
          for (int i = 0; i < 32; ++i) v[i] = gelu_erf(v[i]);
        } else if (p.act == ACT_TANH) {
#pragma unroll
          for (int i = 0; i < 32; ++i) v[i] = tanhf(v[i]);
        } else if (p.act == ACT_QUICK_GELU) {
#pragma unroll
          for (int i = 0; i < 32; ++i) v[i] = quick_gelu(v[i]);
        }
        const bool full_chunk = (col + 32 <= p.N) && p.vec_ok;
        if (p.out_f32) {
          float* o = static_cast<float*>(p.C) + c_off + col;
          const float* rs = p.residual ? static_cast<const float*>(p.residual) + c_off + col : nullptr;
          if (full_chunk) {
#pragma unroll
            for (int i = 0; i < 32; i += 4) {
              float4 o4 = make_float4(v[i], v[i + 1], v[i + 2], v[i + 3]);
              if (rs) {
                const float4 r4 = *reinterpret_cast<const float4*>(rs + i);
                o4.x += r4.x; o4.y += r4.y; o4.z += r4.z; o4.w += r4.w;
              }
              *reinterpret_cast<float4*>(o + i) = o4;
            }
          } else {
            for (int i = 0; i < 32 && col + i < p.N; ++i) o[i] = rs ? v[i] + rs[i] : v[i];
          }
        } else {
          __nv_bfloat16* o = static_cast<__nv_bfloat16*>(p.C) + c_off + col;
          const __nv_bfloat16* rs = p.residual ? static_cast<const __nv_bfloat16*>(p.residual) + c_off + col : nullptr;
          if (full_chunk) {
#pragma unroll
            for (int i = 0; i < 32; i += 8) {
              if (rs) {
                const uint4 r4 = *reinterpret_cast<const uint4*>(rs + i);
                v[i + 0] += bf16_lo(r4.x); v[i + 1] += bf16_hi(r4.x);
                v[i + 2] += bf16_lo(r4.y); v[i + 3] += bf16_hi(r4.y);
                v[i + 4] += bf16_lo(r4.z); v[i + 5] += bf16_hi(r4.z);
                v[i + 6] += bf16_lo(r4.w); v[i + 7] += bf16_hi(r4.w);
              }
              uint4 o4;
              o4.x = pack_bf16x2(v[i + 0], v[i + 1]);
              o4.y = pack_bf16x2(v[i + 2], v[i + 3]);
              o4.z = pack_bf16x2(v[i + 4], v[i + 5]);
              o4.w = pack_bf16x2(v[i + 6], v[i + 7]);
              *reinterpret_cast<uint4*>(o + i) = o4;
            }
          } else {
            for (int i = 0; i < 32 && col + i < p.N; ++i)
              o[i] = __float2bfloat16_rn(rs ? v[i] + __bfloat162float(rs[i]) : v[i]);
          }
        }
      }
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive(tempty_bar(as));
      if (++as == 2) { as = 0; aphase ^= 1u; }
    }
  }

  tc_fence_before();
  __syncthreads();
  if (warp_idx == 2) {
    tc_fence_after();
    tmem_dealloc<Cfg::kTmemCols>(tmem_base);
  }
}

// 4-D bf16 tensor map (cols, rows, inner batch, outer batch); strides in elements.  A batch level of
// extent 1 gets a harmless stride (the coordinate is always 0).
int make_tmap_bf16_4d(CUtensorMap* out, const void* base, uint64_t cols, uint64_t rows, uint64_t bi, uint64_t bo,
                      uint64_t row_stride, uint64_t bi_stride, uint64_t bo_stride, uint32_t box_cols,
                      uint32_t box_rows) {
  EncodeTiledFn enc = get_encode_tiled();
  if (!enc) return VT_ERR_DRIVER;
  const uint64_t safe = row_stride * (rows > 0 ? rows : 1);
  if (bi <= 1 || bi_stride == 0) { bi = 1; bi_stride = safe; }
  if (bo <= 1 || bo_stride == 0) { bo = 1; bo_stride = safe; }
  cuuint64_t dims[4] = {cols, rows, bi, bo};
  cuuint64_t strides[3] = {row_stride * 2, bi_stride * 2, bo_stride * 2};
  cuuint32_t box[4] = {box_cols, box_rows, 1, 1};
  cuuint32_t estr[4] = {1, 1, 1, 1};
  const CUresult r = enc(out, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 4, const_cast<void*>(base), dims, strides, box, estr,
                         CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                         CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  return r == CUDA_SUCCESS ? 0 : VT_ERR_DRIVER;
}

template <int BN, bool B_MN>
int launch_bgemm(const CUtensorMap& ta, const CUtensorMap& tb, const BgemmParams& p, cudaStream_t stream) {
  using Cfg = BgCfg<BN, B_MN>;
  auto kern = bgemm_tcgen05_kernel<BN, B_MN>;
  static int granted[kMaxDevices] = {0};
  if (const int rc = ensure_dynamic_smem(kern, Cfg::kSmemBytes, granted)) return rc;
  int dev = 0, sms = 148;
  cudaGetDevice(&dev);
  cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
  const long long tiles = static_cast<long long>(p.num_m_tiles) * p.num_n_tiles * p.batch_total;
  const int grid = static_cast<int>(tiles < sms ? tiles : sms);
  kern<<<grid, GB_THREADS, Cfg::kSmemBytes, stream>>>(ta, tb, p);
  return static_cast<int>(cudaGetLastError());
}

}  // namespace

// A: bf16 [bo, bi, M, K] K-major (strides sA = {outer, inner, row}, column stride 1).
// B: bf16; b_mn == 0: [bo, bi, N, K] K-major; b_mn != 0: [bo, bi, K, N] with N contiguous (sB = {outer, inner, row}).
// A batch stride of 0 broadcasts the operand along that level; 0 on both levels shares one matrix with all
// batches (weights).
// C / residual: bf16 | f32 [bo, bi, M, N] (sC = {outer, inner, row}); bias f32 [N].
int bgemm_tcgen05(const void* A, const void* B, void* C, const float* bias, const void* residual, int M, int N, int K,
                  int batch_outer, int batch_inner, const long long* sA, const long long* sB, const long long* sC,
                  int b_mn, float scale, int act, int out_dtype, cudaStream_t stream) {
  if (!A || !B || !C || !sA || !sB || !sC || M <= 0 || N <= 0 || K <= 0 || batch_outer <= 0 || batch_inner <= 0)
    return VT_ERR_ARG;
  if (out_dtype != VT_BF16 && out_dtype != VT_F32) return VT_ERR_DTYPE;
  if (act < ACT_NONE || act > ACT_QUICK_GELU) return VT_ERR_ARG;
  if (static_cast<long long>(batch_outer) * batch_inner >= (1LL << 30)) return VT_ERR_UNSUPPORTED;
  // TMA: base 16-byte aligned, every stride a multiple of 16 bytes
  if ((sA[0] % 8) || (sA[1] % 8) || (sA[2] % 8) || (sB[0] % 8) || (sB[1] % 8) || (sB[2] % 8)) return VT_ERR_ALIGN;
  if ((reinterpret_cast<uintptr_t>(A) | reinterpret_cast<uintptr_t>(B)) & 15) return VT_ERR_ALIGN;
  if (sA[2] < K || sB[2] < (b_mn ? N : K)) return VT_ERR_ARG;
  if (reinterpret_cast<uintptr_t>(bias) & 3) return VT_ERR_ALIGN;

  BgemmParams p;
  p.M = M; p.N = N; p.K = K;
  p.batch_inner = batch_inner;
  p.batch_total = batch_outer * batch_inner;
  p.a_inner = sA[1] != 0; p.a_outer = sA[0] != 0;
  p.b_inner = sB[1] != 0; p.b_outer = sB[0] != 0;
  p.C = C;
  p.sCo = sC[0]; p.sCi = sC[1]; p.ldc = sC[2];
  p.residual = residual;
  p.bias = bias;
  p.scale = scale;
  p.act = act;
  p.out_f32 = (out_dtype == VT_F32);
  const int es = p.out_f32 ? 4 : 2;
  const int per16 = 16 / es;
  p.vec_ok = ((sC[0] % per16) == 0 && (sC[1] % per16) == 0 && (sC[2] % per16) == 0 &&
              ((reinterpret_cast<uintptr_t>(C) | reinterpret_cast<uintptr_t>(residual)) & 15) == 0)
                 ? 1 : 0;
  p.num_m_tiles = (M + GB_BM - 1) / GB_BM;

  CUtensorMap ta, tb;
  const uint64_t abi = p.a_inner ? batch_inner : 1, abo = p.a_outer ? batch_outer : 1;
  const uint64_t bbi = p.b_inner ? batch_inner : 1, bbo = p.b_outer ? batch_outer : 1;
  int rc = make_tmap_bf16_4d(&ta, A, K, M, abi, abo, sA[2], sA[1], sA[0], GB_BK, GB_BM);
  if (rc) return rc;
  if (b_mn) {
    p.num_n_tiles = (N + 63) / 64;
    rc = make_tmap_bf16_4d(&tb, B, N, K, bbi, bbo, sB[2], sB[1], sB[0], 64, GB_BK);
    if (rc) return rc;
    return launch_bgemm<64, true>(ta, tb, p, stream);
  }
  p.num_n_tiles = (N + 127) / 128;
  rc = make_tmap_bf16_4d(&tb, B, K, N, bbi, bbo, sB[2], sB[1], sB[0], GB_BK, 128);
  if (rc) return rc;
  return launch_bgemm<128, false>(ta, tb, p, stream);
}

}  // namespace vt
