// K1: persistent, warp-specialised bf16 GEMM on tcgen05 tensor cores with TMEM accumulators.
//
//   out[M,N] = epilogue( A[M,K] . Bt[N,K]^T + bias[N] )        (both operands K-major)
//
// Replaces the Triton `matmul_kernel` (reference vit/kernels/matmul.py:40-108: fp32 accumulate,
// bias add :100-102, exact-erf GELU :104-106) and, through the residual epilogue, the two
// `add_kernel` launches per layer (reference vit/vit.py:140,147).
//
// Structure (one CTA per SM, 384 threads):
//   warp 0      TMA producer: A tile 128x64 and B tile BNx64 per stage, SWIZZLE_128B
//   warp 1      MMA issuer:   one thread issues tcgen05.mma (M=128, N=BN, K=16) x 4 per stage
//   warp 2      TMEM allocator (2 x BN fp32 columns = double-buffered accumulator)
//   warps 4-11  epilogue: tcgen05.ld -> bias / GELU / residual -> bf16|f32 -> global
// Three mbarrier pipelines: smem full/empty, TMEM full/empty, static persistent tile schedule.
#include "common.cuh"
#include "tensormap.h"

namespace vt {

namespace {

constexpr int BM = 128;
constexpr int BK = 64;
constexpr int kEpiWarps = 8;
constexpr int kThreads = 128 + kEpiWarps * 32;

enum : int { EPI_GELU = 1, EPI_RES = 2, EPI_F32 = 4, EPI_QGELU = 8 };   // EPI_QGELU: quick GELU (CLIP)

struct GemmParams {
  int M, N, K;
  int num_m_tiles, num_n_tiles;
  void* out;
  long long ldo;
  const float* bias;
  const void* residual;
  long long ldr;
};

template <int BN>
struct GemmCfg {
  static constexpr int kABytes = BM * BK * 2;
  static constexpr int kBBytes = BN * BK * 2;
  static constexpr int kStageBytes = kABytes + kBBytes;
  static constexpr int kStages = (BN == 256) ? 4 : 6;
  static constexpr int kTmemCols = 2 * BN;
  // 1024 B alignment slack + tiles + barriers
  static constexpr int kSmemBytes = 1024 + kStages * kStageBytes + 256;
};

template <int BN, int EPI>
__global__ void __launch_bounds__(kThreads, 1)
gemm_bf16_tcgen05_kernel(const __grid_constant__ CUtensorMap tma_a,
                         const __grid_constant__ CUtensorMap tma_b, const GemmParams p) {
  using Cfg = GemmCfg<BN>;
  constexpr int kStages = Cfg::kStages;

  extern __shared__ uint8_t smem_raw[];
  const uint32_t smem_base = (smem_u32(smem_raw) + 1023u) & ~1023u;
  uint8_t* smem_gen = smem_raw + (smem_base - smem_u32(smem_raw));

  const uint32_t tiles_addr = smem_base;
  const uint32_t bar_addr = smem_base + kStages * Cfg::kStageBytes;
  // barrier block layout (8 B each): full[kStages], empty[kStages], tfull[2], tempty[2], tmem ptr
  auto full_bar = [&](int s) { return bar_addr + 8u * s; };
  auto empty_bar = [&](int s) { return bar_addr + 8u * (kStages + s); };
  auto tfull_bar = [&](int s) { return bar_addr + 8u * (2 * kStages + s); };
  auto tempty_bar = [&](int s) { return bar_addr + 8u * (2 * kStages + 2 + s); };
  const uint32_t tmem_slot = bar_addr + 8u * (2 * kStages + 4);
  volatile uint32_t* tmem_slot_gen =
      reinterpret_cast<volatile uint32_t*>(smem_gen + kStages * Cfg::kStageBytes +
                                           8 * (2 * kStages + 4));

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
      mbar_init(tempty_bar(s), kEpiWarps);
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

  const int num_tiles = p.num_m_tiles * p.num_n_tiles;
  const int num_kb = (p.K + BK - 1) / BK;

  if (warp_idx == 0) {
    // ------------------------------------------------------------------ TMA producer
    if (lane == 0) {
      int s = 0;
      uint32_t phase = 0;
      for (int t = blockIdx.x; t < num_tiles; t += gridDim.x) {
        const int m_blk = t / p.num_n_tiles;
        const int n_blk = t - m_blk * p.num_n_tiles;
        for (int kb = 0; kb < num_kb; ++kb) {
          mbar_wait(empty_bar(s), phase ^ 1u);
          const uint32_t a_dst = tiles_addr + s * Cfg::kStageBytes;
          const uint32_t b_dst = a_dst + Cfg::kABytes;
          mbar_arrive_expect_tx(full_bar(s), Cfg::kStageBytes);
          tma_load_2d(&tma_a, full_bar(s), a_dst, kb * BK, m_blk * BM, kEvictNormal);
          tma_load_2d(&tma_b, full_bar(s), b_dst, kb * BK, n_blk * BN, kEvictLast);
          if (++s == kStages) { s = 0; phase ^= 1u; }
        }
      }
    }
  } else if (warp_idx == 1) {
    // ------------------------------------------------------------------ MMA issuer
    if (lane == 0) {
      constexpr uint32_t idesc = make_idesc_bf16(BM, BN, 0, 0);
      int s = 0;
      uint32_t phase = 0;
      int as = 0;
      uint32_t aphase = 0;
      for (int t = blockIdx.x; t < num_tiles; t += gridDim.x) {
        mbar_wait(tempty_bar(as), aphase ^ 1u);
        tc_fence_after();
        const uint32_t d_tmem = tmem_base + as * BN;
        for (int kb = 0; kb < num_kb; ++kb) {
          mbar_wait(full_bar(s), phase);
          tc_fence_after();
          const uint32_t a_src = tiles_addr + s * Cfg::kStageBytes;
          const uint32_t b_src = a_src + Cfg::kABytes;
#pragma unroll
          for (int k = 0; k < BK / 16; ++k) {
            const uint64_t adesc = make_desc_kmajor_sw128(a_src + k * 32);
            const uint64_t bdesc = make_desc_kmajor_sw128(b_src + k * 32);
            umma_ss(d_tmem, adesc, bdesc, idesc, (kb | k) != 0 ? 1u : 0u);
          }
          umma_commit(empty_bar(s));
          if (++s == kStages) { s = 0; phase ^= 1u; }
        }
        umma_commit(tfull_bar(as));
        if (++as == 2) { as = 0; aphase ^= 1u; }
      }
    }
  } else if (warp_idx >= 4) {
    // ------------------------------------------------------------------ epilogue
    const int q = warp_idx & 3;            // TMEM lane quarter this warp may read
    const int half = (warp_idx - 4) >> 2;  // which half of the BN columns
    constexpr int kColsPerWarp = BN / 2;
    int as = 0;
    uint32_t aphase = 0;
    for (int t = blockIdx.x; t < num_tiles; t += gridDim.x) {
      const int m_blk = t / p.num_n_tiles;
      const int n_blk = t - m_blk * p.num_n_tiles;
      const int row = m_blk * BM + q * 32 + lane;
      mbar_wait(tfull_bar(as), aphase);
      tc_fence_after();
#pragma unroll 1
      for (int c = 0; c < kColsPerWarp / 32; ++c) {
        const int col_in_tile = half * kColsPerWarp + c * 32;
        const int col = n_blk * BN + col_in_tile;
        uint32_t r[32];
        tmem_ld_32x32(tmem_base + (static_cast<uint32_t>(q * 32) << 16) + as * BN + col_in_tile, r);
        tmem_ld_wait();
        if (col >= p.N) continue;  // warp-uniform
        float v[32];
        if (p.bias != nullptr) {
#pragma unroll
          for (int i = 0; i < 32; i += 4) {
            float4 b4;
            if (col + i + 3 < p.N) {
              b4 = __ldg(reinterpret_cast<const float4*>(p.bias + col + i));
            } else {
              b4.x = (col + i + 0 < p.N) ? __ldg(p.bias + col + i + 0) : 0.f;
              b4.y = (col + i + 1 < p.N) ? __ldg(p.bias + col + i + 1) : 0.f;
              b4.z = (col + i + 2 < p.N) ? __ldg(p.bias + col + i + 2) : 0.f;
              b4.w = 0.f;
            }
            v[i + 0] = __uint_as_float(r[i + 0]) + b4.x;
            v[i + 1] = __uint_as_float(r[i + 1]) + b4.y;
            v[i + 2] = __uint_as_float(r[i + 2]) + b4.z;
            v[i + 3] = __uint_as_float(r[i + 3]) + b4.w;
          }
        } else {
#pragma unroll
          for (int i = 0; i < 32; ++i) v[i] = __uint_as_float(r[i]);
        }
        if (EPI & EPI_GELU) {
#pragma unroll
          for (int i = 0; i < 32; ++i) v[i] = gelu_erf(v[i]);
        }
        if (EPI & EPI_QGELU) {
#pragma unroll
          for (int i = 0; i < 32; ++i) v[i] = quick_gelu(v[i]);
        }
        if (row < p.M) {
          const bool full_chunk = (col + 32 <= p.N);
          if (EPI & EPI_F32) {
            float* o = reinterpret_cast<float*>(p.out) + static_cast<long long>(row) * p.ldo + col;
            const float* rs = (EPI & EPI_RES)
                                  ? reinterpret_cast<const float*>(p.residual) +
                                        static_cast<long long>(row) * p.ldr + col
                                  : nullptr;
            if (full_chunk) {
#pragma unroll
              for (int i = 0; i < 32; i += 4) {
                float4 o4 = make_float4(v[i], v[i + 1], v[i + 2], v[i + 3]);
                if (EPI & EPI_RES) {
                  const float4 r4 = *reinterpret_cast<const float4*>(rs + i);
                  o4.x += r4.x; o4.y += r4.y; o4.z += r4.z; o4.w += r4.w;
                }
                *reinterpret_cast<float4*>(o + i) = o4;
              }
            } else {
              for (int i = 0; i < 32 && col + i < p.N; ++i) {
                float x = v[i];
                if (EPI & EPI_RES) x += rs[i];
                o[i] = x;
              }
            }
          } else {
            __nv_bfloat16* o = reinterpret_cast<__nv_bfloat16*>(p.out) +
                               static_cast<long long>(row) * p.ldo + col;
            const __nv_bfloat16* rs = (EPI & EPI_RES)
                                          ? reinterpret_cast<const __nv_bfloat16*>(p.residual) +
                                                static_cast<long long>(row) * p.ldr + col
                                          : nullptr;
            if (full_chunk) {
#pragma unroll
              for (int i = 0; i < 32; i += 8) {
                if (EPI & EPI_RES) {
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
              for (int i = 0; i < 32 && col + i < p.N; ++i) {
                float x = v[i];
                if (EPI & EPI_RES) x += __bfloat162float(rs[i]);
                o[i] = __float2bfloat16_rn(x);
              }
            }
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

int g_num_sms = 0;
int num_sms() {
  if (g_num_sms == 0) {
    int dev = 0;
    cudaGetDevice(&dev);
    cudaDeviceGetAttribute(&g_num_sms, cudaDevAttrMultiProcessorCount, dev);
    if (g_num_sms <= 0) g_num_sms = 148;
  }
  return g_num_sms;
}

template <int BN, int EPI>
int launch_cfg(const CUtensorMap& ta, const CUtensorMap& tb, const GemmParams& p,
               cudaStream_t stream) {
  using Cfg = GemmCfg<BN>;
  auto kern = gemm_bf16_tcgen05_kernel<BN, EPI>;
  static int granted[kMaxDevices] = {0};
  if (const int rc_attr = ensure_dynamic_smem(kern, Cfg::kSmemBytes, granted)) return rc_attr;
  const int tiles = p.num_m_tiles * p.num_n_tiles;
  const int grid = tiles < num_sms() ? tiles : num_sms();
  kern<<<grid, kThreads, Cfg::kSmemBytes, stream>>>(ta, tb, p);
  return static_cast<int>(cudaGetLastError());
}

template <int BN>
int launch_bn(const CUtensorMap& ta, const CUtensorMap& tb, const GemmParams& p, int epi,
              cudaStream_t stream) {
  switch (epi) {
    case 0: return launch_cfg<BN, 0>(ta, tb, p, stream);
    case EPI_GELU: return launch_cfg<BN, EPI_GELU>(ta, tb, p, stream);
    case EPI_RES: return launch_cfg<BN, EPI_RES>(ta, tb, p, stream);
    case EPI_F32: return launch_cfg<BN, EPI_F32>(ta, tb, p, stream);
    case EPI_F32 | EPI_GELU: return launch_cfg<BN, EPI_F32 | EPI_GELU>(ta, tb, p, stream);
    case EPI_QGELU: return launch_cfg<BN, EPI_QGELU>(ta, tb, p, stream);
    case EPI_F32 | EPI_QGELU: return launch_cfg<BN, EPI_F32 | EPI_QGELU>(ta, tb, p, stream);
    case EPI_F32 | EPI_RES: return launch_cfg<BN, EPI_F32 | EPI_RES>(ta, tb, p, stream);
    default: return VT_ERR_UNSUPPORTED;
  }
}

}  // namespace

// A [M,K] bf16 (row stride lda), Bt [N,K] bf16 (row stride ldb), out [M,N] bf16|f32.
// residual has the dtype of out.  bias is fp32 (may be null).
int gemm_bf16_tcgen05(const void* A, long long lda, const void* Bt, long long ldb, void* out,
                      long long ldo, int out_dtype, const float* bias, const void* residual,
                      long long ldr, int M, int N, int K, int gelu, cudaStream_t stream) {
  if (!A || !Bt || !out || M <= 0 || N <= 0 || K <= 0 || !gemm_act_ok(gelu)) return VT_ERR_ARG;
  if (gelu && residual) return VT_ERR_UNSUPPORTED;
  if ((K % 8) || (lda % 8) || (ldb % 8) || (N % 8) || (ldo % 8) || (residual && (ldr % 8)))
    return VT_ERR_ALIGN;
  if ((reinterpret_cast<uintptr_t>(A) | reinterpret_cast<uintptr_t>(Bt) |
       reinterpret_cast<uintptr_t>(out) | reinterpret_cast<uintptr_t>(residual) |
       reinterpret_cast<uintptr_t>(bias)) & 15)
    return VT_ERR_ALIGN;
  if (out_dtype != VT_BF16 && out_dtype != VT_F32) return VT_ERR_DTYPE;

  const int bn = (N >= 256 || N > 128) ? 256 : 128;
  CUtensorMap ta, tb;
  int rc = make_tmap_bf16_2d(&ta, A, K, M, lda, BK, BM, TMAP_SW_128);
  if (rc) return rc;
  rc = make_tmap_bf16_2d(&tb, Bt, K, N, ldb, BK, bn, TMAP_SW_128);
  if (rc) return rc;

  GemmParams p;
  p.M = M; p.N = N; p.K = K;
  p.num_m_tiles = (M + BM - 1) / BM;
  p.num_n_tiles = (N + bn - 1) / bn;
  p.out = out; p.ldo = ldo;
  p.bias = bias;
  p.residual = residual; p.ldr = ldr;
  int epi = (gelu == kActGelu ? EPI_GELU : gelu == kActQuickGelu ? EPI_QGELU : 0) | (residual ? EPI_RES : 0) | (out_dtype == VT_F32 ? EPI_F32 : 0);
  return bn == 256 ? launch_bn<256>(ta, tb, p, epi, stream) : launch_bn<128>(ta, tb, p, epi, stream);
}

}  // namespace vt
