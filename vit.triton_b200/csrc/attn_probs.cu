// vt_attn_probs: the attention probabilities of every head as a dense bf16 [B, H, N, N] tensor (HF ViTModel's
// output_attentions), from the same fused-QKV activation that vt_flash_attn reads.
//
//   probs[b, h, i, j] = exp2(a_ij - m_i) / sum_j exp2(a_ij - m_i),  a_ij = scale * log2(e) * (q_i . k_j),  m_i = max_j a_ij
//
// One work item is one (image, head, 128-query tile); a CTA of four warps walks items blockIdx.x, + gridDim.x, ...
// (a 1-D persistent grid: B * H is unbounded).  Per item:
//   pass A  for each key block j (bkv <= 256 keys): TMA Q (first block) and K_j, S = Q K_j^T by tcgen05.mma into TMEM
//           (thread = query row = TMEM lane), row max of the block, then the running sum
//           l = l * exp2(m_old - m_new) + sum exp2(a - m_new).  With a single block (N <= 256) the exponentials are
//           written back over the scores in TMEM.
//   pass B  for each key block: (single block) read the exponentials back, or (several blocks) recompute S = Q K_j^T
//           and the exponentials against the final max; multiply by 1 / l, round to bf16 once and stage in shared
//           memory, then store.
// Stores.  Rows of N bf16 are generally not 16-byte aligned (N = 197: 394 bytes), so a 2-D TMA store cannot write
// them.  With a single key block the 32 rows of a warp are one contiguous span of 32 N elements of probs; the warp
// stages it in shared memory at the same offset modulo 16 bytes as its destination and copies it with 16-byte vector
// stores in the middle and scalar head and tail elements.  With several blocks each row's block segment is such a
// span.  No store ever leaves its span.
// The flow inside a CTA is serial (load -> MMA -> passes -> store); two CTAs share an SM (256 TMEM columns and at
// least 80 KB of shared memory each), so one CTA's loads and MMAs overlap the other's exponentials and stores.
// The exponentials run on the MUFU (ex2.approx); the flash kernel's FMA-pipe polynomial is not used here.
#include "../../include/vitb200_attn.h"
#include "common.cuh"
#include "tensormap.h"

namespace vt {

namespace {

constexpr int kPQT = 128;                 // query rows per item (= TMEM lanes)
constexpr int kPThreads = 128;            // four warps, warp w owns TMEM lanes / query rows 32 w .. 32 w + 31
constexpr int kPCols = 256;               // TMEM columns: one block of scores
constexpr int kPSingle = 256;             // N up to this: one key block, scores stay in TMEM between the passes
constexpr int kPBlock = 128;              // longer sequences: key blocks of at most this many keys
constexpr int kPMinSmem = 80 * 1024;      // at most two CTAs per SM: two TMEM allocations of 256 columns fit
constexpr int kPSmemLimit = 232448;

struct ProbsParams {
  int N, H, B;
  int nqt;            // query tiles per (image, head)
  int nblk, bkv;      // key blocks per row, keys per block (multiple of 16)
  int pitch;          // several blocks: staging row pitch in elements (bkv + 8)
  long long total_items;
  float scale_log2;
  uint16_t* probs;
};

// Copy n bf16 elements from shared memory to global memory, cooperatively by one warp.  src and dst have the same
// address modulo 16 bytes: head elements up to dst's first 16-byte boundary, 16-byte vectors, then the tail.
__device__ __forceinline__ void store_span(const uint16_t* src, uint16_t* dst, long long n, int lane) {
  const long long head = min(n, static_cast<long long>((8 - ((reinterpret_cast<uintptr_t>(dst) >> 1) & 7)) & 7));
  if (lane < head) dst[lane] = src[lane];
  const long long nvec = (n - head) >> 3;
  const uint4* sv = reinterpret_cast<const uint4*>(src + head);
  uint4* dv = reinterpret_cast<uint4*>(dst + head);
  for (long long i = lane; i < nvec; i += 32) dv[i] = sv[i];
  const long long t0 = head + (nvec << 3);
  if (t0 + lane < n) dst[t0 + lane] = src[t0 + lane];
}

template <int DH>
__global__ void __launch_bounds__(kPThreads, 1)
attn_probs_kernel(const __grid_constant__ CUtensorMap tma_q, const __grid_constant__ CUtensorMap tma_k,
                  const __grid_constant__ CUtensorMap tma_qt, const __grid_constant__ CUtensorMap tma_kt,
                  const ProbsParams p) {
  static_assert(DH == 64 || DH == 80, "head dim 64 or 80");
  constexpr int kDT = DH - 64;                     // 0 or 16: columns of the SWIZZLE_32B tail
  constexpr int kQBytes = kPQT * 64 * 2;
  constexpr int kQTailBytes = kPQT * kDT * 2;
  extern __shared__ uint8_t smem_raw[];
  const uint32_t smem_base = (smem_u32(smem_raw) + 1023u) & ~1023u;
  uint8_t* smem_gen = smem_raw + (smem_base - smem_u32(smem_raw));

  const int k_bytes = p.bkv * 64 * 2;
  const int kt_bytes = p.bkv * kDT * 2;
  // [Q][K][Q tail][K tail][staging: 4 warps][barriers][tmem slot]
  const uint32_t q_smem = smem_base;
  const uint32_t k_smem = q_smem + kQBytes;
  const uint32_t qt_smem = k_smem + k_bytes;
  const uint32_t kt_smem = qt_smem + kQTailBytes;
  const int stage_off = kQBytes + k_bytes + kQTailBytes + kt_bytes;
  const int stage_elems = p.nblk == 1 ? 32 * p.N + 8 : 32 * p.pitch;   // per warp
  const int stage_warp = (stage_elems + 7) & ~7;
  const int bar_off = stage_off + 4 * stage_warp * 2;
  const uint32_t bar_load = smem_base + bar_off;
  const uint32_t bar_mma = bar_load + 8;
  const uint32_t tmem_slot = bar_load + 16;
  volatile uint32_t* tmem_slot_gen = reinterpret_cast<volatile uint32_t*>(smem_gen + bar_off + 16);

  const int warp = threadIdx.x >> 5;
  const int lane = threadIdx.x & 31;
  uint16_t* stage = reinterpret_cast<uint16_t*>(smem_gen + stage_off) + warp * stage_warp;

  if (threadIdx.x == 0) {
    mbar_init(bar_load, 1);
    mbar_init(bar_mma, 1);
    fence_barrier_init();
    tma_prefetch_desc(&tma_q);
    tma_prefetch_desc(&tma_k);
    if (kDT) {
      tma_prefetch_desc(&tma_qt);
      tma_prefetch_desc(&tma_kt);
    }
  }
  if (warp == 0) {
    tmem_alloc<kPCols>(tmem_slot);
    tmem_relinquish();
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot_gen;
  const uint32_t t_lane = tmem_base + (static_cast<uint32_t>(warp * 32) << 16);
  const uintptr_t probs_elem0 = reinterpret_cast<uintptr_t>(p.probs) >> 1;   // element address of probs[0]

  uint32_t ld_ph = 0, mma_ph = 0;
  // S = Q K_j^T of the current item into TMEM columns [0, nj); every thread returns when it is there
  auto scores = [&](int img, int head, int qt, int j, bool with_q, int nj) {
    if (threadIdx.x == 0) {
      mbar_arrive_expect_tx(bar_load, (with_q ? kQBytes + kQTailBytes : 0) + k_bytes + kt_bytes);
      if (with_q) {
        tma_load_3d(&tma_q, bar_load, q_smem, head * DH, qt * kPQT, img, kEvictFirst);
        if (kDT) tma_load_3d(&tma_qt, bar_load, qt_smem, head * DH + 64, qt * kPQT, img, kEvictFirst);
      }
      tma_load_3d(&tma_k, bar_load, k_smem, head * DH, j * p.bkv, img, kEvictNormal);
      if (kDT) tma_load_3d(&tma_kt, bar_load, kt_smem, head * DH + 64, j * p.bkv, img, kEvictNormal);
      mbar_wait(bar_load, ld_ph);
      tc_fence_after();
      const uint32_t idesc = make_idesc_bf16(kPQT, nj, 0, 0);
      const uint64_t qd = make_desc_kmajor_sw128(q_smem);
      const uint64_t kd = make_desc_kmajor_sw128(k_smem);
#pragma unroll
      for (int k = 0; k < 4; ++k) umma_ss(tmem_base, qd + 2 * k, kd + 2 * k, idesc, k != 0 ? 1u : 0u);
      if (kDT)   // fifth K step on the 16-column SWIZZLE_32B tiles (rows of 32 B, 8-row atoms of 256 B)
        umma_ss(tmem_base, make_smem_desc(qt_smem, 0, 256, 6), make_smem_desc(kt_smem, 0, 256, 6), idesc, 1u);
      umma_commit(bar_mma);
    }
    ld_ph ^= 1u;
    mbar_wait(bar_mma, mma_ph);
    mma_ph ^= 1u;
    tc_fence_after();
  };
  // every thread is done with TMEM and the staging tile: the next MMA / TMA may overwrite them
  auto release = [&]() {
    tc_fence_before();
    __syncthreads();
  };

  const int nv_last = p.N - (p.nblk - 1) * p.bkv;
  for (long long item = blockIdx.x; item < p.total_items; item += gridDim.x) {
    const int qt = static_cast<int>(item % p.nqt);
    const long long bh = item / p.nqt;
    const int head = static_cast<int>(bh % p.H);
    const int img = static_cast<int>(bh / p.H);
    const int r0 = qt * kPQT + warp * 32;             // first query row of this warp
    const int row = r0 + lane;
    const bool live = r0 < p.N;                       // warp-uniform: some row of the warp is a real query
    const bool mine = row < p.N;
    const long long row_elem = (bh * p.N + row) * static_cast<long long>(p.N);   // probs element of (row, 0)

    // ---------------------------------------------------------------- pass A: row max and sum
    float m = -INFINITY, l = 0.f;
    for (int j = 0; j < p.nblk; ++j) {
      const int nv = (j == p.nblk - 1) ? nv_last : p.bkv;
      const int nj = (nv + 15) & ~15;
      scores(img, head, qt, j, j == 0, nj);
      if (live) {
        float mx = -INFINITY;
        for (int c = 0; c < nj; c += 16) {
          uint32_t r[16];
          tmem_ld_32x16(t_lane + c, r);
          tmem_ld_wait();
#pragma unroll
          for (int i = 0; i < 16; ++i)
            if (c + i < nv) mx = fmaxf(mx, __uint_as_float(r[i]));
        }
        const float m_new = fmaxf(m, mx * p.scale_log2);    // scale > 0: max of the products = product of the max
        float sum = 0.f;
        for (int c = 0; c < nj; c += 16) {
          uint32_t r[16];
          tmem_ld_32x16(t_lane + c, r);
          tmem_ld_wait();
#pragma unroll
          for (int i = 0; i < 16; ++i) {
            const float e = (c + i < nv) ? ex2_approx(fmaf(__uint_as_float(r[i]), p.scale_log2, -m_new)) : 0.f;
            sum += e;
            r[i] = __float_as_uint(e);
          }
          if (p.nblk == 1) tmem_st_32x16(t_lane + c, r);
        }
        if (p.nblk == 1) tmem_st_wait();
        l = l * ex2_approx(m - m_new) + sum;      // first block: exp2(-inf) * 0 = 0
        m = m_new;
      }
      release();
    }

    // ---------------------------------------------------------------- pass B: normalise, stage, store
    const float inv = __frcp_rn(l);
    for (int j = 0; j < p.nblk; ++j) {
      const int nv = (j == p.nblk - 1) ? nv_last : p.bkv;
      const int nj = (nv + 15) & ~15;
      if (p.nblk > 1) scores(img, head, qt, j, false, nj);
      if (live) {
        // this thread's row in the staging tile, at its destination's offset modulo 16 bytes
        uint16_t* srow;
        if (p.nblk == 1) {
          const int ph = static_cast<int>((probs_elem0 + (bh * p.N + r0) * static_cast<long long>(p.N)) & 7);
          srow = stage + ph + lane * p.N;
        } else {
          srow = stage + lane * p.pitch + static_cast<int>((probs_elem0 + row_elem + j * p.bkv) & 7);
        }
        for (int c = 0; c < nj; c += 16) {
          uint32_t r[16];
          tmem_ld_32x16(t_lane + c, r);
          tmem_ld_wait();
          if (mine) {
#pragma unroll
            for (int i = 0; i < 16; i += 2) {
              float e0 = __uint_as_float(r[i]), e1 = __uint_as_float(r[i + 1]);
              if (p.nblk > 1) {
                e0 = ex2_approx(fmaf(e0, p.scale_log2, -m));
                e1 = ex2_approx(fmaf(e1, p.scale_log2, -m));
              }
              const uint32_t pk = pack_bf16x2(e0 * inv, e1 * inv);
              if (c + i < nv) srow[c + i] = static_cast<uint16_t>(pk & 0xFFFFu);
              if (c + i + 1 < nv) srow[c + i + 1] = static_cast<uint16_t>(pk >> 16);
            }
          }
        }
        __syncwarp();
        if (p.nblk == 1) {
          const int rows = min(32, p.N - r0);
          const long long e0 = (bh * p.N + r0) * static_cast<long long>(p.N);
          const int ph = static_cast<int>((probs_elem0 + e0) & 7);
          store_span(stage + ph, p.probs + e0, static_cast<long long>(rows) * p.N, lane);
        } else {
          const int rows = min(32, p.N - r0);
          for (int rr = 0; rr < rows; ++rr) {
            const long long e0 = (bh * p.N + r0 + rr) * static_cast<long long>(p.N) + j * p.bkv;
            store_span(stage + rr * p.pitch + static_cast<int>((probs_elem0 + e0) & 7), p.probs + e0, nv, lane);
          }
        }
      }
      release();
    }
  }

  if (warp == 0) {
    tc_fence_after();
    tmem_dealloc<kPCols>(tmem_base);
  }
}

template <int DH>
int launch_attn_probs(const void* q, const void* k, const ProbsParams& p, long long qk_row_stride,
                      long long qk_batch_stride, cudaStream_t stream) {
  constexpr int kDT = DH - 64;
  const int stage_elems = p.nblk == 1 ? 32 * p.N + 8 : 32 * p.pitch;
  int smem = 1024 + kPQT * DH * 2 + p.bkv * DH * 2 + 4 * ((stage_elems + 7) & ~7) * 2 + 32;
  if (smem > kPSmemLimit) return VT_ERR_UNSUPPORTED;
  if (smem < kPMinSmem) smem = kPMinSmem;
  const uint64_t cols = static_cast<uint64_t>(p.H) * DH;
  CUtensorMap tq, tk, tqt, tkt;
  int rc = make_tmap_bf16_3d(&tq, q, cols, p.N, p.B, qk_row_stride, qk_batch_stride, 64, kPQT, TMAP_SW_128);
  if (rc) return rc;
  rc = make_tmap_bf16_3d(&tk, k, cols, p.N, p.B, qk_row_stride, qk_batch_stride, 64, p.bkv, TMAP_SW_128);
  if (rc) return rc;
  if (kDT) {
    rc = make_tmap_bf16_3d(&tqt, q, cols, p.N, p.B, qk_row_stride, qk_batch_stride, 16, kPQT, TMAP_SW_32);
    if (rc) return rc;
    rc = make_tmap_bf16_3d(&tkt, k, cols, p.N, p.B, qk_row_stride, qk_batch_stride, 16, p.bkv, TMAP_SW_32);
    if (rc) return rc;
  } else {
    tqt = tq;   // unused
    tkt = tk;
  }
  auto kern = attn_probs_kernel<DH>;
  static int granted[kMaxDevices] = {0};
  if (const int rc_attr = ensure_dynamic_smem(kern, smem, granted)) return rc_attr;
  int dev = 0, sms = 148;
  cudaGetDevice(&dev);
  cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
  const long long grid = p.total_items < 2LL * sms ? p.total_items : 2LL * sms;
  kern<<<static_cast<unsigned>(grid), kPThreads, smem, stream>>>(tq, tk, tqt, tkt, p);
  return static_cast<int>(cudaGetLastError());
}

}  // namespace

int attn_probs(const void* q, const void* k, void* probs, int B, int H, int N, int dh, long long qk_row_stride,
               long long qk_batch_stride, float scale, cudaStream_t s) {
  if (!q || !k || !probs || B <= 0 || H <= 0 || N <= 0) return VT_ERR_ARG;
  if ((dh != 64 && dh != 80) || !(scale > 0.f) || !(scale < INFINITY)) return VT_ERR_UNSUPPORTED;
  if ((qk_row_stride % 8) || (qk_batch_stride % 8) || qk_row_stride <= 0 || qk_batch_stride <= 0) return VT_ERR_ALIGN;
  if (((reinterpret_cast<uintptr_t>(q) | reinterpret_cast<uintptr_t>(k)) & 15) || (reinterpret_cast<uintptr_t>(probs) & 1))
    return VT_ERR_ALIGN;
  ProbsParams p;
  p.N = N;
  p.H = H;
  p.B = B;
  p.nqt = (N + kPQT - 1) / kPQT;
  p.nblk = N <= kPSingle ? 1 : (N + kPBlock - 1) / kPBlock;
  p.bkv = (((N + p.nblk - 1) / p.nblk) + 15) & ~15;
  if ((p.nblk - 1) * p.bkv >= N) return VT_ERR_UNSUPPORTED;   // the last block must hold at least one key
  p.pitch = p.bkv + 8;
  p.total_items = static_cast<long long>(B) * H * p.nqt;
  p.scale_log2 = scale * 1.4426950408889634f;
  p.probs = static_cast<uint16_t*>(probs);
  if (dh == 64) return launch_attn_probs<64>(q, k, p, qk_row_stride, qk_batch_stride, s);
  return launch_attn_probs<80>(q, k, p, qk_row_stride, qk_batch_stride, s);
}

}  // namespace vt

extern "C" int vt_attn_probs(const void* q, const void* k, void* probs, int32_t B, int32_t H, int32_t N, int32_t dh,
                             int64_t qk_row_stride, int64_t qk_batch_stride, float scale, void* stream) {
  return vt::attn_probs(q, k, probs, B, H, N, dh, qk_row_stride, qk_batch_stride, scale,
                        static_cast<cudaStream_t>(stream));
}
