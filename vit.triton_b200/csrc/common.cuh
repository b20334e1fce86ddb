// Shared device-side helpers for the sm_100a kernels: mbarrier, TMA, tcgen05/TMEM PTX wrappers,
// UMMA descriptor builders and small math utilities.  Everything here is inline PTX for
// compute_100a; nothing is portable to other architectures on purpose.
#pragma once
#include <cstdlib>
#include <utility>

#include <cuda.h>
#include <cuda_bf16.h>
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>

namespace vt {

// ----------------------------------------------------------------------------------------------
// error codes of the C ABI (negative = argument error, positive = cudaError_t)
// ----------------------------------------------------------------------------------------------
enum : int {
  VT_OK = 0,
  VT_ERR_ARG = -1,        // bad shape / null pointer
  VT_ERR_DTYPE = -2,      // unsupported dtype
  VT_ERR_ALIGN = -3,      // pointer / stride alignment
  VT_ERR_UNSUPPORTED = -4,
  VT_ERR_DRIVER = -5,     // cuTensorMapEncode / driver entry point failure
};

enum : int { VT_F32 = 0, VT_BF16 = 1, VT_U8 = 2, VT_E4M3 = 3 };

// GEMM epilogue activations: the VT_ACT_* codes of include/vitb200_clip.h.  vt_bgemm takes all four; the `gelu`
// argument of vt_gemm_bf16, vt_gemm_bf16_ln, vt_gemm_fp8 and vt_gemm_strided takes none, GELU or quick GELU.
enum : int { kActNone = 0, kActGelu = 1, kActTanh = 2, kActQuickGelu = 3 };
inline bool gemm_act_ok(int act) { return act == kActNone || act == kActGelu || act == kActQuickGelu; }

// ----------------------------------------------------------------------------------------------
// host: opt-in dynamic shared memory.  cudaFuncAttributeMaxDynamicSharedMemorySize is a PER-DEVICE
// attribute; `granted` is the call site's own per-device cache (one static array per kernel).
// ----------------------------------------------------------------------------------------------
constexpr int kMaxDevices = 64;
template <typename Kernel>
inline int ensure_dynamic_smem(Kernel kernel, int bytes, int (&granted)[kMaxDevices]) {
  int dev = 0;
  cudaGetDevice(&dev);
  const int slot = (dev >= 0 && dev < kMaxDevices) ? dev : 0;
  if (bytes > granted[slot] || dev != slot) {
    const cudaError_t e = cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, bytes);
    if (e != cudaSuccess) return static_cast<int>(e);
    granted[slot] = bytes;
  }
  return 0;
}

// Programmatic dependent launch of the GEMM and attention kernels (on by default, VT_PDL=0 switches it off).  A kernel launched with the
// attribute may become resident while its predecessor in the stream is still running: its CTAs run their
// prologue (barrier init, TMEM allocation, tensor-map prefetch) on SMs the predecessor has already left and block in
// pdl_wait() until the predecessor's grid has completed and its writes are visible; nothing a kernel reads or
// writes in global memory comes before its pdl_wait(), so a chain of such kernels stays ordered (a kernel past its wait
// implies its predecessor completed).  Both instructions are no-ops in a kernel launched without the attribute.
// Measured (tools/fwd_ab.py, 100 graph replays, two A/B pairs on one box): 8.836 / 8.814 -> 8.739 / 8.767 ms per C2
// forward: the ~5 us between the last CTA of a kernel and the first work of the next shrink by the launch latency.
inline bool pdl_enabled() {
  static const bool v = [] { const char* e = getenv("VT_PDL"); return !(e && e[0] == '0'); }();
  return v;
}
template <typename... KArgs, typename... Args>
inline cudaError_t launch_maybe_pdl(void (*kernel)(KArgs...), dim3 grid, dim3 block, size_t smem, cudaStream_t stream,
                                    Args&&... args) {
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = grid;
  cfg.blockDim = block;
  cfg.dynamicSmemBytes = smem;
  cfg.stream = stream;
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
  attr[0].val.programmaticStreamSerializationAllowed = 1;
  cfg.attrs = attr;
  cfg.numAttrs = pdl_enabled() ? 1 : 0;
  return cudaLaunchKernelEx(&cfg, kernel, std::forward<Args>(args)...);
}
__device__ __forceinline__ void pdl_wait() { asm volatile("griddepcontrol.wait;" ::: "memory"); }
__device__ __forceinline__ void pdl_launch_dependents() { asm volatile("griddepcontrol.launch_dependents;" ::: "memory"); }

// ----------------------------------------------------------------------------------------------
// misc
// ----------------------------------------------------------------------------------------------
__device__ __forceinline__ uint32_t smem_u32(const void* p) {
  return static_cast<uint32_t>(__cvta_generic_to_shared(p));
}

__device__ __forceinline__ uint32_t elect_one_sync() {
  uint32_t pred = 0;
  asm volatile(
      "{\n\t"
      ".reg .b32 rx;\n\t"
      ".reg .pred px;\n\t"
      "elect.sync rx|px, 0xffffffff;\n\t"
      "selp.b32 %0, 1, 0, px;\n\t"
      "}\n"
      : "=r"(pred));
  return pred;
}

// ----------------------------------------------------------------------------------------------
// mbarrier
// ----------------------------------------------------------------------------------------------
__device__ __forceinline__ void mbar_init(uint32_t bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(bar), "r"(count) : "memory");
}

__device__ __forceinline__ void fence_barrier_init() {
  asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
}

__device__ __forceinline__ void fence_proxy_async_smem() {
  asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
}

__device__ __forceinline__ void mbar_arrive(uint32_t bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(bar) : "memory");
}

__device__ __forceinline__ void mbar_arrive_expect_tx(uint32_t bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(bytes)
               : "memory");
}

__device__ __forceinline__ uint32_t mbar_try_wait(uint32_t bar, uint32_t parity) {
  uint32_t done;
  asm volatile(
      "{\n\t"
      ".reg .pred p;\n\t"
      "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
      "selp.b32 %0, 1, 0, p;\n\t"
      "}\n"
      : "=r"(done)
      : "r"(bar), "r"(parity)
      : "memory");
  return done;
}

// Non-blocking phase test (try_wait may suspend the warp for a system-dependent time before it answers).
__device__ __forceinline__ uint32_t mbar_test_wait(uint32_t bar, uint32_t parity) {
  uint32_t done;
  asm volatile(
      "{\n\t"
      ".reg .pred p;\n\t"
      "mbarrier.test_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
      "selp.b32 %0, 1, 0, p;\n\t"
      "}\n"
      : "=r"(done)
      : "r"(bar), "r"(parity)
      : "memory");
  return done;
}

// try_wait with a suspend-time hint (ns): the warp sleeps in hardware until the phase completes or
// the hint expires instead of returning after a few dozen cycles.
__device__ __forceinline__ uint32_t mbar_try_wait_hint(uint32_t bar, uint32_t parity, uint32_t ns) {
  uint32_t done;
  asm volatile(
      "{\n\t"
      ".reg .pred p;\n\t"
      "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2, %3;\n\t"
      "selp.b32 %0, 1, 0, p;\n\t"
      "}\n"
      : "=r"(done)
      : "r"(bar), "r"(parity), "r"(ns)
      : "memory");
  return done;
}

// Bounded wait: a protocol bug must surface as a trapped kernel (a CUDA error the host sees),
// never as a hung GPU.  ~4e9 cycles is about two seconds at boost clocks.  The slow path must stay
// cheap: a polling warp competes for issue slots with the warps doing the work (in the attention
// kernel the un-hinted poll loop with a clock read per iteration was 24 % of all issued
// instructions), so it sleeps on the suspend-time hint and looks at the clock every 256 polls.
__device__ __forceinline__ void mbar_wait(uint32_t bar, uint32_t parity) {
  if (mbar_try_wait(bar, parity)) return;
  long long t0 = 0;
  uint32_t polls = 0;
  while (!mbar_try_wait_hint(bar, parity, 1000000u)) {
    if ((++polls & 255u) == 0) {
      const long long now = clock64();
      if (t0 == 0) t0 = now;
      if (now - t0 > 4000000000LL) {
        printf("vt: mbarrier timeout block (%d,%d,%d) thread %d bar 0x%x parity %u\n", blockIdx.x,
               blockIdx.y, blockIdx.z, threadIdx.x, bar, parity);
        __trap();
      }
    }
  }
}

// ----------------------------------------------------------------------------------------------
// TMA (cp.async.bulk.tensor) — loads complete on an mbarrier, stores use bulk groups
// ----------------------------------------------------------------------------------------------
constexpr uint64_t kEvictNormal = 0x1000000000000000ull;
constexpr uint64_t kEvictFirst = 0x12F0000000000000ull;
constexpr uint64_t kEvictLast = 0x14F0000000000000ull;

__device__ __forceinline__ void tma_prefetch_desc(const CUtensorMap* m) {
  asm volatile("prefetch.tensormap [%0];" ::"l"(reinterpret_cast<uint64_t>(m)) : "memory");
}

__device__ __forceinline__ void tma_load_2d(const CUtensorMap* m, uint32_t bar, uint32_t dst,
                                            int c0, int c1, uint64_t hint) {
  asm volatile(
      "cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes.L2::cache_hint"
      " [%0], [%1, {%3, %4}], [%2], %5;"
      :
      : "r"(dst), "l"(reinterpret_cast<uint64_t>(m)), "r"(bar), "r"(c0), "r"(c1), "l"(hint)
      : "memory");
}

__device__ __forceinline__ void tma_load_3d(const CUtensorMap* m, uint32_t bar, uint32_t dst,
                                            int c0, int c1, int c2, uint64_t hint) {
  asm volatile(
      "cp.async.bulk.tensor.3d.shared::cluster.global.mbarrier::complete_tx::bytes.L2::cache_hint"
      " [%0], [%1, {%3, %4, %5}], [%2], %6;"
      :
      : "r"(dst), "l"(reinterpret_cast<uint64_t>(m)), "r"(bar), "r"(c0), "r"(c1), "r"(c2),
        "l"(hint)
      : "memory");
}

__device__ __forceinline__ void tma_store_2d(const CUtensorMap* m, uint32_t src, int c0, int c1) {
  asm volatile("cp.async.bulk.tensor.2d.global.shared::cta.bulk_group [%0, {%2, %3}], [%1];"
               :
               : "l"(reinterpret_cast<uint64_t>(m)), "r"(src), "r"(c0), "r"(c1)
               : "memory");
}

__device__ __forceinline__ void tma_store_3d(const CUtensorMap* m, uint32_t src, int c0, int c1, int c2) {
  asm volatile("cp.async.bulk.tensor.3d.global.shared::cta.bulk_group [%0, {%2, %3, %4}], [%1];"
               :
               : "l"(reinterpret_cast<uint64_t>(m)), "r"(src), "r"(c0), "r"(c1), "r"(c2)
               : "memory");
}

__device__ __forceinline__ void tma_store_commit() {
  asm volatile("cp.async.bulk.commit_group;" ::: "memory");
}

template <int N>
__device__ __forceinline__ void tma_store_wait_read() {
  asm volatile("cp.async.bulk.wait_group.read %0;" ::"n"(N) : "memory");
}

template <int N>
__device__ __forceinline__ void tma_store_wait() {
  asm volatile("cp.async.bulk.wait_group %0;" ::"n"(N) : "memory");
}

// ----------------------------------------------------------------------------------------------
// tcgen05 / TMEM
// ----------------------------------------------------------------------------------------------
template <int kCols>
__device__ __forceinline__ void tmem_alloc(uint32_t smem_dst) {
  asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_dst),
               "n"(kCols)
               : "memory");
}

__device__ __forceinline__ void tmem_relinquish() {
  asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
}

template <int kCols>
__device__ __forceinline__ void tmem_dealloc(uint32_t taddr) {
  asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(taddr), "n"(kCols)
               : "memory");
}

__device__ __forceinline__ void tc_fence_before() {
  asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
}
__device__ __forceinline__ void tc_fence_after() {
  asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
}

// D[tmem] (+)= A[smem] * B[smem]; issued by ONE thread.
__device__ __forceinline__ void umma_ss(uint32_t d_tmem, uint64_t a_desc, uint64_t b_desc,
                                        uint32_t idesc, uint32_t accumulate) {
  asm volatile(
      "{\n\t"
      ".reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t"
      "}\n"
      :
      : "r"(d_tmem), "l"(a_desc), "l"(b_desc), "r"(idesc), "r"(accumulate)
      : "memory");
}

// D[tmem] (+)= A[tmem] * B[smem]; issued by ONE thread.
__device__ __forceinline__ void umma_ts(uint32_t d_tmem, uint32_t a_tmem, uint64_t b_desc,
                                        uint32_t idesc, uint32_t accumulate) {
  asm volatile(
      "{\n\t"
      ".reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::f16 [%0], [%1], %2, %3, p;\n\t"
      "}\n"
      :
      : "r"(d_tmem), "r"(a_tmem), "l"(b_desc), "r"(idesc), "r"(accumulate)
      : "memory");
}

// Arrives on the mbarrier once every tcgen05.mma issued so far by this thread has completed.
// Implies tcgen05.fence::before_thread_sync.
__device__ __forceinline__ void umma_commit(uint32_t bar) {
  asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(
                   bar)
               : "memory");
}

// 32 lanes x 32 columns of 32-bit: thread t of the warp receives lane (base_lane + t),
// registers r[0..31] = columns col .. col+31.
__device__ __forceinline__ void tmem_ld_32x32(uint32_t taddr, uint32_t (&r)[32]) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
      "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
      "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];"
      : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]),
        "=r"(r[7]), "=r"(r[8]), "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]),
        "=r"(r[14]), "=r"(r[15]), "=r"(r[16]), "=r"(r[17]), "=r"(r[18]), "=r"(r[19]), "=r"(r[20]),
        "=r"(r[21]), "=r"(r[22]), "=r"(r[23]), "=r"(r[24]), "=r"(r[25]), "=r"(r[26]), "=r"(r[27]),
        "=r"(r[28]), "=r"(r[29]), "=r"(r[30]), "=r"(r[31])
      : "r"(taddr)
      : "memory");
}

__device__ __forceinline__ void tmem_ld_32x16(uint32_t taddr, uint32_t (&r)[16]) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x16.b32 "
      "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15}, [%16];"
      : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]),
        "=r"(r[7]), "=r"(r[8]), "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]),
        "=r"(r[14]), "=r"(r[15])
      : "r"(taddr)
      : "memory");
}

__device__ __forceinline__ void tmem_ld_32x8(uint32_t taddr, uint32_t (&r)[8]) {
  asm volatile("tcgen05.ld.sync.aligned.32x32b.x8.b32 {%0, %1, %2, %3, %4, %5, %6, %7}, [%8];"
               : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]),
                 "=r"(r[7])
               : "r"(taddr)
               : "memory");
}

__device__ __forceinline__ void tmem_ld_wait() {
  asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
}

// 32 lanes x 8 columns store (used for bf16-packed P: 16 values per row per call).
__device__ __forceinline__ void tmem_st_32x8(uint32_t taddr, const uint32_t (&r)[8]) {
  asm volatile(
      "tcgen05.st.sync.aligned.32x32b.x8.b32 [%0], {%1, %2, %3, %4, %5, %6, %7, %8};"
      :
      : "r"(taddr), "r"(r[0]), "r"(r[1]), "r"(r[2]), "r"(r[3]), "r"(r[4]), "r"(r[5]), "r"(r[6]),
        "r"(r[7])
      : "memory");
}

__device__ __forceinline__ void tmem_st_32x16(uint32_t taddr, const uint32_t (&r)[16]) {
  asm volatile(
      "tcgen05.st.sync.aligned.32x32b.x16.b32 [%0], "
      "{%1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, %16};"
      :
      : "r"(taddr), "r"(r[0]), "r"(r[1]), "r"(r[2]), "r"(r[3]), "r"(r[4]), "r"(r[5]), "r"(r[6]),
        "r"(r[7]), "r"(r[8]), "r"(r[9]), "r"(r[10]), "r"(r[11]), "r"(r[12]), "r"(r[13]),
        "r"(r[14]), "r"(r[15])
      : "memory");
}

__device__ __forceinline__ void tmem_st_wait() {
  asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory");
}

// ----------------------------------------------------------------------------------------------
// UMMA descriptors (bit layouts: SURVEY.md appendix B)
// ----------------------------------------------------------------------------------------------
// Instruction descriptor for kind::f16, bf16 x bf16 -> f32.
//   a_mn_major / b_mn_major: 0 = K-major operand, 1 = MN-major operand.
__host__ __device__ constexpr uint32_t make_idesc_bf16(int m, int n, int a_mn_major,
                                                       int b_mn_major) {
  return (1u << 4)                                   // C format F32
         | (1u << 7)                                 // A format BF16
         | (1u << 10)                                // B format BF16
         | (static_cast<uint32_t>(a_mn_major) << 15) // A major
         | (static_cast<uint32_t>(b_mn_major) << 16) // B major
         | (static_cast<uint32_t>(n >> 3) << 17)     // N / 8
         | (static_cast<uint32_t>(m >> 4) << 24);    // M / 16
}

// Shared-memory matrix descriptor.  layout_type: 2 = SWIZZLE_128B, 6 = SWIZZLE_32B, 0 = none.
__device__ __forceinline__ uint64_t make_smem_desc(uint32_t saddr, uint32_t lbo_bytes,
                                                   uint32_t sbo_bytes, uint32_t layout_type) {
  uint64_t d = 0;
  d |= static_cast<uint64_t>((saddr & 0x3FFFFu) >> 4);
  d |= static_cast<uint64_t>((lbo_bytes >> 4) & 0x3FFFu) << 16;
  d |= static_cast<uint64_t>((sbo_bytes >> 4) & 0x3FFFu) << 32;
  d |= 1ull << 46;  // descriptor version (sm_100)
  d |= static_cast<uint64_t>(layout_type & 7u) << 61;
  return d;
}

// K-major operand tile stored by TMA with SWIZZLE_128B: rows of 128 bytes (64 bf16 along K),
// 8-row swizzle atoms of 1024 bytes stacked along M/N.
__device__ __forceinline__ uint64_t make_desc_kmajor_sw128(uint32_t saddr) {
  return make_smem_desc(saddr, 0, 1024, 2);
}

// MN-major operand tile stored by TMA with SWIZZLE_128B: each K index is one 128-byte row of 64
// contiguous MN elements; 8 K rows form a 1024-byte atom (SBO); MN groups of 64 are lbo apart.
__device__ __forceinline__ uint64_t make_desc_mnmajor_sw128(uint32_t saddr, uint32_t lbo_bytes) {
  return make_smem_desc(saddr, lbo_bytes, 1024, 2);
}

// ----------------------------------------------------------------------------------------------
// math
// ----------------------------------------------------------------------------------------------
__device__ __forceinline__ float gelu_erf(float x) {
  return 0.5f * x * (1.0f + erff(x * 0.70710678118654752440f));
}

// Exact-erf GELU to 3.3e-7 absolute (Abramowitz-Stegun 7.1.26 for erfc, two MUFU ops + 12 FMA-pipe
// ops): gelu(x) = relu(x) - 0.5|x| * P(t) * exp(-x^2/2), t = 1/(1 + p|x|/sqrt(2)).  Used where the
// result is rounded to bf16 (rounding error >= 2e-3 relative); fp32 outputs use erff.
__device__ __forceinline__ float gelu_erf_fast(float x) {
  const float ax = fabsf(x);
  float t;
  asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(t) : "f"(fmaf(ax, 0.23164189f, 1.0f)));
  float poly = fmaf(t, 1.061405429f, -1.453152027f);
  poly = fmaf(t, poly, 1.421413741f);
  poly = fmaf(t, poly, -0.284496736f);
  poly = fmaf(t, poly, 0.254829592f);
  poly *= t;
  float e;
  asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(e) : "f"(x * x * -0.72134752f));
  return fmaxf(x, 0.0f) - (0.5f * ax) * poly * e;
}

// GELU for results that are immediately rounded to bf16: the 3-term Abramowitz-Stegun 7.1.25 erfc
// (|erf error| <= 2.5e-5, |gelu error| <= 2.6e-5 absolute, i.e. 1/75 of a bf16 ulp at |x| ~ 1) in 11
// instructions, two of them MUFU.  Coefficients are pre-multiplied by 0.5.
__device__ __forceinline__ float gelu_erf_bf16(float x) {
  const float ax = fabsf(x);
  float t;
  asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(t) : "f"(fmaf(ax, 0.33267253f, 1.0f)));
  float poly = fmaf(t, 0.3739278f, -0.0479399f);
  poly = fmaf(t, poly, 0.1740121f);
  const float h = (poly * t) * ax;
  float e;
  asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(e) : "f"(x * x * -0.72134752f));
  return fmaf(-h, e, fmaxf(x, 0.0f));
}

// gelu_erf_bf16 on TWO values with the FMA-pipe work on packed fp32 pairs (FFMA2, sm_100): the same
// formula and constants, nine instructions per element instead of twelve; the fc1 epilogue is bound
// by instruction issue, not by the two MUFU operations per element (profiles/README.md).
__device__ __forceinline__ float2 gelu_erf_bf16_x2(float2 x) {
  const float2 ax = make_float2(fabsf(x.x), fabsf(x.y));
  const float2 u = __ffma2_rn(ax, make_float2(0.33267253f, 0.33267253f), make_float2(1.0f, 1.0f));
  float2 t;
  asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(t.x) : "f"(u.x));
  asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(t.y) : "f"(u.y));
  // coefficients negated: nh = -(poly * t) * |x|
  float2 poly = __ffma2_rn(t, make_float2(-0.3739278f, -0.3739278f), make_float2(0.0479399f, 0.0479399f));
  poly = __ffma2_rn(t, poly, make_float2(-0.1740121f, -0.1740121f));
  const float2 nh = __fmul2_rn(__fmul2_rn(poly, t), ax);
  const float2 ea = __fmul2_rn(__fmul2_rn(x, x), make_float2(-0.72134752f, -0.72134752f));
  float2 e;
  asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(e.x) : "f"(ea.x));
  asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(e.y) : "f"(ea.y));
  return __ffma2_rn(nh, e, make_float2(fmaxf(x.x, 0.0f), fmaxf(x.y, 0.0f)));
}

// Exact-erf GELU with ONE MUFU operation per element:  gelu(x) = relu(x) - 0.5|x| * erfc(|x|/sqrt(2))
// and log2(erfc(a/sqrt(2))) is smooth enough for a degree-5 polynomial without constant term
// (erfc(0) = 1), fitted in the weighted minimax sense (weight = d gelu / d P) on [0, 8]:
// |gelu error| <= 5.6e-7 absolute over [-10, 10] evaluated in fp32 (tests/test_host_logic.py restates
// the arithmetic in numpy), against 2.6e-5 for the Abramowitz-Stegun form above.  The leading
// coefficient is negative and a*(c1 + ... + c5 a^4) < 0 for all a > 0, so the exponential underflows
// to zero for large |x| instead of needing a clamp.  13 instructions per PAIR, two of them MUFU
// (the A&S form: 16 and four): the GELU epilogue was bound by the MUFU pipe (2 x 32768 operations
// per 128 x 256 tile = 4096 of the tile's ~6800 cycles at 16 per clock) plus the issue slots.
__device__ __forceinline__ float2 gelu_erf_poly_x2(float2 x) {
  const float2 a = make_float2(fabsf(x.x), fabsf(x.y));
  float2 p = __ffma2_rn(a, make_float2(-0.00048810223f, -0.00048810223f), make_float2(0.0071987188f, 0.0071987188f));
  p = __ffma2_rn(a, p, make_float2(-0.052146632f, -0.052146632f));
  p = __ffma2_rn(a, p, make_float2(-0.45959586f, -0.45959586f));
  p = __ffma2_rn(a, p, make_float2(-1.1510005f, -1.1510005f));
  p = __fmul2_rn(a, p);
  float2 e;
  asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(e.x) : "f"(p.x));
  asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(e.y) : "f"(p.y));
  const float2 nh = __fmul2_rn(a, make_float2(-0.5f, -0.5f));
  return __ffma2_rn(nh, e, make_float2(fmaxf(x.x, 0.0f), fmaxf(x.y, 0.0f)));
}

// Quick GELU (CLIP's hidden_act="quick_gelu", VT_ACT_QUICK_GELU) for fp32 outputs: x * sigmoid(1.702 x) with expf and
// an IEEE division, within 2e-6 relative + 1e-7 absolute of the fp64 value for every finite x (for x < -52 the
// exponential overflows to +inf and the result is -0, off by less than 1e-36).
__device__ __forceinline__ float quick_gelu(float x) {
  return x / (1.0f + expf(-1.702f * x));
}

// Quick GELU for results that are immediately rounded to bf16 (fc1 epilogue), ONE MUFU operation per element:
// with a = |x| and e2 = 2^(-1.702 a log2(e) / 2), e = e2^2 = exp(-1.702 a),
//   x * sigmoid(1.702 x) = relu(x) - a * e / (1 + e)         (both signs: x - x e/(1+e) for x >= 0, x e/(1+e) below)
// and 1 / (1 + e) on e in [0, 1] is a degree-4 minimax polynomial (relative error <= 3.0e-4; the coefficients below
// are negated so that a * e2 * (e2 * -r) is one FFMA2 into relu(x)).  The product keeps the two factors a * e2 and
// e2 * r apart so that neither underflows before the final FMA: results down to the fp32 subnormal range (x to about
// -60) keep their relative accuracy, and ex2.approx.ftz only flushes e2 where the result is below bf16's range.
// Relative error <= 3.1e-4, under a tenth of a bf16 ulp: within one bf16 ulp of the correctly rounded fp64
// x * sigmoid(1.702 x) for every finite bf16 input (tests/test_abi_clip.py restates the arithmetic in numpy and
// checks all of them).  tanh.approx.f32 (0.5 x + 0.5 x tanh(0.851 x)) needs no second MUFU either, but its
// 2^-11 relative error is amplified by the cancellation at x < 0 and misses that bound.  15 instructions per PAIR,
// two of them MUFU (gelu_erf_poly_x2: 13 and two).
__device__ __forceinline__ float2 quick_gelu_bf16_x2(float2 x) {
  const float2 a = make_float2(fabsf(x.x), fabsf(x.y));
  const float2 t = __fmul2_rn(a, make_float2(-1.2277335f, -1.2277335f));   // -1.702 log2(e) / 2
  float2 e2;
  asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(e2.x) : "f"(t.x));
  asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(e2.y) : "f"(t.y));
  const float2 e = __fmul2_rn(e2, e2);
  float2 r = __ffma2_rn(e, make_float2(-0.15224545f, -0.15224545f), make_float2(0.53285909f, 0.53285909f));
  r = __ffma2_rn(e, r, make_float2(-0.86589509f, -0.86589509f));
  r = __ffma2_rn(e, r, make_float2(0.98483551f, 0.98483551f));
  r = __ffma2_rn(e, r, make_float2(-0.99970269f, -0.99970269f));                // r = -1 / (1 + e)
  return __ffma2_rn(__fmul2_rn(a, e2), __fmul2_rn(e2, r), make_float2(fmaxf(x.x, 0.0f), fmaxf(x.y, 0.0f)));
}

__device__ __forceinline__ float ex2_approx(float x) {
  float y;
  asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
  return y;
}

__device__ __forceinline__ uint32_t pack_bf16x2(float lo, float hi) {
  uint32_t r;
  asm("cvt.rn.bf16x2.f32 %0, %1, %2;" : "=r"(r) : "f"(hi), "f"(lo));
  return r;
}

__device__ __forceinline__ float bf16_lo(uint32_t v) { return __uint_as_float(v << 16); }
__device__ __forceinline__ float bf16_hi(uint32_t v) { return __uint_as_float(v & 0xFFFF0000u); }

__device__ __forceinline__ float warp_sum(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}
__device__ __forceinline__ float warp_max(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v = fmaxf(v, __shfl_xor_sync(0xffffffffu, v, o));
  return v;
}

}  // namespace vt
