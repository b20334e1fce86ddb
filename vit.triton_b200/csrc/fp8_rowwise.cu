// FP8 (e4m3) side kernels of the optional FP8 path (VT_FP8=1; SURVEY.md 8f-3): the bandwidth-bound steps that
// produce e4m3 operands for vt_gemm_fp8 (gemm2_sm100.cu, tcgen05.mma kind::f8f6f4).
//
//   layernorm_e4m3   y8[m,:] = e4m3( LN(x[m,:]) * out_scale )           (bf16 in; the reference's layernorm,
//                    vit/kernels/layernorm.py:51-85, with the quantisation of the GEMM operand fused in)
//   quantize_rows    w8[n,:] = e4m3( w[n,:] / s_n ),  s_n = amax_k |w[n,k]| / 448   (pack time, per output channel)
//
// |LN(x)_i| <= sqrt(dim - 1) (Samuelson), so |gamma_i LN(x)_i + beta_i| <= max|gamma| sqrt(dim - 1) + max|beta|; the
// host picks out_scale per LayerNorm from that bound (packing.fp8_ln_scale: a power of two, at most 16) so that no
// element saturates.  The cast saturates anyway (satfinite).  dim <= 2048 (VPL <= 8).
#include "common.cuh"

namespace vt {

namespace {

__device__ __forceinline__ uint32_t e4m3x4(float a, float b, float c, float d) {
  uint16_t lo, hi;
  asm("cvt.rn.satfinite.e4m3x2.f32 %0, %1, %2;" : "=h"(lo) : "f"(b), "f"(a));
  asm("cvt.rn.satfinite.e4m3x2.f32 %0, %1, %2;" : "=h"(hi) : "f"(d), "f"(c));
  return static_cast<uint32_t>(lo) | (static_cast<uint32_t>(hi) << 16);
}

// one warp per row; the row stays in registers as packed bf16 (VPL 16-byte vectors per lane)
template <int VPL>
__global__ void __launch_bounds__(256)
layernorm_e4m3_kernel(const __nv_bfloat16* __restrict__ x, const __nv_bfloat16* __restrict__ gamma,
                      const __nv_bfloat16* __restrict__ beta, uint8_t* __restrict__ out, long long rows, int dim,
                      long long in_stride, long long out_stride, float eps, float out_scale) {
  const int lane = threadIdx.x & 31;
  const long long row = static_cast<long long>(blockIdx.x) * (blockDim.x >> 5) + (threadIdx.x >> 5);
  if (row >= rows) return;
  const uint4* xr = reinterpret_cast<const uint4*>(x + row * in_stride);
  const int nvec = dim >> 3;
  uint4 d[VPL];
#pragma unroll
  for (int i = 0; i < VPL; ++i) {
    const int vi = lane + i * 32;
    d[i] = (vi < nvec) ? xr[vi] : make_uint4(0u, 0u, 0u, 0u);
  }
  auto up = [](uint32_t w) { return make_float2(bf16_lo(w), bf16_hi(w)); };
  float2 s2 = make_float2(0.f, 0.f);
#pragma unroll
  for (int i = 0; i < VPL; ++i) {
    if (lane + i * 32 < nvec) {
      s2 = __fadd2_rn(s2, up(d[i].x)); s2 = __fadd2_rn(s2, up(d[i].y));
      s2 = __fadd2_rn(s2, up(d[i].z)); s2 = __fadd2_rn(s2, up(d[i].w));
    }
  }
  const float mean = warp_sum(s2.x + s2.y) / static_cast<float>(dim);
  const float2 nmean = make_float2(-mean, -mean);
  float2 q2 = make_float2(0.f, 0.f);
  auto acc = [&](uint32_t w) { const float2 c = __fadd2_rn(up(w), nmean); q2 = __ffma2_rn(c, c, q2); };
#pragma unroll
  for (int i = 0; i < VPL; ++i) {
    if (lane + i * 32 < nvec) {
      acc(d[i].x); acc(d[i].y); acc(d[i].z); acc(d[i].w);
    }
  }
  const float var = warp_sum(q2.x + q2.y) / static_cast<float>(dim);
  const float rstd = 1.0f / sqrtf(var + eps);
  const float2 rstd2 = make_float2(rstd, rstd);
  const float2 os2 = make_float2(out_scale, out_scale);
  uint2* orow = reinterpret_cast<uint2*>(out + row * out_stride);
  const uint4* gp = reinterpret_cast<const uint4*>(gamma);
  const uint4* bp = reinterpret_cast<const uint4*>(beta);
  auto nrm = [&](uint32_t v, uint32_t g, uint32_t b) {
    const float2 t = __fmul2_rn(__fadd2_rn(up(v), nmean), rstd2);
    return __fmul2_rn(__ffma2_rn(up(g), t, up(b)), os2);
  };
#pragma unroll
  for (int i = 0; i < VPL; ++i) {
    const int vi = lane + i * 32;
    if (vi < nvec) {
      const uint4 g = __ldg(gp + vi);
      const uint4 b = __ldg(bp + vi);
      const float2 a0 = nrm(d[i].x, g.x, b.x), a1 = nrm(d[i].y, g.y, b.y);
      const float2 a2 = nrm(d[i].z, g.z, b.z), a3 = nrm(d[i].w, g.w, b.w);
      orow[vi] = make_uint2(e4m3x4(a0.x, a0.y, a1.x, a1.y), e4m3x4(a2.x, a2.y, a3.x, a3.y));
    }
  }
}

// one warp per weight row
__global__ void __launch_bounds__(256)
quantize_rows_e4m3_kernel(const __nv_bfloat16* __restrict__ w, long long ldw, uint8_t* __restrict__ out, long long ldo,
                          float* __restrict__ scales, int N, int K) {
  const int lane = threadIdx.x & 31;
  const int n = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  if (n >= N) return;
  const __nv_bfloat16* wr = w + static_cast<long long>(n) * ldw;
  float amax = 0.f;
  for (int k = lane; k < K; k += 32) amax = fmaxf(amax, fabsf(__bfloat162float(wr[k])));
  amax = warp_max(amax);
  // a zero or subnormal amax / 448 has no usable reciprocal (1 / s overflows to inf, 0 * inf = NaN); such a row
  // (amax < 448 * 2^-126) quantises to zero codes with s = 1
  const float s0 = amax / 448.0f;
  const float s = s0 >= 0x1p-126f ? s0 : 1.0f;
  const float inv = 1.0f / s;
  if (lane == 0) scales[n] = s;
  uint8_t* orow = out + static_cast<long long>(n) * ldo;
  for (int k4 = lane * 4; k4 < K; k4 += 128) {     // K % 4 == 0 (host)
    const float a = __bfloat162float(wr[k4]) * inv, b = __bfloat162float(wr[k4 + 1]) * inv;
    const float c = __bfloat162float(wr[k4 + 2]) * inv, d = __bfloat162float(wr[k4 + 3]) * inv;
    *reinterpret_cast<uint32_t*>(orow + k4) = e4m3x4(a, b, c, d);
  }
}

}  // namespace

int layernorm_e4m3(const void* x, const void* gamma, const void* beta, void* out, long long rows, int dim,
                   long long in_stride, long long out_stride, float eps, float out_scale, cudaStream_t stream) {
  if (!x || !gamma || !beta || !out || rows < 0 || dim <= 0) return VT_ERR_ARG;
  if (rows == 0) return VT_OK;
  if ((dim % 8) || (in_stride % 8) || (out_stride % 8) ||
      ((reinterpret_cast<uintptr_t>(x) | reinterpret_cast<uintptr_t>(gamma) | reinterpret_cast<uintptr_t>(beta)) & 15) ||
      (reinterpret_cast<uintptr_t>(out) & 7))
    return VT_ERR_ALIGN;
  const int vpl = (dim / 8 + 31) / 32;
  const unsigned grid = static_cast<unsigned>((rows + 7) / 8);
  const __nv_bfloat16* xp = static_cast<const __nv_bfloat16*>(x);
  const __nv_bfloat16* gp = static_cast<const __nv_bfloat16*>(gamma);
  const __nv_bfloat16* bp = static_cast<const __nv_bfloat16*>(beta);
  uint8_t* op = static_cast<uint8_t*>(out);
#define VT_LN8_CASE(V)                                                                                            \
  case V:                                                                                                         \
    layernorm_e4m3_kernel<V><<<grid, 256, 0, stream>>>(xp, gp, bp, op, rows, dim, in_stride, out_stride, eps,    \
                                                       out_scale);                                                \
    break;
  switch (vpl) {
    VT_LN8_CASE(1) VT_LN8_CASE(2) VT_LN8_CASE(3) VT_LN8_CASE(4) VT_LN8_CASE(5) VT_LN8_CASE(6) VT_LN8_CASE(7) VT_LN8_CASE(8)
    default: return VT_ERR_UNSUPPORTED;
  }
#undef VT_LN8_CASE
  return static_cast<int>(cudaGetLastError());
}

int quantize_rows_e4m3(const void* w, long long ldw, void* out, long long ldo, float* scales, int N, int K,
                       cudaStream_t stream) {
  if (!w || !out || !scales || N <= 0 || K <= 0) return VT_ERR_ARG;
  if ((K % 4) || (ldo % 4) || (reinterpret_cast<uintptr_t>(out) & 3)) return VT_ERR_ALIGN;
  quantize_rows_e4m3_kernel<<<(N + 7) / 8, 256, 0, stream>>>(static_cast<const __nv_bfloat16*>(w), ldw,
                                                            static_cast<uint8_t*>(out), ldo, scales, N, K);
  return static_cast<int>(cudaGetLastError());
}

}  // namespace vt
