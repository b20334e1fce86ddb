// Bicubic resample of the position table to another patch grid: what lets a checkpoint run at an input resolution
// other than the one it was trained at (HF ViTEmbeddings.interpolate_pos_encoding).  Pack-time work: one launch per
// (weights, grid), the result is cached by the host (vit/vit.py Embeddings.interpolate_pos_encoding).
//
//   out[0, :]               = pos[0, :]                                         (CLS position, copied)
//   out[1 + y * gw + x, :]  = bicubic(grid, y, x)  of the g_in x g_in grid pos[1 + i * g_in + j, :]
//
// bicubic = torch.nn.functional.interpolate(mode="bicubic", align_corners=False) with the channel stored last, in
// fp32 with torch's CPU arithmetic: src = (in / out) * (dst + 0.5) - 0.5 (not clamped), i = floor(src),
// t = src - i, Keys' cubic with A = -0.75, tap indices clamped to [0, in - 1], the 4-tap horizontal pass of each of
// the four source rows first, then the vertical pass.  At gh = gw = g_in the weights are (0, 1, 0, 0) exactly and the
// output reproduces the input bit for bit.
#include "common.cuh"

namespace vt {

namespace {

constexpr float kCubicA = -0.75f;

__device__ __forceinline__ float cubic1(float x) {   // |x| <= 1
  return ((kCubicA + 2.f) * x - (kCubicA + 3.f)) * x * x + 1.f;
}
__device__ __forceinline__ float cubic2(float x) {   // 1 < |x| < 2
  return ((kCubicA * x - 5.f * kCubicA) * x + 8.f * kCubicA) * x - 4.f * kCubicA;
}

__device__ __forceinline__ void cubic_weights(float t, float w[4]) {
  w[0] = cubic2(t + 1.f);
  w[1] = cubic1(t);
  w[2] = cubic1(1.f - t);
  w[3] = cubic2(2.f - t);
}

// source coordinate -> first tap index and the four weights
__device__ __forceinline__ int source_taps(int dst, float scale, float w[4]) {
  const float src = scale * (static_cast<float>(dst) + 0.5f) - 0.5f;
  const float fi = floorf(src);
  cubic_weights(src - fi, w);
  return static_cast<int>(fi) - 1;
}

__device__ __forceinline__ float ldp(const float* p) { return *p; }
__device__ __forceinline__ float ldp(const __nv_bfloat16* p) { return __bfloat162float(*p); }

// blockIdx.x = output token, threads stride over the channels: every tap row is read coalesced.  The table is at
// most a few MB and read from L2; the launch is latency-, not bandwidth-bound.
template <typename T>
__global__ void __launch_bounds__(256)
pos_resample_kernel(const T* __restrict__ pos, float* __restrict__ out, int D, int g_in, int gh, int gw,
                    float scale_h, float scale_w) {
  const int t = blockIdx.x;
  float* dst = out + static_cast<long long>(t) * D;
  if (t == 0) {
    for (int d = threadIdx.x; d < D; d += blockDim.x) dst[d] = ldp(pos + d);
    return;
  }
  const int y = (t - 1) / gw, x = (t - 1) - y * gw;
  float wy[4], wx[4];
  const int y0 = source_taps(y, scale_h, wy);
  const int x0 = source_taps(x, scale_w, wx);
  int rows[4], cols[4];
#pragma unroll
  for (int a = 0; a < 4; ++a) {
    rows[a] = min(max(y0 + a, 0), g_in - 1);
    cols[a] = min(max(x0 + a, 0), g_in - 1);
  }
  const T* grid = pos + D;   // row 1 of the table = grid position (0, 0)
  for (int d = threadIdx.x; d < D; d += blockDim.x) {
    float h[4];
#pragma unroll
    for (int a = 0; a < 4; ++a) {
      const T* row = grid + static_cast<long long>(rows[a]) * g_in * D + d;
      h[a] = ldp(row + static_cast<long long>(cols[0]) * D) * wx[0] + ldp(row + static_cast<long long>(cols[1]) * D) * wx[1] +
             ldp(row + static_cast<long long>(cols[2]) * D) * wx[2] + ldp(row + static_cast<long long>(cols[3]) * D) * wx[3];
    }
    dst[d] = h[0] * wy[0] + h[1] * wy[1] + h[2] * wy[2] + h[3] * wy[3];
  }
}

}  // namespace

// pos: [1 + g_in^2, D] (f32 | bf16), out: f32 [1 + gh * gw, D]; distinct buffers.
int pos_resample(const void* pos, int pos_dtype, float* out, int D, int g_in, int gh, int gw, cudaStream_t stream) {
  if (!pos || !out || D <= 0 || g_in <= 0 || gh <= 0 || gw <= 0) return VT_ERR_ARG;
  const long long tokens = 1 + static_cast<long long>(gh) * gw;
  if (tokens > 0x7fffffffLL) return VT_ERR_UNSUPPORTED;
  const float scale_h = static_cast<float>(g_in) / static_cast<float>(gh);
  const float scale_w = static_cast<float>(g_in) / static_cast<float>(gw);
  const int threads = D >= 256 ? 256 : ((D + 31) / 32) * 32;
  const dim3 grid(static_cast<unsigned>(tokens));
  if (pos_dtype == VT_F32)
    pos_resample_kernel<float><<<grid, threads, 0, stream>>>(static_cast<const float*>(pos), out, D, g_in, gh, gw,
                                                               scale_h, scale_w);
  else if (pos_dtype == VT_BF16)
    pos_resample_kernel<__nv_bfloat16><<<grid, threads, 0, stream>>>(static_cast<const __nv_bfloat16*>(pos), out, D,
                                                                       g_in, gh, gw, scale_h, scale_w);
  else
    return VT_ERR_DTYPE;
  return static_cast<int>(cudaGetLastError());
}

}  // namespace vt
